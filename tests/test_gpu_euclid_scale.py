"""diff_euclid_kernel (csrc/diff_euclid.cu, RGB Euclidean and CIE76) against the f64 oracle at the sizes where its tiling changes.

The kernel walks 64-cell x 64-image tiles in 16 x 16-tile super-blocks (tile_of_block, csrc/kernels.h), sums 16-pixel chunks in
two levels (1,024-pixel partials flushed into a total) and, without repeats, picks the winner in a fused epilogue whose only
protection against the zero padding of the last library tile is the guard `li0 + li < n_lib`. Each test below targets one of those:

  A  tile raster: valid-cell counts below one tile, exactly 64 k, a partial 17th cell tile, past two column blocks; library sizes
     around one tile and one band; both axes past 16 tiles at once; fused epilogue and wavefront / top-K selection.
  B  pixel axis: masks of exactly k active pixels around the 16-pixel chunk and the 1,024-pixel flush, and a flipped shape whose
     active list is the union of four flipped masks.
  C  padding: whole black cells (distance 0 to every padding slot) against libraries that are not a multiple of 64 images.
  D  BASELINE config 3 as specified (4K, 2,000 images @64, CIE76, 3 size levels).
  E  BASELINE config 5 at full size (16K, 20,000 images @128, Puzzle.mcs, detail 50 %, RGB), with repeats for top-K at N = 20,000.
  F  (CPU) the case tables of A-C still cross the boundaries they name.

Criteria (tests/helpers/parity.py): difference sums as check_differences; grids teacher-forced against f64 within the tie band;
wherever the engine's own difference matrix decides the choice (argmin, repeat-penalised selection), exact equality.
GPU tests carry their own mark so that F runs without a device."""
import os

import numpy as np
import pytest

from tests.helpers.parity import TIE_TOL, check_differences, check_grid

TILE = 64          # cells per cell tile = images per library tile (MM_ETC / MM_ETN)
SUPER = 16         # tiles per super-block side (kSuperTiles)
CHUNK = 16         # pixels per chunk (MM_EKP)
FLUSH = 1024       # pixels per first-level partial sum (kFlushChunks chunks)
DIFFS = [pytest.param(0, id="rgb"), pytest.param(1, id="cie76")]

# A: (main rows, main cols, valid 8 px cells, library size, cell tiles, library tiles)
A_CASES = [
    (56, 70, 63, 1, 1, 1),            # one partial tile on each axis, clipped right border
    (56, 70, 63, 64, 1, 1),
    (64, 64, 64, 65, 1, 2),           # exactly one cell tile; one padded library tile
    (64, 64, 64, 63, 1, 1),
    (250, 256, 1024, 1100, 16, 18),   # exactly one column block; second, partial library band
    (251, 263, 1056, 1024, 17, 16),   # partial 17th cell tile (second, partial column block); exactly one band
    (251, 263, 1056, 1025, 17, 17),   # both axes past 16 tiles; a 1-image band
    (360, 366, 2070, 65, 33, 2),      # two full column blocks and a partial one
    (360, 366, 2070, 1100, 33, 18),   # the same against a partial second band
]
A_CELL = 8

# B: (active pixels k, cell size, flips). 70 cells (two tiles) against 130 images (three tiles, the last one 2 images).
B_CASES = [(k, 33 if k <= 33 * 33 else 65, False) for k in (1, 15, 16, 17, 1023, 1024, 1025, 2047, 2048, 2049, 4097)]
B_CASES.append((700, 33, True))  # alternate columns flipped horizontally, rows vertically: the union of four 700-pixel masks
B_N, B_CELLS = 130, 70
B_MAIN = {33: (218, 314), 65: (430, 615)}  # 7 x 10 cells, bottom row and right column clipped

# C: black cells against a library whose last tile is padded
C_NS = [1, 63, 65, 100]
C_MAIN, C_CELL, C_BLACK_ROW = (200, 300), 32, 3


def _ceil(a, b):
    return -(-a // b)


def _square_group(oracle, size):
    return oracle.CellGroup.make(oracle.CellShape.square(size), 100, 0)


def _b_shape(oracle, k, size, flips):
    rng = np.random.default_rng(9000 + k)
    m = np.zeros(size * size, np.uint8)
    m[rng.choice(size * size, k, replace=False)] = 255
    sh = oracle.CellShape.from_mask(m.reshape(size, size))
    sh.alt_col_flip_h = sh.alt_row_flip_v = flips
    return sh


def _valid(state):
    """padded grid positions (y, x) of the valid cells in raster order = row order of the difference matrix"""
    return list(zip(*[a.tolist() for a in np.nonzero(state >= 0)]))


def _active_pixels(oracle, normal, detail, state):
    """The kernel's pixel axis: union of the flipped detail masks that occur among the valid cells (generator.cu, active pixel
    list); returns (its length, the flips that occur)."""
    used = {oracle.flip_at(normal, x - 2, y - 2) for y, x in _valid(state)}
    m4 = detail.masks4()
    return int(np.any([m4[f] > 0 for f in sorted(used)], axis=0).sum()), used


def _c_black_cells(state):
    """Padded grid positions painted black: one whole grid row, the first and the last valid cell."""
    valid = _valid(state)
    row = C_BLACK_ROW + 2
    return sorted({c for c in valid if c[0] == row} | {valid[0], valid[-1]})


# ----------------------------------------------------------------------------- running the engine


def _generator(main, lib, shape, diff, detail=100, steps=0):
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(diff)
    cg = CellGroup()
    cg.setCellShape(shape)
    cg.setDetail(detail)
    cg.setSizeSteps(steps)
    gen.setCellGroup(cg)
    return gen


def _generate(gen, rr, ra, keep=True):
    gen.setRepeat(rr, ra)
    gen.setKeepDifferences(keep)
    assert gen.generateBestFits()
    grids = gen.getBestFits()
    return grids, ([gen.getDifferences(s) for s in range(len(grids))] if keep else None)


def _assert_argmin(D, state, grid):
    """No repeats: every valid cell holds the lowest index of its row minimum in the engine's own D (exact)."""
    valid = state >= 0
    assert (grid[~valid] == -1).all()
    got, want = grid[valid], np.argmin(D, axis=1)
    assert np.array_equal(got, want), "%d cells differ from the argmin of the engine's D, first at %s" % (
        int((got != want).sum()), np.argwhere(got != want)[:3].ravel().tolist())


def _check_case(oracle, label, main, lib, o_shape, diff, state, runs):
    """runs: (rr, ra, grid, D) of one generator. D against the f64 oracle, the grid against the engine's D (exact) and the f64
    oracle (tie band); prints the summary line."""
    og = oracle.CellGroup.make(o_shape, 100, 0)
    want = oracle.generate(main, lib, og, [state], diff, 0, 0, 0, want_D=True, early_exit=False)[0].D
    worst, ties = 0.0, []
    for rr, ra, grid, D in runs:
        assert D.shape == want.shape and np.isfinite(D).all()
        worst = max(worst, float(check_differences(D, want).max()))
        if rr == 0:
            _assert_argmin(D, state, grid)
        else:
            sel = oracle.select_from_D(D.astype(np.float64), state, rr, ra)
            assert np.array_equal(sel, grid), "%d cells differ from the repeat rule on the engine's D" % int((sel != grid).sum())
        n, t, bad = check_grid(want, state, grid, rr, ra, TIE_TOL)
        assert not bad, "repeats %d/%d: %d cells outside the tie band, first %s" % (rr, ra, len(bad), bad[:3])
        ties.append(t)
    print("%s: %d cells x %d images, max relative error %.2e, tie-band cells %s" % (label, n, lib.shape[0], worst,
                                                                                 " / ".join(map(str, ties))))
    return want


# ----------------------------------------------------------------------------- A: tile raster


@pytest.mark.gpu
@pytest.mark.parametrize("diff", DIFFS)
@pytest.mark.parametrize("H,W,n_cells,N,n_ct,n_lt", A_CASES, ids=["%dcells-N%d" % (c[2], c[3]) for c in A_CASES])
def test_tile_raster_boundaries(oracle, H, W, n_cells, N, n_ct, n_lt, diff):
    """Full D of 8 px cells (4 chunks) against f64 at every tile-count boundary of the raster, once through the fused argmin epilogue
    (no repeats) and once through the wavefront (repeats 2/500, top-K candidates when 4 x 13 <= N)."""
    from mosaicmagnifique_b200 import CellShape, synthetic
    main = synthetic.make_main_image(H, W, 3100 + n_cells, block=8)
    lib = synthetic.make_library(N, A_CELL, 3200 + N)
    gen = _generator(main, lib, CellShape(A_CELL), diff)
    state = gen.computeGridState()[0]
    assert np.array_equal(state, oracle.grid_state(_square_group(oracle, A_CELL), main)[0])
    n = int((state >= 0).sum())
    assert (n, _ceil(n, TILE), _ceil(N, TILE)) == (n_cells, n_ct, n_lt)
    runs = []
    for rr, ra in ((0, 0), (2, 500)):
        grids, Ds = _generate(gen, rr, ra)
        runs.append((rr, ra, grids[0], Ds[0]))
    gen.close()
    _check_case(oracle, "A %d cells (%d tiles) x N=%d (%d tiles), diff %d" % (n_cells, n_ct, N, n_lt, diff), main, lib,
                oracle.CellShape.square(A_CELL), diff, state, runs)


# ----------------------------------------------------------------------------- B: pixel axis


@pytest.mark.gpu
@pytest.mark.parametrize("diff", DIFFS)
@pytest.mark.parametrize("k,size,flips", B_CASES, ids=["k%d%s" % (c[0], "-flips" if c[2] else "") for c in B_CASES])
def test_pixel_axis_boundaries(oracle, k, size, flips, diff):
    """Masks of exactly k active pixels: 1 chunk, 16-pixel chunk edges, the 1,024-pixel flush edge, two and four flushes plus a tail."""
    from mosaicmagnifique_b200 import synthetic
    from tests.test_gpu_generator import _to_product_shape
    sh = _b_shape(oracle, k, size, flips)
    H, W = B_MAIN[size]
    main = synthetic.make_main_image(H, W, 3300 + k, block=16)
    lib = synthetic.make_library(B_N, size, 3400 + k)
    gen = _generator(main, lib, _to_product_shape(sh), diff)
    state = gen.computeGridState()[0]
    assert int((state >= 0).sum()) == B_CELLS
    n_active, used = _active_pixels(oracle, sh, sh, state)
    if flips:
        assert used == {0, 1, 2, 3} and k < FLUSH < n_active
    else:
        assert n_active == k
    grids, Ds = _generate(gen, 0, 0)
    gen.close()
    _check_case(oracle, "B k=%d (%d active, %d chunks), diff %d" % (k, n_active, _ceil(n_active, CHUNK), diff), main, lib, sh, diff,
                state, [(0, 0, grids[0], Ds[0])])


# ----------------------------------------------------------------------------- C: black cells against padding


def _black_main(oracle, seed):
    from mosaicmagnifique_b200 import synthetic
    H, W = C_MAIN
    main = synthetic.make_main_image(H, W, seed, block=32)
    sh = oracle.CellShape.square(C_CELL)
    state = oracle.grid_state(_square_group(oracle, C_CELL), None, H, W)[0]
    black = _c_black_cells(state)
    for y, x in black:
        rx, ry, rw, rh = oracle.rect_at(sh, x - 2, y - 2)
        main[max(ry, 0):max(ry + rh, 0), max(rx, 0):max(rx + rw, 0)] = 0
    return main, state, black


@pytest.mark.gpu
@pytest.mark.parametrize("diff", DIFFS)
@pytest.mark.parametrize("rr,ra", [(0, 0), (2, 500)], ids=["fused", "wavefront"])
@pytest.mark.parametrize("N", C_NS)
def test_black_cells_never_pick_padding(oracle, N, rr, ra, diff):
    """A black cell is at distance exactly 0 from every zero padding slot of the last library tile; only the epilogue guard (and
    M = N in the wavefront / top-K) keeps those slots out of the choice."""
    from mosaicmagnifique_b200 import CellShape, capi, synthetic
    main, o_state, black = _black_main(oracle, 3500 + N)
    lib = synthetic.make_library(N, C_CELL, 3600 + N)
    # premises: no library image is black, and the working space of CIE76 maps black to exactly (0, 0, 0) like RGB
    assert (lib.reshape(N, -1).max(axis=1) > 0).all()
    lab = np.full(3, np.nan, np.float32)
    assert capi().mosaic_kernel_bgr_to_lab(0, np.zeros(3, np.uint8).ctypes.data, 1, lab.ctypes.data) == 0
    assert (lab == 0).all(), lab
    assert N % TILE != 0

    gen = _generator(main, lib, CellShape(C_CELL), diff)
    state = gen.computeGridState()[0]
    assert np.array_equal(state, o_state)
    grids, Ds = _generate(gen, rr, ra)
    gen.close()
    grid, D = grids[0], Ds[0]
    index_of = {c: i for i, c in enumerate(_valid(state))}
    for c in black:
        assert 0 <= grid[c] < N, (c, int(grid[c]))
        assert (D[index_of[c]] > 0).all(), c
    want = _check_case(oracle, "C N=%d repeats %d/%d, %d black cells, diff %d" % (N, rr, ra, len(black), diff), main, lib,
                       oracle.CellShape.square(C_CELL), diff, state, [(rr, ra, grid, D)])
    assert all((want[index_of[c]] > 0).all() for c in black)


# ----------------------------------------------------------------------------- D: config 3 as specified


def _f64_rows(oracle, mains, og, step, state, cells, lib_f, diff):
    """Complete f64 difference rows (no early exit) of `cells` (padded grid positions) against the whole working-space library."""
    sub = np.full_like(state, -1)
    for c in cells:
        sub[c] = 0
    ex, bounds, flips, _ = oracle.extract_cells(mains, og, step, sub)
    masks4 = og.detail_cells[step].masks4()
    r = oracle.generate_step(diff, ex, bounds, flips, lib_f, masks4, sub, 0, 0, want_D=True, early_exit=False)
    return r.D, bounds  # rows in raster order of `cells`


def _sample_cells(oracle, og, step, state, n_inner, n_border, H, W):
    """The first and the last valid cell, n_inner cells spread over the interior, n_border cells of the right border column (rows
    spread) and n_border of the bottom row. Returns (cells in raster order, how many of them the image clips)."""
    valid = _valid(state)
    rows = sorted({c[0] for c in valid})
    ends = {r: (min(c for c in valid if c[0] == r), max(c for c in valid if c[0] == r)) for r in rows}
    inner = [c for c in valid if rows[0] < c[0] < rows[-1] and c not in ends[c[0]]]
    right = [ends[r][1] for r in rows[1:-1]]
    bottom = [c for c in valid if c[0] == rows[-1]][1:-1]
    cells = {valid[0], valid[-1]}
    for part, n in ((inner, n_inner), (right, n_border), (bottom, n_border)):
        if part:
            cells |= {part[i] for i in np.linspace(0, len(part) - 1, n).astype(int)}
    ds = og.detail_cells[step].size

    def clipped(c):
        _, _, b = oracle.cell_bounds(og.cells[step], ds, og.detail, c[1] - 2, c[0] - 2, W, H)
        return b[2] < ds or b[3] < ds

    return sorted(cells), sum(map(clipped, cells))


@pytest.mark.gpu
def test_config3_as_specified(oracle):
    """BASELINE config 3: 3840 x 2160 main, 2,000 images @64, CIE76, 3 size levels, no repeats (bench.py `cfg3` seeds). The f32
    working library is halved per step and repacked (pack_library_euclid_kernel after a memset), not the fused 8U packer."""
    from mosaicmagnifique_b200 import CellShape, synthetic
    H, W, N, S, steps = 2160, 3840, 2000, 64, 2
    main, lib = synthetic.make_main_image(H, W, 2003), synthetic.make_library(N, S, 1003)
    gen = _generator(main, lib, CellShape(S), 1, steps=steps)
    states = gen.computeGridState()
    og = oracle.CellGroup.make(oracle.CellShape.square(S), 100, steps)
    o_states = oracle.grid_state(og, main)
    assert len(states) == len(o_states) == steps + 1
    for s, (a, b) in enumerate(zip(states, o_states)):
        assert np.array_equal(a, b), "grid state of step %d" % s
    grids, Ds = _generate(gen, 0, 0)
    gen.close()
    counts = [int((s >= 0).sum()) for s in states]
    # the 64 px cells of the noise blocks split, and so do all their 32 px quarters: step 1 holds no cell, step 2 many column blocks
    assert counts[0] > TILE * SUPER and counts[1] == 0 and counts[2] > 2 * TILE * SUPER, counts

    mains = [oracle.to_working_space(main, oracle.CIE76)]
    lib_f = oracle.preprocess_library(lib, og, oracle.CIE76)
    worst, in_band, n_rows, n_clipped = 0.0, 0, 0, 0
    for s in range(steps + 1):
        if s > 0:
            lib_f = oracle.halve_library(lib_f)
        assert Ds[s].shape == (counts[s], N)
        if counts[s] == 0:
            assert (grids[s] == -1).all()
            continue
        _assert_argmin(Ds[s], states[s], grids[s])
        cells, clipped = _sample_cells(oracle, og, s, states[s], 4, 1, H, W)
        assert len(cells) == 8 and (clipped > 0 or s > 0), (s, cells, clipped)  # 16 px cells tile 3840 x 2160 exactly
        want, _ = _f64_rows(oracle, mains, og, s, states[s], cells, lib_f, oracle.CIE76)
        index_of = {c: i for i, c in enumerate(_valid(states[s]))}
        got = Ds[s][[index_of[c] for c in cells]]
        worst = max(worst, float(check_differences(got, want).max()))
        for c, row in zip(cells, want):
            b, g = int(np.argmin(row)), int(grids[s][c])
            if g != b:
                assert (row[g] - row[b]) / max(row[b], 1e-30) <= TIE_TOL, (s, c, g, b)
                in_band += 1
        n_rows += len(cells)
        n_clipped += clipped
    print("config 3 as specified: cells per step %s, %d complete f64 rows (%d clipped border cells), max relative error %.2e, "
          "tie-band cells %d" % (counts, n_rows, n_clipped, worst, in_band))


# ----------------------------------------------------------------------------- E: config 5 at full size


@pytest.mark.gpu
def test_config5_full_size(oracle):
    """BASELINE config 5 at its own size: 15360 x 8640 main, 20,000 images @128, Puzzle.mcs, detail 50 % (3,032 active pixels = 190
    chunks: two flushes and a 62-chunk tail), RGB; 11,664 cells = 183 cell tiles, 313 library tiles = 19 full bands + 9 tiles.
      (i)   no repeats, D kept: grid = argmin of the engine's D everywhere; without D (the benchmark path) the identical grid;
      (ii)  16 complete f64 rows (first and last cell, clipped right and bottom borders, interior): sums and choices. The first cell
            keeps no active pixel inside the image (its 10 x 10 corner of the mask is empty): an all-zero row, where index 0 must win;
      (iii) repeats 3/2000 (top-K of 25 over 20,000 images, wavefront): grid = the repeat rule applied to the engine's D, exactly.
    CPU: the f64 rows take ~6 s of one core, spread over threads by library batches of 2,000 images."""
    import threading

    from mosaicmagnifique_b200 import load_mcs, synthetic
    from tests.test_gpu_baseline_configs import CELLS, load_shape
    H, W, N, S, detail = 8640, 15360, 20000, 128, 50
    shape = load_mcs(os.path.join(CELLS, "Puzzle.mcs")).resized(S)
    o_shape, _ = load_shape(oracle, "Puzzle")
    o_shape = o_shape.resized(S)
    assert (shape.rowSpacing, shape.colSpacing) == (o_shape.row_spacing, o_shape.col_spacing) == (108, 108)
    main, lib = synthetic.make_main_image(H, W, 2005), synthetic.make_library(N, S, 1005)
    og = oracle.CellGroup.make(o_shape, detail, 0)
    gen = _generator(main, lib, shape, 0, detail=detail)
    state = gen.computeGridState()[0]
    assert np.array_equal(state, oracle.grid_state(og, None, H, W)[0])
    n_cells = int((state >= 0).sum())
    n_active, _ = _active_pixels(oracle, og.cells[0], og.detail_cells[0], state)
    assert state.shape == (82, 145) and n_cells == 11664 and _ceil(n_cells, TILE) == 183 and _ceil(N, TILE) == 313
    assert n_active == 3032 and _ceil(n_active, CHUNK) == 190
    valid = _valid(state)
    index_of = {c: i for i, c in enumerate(valid)}
    sample, clipped = _sample_cells(oracle, og, 0, state, 8, 3, H, W)
    # the first cell (clipped at the top left), three more of the right column, three more of the bottom row and the last cell
    assert len(sample) == 16 and valid[0] in sample and valid[-1] in sample and clipped == 8, (sample, clipped)

    # (i)
    grids, Ds = _generate(gen, 0, 0)
    grid, D = grids[0], Ds[0]
    assert D.shape == (n_cells, N) and np.isfinite(D).all()
    _assert_argmin(D, state, grid)
    got_rows = D[[index_of[c] for c in sample]].copy()
    del D, Ds
    grids_fast, _ = _generate(gen, 0, 0, keep=False)
    assert np.array_equal(grids_fast[0], grid)
    # (iii)
    rr, ra = 3, 2000
    grids3, Ds3 = _generate(gen, rr, ra)
    gen.close()
    sel = oracle.select_from_D(Ds3[0].astype(np.float64), state, rr, ra)
    assert np.array_equal(sel, grids3[0]), "%d cells differ from the repeat rule on the engine's D" % int((sel != grids3[0]).sum())
    n_repeat_diff = int((grids3[0] != grid).sum())
    del Ds3, sel

    # (ii) complete f64 rows, library in batches
    mains = [oracle.to_working_space(main, oracle.RGB_EUCLIDEAN)]
    sub = np.full_like(state, -1)
    for c in sample:
        sub[c] = 0
    ex, bounds, flips, _ = oracle.extract_cells(mains, og, 0, sub)
    del mains
    masks4 = og.detail_cells[0].masks4()
    want = np.empty((len(sample), N))
    batches = [(lo, min(lo + 2000, N)) for lo in range(0, N, 2000)]
    lock = threading.Lock()

    def worker():
        while True:
            with lock:
                if not batches:
                    return
                lo, hi = batches.pop()
            lib_f = oracle.preprocess_library(lib[lo:hi], og, oracle.RGB_EUCLIDEAN)
            want[:, lo:hi] = oracle.generate_step(oracle.RGB_EUCLIDEAN, ex, bounds, flips, lib_f, masks4, sub, 0, 0, want_D=True,
                                                  early_exit=False).D

    threads = [threading.Thread(target=worker) for _ in range(max(2, min(10, (os.cpu_count() or 2) - 1)))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    worst = float(check_differences(got_rows, want).max())
    in_band = 0
    for c, row in zip(sample, want):
        b, g = int(np.argmin(row)), int(grid[c])
        if g != b:
            assert (row[g] - row[b]) / max(row[b], 1e-30) <= TIE_TOL, (c, g, b)
            in_band += 1
    print("config 5 full size: %d cells x %d images; %d complete f64 rows (%d clipped border cells), max relative error %.2e, "
          "tie-band cells %d; repeats %d/%d changed %d cells" % (n_cells, N, len(sample), clipped, worst, in_band, rr, ra,
                                                                 n_repeat_diff))


# ----------------------------------------------------------------------------- F: the case tables (CPU)


def test_case_tables_cross_their_boundaries(oracle):
    """Recomputes the cell, tile, pixel and chunk counts of A-C from the oracle's grid state and masks, so that a change of a
    table (or of the grid geometry) cannot quietly move a case off the boundary it is there for."""
    # A
    seen = set()
    for H, W, n_cells, N, n_ct, n_lt in A_CASES:
        state = oracle.grid_state(_square_group(oracle, A_CELL), None, H, W)[0]
        n = int((state >= 0).sum())
        assert (n, _ceil(n, TILE), _ceil(N, TILE)) == (n_cells, n_ct, n_lt), (H, W, N)
        seen |= {"under one tile" if n < TILE else "", "64k" if n % TILE == 0 else "",
                 "17th tile" if 1025 <= n <= 1088 else "", "past two blocks" if n > 2 * TILE * SUPER else "",
                 "both past 16" if n_ct > SUPER and n_lt > SUPER else "", "partial band" if n_lt > SUPER and n_lt % SUPER else "",
                 "clipped" if (H % A_CELL or W % A_CELL) else ""}
    assert seen >= {"under one tile", "64k", "17th tile", "past two blocks", "both past 16", "partial band", "clipped"}, seen
    assert {c[3] for c in A_CASES} == {1, 63, 64, 65, 1024, 1025, 1100}
    assert any(c[4] > 2 * SUPER and c[4] % SUPER for c in A_CASES)  # a third, partial column block

    # B
    chunks = []
    for k, size, flips in B_CASES:
        sh = _b_shape(oracle, k, size, flips)
        assert int((sh.mask > 0).sum()) == k
        H, W = B_MAIN[size]
        state = oracle.grid_state(_square_group(oracle, size), None, H, W)[0]
        n = int((state >= 0).sum())
        assert n == B_CELLS and _ceil(n, TILE) == 2 and _ceil(B_N, TILE) == 3 and B_N % TILE
        assert H % size and W % size  # clipped border cells
        n_active, used = _active_pixels(oracle, sh, sh, state)
        if flips:
            assert used == {0, 1, 2, 3} and k < FLUSH < n_active
        else:
            assert used == {0} and n_active == k
        chunks.append(_ceil(n_active, CHUNK))
    assert {k for k, _, f in B_CASES if not f} == {1, 15, 16, 17, 1023, 1024, 1025, 2047, 2048, 2049, 4097}
    per_flush = FLUSH // CHUNK
    assert {c // per_flush for c in chunks} == {0, 1, 2, 4}        # no flush, one, two and four flushes
    assert {c % per_flush for c in chunks} >= {0, 1}  # a flush with no tail after it, a 1-chunk tail
    assert {k % CHUNK for k, _, _ in B_CASES} >= {0, 1, CHUNK - 1}  # full, 1-pixel and 15-pixel last chunks

    # C
    H, W = C_MAIN
    state = oracle.grid_state(_square_group(oracle, C_CELL), None, H, W)[0]
    black = _c_black_cells(state)
    valid = _valid(state)
    row = [c for c in valid if c[0] == C_BLACK_ROW + 2]
    assert len(row) == _ceil(W, C_CELL) and set(row) | {valid[0], valid[-1]} == set(black) and len(black) == len(row) + 2
    assert all(N % TILE for N in C_NS) and H % C_CELL and W % C_CELL  # padded library tiles; the last black cell is clipped
