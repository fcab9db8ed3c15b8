"""Mirrored library tiles (mosaic_set_tile_flips, DESIGN.md 4.4).

With flips on, the candidate set is O * N slots, orientation-major: slot = j * N + i for the j-th enabled orientation of image i,
exactly a library given explicitly as [lib, flip_1(lib), ...]. So:
  * without repeats, slot grids and the difference matrix D must be bit-identical to a handle given that explicit library;
  * with repeats, the O orientations of an image share one count: the grid must be the grouped repeat rule applied to the engine's
    own D (exactly), and to the f64 oracle's D of the explicit library (outside the 1e-5 tie band);
  * buildPhotomosaic must equal the oracle's compositing of the explicit library with slot grids, byte for byte.
"""
import os

import numpy as np
import pytest

from tests.helpers.parity import D_TOL_TYPICAL, TIE_TOL, check_differences, rel_err

pytestmark = pytest.mark.gpu
CELLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells")
TRIANGLE = "IsocelesTriangle-45deg"  # alternate rows and columns flip the mask: all four mask flips occur


def orientations(flips):
    return [c for c in range(4) if c & ~flips == 0]


def orient(lib, code):
    out = lib
    if code & 1:
        out = out[:, :, ::-1]  # columns: cv::flip code 1
    if code & 2:
        out = out[:, ::-1]  # rows: cv::flip code 0
    return np.ascontiguousarray(out)


def explicit_library(lib, flips):
    return np.concatenate([orient(lib, c) for c in orientations(flips)])


def slot_grids(images, codes, flips, n):
    order = {c: j for j, c in enumerate(orientations(flips))}
    out = []
    for im, fl in zip(images, codes):
        assert ((im < 0) == (fl < 0)).all()
        j = np.vectorize(lambda c: order.get(int(c), 0))(fl)
        out.append(np.where(im >= 0, j * n + im, -1))
    return out


def product_shape(name, size):
    from mosaicmagnifique_b200 import CellShape, load_mcs
    return CellShape(size) if name == "square" else load_mcs(os.path.join(CELLS, name + ".mcs")).resized(size)


def oracle_shape(oracle, name, size):
    if name == "square":
        return oracle.CellShape.square(size)
    from tests.test_gpu_baseline_configs import load_shape
    return load_shape(oracle, name)[0].resized(size)


def run(main, lib, shape, diff, flips=0, detail=100, steps=0, rr=0, ra=0, keep=True, scheme=0, faithful=True, margins=False):
    """One generate on a fresh handle: (image grids, orientation grids or None, D per step or None, timings)."""
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
    gen = PhotomosaicGenerator(0)
    try:
        gen.setMainImage(main)
        gen.setLibrary(lib)
        gen.setColourDifference(diff)
        gen.setColourScheme(scheme)
        gen.setVariantQuirk(faithful)
        cg = CellGroup()
        cg.setCellShape(shape)
        cg.setDetail(detail)
        cg.setSizeSteps(steps)
        gen.setCellGroup(cg)
        state = gen.computeGridState()
        if flips:
            gen.setTileFlips(bool(flips & 1), bool(flips & 2))
        gen.setRepeat(rr, ra)
        gen.setKeepDifferences(keep)
        gen.setReportMargins(margins)
        assert gen.generateBestFits()
        grids = [g.copy() for g in gen.getBestFits()]
        codes = gen.getBestFitFlips() if flips else None
        Ds = [gen.getDifferences(s) for s in range(len(state))] if keep else None
        return grids, codes, Ds, gen.getTimings()
    finally:
        gen.close()


def window_counts_grouped(grid, x, y, rr, n_images):
    """calculateRepeats occurrence counts with the orientations of an image pooled: slot s counts for image s mod N."""
    rows, cols = grid.shape
    y0 = min(max(y - rr, 0), rows)
    x0 = min(max(x - rr, 0), cols)
    x1 = min(max(x + rr, 0), cols - 1)
    vals = np.concatenate([grid[y0:y, x0:x1 + 1].ravel(), grid[y, x0:x]])
    vals = vals[vals >= 0] % n_images
    return np.bincount(vals, minlength=n_images) if vals.size else np.zeros(n_images, np.int64)


def grouped_rule(D, state, rr, ra, n_images):
    """The grouped repeat rule in raster order on D (f64), from scratch: what the wavefront must reproduce exactly."""
    grid = np.where(state >= 0, 0, -1).astype(np.int64)
    O = D.shape[1] // n_images
    c = 0
    for y in range(grid.shape[0]):
        for x in range(grid.shape[1]):
            if grid[y, x] < 0:
                continue
            v = D[c].astype(np.float64)
            if rr > 0 and ra:
                v = v + ra * np.tile(window_counts_grouped(grid, x, y, rr, n_images), O)
            grid[y, x] = int(np.argmin(v))
            c += 1
    return grid


def check_grid_grouped(D_oracle, state, gpu_slots, rr, ra, n_images, tol=TIE_TOL):
    """tests/helpers/parity.check_grid with grouped counts: teacher-forced, (n_cells, n_tie_band, mismatches)."""
    O = D_oracle.shape[1] // n_images
    ties, bad, c = 0, [], 0
    for y in range(state.shape[0]):
        for x in range(state.shape[1]):
            if state[y, x] < 0:
                assert gpu_slots[y, x] == -1
                continue
            v = D_oracle[c].astype(np.float64)
            if rr > 0 and ra:
                v = v + ra * np.tile(window_counts_grouped(gpu_slots, x, y, rr, n_images), O)
            best, got = int(np.argmin(v)), int(gpu_slots[y, x])
            if got != best:
                gap = (v[got] - v[best]) / max(v[best], 1e-30) if 0 <= got < v.size else np.inf
                if gap <= tol:
                    ties += 1
                else:
                    bad.append((y, x, got, best, float(gap)))
            c += 1
    return c, ties, bad


# ----------------------------------------------------------------------------- bit-identity without repeats

CASES = [  # shape, cell, detail, steps, scheme, faithful
    ("square", 64, 100, 0, 0, True),
    ("square", 64, 50, 0, 0, True),
    ("square", 64, 70, 0, 0, True),  # fractional INTER_AREA (64 -> 44)
    (TRIANGLE, 64, 100, 2, 0, True),  # all four mask flips, f32 halving over two size steps
    (TRIANGLE, 64, 50, 0, 0, True),
    ("square", 64, 100, 0, 2, False),  # triadic scheme, every variant compared
]


@pytest.mark.parametrize("flips", [1, 2, 3])
@pytest.mark.parametrize("diff", [0, 1, 2])
@pytest.mark.parametrize("case", CASES, ids=["sq-d100", "sq-d50", "sq-d70", "tri-steps2", "tri-d50", "sq-triadic"])
def test_bit_identical_to_explicit_library(case, diff, flips):
    from mosaicmagnifique_b200 import synthetic
    name, cell, detail, steps, scheme, faithful = case
    main = synthetic.make_main_image(320, 448, 500 + diff, block=32)
    lib = synthetic.make_library(13, cell, 600 + flips)
    ext = explicit_library(lib, flips)
    shape = product_shape(name, cell)
    kw = dict(detail=detail, steps=steps, scheme=scheme, faithful=faithful)
    for keep in (True, False):  # D-writing launch, then the fused-argmin launch (CIEDE2000 without D)
        g_ext, _, D_ext, tm_ext = run(main, ext, shape, diff, 0, keep=keep, **kw)
        g, codes, D, tm = run(main, lib, shape, diff, flips, keep=keep, **kw)
        for a, b in zip(slot_grids(g, codes, flips, len(lib)), g_ext):
            assert np.array_equal(a, b)
        if keep:
            for a, b in zip(D, D_ext):
                assert a.shape == (b.shape[0], len(ext)) and np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert tm["pixel_diffs"] == tm_ext["pixel_diffs"]


# ----------------------------------------------------------------------------- repeats count per source image


@pytest.mark.parametrize("rr,n_lib", [(2, 60), (8, 600)])  # 4 * (O * W + 1) <= O * N: the CIEDE2000 run prunes
@pytest.mark.parametrize("diff", [2, 0])
def test_grouped_repeats(oracle, diff, rr, n_lib):
    from mosaicmagnifique_b200 import CellShape, synthetic
    ra, flips, cell = 500, 3, 32  # 32 px: a single exactly-opposite-hue pixel pair (parity.py) stays inside D_TOL of a whole sum
    main = synthetic.make_main_image(448, 576, 700 + rr, block=32)
    lib = synthetic.make_library(n_lib, cell, 701 + rr)
    O = len(orientations(flips))
    assert 4 * (O * (2 * rr * rr + 2 * rr) + 1) <= O * n_lib
    g, codes, D, _ = run(main, lib, CellShape(cell), diff, flips, rr=rr, ra=ra, keep=True)
    slots = slot_grids(g, codes, flips, n_lib)[0]
    state = np.where(g[0] >= 0, 0, -1)
    # (a) the grouped rule on the engine's own D, exactly
    assert np.array_equal(slots, grouped_rule(D[0], state, rr, ra, n_lib))
    # (b) the pruned / D-less run chooses the same grid
    g2, codes2, _, tm = run(main, lib, CellShape(cell), diff, flips, rr=rr, ra=ra, keep=False)
    assert np.array_equal(slot_grids(g2, codes2, flips, n_lib)[0], slots)
    if diff == 2:
        assert tm["evaluated_pixel_diffs"] < tm["pixel_diffs"]
    # (c) the f64 oracle's D on the explicit library, teacher-forced with grouped counts
    og = oracle.CellGroup.make(oracle.CellShape.square(cell), 100, 0)
    ostate = oracle.grid_state(og, main)
    assert np.array_equal(ostate[0], state)
    want = oracle.generate(main, explicit_library(lib, flips), og, ostate, diff, 0, 0, 0, early_exit=False)[0]
    # 99 % of the sums within what FP32 explains. The maximum is not bounded by D_TOL here: a single exactly-opposite-hue pixel pair
    # (the discontinuity parity.py describes) weighs 4.5 x more in these 1,024-pixel sums than in a 4,608-pixel cell. D itself is the
    # explicit-library run's bit for bit (test_bit_identical_to_explicit_library).
    e = rel_err(D[0], want.D)
    assert np.quantile(e, 0.99) < D_TOL_TYPICAL, np.quantile(e, 0.99)
    n, ties, bad = check_grid_grouped(want.D, state, slots, rr, ra, n_lib)
    assert not bad, bad[:3]
    print("rr %d N %d: %d cells, %d in the tie band, max rel err of D %.2e, orientations used %s" % (
        rr, n_lib, n, ties, e.max(), np.unique(codes[0]).tolist()))


def test_margins_with_flips():
    """report_margins widens K to O * W + 2; the grid is unchanged and the best margin is the chosen slot's penalised score."""
    from mosaicmagnifique_b200 import CellShape, synthetic
    main = synthetic.make_main_image(256, 320, 810, block=16)
    lib = synthetic.make_library(80, 16, 811)
    a = run(main, lib, CellShape(16), 2, 3, rr=2, ra=500, keep=False)
    b = run(main, lib, CellShape(16), 2, 3, rr=2, ra=500, keep=False, margins=True)
    assert np.array_equal(a[0][0], b[0][0]) and np.array_equal(a[1][0], b[1][0])


# ----------------------------------------------------------------------------- ties


def test_self_mirror_images_are_placed_unflipped():
    from mosaicmagnifique_b200 import CellShape, synthetic
    S = 32
    rng = np.random.default_rng(900)
    sym = []
    for _ in range(10):  # mirror-symmetric in both axes: one quadrant mirrored
        q = rng.integers(0, 256, (S // 2, S // 2, 3), np.uint8)
        half = np.concatenate([q, q[:, ::-1]], axis=1)
        sym.append(np.concatenate([half, half[::-1]], axis=0))
    uniform = [np.full((S, S, 3), rng.integers(0, 256, 3), np.uint8) for _ in range(10)]
    lib = np.ascontiguousarray(np.stack(sym + uniform + list(synthetic.make_library(12, S, 901))))
    main = synthetic.make_main_image(320, 448, 902, block=32)
    for diff in (0, 2):
        g, codes, _, _ = run(main, lib, CellShape(S), diff, 3, keep=False)
        chosen_sym = g[0] < 20
        chosen_sym &= g[0] >= 0
        assert chosen_sym.any()
        assert (codes[0][chosen_sym] == 0).all()
        assert ((codes[0] >= 0) == (g[0] >= 0)).all()


# ----------------------------------------------------------------------------- sharding


@pytest.mark.parametrize("world", [2, 4])
def test_emulated_ranks(world):
    import torch
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator, synthetic
    from mosaicmagnifique_b200.parallel import device_view
    main = synthetic.make_main_image(520, 700, 950 + world, block=32)
    lib = synthetic.make_library(70, 32, 951)
    rr, ra, flips = 2, 400, 3
    want, want_codes, _, _ = run(main, lib, CellShape(32), 2, flips, rr=rr, ra=ra, keep=False)
    dev = torch.device("cuda", 0)
    gens = []
    for r in range(world):
        g = PhotomosaicGenerator(0)
        g.setMainImage(main)
        g.setLibrary(lib)
        g.setColourDifference(2)
        cg = CellGroup()
        cg.setCellShape(CellShape(32))
        g.setCellGroup(cg)
        g.setRepeat(rr, ra)
        g.setTileFlips(True, True)
        g.computeGridState()
        g.setShard(r, world)
        g.generateCandidates()
        gens.append(g)
    blocks = [g.candidateBlock(0) for g in gens]
    k, rpr = blocks[0]["k"], blocks[0]["rows_per_rank"]
    assert k == min(4 * len(lib), 4 * (2 * rr * rr + 2 * rr) + 1)
    gathered = torch.cat([device_view(b["ptr"], (b["bytes"] // 4,), torch.int32, dev).clone() for b in blocks]).contiguous()
    torch.cuda.synchronize()
    for g in gens:
        g.selectFromGathered(0, gathered.data_ptr(), k, rpr)
        assert np.array_equal(g.getBestFits()[0], want[0])
        assert np.array_equal(g.getBestFitFlips()[0], want_codes[0])
        g.close()


# ----------------------------------------------------------------------------- compositing


@pytest.mark.parametrize("name,steps,bg", [("square", 2, (0, 0, 0, 0)), (TRIANGLE, 2, (17, 200, 90, 255)), (TRIANGLE, 0, (3, 4, 5, 6))])
@pytest.mark.parametrize("flips", [1, 3])
def test_build_photomosaic_equals_explicit_library(oracle, name, steps, bg, flips):
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator, synthetic
    S = 64
    main = synthetic.make_main_image(300, 430, 960 + steps, block=32)
    lib = synthetic.make_library(11, S, 961)
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(2)
    cg = CellGroup()
    cg.setCellShape(product_shape(name, S))
    cg.setSizeSteps(steps)
    gen.setCellGroup(cg)
    gen.computeGridState()
    gen.setTileFlips(bool(flips & 1), bool(flips & 2))
    gen.setRepeat(1, 300)
    assert gen.generateBestFits()
    slots = slot_grids(gen.getBestFits(), gen.getBestFitFlips(), flips, len(lib))
    assert any((np.asarray(c) > 0).any() for c in gen.getBestFitFlips())
    got = gen.buildPhotomosaic(bg)
    gen.close()
    og = oracle.CellGroup.make(oracle_shape(oracle, name, S), 100, steps)
    want = oracle.build_photomosaic(main.shape, explicit_library(lib, flips), og, slots, bg)
    assert np.array_equal(got, want)


# ----------------------------------------------------------------------------- at size


def _f64_rows(oracle, main, ext, og, state, diff, cells):
    from tests.test_gpu_euclid_scale import _f64_rows as rows
    mains = [oracle.to_working_space(main, diff)]
    D, _ = rows(oracle, mains, og, 0, state, cells, oracle.preprocess_library(ext, og, diff), diff)
    return D


def _at_size(oracle, cfg_name, flips):
    import bench
    from tests.test_gpu_baseline_configs import load_shape
    cfg = bench.WORKLOADS[cfg_name]
    main, lib = bench.make_inputs(cfg)
    N, O = len(lib), len(orientations(flips))
    g, codes, D, tm = run(main, lib, bench.make_shape(cfg), cfg["diff"], flips, detail=cfg["detail"], rr=cfg["rr"], ra=cfg["ra"])
    slots = slot_grids(g, codes, flips, N)[0]
    state = np.where(g[0] >= 0, 0, -1)
    D = D[0]
    assert D.shape == (int((state >= 0).sum()), O * N) and np.isfinite(D).all()
    assert np.array_equal(slots, grouped_rule(D, state, cfg["rr"], cfg["ra"], N))
    o_shape = load_shape(oracle, cfg["shape"])[0].resized(cfg["cell"])
    og = oracle.CellGroup.make(o_shape, cfg["detail"], 0)
    valid = [tuple(c) for c in np.argwhere(state >= 0)]
    pick = sorted({valid[i] for i in np.linspace(0, len(valid) - 1, 8).astype(int)})
    index_of = {c: i for i, c in enumerate(valid)}
    want = _f64_rows(oracle, main, explicit_library(lib, flips), og, state, cfg["diff"], pick)
    check_differences(D[[index_of[c] for c in pick]], want)
    print("%s flips %d: %d cells x %d slots, orientation counts %s" % (cfg_name, flips, len(valid), O * N,
                                                                       np.bincount(codes[0][codes[0] >= 0], minlength=4).tolist()))
    return tm


def test_config2_as_specified_flips_hv(oracle):
    _at_size(oracle, "cfg2", 3)


def test_config5_full_size_flips_h(oracle):
    _at_size(oracle, "cfg5", 1)


# ----------------------------------------------------------------------------- invalid input


def test_invalid_input():
    import ctypes
    from mosaicmagnifique_b200 import CellGroup, CellShape, MosaicError, PhotomosaicGenerator, synthetic
    main = synthetic.make_main_image(256, 320, 990, block=32)
    lib = synthetic.make_library(9, 32, 991)
    gen = PhotomosaicGenerator(0)
    L, h = gen._L, gen._h
    assert L.mosaic_set_tile_flips(h, -1) == -1 and L.mosaic_set_tile_flips(h, 4) == -1
    gen.setMainImage(main)
    gen.setLibrary(lib)
    cg = CellGroup()
    cg.setCellShape(CellShape(32))
    gen.setCellGroup(cg)
    state = gen.computeGridState()
    gen.setTileFlips(True, False)
    out = np.empty(state[0].shape, np.int8)
    assert L.mosaic_get_best_fit_flips(h, 0, out.ctypes.data, out.shape[0], out.shape[1]) == -4
    with pytest.raises(MosaicError):
        gen.getBestFitFlips()
    # a library stored at the detail size cannot be re-oriented
    assert L.mosaic_set_library_shard(h, lib.ctypes.data, 0, len(lib), len(lib), 32, len(lib)) == -5
    assert "re-oriented" in L.mosaic_last_error(h).decode()
    gen.setKeepDifferences(True)
    assert gen.generateBestFits()
    n = L.mosaic_get_valid_cell_count(h, 0)
    D = np.empty((n, 2 * len(lib)), np.float32)
    assert L.mosaic_get_differences(h, 0, D.ctypes.data, ctypes.c_int64(n), ctypes.c_int64(len(lib))) == -1
    assert L.mosaic_get_differences(h, 0, D.ctypes.data, ctypes.c_int64(n), ctypes.c_int64(2 * len(lib))) == 0
    assert gen.getDifferences(0).shape == (n, 2 * len(lib))
    # back to 0: the same grids as a handle that never had flips
    gen.setTileFlips(False, False)
    assert gen.generateBestFits()
    again = gen.getBestFits()[0]
    assert (gen.getBestFitFlips()[0][again >= 0] == 0).all()
    gen.close()
    fresh, _, _, _ = run(main, lib, CellShape(32), 0, 0, keep=False)
    assert np.array_equal(again, fresh[0])
    # a sharded library, then flips: generate refuses
    g2 = PhotomosaicGenerator(0)
    g2.setMainImage(main)
    g2.setCellGroup(cg)
    g2.computeGridState()
    g2.setLibraryShardPtr(lib.ctypes.data, 0, len(lib), len(lib), 32, len(lib))
    g2.setTileFlips(False, True)
    with pytest.raises(MosaicError) as e:
        g2.generateBestFits()
    assert e.value.code == -5
    g2.close()
