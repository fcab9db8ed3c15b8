"""Usage limit (mosaic_set_usage_limit, DESIGN.md 4.4): each library image is chosen at most M times per generate.

The rule is sequential: cells are decided step by step in raster order, each taking the lowest (D + A * window count, slot) over the
slots whose image has been chosen fewer than M times so far. So:
  * the grids must equal that rule applied to the engine's own D (tests/helpers/usage_limit.capped_rule) exactly, with the use counts
    carried across the size steps, and to the f64 oracle's D teacher-forced outside the 1e-5 tie band;
  * no image is used more than M times, and exactly M times when M * N equals the number of cells;
  * a cap that cannot bind gives the grids of the uncapped engine bit for bit (the capped kernel against the wavefront);
  * the pruned and sharded paths choose exactly what the complete, unsharded path chooses.
"""
import numpy as np
import pytest

from tests.helpers.parity import TIE_TOL
from tests.helpers.usage_limit import PREFIX_MAX, capped_rule, exhausted_bound, k_bound, window_counts

pytestmark = pytest.mark.gpu


def make_gen(main, lib, diff, detail=100, steps=0, shape=None, scheme=0, faithful=True):
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(diff)
    gen.setColourScheme(scheme)
    gen.setVariantQuirk(faithful)
    cg = CellGroup()
    cg.setCellShape(shape if shape is not None else CellShape(lib.shape[1]))
    cg.setDetail(detail)
    cg.setSizeSteps(steps)
    gen.setCellGroup(cg)
    state = gen.computeGridState()
    return gen, state


def run(main, lib, diff, M, rr=0, ra=0, flips=0, keep=True, margins=False, **kw):
    """One generate on a fresh handle: (slot grids, state, D per step or None, margins per step or None, timings)."""
    gen, state = make_gen(main, lib, diff, **kw)
    try:
        if flips:
            gen.setTileFlips(bool(flips & 1), bool(flips & 2))
        gen.setRepeat(rr, ra)
        gen.setUsageLimit(M)
        gen.setKeepDifferences(keep)
        gen.setReportMargins(margins)
        assert gen.generateBestFits()
        grids = [g.copy() for g in gen.getBestFits()]
        if flips:  # slot = orientation index * N + image
            codes = gen.getBestFitFlips()
            order = {c: j for j, c in enumerate(c for c in range(4) if c & ~flips == 0)}
            grids = [np.where(g >= 0, np.vectorize(lambda c: order.get(int(c), 0))(f) * len(lib) + g, -1) for g, f in zip(grids, codes)]
        Ds = [gen.getDifferences(s) for s in range(len(state))] if keep else None
        ms = [gen.getMargins(s) for s in range(len(state))] if margins else None
        return grids, state, Ds, ms, gen.getTimings()
    finally:
        gen.close()


def n_cells(state):
    return int(sum((np.asarray(s) >= 0).sum() for s in state))


def uses(grids, n_images):
    v = np.concatenate([g[g >= 0].ravel() for g in grids]) % n_images
    return np.bincount(v, minlength=n_images)


# ----------------------------------------------------------------------------- exact against the rule on the engine's D

# diff, M, (rr, ra), flips, steps, library images per allowed cell (> 1: K_s stays small, the candidates come from top-K)
CASES = [(d, M, rep, fl, st, wide)
         for d in (0, 1, 2) for M in (1, 2, 3) for rep, fl, st, wide in
         (((0, 0), 0, 2, 1.1), ((2, 500), 3, 0, 8.0), ((8, 500), 3, 2, 1.3))]


@pytest.mark.parametrize("case", CASES, ids=["d%d-M%d-r%d-f%d-s%d-%g" % (d, M, r[0], f, s, w) for d, M, r, f, s, w in CASES])
def test_grid_equals_rule_on_engine_D(case):
    from mosaicmagnifique_b200 import synthetic
    diff, M, (rr, ra), flips, steps, wide = case
    main = synthetic.make_main_image(320, 448, 40 + diff + 3 * M, block=32)
    probe, state = make_gen(main, synthetic.make_library(1, 32, 1), diff, detail=50, steps=steps)
    probe.close()
    U = n_cells(state)
    N = int(np.ceil(U / M * wide))
    lib = synthetic.make_library(N, 32, 50 + M)
    grids, state, Ds, _, _ = run(main, lib, diff, M, rr, ra, flips, detail=50, steps=steps)
    want, _ = capped_rule(Ds, state, rr, ra, N, M)
    for s, (a, b) in enumerate(zip(grids, want)):
        assert np.array_equal(a, b), "step %d: %d cells differ" % (s, int((a != b).sum()))
    assert uses(grids, N).max() <= M
    # the run that does not keep D (pruned where CIEDE2000 allows it) chooses the same
    g2 = run(main, lib, diff, M, rr, ra, flips, keep=False, detail=50, steps=steps)[0]
    assert all(np.array_equal(a, b) for a, b in zip(g2, grids))


def test_colour_scheme_every_variant():
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(256, 320, 61, block=32)
    lib = synthetic.make_library(120, 32, 62)
    grids, state, Ds, _, _ = run(main, lib, 2, 1, 2, 500, scheme=2, faithful=False)
    assert n_cells(state) <= len(lib)
    assert np.array_equal(grids[0], capped_rule(Ds, state, 2, 500, len(lib), 1)[0][0])
    assert uses(grids, len(lib)).max() == 1


# ----------------------------------------------------------------------------- exact against f64


@pytest.mark.parametrize("diff,rr,ra", [(2, 2, 500), (0, 0, 0), (1, 8, 500)])
def test_teacher_forced_against_f64(oracle, diff, rr, ra):
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(384, 512, 70 + diff, block=32)
    lib = synthetic.make_library(260, 32, 71)
    M = 1
    grids, state, Ds, _, _ = run(main, lib, diff, M, rr, ra)
    og = oracle.CellGroup.make(oracle.CellShape.square(32), 100, 0)
    ostate = oracle.grid_state(og, main)
    assert np.array_equal(ostate[0], state[0]) and n_cells(state) <= len(lib)
    Do = oracle.generate(main, lib, og, ostate, diff, 0, 0, 0, early_exit=False)[0].D
    grid, used = grids[0], np.zeros(len(lib), np.int64)
    ties, bad, c = 0, [], 0
    for y in range(grid.shape[0]):
        for x in range(grid.shape[1]):
            if state[0][y, x] < 0:
                assert grid[y, x] == -1
                continue
            got = int(grid[y, x])
            assert used[got] < M
            v = Do[c] + (ra * window_counts(grid, x, y, rr, len(lib)) if rr and ra else 0)
            v = np.where(used < M, v, np.inf)
            best = int(np.argmin(v))
            if got != best:
                gap = (v[got] - v[best]) / max(v[best], 1e-30)
                ties += gap <= TIE_TOL
                if gap > TIE_TOL:
                    bad.append((y, x, got, best, gap))
            used[got] += 1
            c += 1
    assert not bad, bad[:3]
    print("diff %d: %d cells, %d in the tie band" % (diff, c, ties))


# ----------------------------------------------------------------------------- counts and a cap that cannot bind


@pytest.mark.parametrize("M", [1, 2, 3])
def test_every_image_used_M_times_when_MN_equals_cells(M):
    """N = ceil(U / M): every image is used M times, except that the d = M * N - U placements nobody needs are missing"""
    from mosaicmagnifique_b200 import MosaicError, synthetic
    main = synthetic.make_main_image(320, 448, 80 + M, block=32)
    for steps in (0, 2):
        probe, state = make_gen(main, synthetic.make_library(1, 32, 1), 2, steps=steps)
        probe.close()
        U = n_cells(state)
        N = -(-U // M)
        d = M * N - U
        lib = synthetic.make_library(N, 32, 81)
        grids, state, Ds, _, _ = run(main, lib, 2, M, 2, 500, steps=steps)
        cnt = uses(grids, N)
        assert cnt.sum() == U and cnt.max() == M and (M - cnt).sum() == d
        if d == 0:
            assert (cnt == M).all()
        assert all(np.array_equal(a, b) for a, b in zip(grids, capped_rule(Ds, state, 2, 500, N, M)[0]))
        with pytest.raises(MosaicError) as e:  # one image fewer cannot cover the cells
            run(main, lib[:-1], 2, M, 2, 500, steps=steps)
        assert e.value.code == -1


@pytest.mark.parametrize("diff,rr,ra,flips", [(2, 2, 500, 0), (0, 0, 0, 0), (2, 0, 0, 3), (1, 8, 500, 1)])
def test_non_binding_cap_is_bit_identical_to_no_cap(diff, rr, ra, flips):
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(320, 448, 90 + diff, block=32)
    lib = synthetic.make_library(200, 32, 91)
    base = run(main, lib, diff, 0, rr, ra, flips, keep=False, margins=True, steps=2)
    U = n_cells(base[1])
    capped = run(main, lib, diff, U, rr, ra, flips, keep=False, margins=True, steps=2)
    for a, b in zip(base[0], capped[0]):
        assert np.array_equal(a, b)
    for (b0, s0), (b1, s1) in zip(base[3], capped[3]):
        assert np.array_equal(b0, b1) and np.array_equal(s0, s1)


# ----------------------------------------------------------------------------- the fallback past the sorted prefix


@pytest.mark.parametrize("N", [1500, 6000])  # K_s * 4 > N: prefixes of D rows; K_s * 4 <= N: prefixes of top-K lists
def test_fallback_past_the_prefix(N):
    """A flat main image: every cell has the same D row, so with M = 1 cell c takes the c-th best image, and from cell 1,024 on every
    image of the sorted prefix is exhausted."""
    from mosaicmagnifique_b200 import synthetic
    main = np.full((16 * 30, 16 * 40, 3), (90, 140, 200), np.uint8)
    lib = synthetic.make_library(N, 16, 100)
    grids, state, Ds, _, _ = run(main, lib, 0, 1)
    U = n_cells(state)
    assert U > PREFIX_MAX + 64 and U < N
    K = k_bound(1, N, 0, exhausted_bound(0, U, 1))
    assert (K * 4 <= N) == (N == 6000)
    want, fallbacks = capped_rule(Ds, state, 0, 0, N, 1, scan=([(min(K, PREFIX_MAX), K if K * 4 <= N else N)], False))
    assert np.array_equal(grids[0], want[0])
    assert fallbacks >= U - PREFIX_MAX - 32
    assert uses(grids, N).max() == 1
    order = np.lexsort((np.arange(N), Ds[0][0]))
    assert np.array_equal(grids[0][state[0] >= 0], order[:U])  # raster order walks down the shared ranking
    print("N %d: %d cells, %d fell back past the prefix" % (N, U, fallbacks))


# ----------------------------------------------------------------------------- pruned equals complete


def test_pruned_equals_complete():
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(448, 576, 110, block=32)
    lib = synthetic.make_library(900, 32, 111)
    M, rr, ra = 2, 2, 500
    full = run(main, lib, 2, M, rr, ra, keep=True, margins=True)
    pruned = run(main, lib, 2, M, rr, ra, keep=False, margins=True)
    U = n_cells(full[1])
    assert 4 * k_bound(1, len(lib), rr, exhausted_bound(0, U, M), margins=True) <= len(lib)
    assert pruned[4]["evaluated_pixel_diffs"] < pruned[4]["pixel_diffs"]  # pruning triggered
    assert np.array_equal(full[0][0], pruned[0][0])
    assert np.array_equal(full[3][0][0], pruned[3][0][0]) and np.array_equal(full[3][0][1], pruned[3][0][1])
    assert np.array_equal(full[0][0], capped_rule(full[2], full[1], rr, ra, len(lib), M)[0][0])
    print("executed share %.3f" % (pruned[4]["evaluated_pixel_diffs"] / pruned[4]["pixel_diffs"]))


# ----------------------------------------------------------------------------- sharded


@pytest.mark.parametrize("world", [2, 4])
def test_emulated_ranks(world):
    import torch
    from mosaicmagnifique_b200 import CellShape, synthetic
    from mosaicmagnifique_b200.parallel import device_view
    main = synthetic.make_main_image(520, 700, 120 + world, block=32)
    M, rr, ra, steps = 1, 2, 400, 2
    probe, state = make_gen(main, synthetic.make_library(1, 32, 1), 2, steps=steps)
    probe.close()
    lib = synthetic.make_library(int(n_cells(state) * 1.2), 32, 121)
    want = run(main, lib, 2, M, rr, ra, keep=False, steps=steps)[0]
    dev = torch.device("cuda", 0)
    gens = []
    for r in range(world):
        g, _ = make_gen(main, lib, 2, steps=steps)
        g.setRepeat(rr, ra)
        g.setUsageLimit(M)
        g.setShard(r, world)
        g.generateCandidates()
        gens.append(g)
    gathered = []
    for s in range(len(state)):
        blocks = [g.candidateBlock(s) for g in gens]
        gathered.append((torch.cat([device_view(b["ptr"], (b["bytes"] // 4,), torch.int32, dev).clone() for b in blocks]).contiguous()
                         if blocks[0]["n_valid"] else None, blocks[0]["k"], blocks[0]["rows_per_rank"]))
    torch.cuda.synchronize()
    non_empty = [s for s in range(len(state)) if gathered[s][0] is not None]
    for g in gens:
        for s in non_empty:
            buf, k, rpr = gathered[s]
            g.selectFromGathered(s, buf.data_ptr(), k, rpr)
        got = g.getBestFits()
        assert all(np.array_equal(a, b) for a, b in zip(got, want))
    # out of order: selecting a step at or below the last one restarts the use counts, and then a step whose predecessor with cells
    # has not been selected since is refused; selecting the steps in order again gives the same grids
    assert len(non_empty) == 2
    g, sel = gens[0], lambda g, s: g._L.mosaic_select_from_gathered(g._h, s, gathered[s][0].data_ptr(), gathered[s][1], gathered[s][2])
    assert sel(g, non_empty[1]) == -4
    for s in non_empty:
        assert sel(g, s) == 0
    assert all(np.array_equal(a, b) for a, b in zip(g.getBestFits(), want))
    for g in gens:
        g.close()


# ----------------------------------------------------------------------------- at size


def _at_size(cfg_name, prune_too):
    import bench
    cfg = bench.WORKLOADS[cfg_name]
    main, lib = bench.make_inputs(cfg)
    kw = dict(detail=cfg["detail"], steps=cfg.get("steps", 0), shape=bench.make_shape(cfg))
    grids, state, Ds, _, tm = run(main, lib, cfg["diff"], 1, cfg["rr"], cfg["ra"], **kw)
    want, _ = capped_rule(Ds, state, cfg["rr"], cfg["ra"], len(lib), 1)
    for a, b in zip(grids, want):
        assert np.array_equal(a, b), "%d cells differ" % int((a != b).sum())
    assert uses(grids, len(lib)).max() == 1
    if prune_too:
        g2, _, _, _, tm2 = run(main, lib, cfg["diff"], 1, cfg["rr"], cfg["ra"], keep=False, **kw)
        assert all(np.array_equal(a, b) for a, b in zip(g2, grids))
        print("executed share %.3f" % (tm2["evaluated_pixel_diffs"] / tm2["pixel_diffs"]))
    print("%s M 1: %d cells, %d images" % (cfg_name, n_cells(state), len(lib)))


def test_config4_no_duplicates():
    _at_size("cfg4", True)


def test_config5_no_duplicates():
    _at_size("cfg5", False)


# ----------------------------------------------------------------------------- invalid input


def test_invalid_input():
    from mosaicmagnifique_b200 import MosaicError, synthetic
    main = synthetic.make_main_image(256, 320, 130, block=32)
    lib = synthetic.make_library(60, 32, 131)
    gen, state = make_gen(main, lib[:20], 2)
    U = n_cells(state)
    L, h = gen._L, gen._h
    assert L.mosaic_set_usage_limit(h, -1) == -1
    with pytest.raises(MosaicError):
        gen.setUsageLimit(-3)
    M = (U - 1) // 20  # M * N < U
    assert M >= 1
    gen.setUsageLimit(M)
    with pytest.raises(MosaicError) as e:
        gen.generateBestFits()
    msg = str(e.value)
    assert e.value.code == -1 and " %d valid cells" % U in msg and "x 20 images" in msg, msg
    gen.setUsageLimit(M + 1)
    assert gen.generateBestFits()
    gen.close()
    # changing M between two generates on one handle: each generate equals a fresh handle's
    lib = synthetic.make_library(U, 32, 132)
    gen, _ = make_gen(main, lib, 2)
    gen.setRepeat(2, 500)
    got = []
    for M in (1, 2, 0, 1):
        gen.setUsageLimit(M)
        assert gen.generateBestFits()
        got.append(gen.getBestFits()[0].copy())
    gen.close()
    for M, g in zip((1, 2, 0, 1), got):
        assert np.array_equal(g, run(main, lib, 2, M, 2, 500, keep=False)[0][0])
    assert (uses([got[0]], U) == 1).all()
