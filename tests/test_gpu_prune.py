"""Exact pruning of the CIEDE2000 difference sums on the top-K paths (DESIGN.md 7).

A pruned run (the default) and a run with setKeepDifferences(True) (complete D, same segment passes) must choose the same grid,
and every sum the pruned run completed must equal the complete run's bit for bit. Pruned pairs hold +inf and must lie strictly
above the K-th smallest sum of their cell, so the K smallest (score, index) entries of every cell -- what top-K hands to the
wavefront -- are identical."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _k_smallest(D, K):
    order = np.lexsort((np.broadcast_to(np.arange(D.shape[1]), D.shape), D), axis=1)[:, :K]
    return np.sort(order, axis=1)


def _check_pruned(full, pruned, K):
    assert full.shape == pruned.shape and np.isfinite(full).all()
    done = np.isfinite(pruned)
    assert np.array_equal(pruned[done].view(np.uint32), full[done].view(np.uint32))
    kth = np.sort(full, axis=1)[:, K - 1:K]
    assert (full[~done] > np.broadcast_to(kth, full.shape)[~done]).all()
    assert np.array_equal(_k_smallest(full, K), _k_smallest(pruned, K))
    return done.mean()


def _generate(main, lib, rr, ra, keep, shape=None, detail=100, steps=0, cell=32, diff=2):
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(diff)
    cg = CellGroup()
    cg.setCellShape(shape if shape is not None else CellShape(cell))
    cg.setDetail(detail)
    cg.setSizeSteps(steps)
    gen.setCellGroup(cg)
    state = gen.computeGridState()
    gen.setRepeat(rr, ra)
    gen.setKeepDifferences(keep)
    assert gen.generateBestFits()
    grids = [g.copy() for g in gen.getBestFits()]
    Ds = [gen.getDifferences(s) for s in range(len(state))]
    tm = gen.getTimings()
    gen.close()
    return grids, Ds, tm


def _pair(main, lib, rr, ra, **kw):
    g_full, D_full, tm_full = _generate(main, lib, rr, ra, True, **kw)
    g_pr, D_pr, tm_pr = _generate(main, lib, rr, ra, False, **kw)
    for a, b in zip(g_full, g_pr):
        assert np.array_equal(a, b)
    assert tm_full["evaluated_pixel_diffs"] == tm_full["pixel_diffs"]
    assert tm_pr["pixel_diffs"] == tm_full["pixel_diffs"]
    K = min(len(lib), 2 * rr * rr + 2 * rr + 1)
    fracs = [_check_pruned(a, b, K) for a, b in zip(D_full, D_pr)]
    return fracs, tm_pr


def test_config4_full_size_pruned_equals_complete():
    import bench
    cfg = bench.WORKLOADS["cfg4"]
    main, lib = bench.make_inputs(cfg)
    fracs, tm = _pair(main, lib, cfg["rr"], cfg["ra"], shape=bench.make_shape(cfg))
    assert tm["evaluated_pixel_diffs"] < tm["pixel_diffs"]
    print("config 4: pairs completed %.3f, evaluated / nominal %.3f" % (fracs[0], tm["evaluated_pixel_diffs"] / tm["pixel_diffs"]))


def test_config2_as_specified_pruned_equals_complete():
    import bench
    cfg = bench.WORKLOADS["cfg2"]
    main, lib = bench.make_inputs(cfg)
    fracs, tm = _pair(main, lib, cfg["rr"], cfg["ra"], shape=bench.make_shape(cfg), detail=cfg["detail"])
    assert tm["evaluated_pixel_diffs"] <= tm["pixel_diffs"]


@pytest.mark.parametrize("n_lib,rr,steps,cell", [
    (70, 2, 0, 32),    # N mod 8 = 6
    (20, 1, 0, 32),    # 4 K = N: smallest library that prunes, M clipped to N
    (19, 1, 0, 32),    # 4 K > N: no pruning, wavefront over whole rows
    (203, 3, 1, 64),   # two size steps, ragged last tile
    (64, 2, 0, 128),   # 128 chunks: the default eight segments of 16
])
def test_seeded_pruned_equals_complete(n_lib, rr, steps, cell):
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(300, 420, 90 + n_lib, block=32)
    lib = synthetic.make_library(n_lib, cell, 91 + n_lib)
    _pair(main, lib, rr, 300, steps=steps, cell=cell)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_emulated_ranks_pruned_candidates_equal_complete(world):
    """Sharded top-K path (candidates_only): every rank's candidate block, pruned and complete, bit-identical."""
    import torch
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator, synthetic
    from mosaicmagnifique_b200.parallel import device_view
    main = synthetic.make_main_image(520, 700, 80 + world, block=32)
    lib = synthetic.make_library(150, 32, 81)
    rr, ra = 3, 400
    want, _, _ = _generate(main, lib, rr, ra, False)
    dev = torch.device("cuda", 0)
    blocks = {}
    for keep in (False, True):
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
            g.computeGridState()
            g.setKeepDifferences(keep)
            g.setShard(r, world)
            g.generateCandidates()
            gens.append(g)
        infos = [g.candidateInfo(0) for g in gens]
        k = infos[0]["k"]
        scores = torch.cat([device_view(i["scores_ptr"], (i["n_cells"], k), torch.float32, dev).clone() for i in infos]).contiguous()
        idx = torch.cat([device_view(i["indices_ptr"], (i["n_cells"], k), torch.int32, dev).clone() for i in infos]).contiguous()
        torch.cuda.synchronize()
        blocks[keep] = (scores.cpu().numpy(), idx.cpu().numpy())
        for g in gens:
            g.selectFromCandidates(0, scores.data_ptr(), idx.data_ptr(), k)
            assert np.array_equal(g.getBestFits()[0], want[0])
            g.close()
    assert np.array_equal(blocks[False][1], blocks[True][1])
    assert np.array_equal(blocks[False][0].view(np.uint32), blocks[True][0].view(np.uint32))


def test_cancel_during_a_later_pass_drains():
    import threading
    import time
    from mosaicmagnifique_b200 import synthetic
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator
    main = synthetic.make_main_image(2160, 3840, 95)
    lib = synthetic.make_library(4000, 128, 96)
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(2)
    cg = CellGroup()
    cg.setCellShape(CellShape(128))
    gen.setCellGroup(cg)
    gen.computeGridState()
    gen.setRepeat(8, 500)
    seen, t_cancel = [], []

    def on_progress(v):
        seen.append(v)
        # the first pass covers 1/8 of the step's rows: cancel once later passes are running
        if not t_cancel and v * 8 > gen.getMaxProgress() * 3:
            t_cancel.append(time.perf_counter())
            gen.cancel()

    gen.setProgressCallback(on_progress)
    assert not gen.generateBestFits()
    t_end = time.perf_counter()
    assert t_cancel and t_end - t_cancel[0] < 0.1
    assert all(a < b for a, b in zip(seen, seen[1:]))
    gen.close()
