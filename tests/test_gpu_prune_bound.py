"""Lightness bound of the CIEDE2000 segments not yet summed (DESIGN.md 4.1).

A row of the segment passes dies once every pair has partial sum + R > T, R a lower bound of what the remaining segments add. The
bound must never exceed what the kernels actually sum, including their rounding: R[s] is checked directly against the summed
segments, and the pruned generate is checked against the complete one (setKeepDifferences(True)) where the bound is tightest --
achromatic cells and libraries, where dE00 = |dL| / S_L exactly -- with near-duplicate images that nearly tie at the K-th sum, and
where weights are not uniform over a block (clipped edge cells, a shape whose four flips occur)."""
import numpy as np
import pytest

from tests.test_gpu_prune import _pair

pytestmark = pytest.mark.gpu

SLACK = 1 - 2.0 ** -8


def _bound_and_rest(cells, lib, seg_chunks, target_area=None):
    """R [n_segs - 1][n_cells][n_lib] from the bound kernels, and the sums of segments s .. end from the difference kernel"""
    from mosaicmagnifique_b200 import capi
    L = capi()
    n_cells, size = cells.shape[0], cells.shape[1]
    n_lib = lib.shape[0]
    rows_per_seg = seg_chunks * 128 // size
    n_segs = size // rows_per_seg
    ta = None if target_area is None else np.asarray(target_area, np.int32)
    cells = np.ascontiguousarray(cells, np.float32)
    lib = np.ascontiguousarray(lib, np.float32)
    mask = np.full((size, size), 255, np.uint8)
    R = np.empty((n_segs - 1, n_cells, n_lib), np.float32)
    assert L.mosaic_kernel_prune_bound(0, cells.ctypes.data, n_cells, lib.ctypes.data, n_lib, mask.ctypes.data, size,
                                       None if ta is None else ta.ctypes.data, seg_chunks, R.ctypes.data) == 0
    seg = np.empty((n_segs, n_cells, n_lib))
    out = np.empty(n_lib, np.float32)
    for s in range(n_segs):
        m = np.zeros((size, size), np.uint8)
        m[s * rows_per_seg:(s + 1) * rows_per_seg] = 255
        for c in range(n_cells):
            assert L.mosaic_kernel_image_difference_sum(0, 2, cells[c].ctypes.data, lib.ctypes.data, n_lib, m.ctypes.data, size,
                                                        None if ta is None else ta.ctypes.data, out.ctypes.data) == 0
            seg[s, c] = out
    rest = np.cumsum(seg[::-1], 0)[::-1][1:]  # rest[s - 1] = segments s .. end
    return R, rest


def _lab(bgr):
    import cv2
    return cv2.cvtColor(bgr.reshape(-1, bgr.shape[-2], 3).astype(np.float32) / 255, cv2.COLOR_BGR2Lab).reshape(bgr.shape)


def test_bound_below_remaining_segments_config4_shape():
    """128 px cells, 8 segments of 16 chunks (config 4's passes), seeded synthetic cells and library: R[s] stays below the sum the
    difference kernel computes for segments s .. 7 by the slack, and is a useful fraction of it."""
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(512, 768, 2004)
    cells = np.stack([_lab(main[y:y + 128, x:x + 128]) for y in (0, 256, 384) for x in (0, 320, 640)])
    lib = _lab(synthetic.make_library(160, 128, 1004))
    R, rest = _bound_and_rest(cells, lib, 16)
    assert (R >= 0).all() and (R <= rest * (1 - 2.0 ** -9)).all(), (R / rest).max()
    assert (R[0] / rest[0]).mean() > 0.2


def test_bound_below_remaining_segments_target_area():
    """A detail-space bound that cuts through blocks (rows 0..99, columns 3..124): those blocks' weights are not uniform and add 0."""
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(256, 256, 77)
    cells = np.stack([_lab(main[y:y + 128, x:x + 128]) for y in (0, 128) for x in (0, 128)])
    lib = _lab(synthetic.make_library(48, 128, 78))
    R, rest = _bound_and_rest(cells, lib, 16, target_area=[0, 100, 3, 125])
    assert (R >= 0).all() and (R <= rest * (1 - 2.0 ** -9)).all()
    # segments 7 (rows 112..127) lie outside the bound: nothing is summed there and the bound is 0
    assert (R[6] == 0).all() and (rest[6] == 0).all()


def test_bound_is_tight_on_achromatic_pairs():
    """a = b = 0 and L_cell + L_lib = 100 at every pixel: dE00 = |dL| exactly, S_L = 1 at the block's worst mean lightness, and
    every block's dL has one sign, so the bound equals the sum up to rounding: R / rest must sit at the slack, not below, not above."""
    rng = np.random.default_rng(5)
    size, n_cells, n_lib = 128, 4, 24
    # L_cell = 50 - x, x constant on runs of 16 pixels (one block), its sign and size varying from block to block; multiples of
    # 1/64 keep Lh = L/2 - 25 and the block sums exact. Library image i is 100 - L of cell i % n_cells, so for those pairs
    # Lbar = 50 everywhere and dL = 2 x.
    x = rng.integers(-2000, 2000, (n_cells, size * size // 16)) / 64.0
    cells = np.zeros((n_cells, size, size, 3), np.float32)
    cells[..., 0] = 50 - np.repeat(x, 16, axis=1).reshape(n_cells, size, size)
    lib = np.zeros((n_lib, size, size, 3), np.float32)
    for i in range(n_lib):
        lib[i, ..., 0] = 100 - cells[i % n_cells, ..., 0]
    R, rest = _bound_and_rest(cells, lib, 16)
    idx = np.arange(n_lib)
    for c in range(n_cells):
        mine = idx % n_cells == c
        q = R[:, c, mine] / rest[:, c, mine]
        assert (q <= SLACK * (1 + 1e-4)).all() and (q >= SLACK * (1 - 1e-4)).all(), (q.min(), q.max())
    assert (R <= rest * (1 - 2.0 ** -9)).all()


def _grey(img):
    return np.repeat(img[..., None], 3, axis=-1).astype(np.uint8)


def _grey_inputs(n_lib, cell, seed, h=352, w=480):
    """grey main image and grey library with near-duplicate pairs (image 2k + 1 = image 2k with a few pixels one level apart), so
    that the K-th and (K + 1)-th sums of a cell nearly tie"""
    rng = np.random.default_rng(seed)
    base = rng.integers(20, 236, (h // 16 + 1, w // 16 + 1))
    main = np.kron(base, np.ones((16, 16), np.int64))[:h, :w] + rng.integers(-12, 13, (h, w))
    lib = np.empty((n_lib, cell, cell), np.int64)
    for i in range(0, n_lib, 2):
        lv = rng.integers(20, 236, (cell // 8, cell // 8))
        lib[i] = np.kron(lv, np.ones((8, 8), np.int64)) + rng.integers(-6, 7, (cell, cell))
        if i + 1 < n_lib:
            lib[i + 1] = lib[i]
            p = rng.integers(0, cell, (3, 2))
            lib[i + 1][p[:, 0], p[:, 1]] += 1
    return _grey(np.clip(main, 0, 255)), _grey(np.clip(lib, 0, 255))


@pytest.mark.parametrize("rr,cell", [(2, 32), (3, 64)])
def test_achromatic_near_duplicates_pruned_equals_complete(rr, cell):
    main, lib = _grey_inputs(120, cell, 11 + rr)
    _pair(main, lib, rr, 400, cell=cell)


def test_achromatic_near_duplicates_sharded_candidates_equal_complete():
    """candidates_only path, 2 emulated ranks: the candidate blocks of pruned and complete runs are bit-identical"""
    import torch
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator
    from mosaicmagnifique_b200.parallel import device_view
    main, lib = _grey_inputs(120, 32, 21)
    rr, ra = 2, 400
    dev = torch.device("cuda", 0)
    blocks = {}
    for keep in (False, True):
        parts = []
        for r in range(2):
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
            g.setShard(r, 2)
            g.generateCandidates()
            i = g.candidateInfo(0)
            s = device_view(i["scores_ptr"], (i["n_cells"], i["k"]), torch.float32, dev).clone()
            x = device_view(i["indices_ptr"], (i["n_cells"], i["k"]), torch.int32, dev).clone()
            torch.cuda.synchronize()
            parts.append((s.cpu().numpy(), x.cpu().numpy()))
            g.close()
        blocks[keep] = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]))
    assert np.array_equal(blocks[False][1], blocks[True][1])
    assert np.array_equal(blocks[False][0].view(np.uint32), blocks[True][0].view(np.uint32))


def test_clipped_edge_cells_pruned_equals_complete():
    """main image not a multiple of the cell: the last row and column of cells are clipped, their blocks partly weighted"""
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(300, 430, 31, block=32)
    lib = synthetic.make_library(96, 64, 32)
    _pair(main, lib, 2, 400, cell=64)


def test_flipped_mask_shape_pruned_equals_complete():
    """IsocelesTriangle-45deg switches all four flips: the compacted pixels are the union of the four masks, so every cell has
    zero-weight pixels inside blocks"""
    import bench
    from mosaicmagnifique_b200 import synthetic
    cfg = dict(bench.WORKLOADS["cfg2"], shape="IsocelesTriangle-45deg", cell=64)
    main = synthetic.make_main_image(384, 512, 41, block=32)
    lib = synthetic.make_library(96, 64, 42)
    _pair(main, lib, 2, 400, shape=bench.make_shape(cfg))
