"""BASELINE.json configs[1] and configs[4] AS SPECIFIED -- on the reference's real cell shapes.

The ten `Cells/*.mcs` of the reference are committed under tests/golden/cells/ (reference-held fixtures) and read with the
product's own reader (mosaic_mcs_load: QDataStream layout + PNG codec in csrc/containers.cpp). The CUDA path is compared with
the reference generator's answer -- its own object code where oracle/_ref/libref_core.so is built, else the stored answer in
tests/golden/reference_grids.npz (which records its source) -- exactly as tests/test_gpu_generator.py::_direct_reference_case does: identical grid states, identical best-fit grids outside the tie band.

  config 2  Hexagon.mcs @128 (spacing 96/110, odd-row offset 55), detail 50 %, CIEDE2000, SampleImages main image
            (tst_Generator.h:80-90, 327-371: CreateHexagonCellGroup(128, 0, 50)); IsocelesTriangle(-45deg) as the flip case
  config 5  Puzzle.mcs @128 (spacing 108), detail 50 %, RGB Euclidean
"""
import os

import numpy as np
import pytest

from tests.test_gpu_generator import _direct_reference_case

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
CELLS = os.path.join(HERE, "golden", "cells")
SAMPLE = os.path.join(HERE, "golden", "images", "edgar-perez-424673-unsplash.jpg")
ALL_SHAPES = ["4PointStar", "6PointStar-1", "6PointStar-2", "6PointStar-3", "Circle", "Hexagon", "IsocelesTriangle-45deg",
              "IsocelesTriangle", "Puzzle", "YinAndYang"]


def load_shape(oracle, name):
    """(oracle CellShape built from the PRODUCT's reading of the file, product CellShape)"""
    from mosaicmagnifique_b200 import load_mcs
    p = load_mcs(os.path.join(CELLS, name + ".mcs"))
    o = oracle.CellShape.from_mask(p.getCellMask())
    o.row_spacing, o.col_spacing = p.rowSpacing, p.colSpacing
    o.alt_row_spacing, o.alt_col_spacing = p.alternateRowSpacing, p.alternateColSpacing
    o.alt_row_offset, o.alt_col_offset = p.alternateRowOffset, p.alternateColOffset
    o.alt_col_flip_h, o.alt_col_flip_v = p.alternateColFlipHorizontal, p.alternateColFlipVertical
    o.alt_row_flip_h, o.alt_row_flip_v = p.alternateRowFlipHorizontal, p.alternateRowFlipVertical
    return o, p


def sample_image(scale):
    import cv2
    img = cv2.imread(SAMPLE, cv2.IMREAD_COLOR)
    assert img is not None and img.shape == (4000, 5000, 3)
    return cv2.resize(img, None, fx=scale, fy=scale, interpolation=cv2.INTER_AREA)


def test_product_reader_equals_checker_reader(oracle):
    """mosaic_mcs_load (own PNG codec) against the cv2-based checker on every committed shape file (no GPU work, but kept with the
    config tests so that the fixtures the GPU cases run on are known to be read correctly on the box)."""
    for name in ALL_SHAPES:
        o, p = load_shape(oracle, name)
        want = oracle.load_mcs(os.path.join(CELLS, name + ".mcs"))
        assert np.array_equal(p.getCellMask(), want.mask) and o.params() == want.params(), name


def test_config2_hexagon_mcs_ciede2000_detail50_sample_image(oracle):
    """configs[1]: SampleImages main image (x0.25 so that the CPU reference finishes in seconds), Hexagon.mcs resized to 128,
    detail 50 %, CIEDE2000, a 160-image substitute library (big-lib.mil is absent from the reference checkout: seeded crops of the
    sample image itself through the reference-equivalent ingest + synthetic images), repeats on."""
    from mosaicmagnifique_b200 import synthetic
    o, _ = load_shape(oracle, "Hexagon")
    sh = o.resized(128)
    assert (sh.row_spacing, sh.col_spacing, sh.alt_row_offset) == (96, 110, 55)
    main = sample_image(0.25)
    lib = synthetic.make_photo_library(sample_image(0.5), 96, 128, seed=2002)
    lib = np.concatenate([lib, synthetic.make_library(64, 128, 2003)])
    n, n_diff = _direct_reference_case(oracle, "baseline-config2_hexagon", main, lib, sh, 2, 50, 0, 2, 500)
    assert n > 100
    print("config 2 (Hexagon.mcs, sample image): %d of %d cells differ from the reference (tie band)" % (n_diff, n))


def test_config5_puzzle_mcs_rgb_detail50(oracle):
    """configs[4] shape: Puzzle.mcs resized to 128 (spacing 108, 72 % active), detail 50 %, RGB Euclidean."""
    from mosaicmagnifique_b200 import synthetic
    o, _ = load_shape(oracle, "Puzzle")
    sh = o.resized(128)
    assert (sh.row_spacing, sh.col_spacing) == (108, 108)
    main = synthetic.make_main_image(1100, 1500, 505, block=64)
    lib = synthetic.make_library(300, 128, 506)
    for rr, ra in ((0, 0), (3, 2000)):  # BASELINE's config 5 has no repeats (fused argmin epilogue); and with the wavefront
        n, n_diff = _direct_reference_case(oracle, "baseline-config5_puzzle-rr%d" % rr, main, lib, sh, 0, 50, 0, rr, ra)
        assert n > 120
        print("config 5 shape (Puzzle.mcs) repeats %d/%d: %d of %d cells differ from the reference (tie band)" % (rr, ra, n_diff, n))


@pytest.mark.parametrize("name", ALL_SHAPES)
def test_every_reference_cell_shape(oracle, name):
    """All ten shipped shapes (flips on IsocelesTriangle: colV/rowV, IsocelesTriangle-45deg: all four, YinAndYang: colH/colV with
    alternate column spacing 0 -> clamped to 1 by resized()), resized to 64, detail 50 % and 100 %, one size step for half of them."""
    from mosaicmagnifique_b200 import synthetic
    o, _ = load_shape(oracle, name)
    k = ALL_SHAPES.index(name)
    sh = o.resized(64)
    main = synthetic.make_main_image(300, 420, 600 + k, block=32)
    lib = synthetic.make_library(48, 64, 700 + k)
    diff = (2, 0, 1)[k % 3]
    detail = 50 if k % 2 == 0 else 100
    steps = 1 if k % 4 == 1 else 0
    n, n_diff = _direct_reference_case(oracle, "baseline-shape-" + name, main, lib, sh, diff, detail, steps, 2, 300)
    assert n > 10
    print("%s: %d of %d cells differ from the reference (tie band)" % (name, n_diff, n))


@pytest.mark.parametrize("all_four", [False, True])
def test_isoceles_45deg_flips_config2_style(oracle, all_four):
    """The flip case of config 2 at its own size: IsocelesTriangle-45deg.mcs @128, detail 50 %, CIEDE2000. The file switches all four
    flip flags on, which (column and row flips XOR-ed, GridUtility.cpp:101-132) yields the unflipped and the doubly flipped mask;
    with the alternate-row vertical flip switched off all four flipped masks occur in the grid (checked)."""
    import ctypes

    from mosaicmagnifique_b200 import capi, synthetic
    from mosaicmagnifique_b200._capi import CellShapeC
    o, _ = load_shape(oracle, "IsocelesTriangle-45deg")
    assert o.alt_col_flip_h and o.alt_col_flip_v and o.alt_row_flip_h and o.alt_row_flip_v
    if all_four:
        o.alt_row_flip_v = False
    sh = o.resized(128)
    L = capi()
    cs = CellShapeC(*sh.params())
    flips = {L.mosaic_flip_at(ctypes.byref(cs), x, y) for x in range(4) for y in range(4)}
    assert flips == ({0, 1, 2, 3} if all_four else {0, 3})
    main = synthetic.make_main_image(700, 900, 811, block=64)
    lib = synthetic.make_library(80, 128, 812)
    n, n_diff = _direct_reference_case(oracle, "baseline-isoceles45-all_four%d" % all_four, main, lib, sh, 2, 50, 0, 2, 500)
    assert n > 60
    print("IsocelesTriangle-45deg @128 (flip states %s): %d of %d cells differ from the reference (tie band)" % (sorted(flips), n_diff, n))
