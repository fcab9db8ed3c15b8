"""CellShape / CellGroup / ImageLibrary and the .mcs / .mil containers, pinned on the reference's own object code:
src/CellShape/CellShape.cpp, CellGroup.cpp, src/ImageLibrary/ImageLibrary.cpp and src/Other/CustomQDataStream.h are compiled
unmodified into oracle/_ref/libref_core.so (Qt = the stand-ins of oracle/shim/qt_standins.h, OpenCV resize / PNG codec = cv2
through callbacks). Checked against them: the oracle (CellShape.resized, CellGroup.make, load_mcs), the product's Python
mirror and readers / writers (mosaicmagnifique_b200.CellShape.resized, formats.py), and the ingest procedure the GPU tests
use as their expectation."""
import glob
import os

import numpy as np
import pytest

CELLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells")  # the reference's Cells/*.mcs
FIELDS = ("row_spacing", "col_spacing", "alt_row_spacing", "alt_col_spacing", "alt_row_offset", "alt_col_offset",
          "alt_col_flip_h", "alt_col_flip_v", "alt_row_flip_h", "alt_row_flip_v")


@pytest.fixture(scope="module")
def ref(oracle):
    if not oracle.reference_generator_available():
        pytest.skip("oracle/_ref/libref_core.so (reference object code) is not built")
    return oracle


def _shapes(o):
    from mosaicmagnifique_b200 import synthetic
    tri = o.CellShape.from_mask(synthetic.triangle_mask(64))
    tri.row_spacing = tri.alt_row_spacing = 64
    tri.col_spacing = tri.alt_col_spacing = 32
    tri.alt_col_flip_v = True
    tri.alt_row_flip_h = True
    hx = o.CellShape.from_mask(synthetic.hexagon_mask(128))
    hx.row_spacing = hx.alt_row_spacing = 96
    hx.col_spacing = hx.alt_col_spacing = 110
    hx.alt_row_offset = 55
    hx.alt_col_offset = 3
    return [o.CellShape.square(64), tri, hx]


def _same_shape(a, b):
    return a.size == b.size and np.array_equal(a.mask, b.mask) and all(getattr(a, f) == getattr(b, f) for f in FIELDS)


def test_cell_shape_resized_matches_reference_object_code(ref):
    """CellShape::resized (CellShape.cpp:281-312), shrinking (INTER_AREA) and growing (INTER_CUBIC): oracle and the product's
    Python mirror against the reference's code, masks for all four flips included."""
    from mosaicmagnifique_b200 import CellShape as ProductShape
    for sh in _shapes(ref):
        for new in (sh.size, sh.size // 2, 25, 37, sh.size + 19, 2 * sh.size):
            want, m4 = ref.reference_cell_shape_resized(sh, new)
            got = sh.resized(new)
            assert _same_shape(got, want), (sh.size, new)
            assert np.array_equal(got.masks4(), m4)
            ps = ProductShape(sh.mask)
            ps.rowSpacing, ps.colSpacing = sh.row_spacing, sh.col_spacing
            ps.alternateRowSpacing, ps.alternateColSpacing = sh.alt_row_spacing, sh.alt_col_spacing
            ps.alternateRowOffset, ps.alternateColOffset = sh.alt_row_offset, sh.alt_col_offset
            pr = ps.resized(new)
            assert np.array_equal(pr.getCellMask(), want.mask)
            assert (pr.rowSpacing, pr.colSpacing, pr.alternateRowSpacing, pr.alternateColSpacing, pr.alternateRowOffset,
                    pr.alternateColOffset) == (want.row_spacing, want.col_spacing, want.alt_row_spacing, want.alt_col_spacing,
                                               want.alt_row_offset, want.alt_col_offset)


@pytest.mark.parametrize("detail,steps", [(100, 0), (50, 2), (33, 1), (20, 3), (3, 1)])
def test_cell_group_matches_reference_object_code(ref, detail, steps):
    """CellGroup::setCellShape / setDetail / setSizeSteps (CellGroup.cpp:29-128): every step's normal and detail cell."""
    for sh in _shapes(ref):
        group = ref.CellGroup.make(sh, detail, steps)
        for s in range(steps + 1):
            for is_detail, mine in ((False, group.cells[s]), (True, group.detail_cells[s])):
                want, m4 = ref.reference_cell_group_cell(group, s, is_detail)
                assert _same_shape(mine, want), (sh.size, detail, s, is_detail)
                assert np.array_equal(mine.masks4(), m4)


def test_product_group_matches_reference_object_code(ref):
    """The product's host model (csrc/host_model.cpp Group::build, through mosaic_host_grid_state's step sizes) is already
    tested against the oracle; here its per-step grid geometry is tied to the reference's CellGroup via the grid sizes."""
    from mosaicmagnifique_b200 import synthetic
    main = synthetic.make_main_image(260, 390, 5, block=32)
    for sh in _shapes(ref):
        group = ref.CellGroup.make(sh, 50, 2)
        want = ref.reference_grid_state(group, main)
        got = ref.grid_state(group, main)
        assert [g.shape for g in got] == [g.shape for g in want]


def test_mcs_files_of_the_reference(ref, tmp_path):
    """Every Cells/*.mcs of the reference: the reference's own loadFromFile vs the product reader (formats.load_mcs) and the
    oracle reader; then both writers round-trip through the other side's reader."""
    from mosaicmagnifique_b200 import formats
    files = sorted(glob.glob(os.path.join(CELLS, "*.mcs")))
    assert len(files) >= 10
    for path in files:
        want, m4 = ref.reference_load_mcs(path)
        f = formats.load_mcs(path)
        assert f["name"] == want.name
        assert np.array_equal(f["mask"], want.mask)
        assert all(f[k] == getattr(want, k) for k in FIELDS), path
        o = ref.load_mcs(path)
        assert _same_shape(o, want) and np.array_equal(o.masks4(), m4)
        # product writer -> reference reader
        p1 = str(tmp_path / "product.mcs")
        formats.save_mcs(p1, f)
        back, _ = ref.reference_load_mcs(p1)
        assert _same_shape(back, want) and back.name == want.name
        # reference writer -> product reader
        p2 = str(tmp_path / "reference.mcs")
        ref.reference_save_mcs(p2, want, want.name)
        f2 = formats.load_mcs(p2)
        assert f2["name"] == want.name and np.array_equal(f2["mask"], want.mask) and all(f2[k] == f[k] for k in FIELDS)


def test_mcs_rejections_match(ref, tmp_path):
    from mosaicmagnifique_b200 import formats
    bad = str(tmp_path / "bad.mcs")
    open(bad, "wb").write(b"\x00\x01\x02\x03" * 8)
    with pytest.raises(ValueError):
        ref.reference_load_mcs(bad)
    with pytest.raises(ValueError):
        formats.load_mcs(bad)


def _procedure(o, im, size):
    """What tests/test_gpu_kernels.py expects of mosaic_library_ingest: centre crop + resizeImage EXACT."""
    r, c = im.shape[:2]
    if c < r:
        d = (r - c) // 2
        im = im[d:c + d, :c]
    elif c > r:
        d = (c - r) // 2
        im = im[:r, d:r + d]
    return o.resize_image_exact(np.ascontiguousarray(im), size, size)


def test_image_library_add_and_resize_match_reference_object_code(ref):
    """ImageLibrary::addImage / setImageSize (ImageLibrary.cpp:42-86) from the reference's code: the crop + resize procedure
    the GPU ingest is checked against IS what the reference computes (tall, wide, square, smaller and equal-size inputs)."""
    rng = np.random.default_rng(21)
    lib = ref.ReferenceImageLibrary(48)
    srcs = {}
    for i, (r, c) in enumerate([(100, 80), (48, 48), (30, 45), (200, 200), (97, 41), (64, 129)]):
        im = rng.integers(0, 256, (r, c, 3), dtype=np.uint8)
        srcs["im%d" % i] = im
        lib.add_image(im, "im%d" % i)
    items = lib.items()
    assert sorted(n for n, _ in items) == sorted(srcs)  # inserted at random indices (std::random_device)
    for name, img in items:
        assert np.array_equal(img, _procedure(ref, srcs[name], 48)), name
    before = dict(items)
    lib.set_image_size(32)  # batchResizeMat on the stored (already 48 px) images
    for name, img in lib.items():
        assert np.array_equal(img, ref.resize_image_exact(before[name], 32, 32)), name
    with pytest.raises(ValueError):
        lib.add_image(np.zeros((0, 0, 3), np.uint8))
    lib.close()


def test_mil_container_round_trips_with_reference_object_code(ref, tmp_path):
    """.mil (ImageLibrary.cpp:117-236): reference writer -> product reader, product writer -> reference reader, and the
    product's ImageLibrary mirror on a reference-written file."""
    from mosaicmagnifique_b200 import ImageLibrary, formats
    rng = np.random.default_rng(22)
    lib = ref.ReferenceImageLibrary(24)
    for i in range(7):
        lib.add_image(rng.integers(0, 256, (24, 24, 3), dtype=np.uint8), "image \u00e9 %d" % i)  # non-ASCII name: UTF-16 on the wire
    p1 = str(tmp_path / "reference.mil")
    lib.save(p1)
    items = lib.items()
    images, names, size = formats.load_mil(p1)
    assert size == 24 and names == [n for n, _ in items]
    assert all(np.array_equal(a, b) for a, (_, b) in zip(images, items))
    mirror = ImageLibrary(1)
    mirror.loadFromFile(p1)
    assert mirror.getImageSize() == 24 and mirror.getNames() == names and np.array_equal(mirror.asArray(), images)
    p2 = str(tmp_path / "product.mil")
    formats.save_mil(p2, images, names)
    lib2 = ref.ReferenceImageLibrary(99)
    lib2.load(p2)
    assert lib2.image_size() == 24
    got = lib2.items()
    assert [n for n, _ in got] == names and all(np.array_equal(a, b) for a, (_, b) in zip(images, got))
    bad = str(tmp_path / "bad.mil")
    open(bad, "wb").write(b"\x00" * 32)
    with pytest.raises(ValueError):
        lib2.load(bad)
    with pytest.raises(ValueError):
        formats.load_mil(bad)
    lib.close()
    lib2.close()


@pytest.mark.parametrize("scheme", [0, 1, 2, 3, 4, 5])
def test_colour_scheme_variants_match_reference_object_code(ref, scheme):
    """ColourScheme.cpp:36-177 compiled unmodified: number of variants, their order and every byte of every variant equal the
    oracle's cv2 restatement (the product's hue_rotate kernel is checked against the same cv2 steps on the GPU)."""
    from mosaicmagnifique_b200 import synthetic
    img = synthetic.make_main_image(70, 93, 40 + scheme, block=16)  # odd width: exercises OpenCV's SIMD row tails
    want = ref.reference_colour_scheme_variants(img, scheme)
    got = ref.colour_scheme_variants(img, scheme)
    assert len(got) == len(want) == {0: 1, 1: 2, 2: 3, 3: 3, 4: 4, 5: 4}[scheme]
    for a, b in zip(got, want):
        assert np.array_equal(np.asarray(a), b)


@pytest.mark.parametrize("detail,steps", [(100, 0), (50, 2), (33, 1), (3, 1)])
def test_product_cell_group_mirror_matches_reference_object_code(ref, detail, steps):
    """mosaicmagnifique_b200.CellGroup.getCell (host arithmetic of libmosaic_b200.so) against the reference's CellGroup.cpp."""
    from mosaicmagnifique_b200 import CellGroup, CellShape
    for sh in _shapes(ref):
        ps = CellShape(sh.mask)
        ps.rowSpacing, ps.colSpacing = sh.row_spacing, sh.col_spacing
        ps.alternateRowSpacing, ps.alternateColSpacing = sh.alt_row_spacing, sh.alt_col_spacing
        ps.alternateRowOffset, ps.alternateColOffset = sh.alt_row_offset, sh.alt_col_offset
        ps.alternateColFlipHorizontal, ps.alternateColFlipVertical = sh.alt_col_flip_h, sh.alt_col_flip_v
        ps.alternateRowFlipHorizontal, ps.alternateRowFlipVertical = sh.alt_row_flip_h, sh.alt_row_flip_v
        cg = CellGroup()
        cg.setCellShape(ps)
        cg.setDetail(detail)
        cg.setSizeSteps(steps)
        group = ref.CellGroup.make(sh, detail, steps)
        for s in range(steps + 1):
            for is_detail in (False, True):
                want, m4 = ref.reference_cell_group_cell(group, s, is_detail)
                got = cg.getCell(s, is_detail)
                assert got.getSize() == want.size == cg.getCellSize(s, is_detail)
                assert np.array_equal(got.getCellMask(), want.mask)
                assert np.array_equal(got.getCellMask(True, False), m4[1]) and np.array_equal(got.getCellMask(False, True), m4[2])
                assert (got.rowSpacing, got.colSpacing, got.alternateRowSpacing, got.alternateColSpacing, got.alternateRowOffset,
                        got.alternateColOffset) == (want.row_spacing, want.col_spacing, want.alt_row_spacing,
                                                    want.alt_col_spacing, want.alt_row_offset, want.alt_col_offset)
                assert (got.alternateColFlipHorizontal, got.alternateColFlipVertical, got.alternateRowFlipHorizontal,
                        got.alternateRowFlipVertical) == (want.alt_col_flip_h, want.alt_col_flip_v, want.alt_row_flip_h,
                                                          want.alt_row_flip_v)
        with pytest.raises(IndexError):
            cg.getCell(steps + 1)


# ---------------------------------------------------------------- the C ABI's own container readers / writers (csrc/containers.cpp)

def _capi_mcs_load(L, path):
    import ctypes
    from mosaicmagnifique_b200._capi import CellShapeC
    c = CellShapeC()
    name = ctypes.create_string_buffer(512)
    rc = L.mosaic_mcs_load(path.encode(), ctypes.byref(c), None, 0, name, 512)
    if rc:
        raise ValueError(L.mosaic_io_last_error().decode())
    mask = np.empty((c.size, c.size), np.uint8)
    assert L.mosaic_mcs_load(path.encode(), ctypes.byref(c), mask.ctypes.data, mask.size, name, 512) == 0
    return c, mask, name.value.decode()


def test_capi_mcs_reader_and_writer_against_reference_object_code(ref, tmp_path):
    """mosaic_mcs_load / mosaic_mcs_save (own QDataStream layout, own PNG codec incl. inflate) on every Cells/*.mcs of the
    reference: equal to the reference's loadFromFile; the library's writer is read back by the reference."""
    import ctypes
    from mosaicmagnifique_b200 import capi
    L = capi()
    for path in sorted(glob.glob(os.path.join(CELLS, "*.mcs"))):
        want, _ = ref.reference_load_mcs(path)
        c, mask, name = _capi_mcs_load(L, path)
        assert name == want.name and np.array_equal(mask, want.mask)
        assert [c.size, c.row_spacing, c.col_spacing, c.alt_row_spacing, c.alt_col_spacing, c.alt_row_offset, c.alt_col_offset,
                c.alt_col_flip_h, c.alt_col_flip_v, c.alt_row_flip_h, c.alt_row_flip_v] == [int(v) for v in want.params()]
        out = str(tmp_path / "capi.mcs")
        assert L.mosaic_mcs_save(out.encode(), ctypes.byref(c), mask.ctypes.data, name.encode()) == 0
        back, _ = ref.reference_load_mcs(out)
        assert _same_shape(back, want) and back.name == want.name
    bad = str(tmp_path / "bad.mcs")
    open(bad, "wb").write(b"\x00" * 40)
    with pytest.raises(ValueError):
        _capi_mcs_load(L, bad)
    assert b".mcs" in L.mosaic_io_last_error()


def test_capi_mil_reader_and_writer_against_reference_object_code(ref, tmp_path):
    """mosaic_mil_info / _load / _save against the reference's own ImageLibrary::saveToFile / loadFromFile (cv2-compressed PNG
    payloads in: dynamic-Huffman inflate; stored-block PNG out: decoded by the real codec on the reference side)."""
    import ctypes
    from mosaicmagnifique_b200 import capi, synthetic
    L = capi()
    lib = ref.ReferenceImageLibrary(40)
    rng = np.random.default_rng(5)
    smooth = synthetic.make_library(5, 40, 77)  # compressible: exercises back-references of the inflate
    for i in range(5):
        lib.add_image(smooth[i], "smooth %d" % i)
    lib.add_image(rng.integers(0, 256, (40, 40, 3), dtype=np.uint8), "noise \u00fc")
    p1 = str(tmp_path / "reference.mil")
    lib.save(p1)
    items = lib.items()
    n, size, nb = ctypes.c_int64(), ctypes.c_int(), ctypes.c_size_t()
    assert L.mosaic_mil_info(p1.encode(), ctypes.byref(n), ctypes.byref(size), ctypes.byref(nb)) == 0
    assert (n.value, size.value) == (6, 40)
    images = np.empty((6, 40, 40, 3), np.uint8)
    names = ctypes.create_string_buffer(nb.value)
    assert L.mosaic_mil_load(p1.encode(), images.ctypes.data, images.size, names, nb.value) == 0
    got_names = names.raw[:nb.value].split(b"\x00")[:-1]
    assert [g.decode() for g in got_names] == [nm for nm, _ in items]
    assert all(np.array_equal(a, b) for a, (_, b) in zip(images, items))
    # library writer -> reference reader
    p2 = str(tmp_path / "capi.mil")
    assert L.mosaic_mil_save(p2.encode(), images.ctypes.data, 6, 40, names.raw[:nb.value]) == 0
    lib2 = ref.ReferenceImageLibrary(1)
    lib2.load(p2)
    got = lib2.items()
    assert lib2.image_size() == 40 and [nm for nm, _ in got] == [nm for nm, _ in items]
    assert all(np.array_equal(a, b) for a, (_, b) in zip(images, got))
    # ... and the Python reader agrees with the C one
    from mosaicmagnifique_b200 import formats
    im2, nm2, sz2 = formats.load_mil(p2)
    assert sz2 == 40 and nm2 == [nm for nm, _ in items] and np.array_equal(im2, images)
    bad = str(tmp_path / "bad.mil")
    open(bad, "wb").write(b"\x01" * 40)
    assert L.mosaic_mil_info(bad.encode(), None, None, None) == -1
    lib.close()
    lib2.close()
