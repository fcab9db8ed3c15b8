"""File formats either side of the path (.mil library, .mcs cell shape): round trips like the reference's
ImageLibrary.SaveAndLoad / CellShape.SaveAndLoad tests (test/tst_ImageLibrary.h, test/tst_CellShape.h), and the
reference's own Cells/*.mcs files (committed under tests/golden/cells)."""
import glob
import os

import numpy as np
import pytest

pytest.importorskip("cv2")

CELLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells")


def test_mil_round_trip(tmp_path):
    from mosaicmagnifique_b200 import formats, synthetic
    lib = synthetic.make_library(9, 24, 3)
    names = ["img %d é" % i for i in range(9)]
    p = str(tmp_path / "lib.mil")
    formats.save_mil(p, lib, names)
    got, got_names, size = formats.load_mil(p)
    assert size == 24 and got_names == names
    assert np.array_equal(got, lib)
    raw = open(p, "rb").read()
    assert raw[:4] == bytes.fromhex("ADBE2480") and raw[4:8] == (6).to_bytes(4, "big")
    with pytest.raises(ValueError):
        open(p, "wb").write(b"\x00" * 16)
        formats.load_mil(p)


def test_mcs_round_trip(tmp_path):
    from mosaicmagnifique_b200 import formats, load_mcs, synthetic
    f = {"name": "Hex", "mask": synthetic.hexagon_mask(64), "row_spacing": 48, "col_spacing": 55, "alt_row_spacing": 48,
         "alt_col_spacing": 55, "alt_row_offset": 27, "alt_col_offset": 0, "alt_col_flip_h": False, "alt_col_flip_v": True,
         "alt_row_flip_h": True, "alt_row_flip_v": False}
    p = str(tmp_path / "hex.mcs")
    formats.save_mcs(p, f)
    g = formats.load_mcs(p)
    for k, v in f.items():
        assert np.array_equal(g[k], v), k
    s = load_mcs(p)
    assert (s.getSize(), s.rowSpacing, s.colSpacing, s.alternateRowOffset) == (64, 48, 55, 27)
    assert s.alternateColFlipVertical and s.alternateRowFlipHorizontal and not s.alternateColFlipHorizontal


def test_reference_cell_fixtures(oracle):
    files = sorted(glob.glob(os.path.join(CELLS, "*.mcs")))
    from mosaicmagnifique_b200 import formats
    assert len(files) == 10
    for p in files:
        f = formats.load_mcs(p)
        o = oracle.load_mcs(p)
        assert f["version"] == 8 and f["mask"].shape == (512, 512)
        assert np.array_equal(np.where(f["mask"] > 127, 255, 0), o.mask)
        assert [f[k] for k in ("row_spacing", "col_spacing", "alt_row_spacing", "alt_col_spacing", "alt_row_offset", "alt_col_offset")] == o.params()[1:7]
    hexa = formats.load_mcs(os.path.join(CELLS, "Hexagon.mcs"))
    assert (hexa["row_spacing"], hexa["col_spacing"], hexa["alt_row_offset"]) == (385, 440, 220)  # SURVEY.md section 8a


def test_container_readers_survive_corrupt_files(tmp_path):
    """csrc/containers.cpp parses files from disk: truncated, bit-flipped and size-lying inputs must come back as an error (or a
    successful parse), never as a crash or an unbounded allocation. Runs in a child process so that a crash is a test failure,
    not the end of the test run."""
    import subprocess
    import sys
    from mosaicmagnifique_b200 import formats, synthetic
    good = str(tmp_path / "good.mcs")
    formats.save_mcs(good, {"name": "t", "mask": synthetic.hexagon_mask(64), "row_spacing": 48, "col_spacing": 55, "alt_row_spacing": 48,
                            "alt_col_spacing": 55, "alt_row_offset": 27, "alt_col_offset": 0, "alt_col_flip_h": False,
                            "alt_col_flip_v": False, "alt_row_flip_h": True, "alt_row_flip_v": False})
    mil = str(tmp_path / "good.mil")
    formats.save_mil(mil, synthetic.make_library(3, 24, 5), ["a", "b", "c"])
    script = r'''
import ctypes, sys
import numpy as np
from mosaicmagnifique_b200 import capi
from mosaicmagnifique_b200._capi import CellShapeC
L = capi()
rng = np.random.default_rng(123)
outcomes = {0: 0, -1: 0}
for path, is_mcs in ((sys.argv[1], True), (sys.argv[2], False)):
    data = bytearray(open(path, "rb").read())
    variants = [bytes(data[:n]) for n in range(0, len(data), max(1, len(data) // 60))]
    for _ in range(300):
        d = bytearray(data)
        for _ in range(int(rng.integers(1, 6))):
            d[int(rng.integers(0, len(d)))] = int(rng.integers(0, 256))
        variants.append(bytes(d))
    lying = bytearray(data)            # IHDR claiming a gigantic image
    i = bytes(lying).find(b"IHDR")
    lying[i + 4:i + 12] = b"\xff\xff\xff\xff\xff\xff\xff\xff"
    variants.append(bytes(lying))
    for v in variants:
        p = sys.argv[3]
        open(p, "wb").write(v)
        if is_mcs:
            c = CellShapeC()
            mask = np.zeros(1 << 16, np.uint8)
            rc = L.mosaic_mcs_load(p.encode(), ctypes.byref(c), mask.ctypes.data, mask.size, None, 0)
        else:
            rc = L.mosaic_mil_info(p.encode(), None, None, None)
        assert rc in (0, -1), rc
        outcomes[rc] += 1
print(outcomes[0], outcomes[-1])
'''
    out = subprocess.run([sys.executable, "-c", script, good, mil, str(tmp_path / "variant.bin")], capture_output=True, text=True,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert out.returncode == 0, out.stdout + out.stderr
    ok, rejected = (int(v) for v in out.stdout.split())
    assert rejected > 300  # nearly every corruption is caught (CRC / Adler / structure); the rest parse as valid files


def test_png_writer_compresses_and_round_trips(tmp_path):
    """The library's own PNG writer (csrc/containers.cpp: row filters + fixed-Huffman deflate with LZ77; round 1 wrote stored blocks):
    what it writes is read back identically by the library's reader AND by OpenCV, a 512 px cell mask lands in the few-KB range of
    the reference's own .mcs files, and library images come out smaller than their raw pixels."""
    import ctypes

    import cv2
    from mosaicmagnifique_b200 import capi, formats, load_mcs, synthetic
    from mosaicmagnifique_b200._capi import CellShapeC
    L = capi()
    # masks: every shipped shape, re-saved by the library
    cells = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells")
    for name in ("Puzzle", "Hexagon", "YinAndYang"):
        src = load_mcs(os.path.join(cells, name + ".mcs"))
        out = str(tmp_path / (name + ".mcs"))
        c = src._c()
        m = src.getCellMask()
        assert L.mosaic_mcs_save(out.encode(), ctypes.byref(c), m.ctypes.data, name.encode()) == 0
        assert os.path.getsize(out) < 12000, os.path.getsize(out)          # stored blocks would be 262 KB
        back = load_mcs(out)
        assert np.array_equal(back.getCellMask(), m) and back.name == name
        assert np.array_equal(formats.load_mcs(out)["mask"], m)              # cv2's decoder agrees
    # photographs: a small .mil, noisy and smooth images, odd size (row filters at the borders)
    rng = np.random.default_rng(3)
    lib = synthetic.make_library(6, 37, 9)
    lib[1] = rng.integers(0, 256, lib[1].shape, dtype=np.uint8)                # incompressible noise still round-trips
    lib[2] = 200
    out = str(tmp_path / "lib.mil")
    names = b"".join(("img%d" % i).encode() + b"\0" for i in range(len(lib)))
    assert L.mosaic_mil_save(out.encode(), lib.ctypes.data, len(lib), 37, names) == 0
    got, got_names, size = formats.load_mil(out)
    assert size == 37 and got_names == ["img%d" % i for i in range(len(lib))] and np.array_equal(got, lib)
    smooth = synthetic.make_library(8, 128, 10)
    out2 = str(tmp_path / "lib128.mil")
    names = b"".join(("s%d" % i).encode() + b"\0" for i in range(len(smooth)))
    assert L.mosaic_mil_save(out2.encode(), smooth.ctypes.data, len(smooth), 128, names) == 0
    assert os.path.getsize(out2) < 0.9 * smooth.size
