"""Scaled compositing (mosaic_set_render_library + mosaic_build_photomosaic_scaled, include/mosaic_b200.h "scaled compositing").

The scaled build at k = R / S must be byte for byte the reference's buildPhotomosaic procedure (oracle.build_photomosaic) on a
k-times larger main image with the render library and the k-scaled cell group (tests/helpers/render_scale.py); at k = 1 with the
matching library it is the plain build. A render library that is the matching library upsampled by nearest neighbour gives the
plain build upsampled (no size steps: halving does not commute with upsampling), which is checked at configs 4 and 5 full size.
"""
import os

import numpy as np
import pytest

from tests.helpers.render_scale import scaled_group
from tests.test_gpu_tile_flips import TRIANGLE, explicit_library, oracle_shape, product_shape, slot_grids

pytestmark = pytest.mark.gpu
HEXAGON = "Hexagon"
BG = (17, 200, 90, 255)


def generate(main, lib, shape, diff=0, detail=100, steps=0, flips=0, rr=1, ra=300):
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
    gen.computeGridState()
    if flips:
        gen.setTileFlips(bool(flips & 1), bool(flips & 2))
    gen.setRepeat(rr, ra)
    assert gen.generateBestFits()
    return gen


def oracle_slots(gen, flips, n):
    grids = gen.getBestFits()
    return slot_grids(grids, gen.getBestFitFlips(), flips, n) if flips else grids


# ----------------------------------------------------------------------------- k = 1


@pytest.mark.parametrize("name", ["square", HEXAGON, TRIANGLE])
@pytest.mark.parametrize("steps", [0, 2])
@pytest.mark.parametrize("detail", [100, 50])
@pytest.mark.parametrize("flips", [0, 3])
def test_scale1_equals_plain_build(name, steps, detail, flips):
    from mosaicmagnifique_b200 import synthetic
    S = 64
    main = synthetic.make_main_image(300, 430, 1100 + steps, block=32)
    lib = synthetic.make_library(11, S, 1101)
    gen = generate(main, lib, product_shape(name, S), 2, detail, steps, flips)
    plain = gen.buildPhotomosaic(BG)
    gen.setRenderLibrary(lib)
    got = gen.buildPhotomosaicScaled(BG)
    gen.close()
    assert got.shape == plain.shape and np.array_equal(got, plain)


def test_scale1_other_render_library(oracle):
    from mosaicmagnifique_b200 import synthetic
    S = 64
    main = synthetic.make_main_image(300, 430, 1110, block=32)
    lib = synthetic.make_library(13, S, 1111)
    render = synthetic.make_library(13, S, 1112)
    gen = generate(main, lib, product_shape(HEXAGON, S), 0, 100, 2)
    gen.setRenderLibrary(render)
    got = gen.buildPhotomosaicScaled(BG)
    grids = gen.getBestFits()
    gen.close()
    og = oracle.CellGroup.make(oracle_shape(oracle, HEXAGON, S), 100, 2)
    assert np.array_equal(got, oracle.build_photomosaic(main.shape, render, og, grids, BG))


# ----------------------------------------------------------------------------- k > 1 against the reference procedure


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("name,steps,flips", [("square", 1, 0), (HEXAGON, 2, 1), (TRIANGLE, 1, 3), (TRIANGLE, 2, 0)])
def test_scaled_equals_reference_procedure(oracle, k, name, steps, flips):
    from mosaicmagnifique_b200 import synthetic
    S = 32
    main = synthetic.make_main_image(250, 370, 1120 + k, block=16)  # not a multiple of any spacing: clipped edge cells
    lib = synthetic.make_library(9, S, 1121)
    render = synthetic.make_library(9, k * S, 1122 + k)
    gen = generate(main, lib, product_shape(name, S), 1, 100, steps, flips)
    gen.setRenderLibrary(render)  # the N images, unoriented: the build mirrors them by the slots' orientations
    got = gen.buildPhotomosaicScaled(BG)
    slots = oracle_slots(gen, flips, len(lib))
    gen.close()
    assert got.shape == (k * main.shape[0], k * main.shape[1], 4)
    og = oracle.CellGroup.make(oracle_shape(oracle, name, S), 100, steps)
    want = oracle.build_photomosaic((k * main.shape[0], k * main.shape[1]), explicit_library(render, flips), scaled_group(oracle, og, k),
                                    slots, BG)
    assert np.array_equal(got, want)


def test_config3_as_specified_k2(oracle):
    import bench
    from mosaicmagnifique_b200 import synthetic
    cfg = bench.WORKLOADS["cfg3"]
    main, lib = bench.make_inputs(cfg)
    k = 2
    render = synthetic.make_library(len(lib), k * cfg["cell"], 1130)
    gen = generate(main, lib, bench.make_shape(cfg), cfg["diff"], cfg["detail"], cfg["steps"], 0, cfg["rr"], cfg["ra"])
    gen.setRenderLibrary(render)
    got = gen.buildPhotomosaicScaled(BG)
    grids = gen.getBestFits()
    gen.close()
    assert len(grids) == 3 and (grids[0] >= 0).any() and any((g >= 0).any() for g in grids[1:])  # cells after a size step
    og = oracle.CellGroup.make(oracle.CellShape.square(cfg["cell"]), 100, cfg["steps"])
    want = oracle.build_photomosaic((k * main.shape[0], k * main.shape[1]), render, scaled_group(oracle, og, k), grids, BG)
    assert np.array_equal(got, want)


# ----------------------------------------------------------------------------- full size, device output


def upsampled_on_gpu(t, k):
    return t.repeat_interleave(k, 0).repeat_interleave(k, 1)


@pytest.mark.parametrize("cfg_name", ["cfg4", "cfg5"])
def test_full_size_device_output_k4(cfg_name):
    import bench
    import torch
    k = 4
    cfg = bench.WORKLOADS[cfg_name]
    assert cfg.get("steps", 0) == 0
    main, lib = bench.make_inputs(cfg)
    H, W = main.shape[:2]
    gen = generate(main, lib, bench.make_shape(cfg), cfg["diff"], cfg["detail"], 0, 0, cfg["rr"], cfg["ra"])
    plain = torch.from_numpy(gen.buildPhotomosaic(BG)).cuda()
    dev = torch.device("cuda", 0)
    lib_t = torch.from_numpy(lib).to(dev)
    render = lib_t.repeat_interleave(k, 1).repeat_interleave(k, 2).contiguous()  # N x kS x kS x 3, nearest neighbour
    del lib_t
    torch.cuda.synchronize()  # the handle copies on its own stream, which does not wait for torch's
    gen.setRenderLibraryPtr(render.data_ptr(), len(lib), k * cfg["cell"])
    del render
    torch.cuda.empty_cache()
    out = torch.empty((k * H, k * W, 4), dtype=torch.uint8, device=dev)
    assert out.numel() == k * k * H * W * 4
    gen.buildPhotomosaicScaled(BG, out=out)
    gen.close()
    torch.cuda.synchronize()
    band = 256
    for r0 in range(0, H, band):
        r1 = min(H, r0 + band)
        assert torch.equal(out[k * r0:k * r1], upsampled_on_gpu(plain[r0:r1], k)), "rows %d..%d" % (r0, r1)
    print("%s k=%d: %d x %d output, %.2f GB" % (cfg_name, k, k * H, k * W, out.numel() / 1e9))


# ----------------------------------------------------------------------------- host output through bands


@pytest.mark.parametrize("pinned", [False, True])
def test_host_bands_equal_device_output(monkeypatch, pinned):
    import torch
    from mosaicmagnifique_b200 import synthetic
    S, k, pad = 32, 3, 5
    main = synthetic.make_main_image(300, 410, 1140, block=16)
    lib = synthetic.make_library(12, S, 1141)
    render = synthetic.make_library(12, k * S, 1142)
    gen = generate(main, lib, product_shape(TRIANGLE, S), 2, 100, 1, 3)
    gen.setRenderLibrary(render)
    rows, cols = k * main.shape[0], k * main.shape[1]
    dev_out = torch.empty((rows, cols, 4), dtype=torch.uint8, device="cuda")
    gen.buildPhotomosaicScaled(BG, out=dev_out)
    want = dev_out.cpu().numpy()
    band_rows = 64  # 15 bands, the last of 4 rows
    assert rows // band_rows >= 5 and rows % band_rows
    monkeypatch.setenv("MM_BUILD_BAND_ROWS", str(band_rows))
    if pinned:
        buf = torch.full((rows, cols + pad, 4), 0xA5, dtype=torch.uint8, pin_memory=True)
        gen.buildPhotomosaicScaled(BG, out=buf[:, :cols])
        buf = buf.numpy()
    else:
        buf = np.full((rows, cols + pad, 4), 0xA5, np.uint8)
        gen.buildPhotomosaicScaled(BG, out=buf[:, :cols])
    gen.close()
    assert np.array_equal(buf[:, :cols], want)
    assert (buf[:, cols:] == 0xA5).all()


@pytest.mark.parametrize("scaled", [False, True])
def test_unaligned_device_output(scaled):
    """A device output at an odd address goes through the band path (no 4-byte stores at an unaligned address): both entry points
    give the bytes of an aligned host build, and the bytes before the image and past each row are left untouched."""
    import torch
    from mosaicmagnifique_b200 import synthetic
    S, k, pad = 32, 2 if scaled else 1, 8
    main = synthetic.make_main_image(150, 210, 1145, block=16)
    lib = synthetic.make_library(10, S, 1146)
    gen = generate(main, lib, product_shape(HEXAGON, S), 0, 100, 1, 1)
    render = synthetic.make_library(10, k * S, 1147)
    gen.setRenderLibrary(render)
    want = gen.buildPhotomosaicScaled(BG) if scaled else gen.buildPhotomosaic(BG)
    rows, cols = want.shape[:2]
    stride = cols * 4 + pad
    buf = torch.full((1 + rows * stride,), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()  # the fill runs on torch's stream, the build on the handle's
    fn = gen._L.mosaic_build_photomosaic_scaled if scaled else gen._L.mosaic_build_photomosaic
    bg = np.asarray(BG, np.uint8)
    assert fn(gen._h, bg.ctypes.data, buf.data_ptr() + 1, rows, cols, stride) == 0, gen._L.mosaic_last_error(gen._h)
    gen.close()
    got = buf.cpu().numpy()
    assert got[0] == 0xA5
    img = got[1:].reshape(rows, stride)
    assert np.array_equal(img[:, :cols * 4].reshape(rows, cols, 4), want)
    assert (img[:, cols * 4:] == 0xA5).all()


# ----------------------------------------------------------------------------- sharded handles


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_ranks_build(world):
    import torch
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator, load_mcs, synthetic
    from mosaicmagnifique_b200.parallel import device_view
    cell, detail, k = 32, 50, 2
    main = synthetic.make_main_image(300, 410, 1150 + world, block=32)
    lib = synthetic.make_library(61, cell, 1151)
    render = synthetic.make_library(61, k * cell, 1152)
    sh = load_mcs(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells", HEXAGON + ".mcs")).resized(cell)

    def configure(g):
        g.setColourDifference(2)
        cg = CellGroup()
        cg.setCellShape(sh)
        cg.setDetail(detail)
        g.setCellGroup(cg)
        g.setRepeat(2, 400)

    ref = PhotomosaicGenerator(0)
    configure(ref)
    ref.setMainImage(main)
    ref.setLibrary(lib)
    state = ref.computeGridState()
    assert ref.generateBestFits()
    ref.setRenderLibrary(render)
    want = ref.buildPhotomosaicScaled(BG)
    ref.close()

    dev = torch.device("cuda", 0)
    n, per_lib = len(lib), -(-len(lib) // world)
    gens = []
    for r in range(world):
        g = PhotomosaicGenerator(0)
        configure(g)
        g.setGridState(state)
        g.setShard(r, world)
        g.setMainImage(main)
        a, b = min(n, r * per_lib), min(n, (r + 1) * per_lib)
        sl = np.ascontiguousarray(lib[a:b])
        g.setLibraryShardPtr(sl.ctypes.data if b > a else 0, a, b - a, n, cell, world * per_lib)
        gens.append(g)
    infos = [g.libraryDevice() for g in gens]
    assert infos[0]["stored_size"] == cell * detail // 100
    stored_row = infos[0]["stored_size"] ** 2 * 3
    views = [device_view(i["ptr"], (world * per_lib, stored_row), torch.uint8, dev) for i in infos]
    for r in range(world):
        for q in range(world):
            if q != r:
                views[q][r * per_lib:(r + 1) * per_lib].copy_(views[r][r * per_lib:(r + 1) * per_lib])
    torch.cuda.synchronize()
    for g in gens:
        g.generateCandidates()
    blks = [g.candidateBlock(0) for g in gens]
    gathered = torch.cat([device_view(b["ptr"], (b["bytes"] // 4,), torch.int32, dev).clone() for b in blks]).contiguous()
    torch.cuda.synchronize()
    for g in gens:
        g.selectFromGathered(0, gathered.data_ptr(), blks[0]["k"], blks[0]["rows_per_rank"])
        L, h = g._L, g._h
        out = np.empty(main.shape[:2] + (4,), np.uint8)
        bg = np.asarray(BG, np.uint8)
        assert L.mosaic_build_photomosaic(h, bg.ctypes.data, out.ctypes.data, out.shape[0], out.shape[1], out.strides[0]) == -4
        g.setRenderLibrary(render)
        assert np.array_equal(g.buildPhotomosaicScaled(BG), want)
        g.close()


# ----------------------------------------------------------------------------- invalid input


def test_invalid_input():
    from mosaicmagnifique_b200 import CellShape, MosaicError, PhotomosaicGenerator, synthetic
    S, k = 32, 2
    main = synthetic.make_main_image(200, 260, 1160, block=32)
    lib = synthetic.make_library(7, S, 1161)
    render = synthetic.make_library(7, k * S, 1162)
    bg = np.asarray(BG, np.uint8)
    H, W = main.shape[:2]

    fresh = PhotomosaicGenerator(0)
    L, h = fresh._L, fresh._h
    out = np.empty((k * H, k * W, 4), np.uint8)
    assert L.mosaic_set_render_library(h, render.ctypes.data, -1, k * S) == -1
    assert L.mosaic_set_render_library(h, render.ctypes.data, len(render), 0) == -1
    assert L.mosaic_set_render_library(h, None, len(render), k * S) == -1
    assert L.mosaic_set_render_library(h, render.ctypes.data, len(render), k * S) == 0  # no cell group yet: nothing checked here
    assert L.mosaic_build_photomosaic_scaled(h, bg.ctypes.data, out.ctypes.data, k * H, k * W, k * W * 4) == -4  # no best fits
    fresh.close()

    gen = generate(main, lib, CellShape(S), 0, 100, 0, 0)
    L, h = gen._L, gen._h
    plain = gen.buildPhotomosaic(BG)
    with pytest.raises(MosaicError) as e:
        gen.buildPhotomosaicScaled(BG)
    assert e.value.code == -4  # no render library

    def scaled(rows=k * H, cols=k * W, stride=None):
        return L.mosaic_build_photomosaic_scaled(h, bg.ctypes.data, out.ctypes.data, rows, cols, k * W * 4 if stride is None else stride)

    def err():
        return L.mosaic_last_error(h).decode()

    gen.setRenderLibrary(render[:6])
    assert scaled() == -1 and "6" in err() and "7" in err()
    big = np.zeros((7, 70, 70, 3), np.uint8)
    gen.setRenderLibrary(big)
    assert scaled() == -1 and "70" in err() and "32" in err()
    gen.setRenderLibrary(render)
    assert np.array_equal(gen.buildPhotomosaic(BG), plain)  # the render library changes nothing in the plain build
    assert scaled(rows=k * H + 1) == -1 and str(k * H) in err()
    assert scaled(cols=k * W - 1) == -1 and str(k * W) in err()
    assert scaled(stride=k * W * 4 - 4) == -1
    assert scaled(stride=k * W * 4 + 2) == -1
    assert scaled() == 0
    assert L.mosaic_build_photomosaic_scaled(h, None, out.ctypes.data, k * H, k * W, k * W * 4) == -1
    assert L.mosaic_build_photomosaic_scaled(h, bg.ctypes.data, None, k * H, k * W, k * W * 4) == -1
    gen.setRenderLibrary(None)
    assert scaled() == -4
    assert np.array_equal(gen.buildPhotomosaic(BG), plain)
    gen.close()


def test_scale_overflowing_int():
    """k * W above INT_MAX is refused: a 2 x 300,000 main image with 2-pixel cells and a one-image render library at side 2 * 7,159
    (k * W = 2,147,700,000)"""
    import torch
    from mosaicmagnifique_b200 import CellGroup, CellShape, PhotomosaicGenerator
    W, S, k = 300_000, 2, 7159
    assert k * W > 2**31 - 1 > (k - 1) * W
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(np.zeros((S, W, 3), np.uint8))
    gen.setLibrary(np.zeros((1, S, S, 3), np.uint8))
    cg = CellGroup()
    cg.setCellShape(CellShape(S))
    gen.setCellGroup(cg)
    gen.computeGridState()
    assert gen.generateBestFits()
    render = torch.zeros((1, k * S, k * S, 3), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    gen.setRenderLibraryPtr(render.data_ptr(), 1, k * S)
    L, h = gen._L, gen._h
    bg, out = np.zeros(4, np.uint8), np.zeros(16, np.uint8)
    assert L.mosaic_build_photomosaic_scaled(h, bg.ctypes.data, out.ctypes.data, 4, 4, 16) == -1
    assert str(k * W) in L.mosaic_last_error(h).decode()
    gen.close()
