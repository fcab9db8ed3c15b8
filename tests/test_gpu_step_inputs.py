"""The packed inputs of the difference kernels, bit for bit against the OpenCV preprocessing of the oracle.

mosaic_debug_step_inputs returns what a generate packs for one size step -- library tiles, cell tiles with weights, the active-pixel
list and the library's colour order -- without running a difference kernel. Every path that builds them is compared here with
oracle.preprocess_library / halve_library / extract_cells (cv2 for every OpenCV call) as uint32 bit patterns:

  fused     one size step: the 8U library packers (pack_library_ciede_kernel<true>, pack_library_euclid_u8_kernel) reduce the
            library k-fold on the fly (area_pixel_u8) and convert it; k = S / ds in {1, 2, 3, 4, 5, 8}, every colour difference,
            CIEDE2000 with and without the colour order, slot counts around the 8- and 64-image library tiles, tile flips 0 / 1 / 3.
  unfused   size steps: area_u8 / area_general_u8 -> to_working_space -> pack_library, the f32 library halved by area_f32 before
            every later step; every step is checked.
  sweep     every integer detail percent at cell sizes 64 and 120 (fractional INTER_AREA tables of library and cells).
  cells     extract_cells_kernel: cells clipped on all four borders (zero fill inside the area average), an offset hexagon and the
            flipped IsocelesTriangle-45deg masks, a triadic scheme with and without the shared-buffer quirk, n_active around the
            16- and 128-pixel chunks.
Stored values: CIEDE2000 (L/2 - 25, a/50, b/50, C/50) with C = sqrt in f64, weight 50; Euclidean (x0, x1, x2), library negated,
weight 1. Padding slots, pixels and rows must be zero (either sign: the fused Euclidean packer writes -0.0, the memset +0.0).
The CPU tests check that the case tables still cross what they name and round-trip the decoder on tiles packed in numpy."""
import ctypes
import os
import re
import zlib
from collections import namedtuple

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS_H = os.path.join(os.path.dirname(HERE), "mosaicmagnifique_b200", "csrc", "kernels.h")
RGB, CIE76, CIEDE = 0, 1, 2
LAYOUT_CIEDE, LAYOUT_EUCLID = 0, 1


def _kernel_constants():
    text = open(KERNELS_H).read()
    return {n: int(re.search(r"#define %s (\d+)" % n, text).group(1)) for n in ("MM_TCB", "MM_TNB", "MM_KP", "MM_ETC", "MM_ETN", "MM_EKP")}


K = _kernel_constants()
# (cells per tile, library slots per tile, pixels per chunk) of each layout
TILES = {LAYOUT_CIEDE: (K["MM_TCB"], K["MM_TNB"], K["MM_KP"]), LAYOUT_EUCLID: (K["MM_ETC"], K["MM_ETN"], K["MM_EKP"])}


def _layout(diff):
    return LAYOUT_CIEDE if diff == CIEDE else LAYOUT_EUCLID


# ----------------------------------------------------------------------------- cases

Case = namedtuple("Case", "name diff S detail N steps flips repeats shape scheme quirk mask_k")


def _case(name, diff, S, detail, N, steps=0, flips=0, repeats=False, shape="square", scheme=0, quirk=True, mask_k=0):
    return Case(name, diff, S, detail, N, steps, flips, repeats, shape, scheme, quirk, mask_k)


# fused 8U packers: (cell size, detail percent) with S / ds = k
FUSED_K = {1: (16, 100), 2: (16, 50), 3: (30, 34), 4: (32, 25), 5: (40, 20), 8: (64, 13)}
FUSED = [
    _case("fused-rgb-k1", RGB, *FUSED_K[1], N=65),
    _case("fused-cie76-k2", CIE76, *FUSED_K[2], N=63),
    _case("fused-rgb-k3", RGB, *FUSED_K[3], N=130),
    _case("fused-cie76-k4-hv", CIE76, *FUSED_K[4], N=9, flips=3),
    _case("fused-rgb-k5-h", RGB, *FUSED_K[5], N=7, flips=1),
    _case("fused-cie76-k8", CIE76, *FUSED_K[8], N=1),
    _case("fused-ciede-k1-order", CIEDE, *FUSED_K[1], N=1, repeats=True),
    _case("fused-ciede-k2", CIEDE, *FUSED_K[2], N=8),
    _case("fused-ciede-k3-order-h", CIEDE, *FUSED_K[3], N=7, flips=1, repeats=True),
    _case("fused-ciede-k4", CIEDE, *FUSED_K[4], N=65),
    _case("fused-ciede-k5-order", CIEDE, *FUSED_K[5], N=63, repeats=True),
    _case("fused-ciede-k8-hv", CIEDE, *FUSED_K[8], N=9, flips=3),
]
# f32 library halved per size step: integer and fractional detail
UNFUSED = [
    _case("steps2-rgb-k2", RGB, 32, 50, N=9, steps=2),
    _case("steps1-cie76-k1-h", CIE76, 32, 100, N=65, steps=1, flips=1),
    _case("steps2-ciede-k4-order", CIEDE, 48, 25, N=63, steps=2, repeats=True),
    _case("steps2-rgb-frac", RGB, 48, 75, N=7, steps=2),
    _case("steps1-cie76-frac", CIE76, 40, 60, N=130, steps=1),
    _case("steps1-ciede-frac-hv", CIEDE, 48, 75, N=9, steps=1, flips=3),
]
# cell extraction: borders, shapes, colour-scheme variants, chunk edges of the active-pixel axis
CELLS = [
    _case("hexagon-ciede-order", CIEDE, 32, 100, N=9, shape="Hexagon", repeats=True),
    _case("hexagon-rgb-frac", RGB, 32, 70, N=8, shape="Hexagon"),
    _case("triangle45-cie76-k2", CIE76, 32, 50, N=8, shape="IsocelesTriangle-45deg"),
    _case("triangle45-ciede", CIEDE, 32, 100, N=7, shape="IsocelesTriangle-45deg"),
    _case("triangle45-4masks-ciede", CIEDE, 32, 100, N=9, shape="IsocelesTriangle-45deg:one-flag-off"),
    _case("triangle45-4masks-rgb-frac", RGB, 32, 70, N=8, shape="IsocelesTriangle-45deg:one-flag-off"),
    _case("triadic-quirk-rgb-d100", RGB, 24, 100, N=9, scheme=2, quirk=True),
    _case("triadic-ciede-d100", CIEDE, 24, 100, N=9, scheme=2, quirk=False),
    _case("triadic-quirk-ciede-d50", CIEDE, 24, 50, N=9, scheme=2, quirk=True),
    _case("triadic-rgb-d50", RGB, 24, 50, N=9, scheme=2, quirk=False),
] + [_case("active%d-%s" % (k, "ciede" if k > 100 else "rgb"), CIEDE if k > 100 else RGB, 24, 100, N=9, shape="mask", mask_k=k)
     for k in (15, 16, 17, 127, 128, 129)]
CASES = FUSED + UNFUSED + CELLS
SWEEP_SIZES = (64, 120)
SWEEP_N = 9


def _main_size(S):
    """a main image that no cell size divides: border cells are clipped on the right and at the bottom (and, for offset shapes, on
    the left and at the top)"""
    return 3 * S + S // 2 + 3, 4 * S + S // 3 + 5


def _seed(name):
    return zlib.crc32(name.encode()) % 100000


def _o_shape(oracle, case):
    """the case's oracle cell shape at its cell size"""
    if case.shape == "square":
        return oracle.CellShape.square(case.S)
    if case.shape == "mask":
        rng = np.random.default_rng(7000 + case.mask_k)
        m = np.zeros(case.S * case.S, np.uint8)
        m[rng.choice(m.size, case.mask_k, replace=False)] = 255
        return oracle.CellShape.from_mask(m.reshape(case.S, case.S))
    from tests.test_gpu_baseline_configs import load_shape
    name, _, variant = case.shape.partition(":")
    o = load_shape(oracle, name)[0].resized(case.S)
    if variant == "one-flag-off":  # the shipped flags give flips {0, 3}; without one of them all four masks occur
        o.alt_row_flip_h = False
    return o


def _states(oracle, og, H, W, seed):
    """grid state per size step: every cell that meets the image at step 0 (so that all clipped border cells are there), a seeded
    two thirds of them at later steps"""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(og.size_steps + 1):
        one = oracle.CellGroup(cells=[og.cells[s]], detail_cells=[og.detail_cells[s]], detail=og.detail, size_steps=0)
        st = oracle.grid_state(one, None, H, W)[0]
        if s > 0:
            drop = (st >= 0) & (rng.random(st.shape) < 1 / 3)
            if drop.sum() < (st >= 0).sum():
                st[drop] = -1
        out.append(st)
    return out


def _valid(state):
    return [(y, x) for y, x in zip(*np.nonzero(state >= 0))]


def _active_pixels(oracle, normal, detail_shape, state):
    """the kernels' pixel axis: union of the flipped detail masks that occur among the step's valid cells, raster order"""
    used = sorted({oracle.flip_at(normal, x - 2, y - 2) for y, x in _valid(state)})
    m4 = detail_shape.masks4()
    return np.flatnonzero(np.any([m4[f] > 0 for f in used], axis=0)) if used else np.zeros(0, np.int64)


def _orientations(flips):
    return [c for c in range(4) if (c & ~flips) == 0]


def _oriented_library(lib, flips):
    """slot j * N + i = image i under the j-th enabled orientation (1: columns mirrored, 2: rows mirrored)"""
    import cv2
    code = {0: None, 1: 1, 2: 0, 3: -1}
    return np.concatenate([lib if c == 0 else np.stack([cv2.flip(im, code[c]) for im in lib]) for c in _orientations(flips)])


def _library_order(lib8, n_pad):
    """the documented colour order: key = Morton code (B in bit 0, G, R) of the 10-bit min(1023, sum * 1024 / (S^2 * 256)) per
    channel, stable sort; padding slots map to themselves"""
    n, S = lib8.shape[0], lib8.shape[1]
    sums = lib8.reshape(n, -1, 3).astype(np.int64).sum(axis=1)
    q = np.minimum(1023, sums * 1024 // (S * S * 256))
    key = np.zeros(n, np.int64)
    for b in range(10):
        for c in range(3):
            key |= ((q[:, c] >> b) & 1) << (3 * b + c)
    return np.concatenate([np.argsort(key, kind="stable"), np.arange(n, n_pad)]).astype(np.int32)


def _stored(x, layout):
    """working-space pixels [..., 3] f32 -> the channels the tiles hold"""
    if layout == LAYOUT_EUCLID:
        return x
    L, a, b = x[..., 0], x[..., 1], x[..., 2]
    C = np.sqrt(a.astype(np.float64) ** 2 + b.astype(np.float64) ** 2).astype(np.float32)
    s = np.float32(0.02)
    return np.stack([np.float32(0.5) * L - np.float32(25.0), s * a, s * b, s * C], axis=-1)


# ----------------------------------------------------------------------------- tile layouts

Geom = namedtuple("Geom", "layout n_chunks n_cell_tiles n_lib_tiles tcb tnb kp")


def _decode_lib(raw, g):
    """library tiles -> [slot][compacted pixel][channel] as stored (Euclidean: negated)"""
    f = np.frombuffer(raw, np.float32)
    if g.layout == LAYOUT_CIEDE:
        # [tile][chunk][pair][2][KP] float4: (L0, L1, a0, a1), (b0, b1, C0, C1) -> channel 2 * float4 + half, image j of the pair
        a = f.reshape(g.n_lib_tiles, g.n_chunks, g.tnb // 2, 2, g.kp, 2, 2)
        return a.transpose(0, 2, 6, 1, 4, 3, 5).reshape(g.n_lib_tiles * g.tnb, g.n_chunks * g.kp, 4)
    a = f.reshape(g.n_lib_tiles, g.n_chunks, g.kp, 3, g.tnb)  # pixel-major [tile][chunk][pixel][x0, x1, x2][images]
    return a.transpose(0, 4, 1, 2, 3).reshape(g.n_lib_tiles * g.tnb, g.n_chunks * g.kp, 3)


def _decode_cells(raw, g):
    """cell tiles -> ([row][compacted pixel][channel], weights [row][compacted pixel])"""
    f = np.frombuffer(raw, np.float32)
    R, Q = g.n_cell_tiles * g.tcb, g.n_chunks * g.kp
    if g.layout == LAYOUT_CIEDE:
        # per (tile, chunk): float4 [TCB][KP], then float w [TCB][KP]
        a = f.reshape(g.n_cell_tiles, g.n_chunks, g.tcb * g.kp * 5)
        v = a[..., :g.tcb * g.kp * 4].reshape(g.n_cell_tiles, g.n_chunks, g.tcb, g.kp, 4)
        w = a[..., g.tcb * g.kp * 4:].reshape(g.n_cell_tiles, g.n_chunks, g.tcb, g.kp)
        return v.transpose(0, 2, 1, 3, 4).reshape(R, Q, 4), w.transpose(0, 2, 1, 3).reshape(R, Q)
    a = f.reshape(g.n_cell_tiles, g.n_chunks, g.kp, 4, g.tcb).transpose(0, 4, 1, 2, 3).reshape(R, Q, 4)  # [pixel][x0, x1, x2, w][cells]
    return a[..., :3], a[..., 3]


def _pack_lib_numpy(vals, g):
    """the layout comments of pack_library_ciede_kernel / pack_library_euclid_kernel, element by element"""
    out = np.zeros(g.n_lib_tiles * g.n_chunks * g.tnb * g.kp * (4 if g.layout == LAYOUT_CIEDE else 3), np.float32)
    for t in range(vals.shape[0]):
        tile, ti = divmod(t, g.tnb)
        for q in range(vals.shape[1]):
            chunk, pi = divmod(q, g.kp)
            if g.layout == LAYOUT_CIEDE:
                tp, j = divmod(ti, 2)
                blk = ((tile * g.n_chunks + chunk) * g.tnb * g.kp) * 4
                L, a, b, C = vals[t, q]
                out[blk + ((tp * 2 + 0) * g.kp + pi) * 4 + j] = L
                out[blk + ((tp * 2 + 0) * g.kp + pi) * 4 + 2 + j] = a
                out[blk + ((tp * 2 + 1) * g.kp + pi) * 4 + j] = b
                out[blk + ((tp * 2 + 1) * g.kp + pi) * 4 + 2 + j] = C
            else:
                blk = (tile * g.n_chunks + chunk) * g.kp * 3 * g.tnb
                for c in range(3):
                    out[blk + (pi * 3 + c) * g.tnb + ti] = vals[t, q, c]
    return out.tobytes()


def _pack_cells_numpy(vals, w, g):
    """the layout comments of extract_cells_kernel, element by element"""
    out = np.zeros(g.n_cell_tiles * g.n_chunks * g.tcb * g.kp * (5 if g.layout == LAYOUT_CIEDE else 4), np.float32)
    for r in range(vals.shape[0]):
        tile, ti = divmod(r, g.tcb)
        for q in range(vals.shape[1]):
            chunk, pi = divmod(q, g.kp)
            if g.layout == LAYOUT_CIEDE:
                blk = (tile * g.n_chunks + chunk) * g.tcb * g.kp * 5
                out[blk + (ti * g.kp + pi) * 4: blk + (ti * g.kp + pi) * 4 + 4] = vals[r, q]
                out[blk + g.tcb * g.kp * 4 + ti * g.kp + pi] = w[r, q]
            else:
                blk = (tile * g.n_chunks + chunk) * g.kp * 4 * g.tcb
                for c in range(3):
                    out[blk + (pi * 4 + c) * g.tcb + ti] = vals[r, q, c]
                out[blk + (pi * 4 + 3) * g.tcb + ti] = w[r, q]
    return out.tobytes()


# ----------------------------------------------------------------------------- comparison


def _expect_bits(label, what, got, want, names):
    """bit equality of float32 arrays; the message names the first differing index and both values"""
    got, want = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(want, np.float32)
    assert got.shape == want.shape, (label, what, got.shape, want.shape)
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
    if len(bad):
        i = tuple(int(v) for v in bad[0])
        where = ", ".join("%s %d" % (n, v) for n, v in zip(names, i))
        raise AssertionError("%s: %s: %d of %d values differ, first at %s: engine %r (0x%08x), reference %r (0x%08x)" % (
            label, what, len(bad), got.size, where, float(got[i]), int(got.view(np.uint32)[i]), float(want[i]),
            int(want.view(np.uint32)[i])))
    return got.size


def _expect_zero(label, what, got, names, offset=()):
    """padding: +0.0 or -0.0"""
    got = np.ascontiguousarray(got, np.float32)
    bad = np.argwhere((got.view(np.uint32) & 0x7FFFFFFF) != 0)
    if len(bad):
        i = tuple(int(v) for v in bad[0])
        where = ", ".join("%s %d" % (n, v + (offset[k] if k < len(offset) else 0)) for k, (n, v) in enumerate(zip(names, i)))
        raise AssertionError("%s: %s padding: %d of %d values are not zero, first at %s: %r" % (label, what, len(bad), got.size, where,
                                                                                              float(got[i])))
    return got.size


# ----------------------------------------------------------------------------- the engine


def _step_inputs(gen, step):
    """(info, cells bytes, library bytes, active-pixel list, perm or None) of mosaic_debug_step_inputs"""
    from mosaicmagnifique_b200._capi import StepInputs
    L = gen._L
    info = StepInputs()
    gen._ck(L.mosaic_debug_step_inputs(gen._h, step, ctypes.byref(info), None, 0, None, 0, None, None))
    cells = np.empty(info.cell_bytes, np.uint8)
    lib = np.empty(info.lib_bytes, np.uint8)
    pix = np.empty(max(info.n_active, 1), np.int32)
    perm = np.full(info.n_lib_tiles * info.slots_per_tile, -1, np.int32)
    again = StepInputs()
    gen._ck(L.mosaic_debug_step_inputs(gen._h, step, ctypes.byref(again), cells.ctypes.data, cells.size, lib.ctypes.data, lib.size,
                                       pix.ctypes.data, perm.ctypes.data))
    assert bytes(again) == bytes(info), "the second call reports other sizes"
    assert (info.cells_per_tile, info.slots_per_tile, info.pixels_per_chunk) == TILES[info.layout]
    return info, cells.tobytes(), lib.tobytes(), pix[:info.n_active], (perm if info.has_perm else None)


def _generator(main, lib, shape, case):
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
    gen = PhotomosaicGenerator(0)
    gen.setMainImage(main)
    gen.setLibrary(lib)
    gen.setColourDifference(case.diff)
    gen.setColourScheme(case.scheme)
    gen.setVariantQuirk(case.quirk)
    gen.setTileFlips(bool(case.flips & 1), bool(case.flips & 2))
    gen.setRepeat(*((2, 500) if case.repeats else (0, 0)))
    cg = CellGroup()
    cg.setCellShape(shape)
    cg.setDetail(case.detail)
    cg.setSizeSteps(case.steps)
    gen.setCellGroup(cg)
    return gen


class _Inputs:
    """one case's engine and oracle inputs"""

    def __init__(self, oracle, case):
        from tests.test_gpu_generator import _to_product_shape
        from mosaicmagnifique_b200 import synthetic
        self.case = case
        seed = _seed(case.name)
        self.H, self.W = _main_size(case.S)
        self.main = synthetic.make_main_image(self.H, self.W, seed, block=max(8, case.S // 2))
        self.lib = synthetic.make_library(case.N, case.S, seed + 1)
        o_shape = _o_shape(oracle, case)
        self.og = oracle.CellGroup.make(o_shape, case.detail, case.steps)
        self.states = _states(oracle, self.og, self.H, self.W, seed + 2)
        self.shape = _to_product_shape(o_shape)

    def generator(self, case=None):
        gen = _generator(self.main, self.lib, self.shape, case or self.case)
        gen.setGridState(self.states)
        return gen


def _check_step(oracle, label, inp, step, got, lib_f, mains):
    """compares one step's packed inputs with the oracle; returns the number of values compared"""
    case, og = inp.case, inp.og
    info, cells_raw, lib_raw, pix, perm = got
    layout = _layout(case.diff)
    assert info.layout == layout, label
    normal, dshape = og.cells[step], og.detail_cells[step]
    ds = dshape.size
    P = ds * ds
    state = inp.states[step]
    want_pix = _active_pixels(oracle, normal, dshape, state)
    assert np.array_equal(pix, want_pix), "%s: active pixels: %d of the engine, %d of the reference, first difference at %s" % (
        label, len(pix), len(want_pix), np.flatnonzero(pix[:len(want_pix)] != want_pix[:len(pix)])[:1].tolist())
    na = len(want_pix)
    g = Geom(layout, info.n_chunks, info.n_cell_tiles, info.n_lib_tiles, *TILES[layout])
    assert info.n_chunks == max(1, -(-na // g.kp)), label
    n_slots = case.N * len(_orientations(case.flips))
    assert info.n_slots == n_slots and info.n_lib_tiles == -(-n_slots // g.tnb), label
    n_compared = na

    # library
    n_pad = info.n_lib_tiles * g.tnb
    want_order = _library_order(_oriented_library(inp.lib, case.flips), n_pad)
    assert (perm is not None) == (case.diff == CIEDE and (case.repeats or info.n_variants > 1)), label
    if perm is not None:
        assert np.array_equal(perm, want_order), "%s: colour order differs at slots %s" % (
            label, np.flatnonzero(perm != want_order)[:5].tolist())
        n_compared += n_pad
    order = perm[:n_slots] if perm is not None else np.arange(n_slots)
    assert lib_f.shape == (n_slots, ds, ds, 3), (label, lib_f.shape)
    want = _stored(lib_f.reshape(n_slots, P, 3)[order][:, want_pix], layout)
    if layout == LAYOUT_EUCLID:
        want = -want
    dec = _decode_lib(lib_raw, g)
    n_compared += _expect_bits(label, "library", dec[:n_slots, :na], want, ("slot", "compacted pixel", "channel"))
    n_compared += _expect_zero(label, "library slots", dec[n_slots:], ("slot", "pixel", "channel"), (n_slots,))
    n_compared += _expect_zero(label, "library pixels", dec[:n_slots, na:], ("slot", "pixel", "channel"), (0, na))

    # cells
    ex, bounds, flips, _ = oracle.extract_cells(mains, og, step, state, shared_buffer_quirk=case.quirk)
    n, V = ex.shape[0], info.n_variants
    if ex.shape[1] != V:  # the faithful quirk compares one variant: every shared-buffer variant holds the last rotation
        assert case.quirk and V == 1, label
        ex = ex[:, -1:]
    assert info.n_rows == n * V and info.n_cell_tiles == -(-n * V // g.tcb), label
    want = _stored(ex.reshape(n * V, P, 3)[:, want_pix], layout)
    m4 = dshape.masks4().reshape(4, P) > 0
    py, px = want_pix // ds, want_pix % ds
    bx, by, bw, bh = (bounds[:, i:i + 1] for i in range(4))
    inside = (px >= bx) & (px < bx + bw) & (py >= by) & (py < by + bh)
    w_on = np.float32(50.0 if layout == LAYOUT_CIEDE else 1.0)
    want_w = np.repeat(np.where(m4[flips][:, want_pix] & inside, w_on, np.float32(0.0)), V, axis=0)
    vals, w = _decode_cells(cells_raw, g)
    R = n * V
    n_compared += _expect_bits(label, "cells", vals[:R, :na], want, ("row", "compacted pixel", "channel"))
    n_compared += _expect_bits(label, "cell weights", w[:R, :na], want_w, ("row", "compacted pixel"))
    n_compared += _expect_zero(label, "cell rows", vals[R:], ("row", "pixel", "channel"), (R,))
    n_compared += _expect_zero(label, "cell weight rows", w[R:], ("row", "pixel"), (R,))
    n_compared += _expect_zero(label, "cell pixels", vals[:R, na:], ("row", "pixel", "channel"), (0, na))
    n_compared += _expect_zero(label, "cell weight pixels", w[:R, na:], ("row", "pixel"), (0, na))
    return n_compared


def _path(info, normal_size, ds):
    lib = "fused k=%d" % info.fused_k if info.fused else "unfused"
    cells = "k=%d" % (normal_size // ds) if normal_size % ds == 0 else "%d/%d" % (normal_size, ds)
    return "library %s, cells %s" % (lib, cells)


def _run(oracle, inp, gen, label):
    """every step of one case: returns the decoded library tiles of each step"""
    case, og = inp.case, inp.og
    mains = [oracle.to_working_space(v, case.diff) for v in oracle.colour_scheme_variants(inp.main, case.scheme)]
    lib_f = oracle.preprocess_library(_oriented_library(inp.lib, case.flips), og, case.diff)
    libs = []
    for s in range(case.steps + 1):
        if s > 0:
            lib_f = oracle.halve_library(lib_f)
        got = _step_inputs(gen, s)
        info = got[0]
        assert bool(info.fused) == (case.steps == 0), label
        n = _check_step(oracle, "%s step %d" % (label, s), inp, s, got, lib_f, mains)
        print("%s step %d: %s; N %d (%d slots), V %d, %d rows, n_active %d (%d chunks), %d values compared" % (
            label, s, _path(info, og.cells[s].size, og.detail_cells[s].size), case.N, info.n_slots, info.n_variants, info.n_rows,
            info.n_active, info.n_chunks, n))
        libs.append((info, got[2], got[4]))
    return libs


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_packed_inputs_match_opencv(oracle, case):
    inp = _Inputs(oracle, case)
    gen = inp.generator()
    try:
        _run(oracle, inp, gen, case.name)
    finally:
        gen.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S", SWEEP_SIZES)
def test_every_detail_percent(oracle, S):
    """RGB library and cells at every integer detail percent the engine accepts (fractional INTER_AREA tables; the integer ratios
    among them take the fused packer)"""
    from mosaicmagnifique_b200 import CellGroup, MosaicError
    case = _case("sweep-%d" % S, RGB, S, 100, N=SWEEP_N)
    inp = _Inputs(oracle, case)
    gen = inp.generator()
    refused = []
    try:
        for p in range(1, 101):
            inp.case = case._replace(name="sweep-%d-d%d" % (S, p), detail=p)
            inp.og = oracle.CellGroup.make(oracle.CellShape.square(S), p, 0)
            cg = CellGroup()
            cg.setCellShape(inp.shape)
            cg.setDetail(p)
            try:
                gen.setCellGroup(cg)
                gen.setGridState(inp.states)
                _run(oracle, inp, gen, inp.case.name)
            except MosaicError as e:
                refused.append((p, str(e)))
    finally:
        gen.close()
    print("sweep at cell size %d: %d detail percents compared, refused: %s" % (S, 100 - len(refused), refused or "none"))
    assert not refused


@pytest.mark.gpu
@pytest.mark.parametrize("diff", [RGB, CIE76, CIEDE], ids=["rgb", "cie76", "ciede"])
def test_fused_equals_unfused(oracle, diff):
    """the library tiles of step 0 are the same bits whether the 8U packer reduces and converts on the fly (no size step) or the f32
    working library is materialised first (one size step): no reference involved"""
    case = _case("fused-vs-unfused", diff, 32, 50, N=9, repeats=diff == CIEDE)
    a = _Inputs(oracle, case)
    b = _Inputs(oracle, case._replace(steps=1))
    b.main, b.lib = a.main, a.lib
    b.states[0] = a.states[0]
    got = []
    for inp in (a, b):
        gen = inp.generator()
        try:
            got.append(_step_inputs(gen, 0))
        finally:
            gen.close()
    (ia, _, la, pa, oa), (ib, _, lb, pb, ob) = got
    assert (ia.fused, ib.fused) == (1, 0) and ia.fused_k == 2
    assert np.array_equal(pa, pb) and (oa is None) == (ob is None) and (oa is None or np.array_equal(oa, ob))
    assert (ia.n_lib_tiles, ia.n_chunks, ia.n_active) == (ib.n_lib_tiles, ib.n_chunks, ib.n_active)
    layout = _layout(diff)
    g = Geom(layout, ia.n_chunks, ia.n_cell_tiles, ia.n_lib_tiles, *TILES[layout])
    n = _expect_bits("fused vs unfused, diff %d" % diff, "library", _decode_lib(la, g)[:ia.n_slots, :ia.n_active],
                     _decode_lib(lb, g)[:ia.n_slots, :ia.n_active], ("slot", "compacted pixel", "channel"))
    print("fused = unfused, diff %d: %d library values" % (diff, n))


@pytest.mark.gpu
def test_results_kept(oracle):
    """the tap runs the preprocessing on the handle's workspace but leaves a generate's results as they were"""
    case = _case("results-kept", CIEDE, 32, 50, N=9, steps=1, flips=1, repeats=True)
    inp = _Inputs(oracle, case)
    gen = inp.generator()
    try:
        gen.setKeepDifferences(True)
        assert gen.generateBestFits()
        before = (gen.getBestFits(), gen.getBestFitFlips(), [gen.getDifferences(s) for s in range(2)], gen.getTimings())
        gen.setTileFlips(False, False)  # the tap then runs with another slot count than the generate's
        for s in (1, 0):
            _step_inputs(gen, s)
        gen.setTileFlips(True, False)
        after =(gen.getBestFits(), gen.getBestFitFlips(), [gen.getDifferences(s) for s in range(2)], gen.getTimings())
    finally:
        gen.close()
    for a, b in zip(before[0] + before[1] + before[2], after[0] + after[1] + after[2]):
        assert np.array_equal(a, b)
    assert before[3] == after[3]


# ----------------------------------------------------------------------------- CPU: the tables and the decoder


def test_case_tables_cross_their_edges(oracle):
    """recomputes from the oracle what each case is there for, so that an edit of a table cannot quietly move it off its edge"""
    fused_k = {LAYOUT_CIEDE: set(), LAYOUT_EUCLID: set()}
    for c in FUSED:
        og = oracle.CellGroup.make(oracle.CellShape.square(c.S), c.detail, 0)
        ds = og.detail_cells[0].size
        assert c.S % ds == 0, c.name
        fused_k[_layout(c.diff)].add(c.S // ds)
    assert fused_k[LAYOUT_CIEDE] == fused_k[LAYOUT_EUCLID] == set(FUSED_K), fused_k
    assert {c.diff for c in FUSED} == {c.diff for c in UNFUSED} == {RGB, CIE76, CIEDE}
    assert {c.repeats for c in FUSED if c.diff == CIEDE} == {True, False}
    assert {c.N for c in FUSED} >= {1, 7, 8, 9, 63, 65, 130} and {c.flips for c in FUSED} == {0, 1, 3}

    # slot remainders of the library tiles (8 and 64 images)
    rem = {LAYOUT_CIEDE: set(), LAYOUT_EUCLID: set()}
    for c in FUSED + UNFUSED:
        lay = _layout(c.diff)
        rem[lay].add(c.N * len(_orientations(c.flips)) % TILES[lay][1])
    assert rem[LAYOUT_CIEDE] >= {0, 1, TILES[LAYOUT_CIEDE][1] - 1}, rem
    assert rem[LAYOUT_EUCLID] >= {1, 2, TILES[LAYOUT_EUCLID][1] - 1}, rem

    # size steps: integer and fractional ratios, the library size even wherever it is halved
    kinds = set()
    for c in UNFUSED:
        og = oracle.CellGroup.make(oracle.CellShape.square(c.S), c.detail, c.steps)
        sizes = [d.size for d in og.detail_cells]
        assert all(sizes[s] == 2 * sizes[s + 1] for s in range(c.steps)), (c.name, sizes)
        kinds |= {(c.diff, c.S % sizes[0] == 0)}
    assert kinds == {(d, k) for d in (RGB, CIE76, CIEDE) for k in (True, False)}, kinds

    # the sweep meets both kinds of ratio, odd integer ones among them
    ks = set()
    for S in SWEEP_SIZES:
        ds = {max(int(S * (p / 100.0)), 1) for p in range(1, 101)}
        ks |= {S // d for d in ds if S % d == 0}
        assert len({d for d in ds if S % d}) > 30, S
    assert ks >= {1, 2, 3, 4, 5, 8}, ks

    # the active-pixel axis: below, at and above a chunk of each layout; the flipped triangle uses its union of four masks
    chunk_rem = {LAYOUT_CIEDE: set(), LAYOUT_EUCLID: set()}
    clipped = set()
    for c in CASES:
        inp_shape = _o_shape(oracle, c)
        og = oracle.CellGroup.make(inp_shape, c.detail, c.steps)
        H, W = _main_size(c.S)
        states = _states(oracle, og, H, W, _seed(c.name) + 2)
        for s, st in enumerate(states):
            assert (st >= 0).any(), (c.name, s)
            pix = _active_pixels(oracle, og.cells[s], og.detail_cells[s], st)
            kp = TILES[_layout(c.diff)][2]
            chunk_rem[_layout(c.diff)].add(len(pix) % kp)
            if c.shape == "mask":
                assert len(pix) == c.mask_k, c.name
            if c.shape.startswith("IsocelesTriangle-45deg") and s == 0:
                used = {oracle.flip_at(og.cells[0], x - 2, y - 2) for y, x in _valid(st)}
                assert used == ({0, 1, 2, 3} if c.shape.endswith("one-flag-off") else {0, 3}), (c.name, used)
                assert len(pix) > int((og.detail_cells[0].mask > 0).sum()), c.name
            for y, x in _valid(st):
                rx, ry, rw, rh = oracle.rect_at(og.cells[s], x - 2, y - 2)
                clipped |= {(c.name, side) for side, cut in
                            (("left", rx < 0), ("top", ry < 0), ("right", rx + rw > W), ("bottom", ry + rh > H)) if cut}
    for lay, (_, _, kp) in TILES.items():
        assert chunk_rem[lay] >= {kp - 1, 0, 1}, (lay, chunk_rem[lay])
    for name in ("hexagon-ciede-order", "hexagon-rgb-frac"):
        assert {side for n, side in clipped if n == name} == {"left", "top", "right", "bottom"}, name
    assert all((c.name, "right") in clipped and (c.name, "bottom") in clipped for c in CASES)
    quirk = {(c.quirk, c.detail) for c in CELLS if c.scheme}
    assert quirk == {(q, d) for q in (True, False) for d in (100, 50)}, quirk


@pytest.mark.parametrize("layout", [LAYOUT_CIEDE, LAYOUT_EUCLID], ids=["ciede", "euclid"])
def test_decoder_round_trip(layout):
    """tiles packed element by element from the layout comments decode back to the values: a decoder bug cannot pass for an engine
    bug. Two tiles on each axis and two chunks, distinct values everywhere."""
    tcb, tnb, kp = TILES[layout]
    g = Geom(layout, 2, 2, 2, tcb, tnb, kp)
    rng = np.random.default_rng(layout)
    C = 4 if layout == LAYOUT_CIEDE else 3
    lib = rng.standard_normal((2 * tnb, 2 * kp, C)).astype(np.float32)
    cells = rng.standard_normal((2 * tcb, 2 * kp, C)).astype(np.float32)
    w = rng.standard_normal((2 * tcb, 2 * kp)).astype(np.float32)
    assert np.array_equal(_decode_lib(_pack_lib_numpy(lib, g), g), lib)
    v, ww = _decode_cells(_pack_cells_numpy(cells, w, g), g)
    assert np.array_equal(v, cells) and np.array_equal(ww, w)
    # block sizes as kernels.h's tile_geom states them (bytes of one tile x chunk block)
    assert len(_pack_lib_numpy(lib, g)) == g.n_lib_tiles * g.n_chunks * (tnb * kp * 16 if layout == LAYOUT_CIEDE else kp * 3 * tnb * 4)
    assert len(_pack_cells_numpy(cells, w, g)) == g.n_cell_tiles * g.n_chunks * (tcb * kp * 20 if layout == LAYOUT_CIEDE else kp * 4 * tcb * 4)


def test_stored_channels():
    """the CIEDE2000 channels: 0.5f * L - 25 is one rounding (what fmaf gives, 0.5 * L being exact), C rounds a f64 square root"""
    x = np.array([[[53.2421875, 80.09375, 67.203125]], [[100.0, -0.5, 0.25]]], np.float32)
    s = _stored(x, LAYOUT_CIEDE)
    assert s.dtype == np.float32
    assert s[0, 0, 0] == np.float32(np.float64(x[0, 0, 0]) * 0.5 - 25.0)
    assert s[0, 0, 3] == np.float32(0.02) * np.float32(np.hypot(80.09375, 67.203125))
    assert np.array_equal(_stored(x, LAYOUT_EUCLID), x)
