"""Debug / analysis: executed share of the CIEDE2000 segment passes on config 4's seeded inputs when a row's alive test adds a
lightness lower bound of the segments not yet summed (DESIGN.md 4.1), for blocks of 8, 16 and 32 compacted pixels.

    python tools/debug/prune_bound_sim.py [SUB]

CPU restatement, f64: the Sharma CIEDE2000, every SUB-th library image (default 10) with K scaled to keep K / N, 8 cells spread
over the grid, 8 segments of 16 pixel rows, library tiles of 8 images in colour order, candidates = the 1.25 K + 8 smallest
`pass-0 partial + bound of segments 1..7`. Config 4's cell is the whole square, so the compacted pixel order is the raster order
and a block is a run of B pixels of one pixel row. Per block the bound is |sum dL| / S_L(m), m = max(|lo|, |hi|) where [lo, hi]
bounds Lbar - 50 from the two blocks' minimum and maximum L, with S_L either exact or bounded by 1 + 0.015 m (the kernel's form,
since sqrt(20 + m^2) >= m)."""
import os
import sys
import time

import cv2
import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from mosaicmagnifique_b200 import synthetic  # noqa: E402

NFULL, S, KFULL, SEGS = 10000, 128, 145, 8
SUB = int(sys.argv[1]) if len(sys.argv) > 1 else 10
N = NFULL // SUB
K = max(3, round(KFULL / SUB))
BLOCKS = (8, 16, 32)
CELLS = [(3, 5), (10, 20), (20, 40), (30, 55), (15, 33), (8, 48), (25, 10), (2, 58)]


def ciede(L1, a1, b1, L2, a2, b2):
    C1 = np.hypot(a1, b1)
    C2 = np.hypot(a2, b2)
    Cb7 = ((C1 + C2) / 2) ** 7
    G = 0.5 * (1 - np.sqrt(Cb7 / (Cb7 + 25.0 ** 7)))
    a1p, a2p = a1 * (1 + G), a2 * (1 + G)
    C1p, C2p = np.hypot(a1p, b1), np.hypot(a2p, b2)
    h1 = np.mod(np.arctan2(b1, a1p), 2 * np.pi)
    h2 = np.mod(np.arctan2(b2, a2p), 2 * np.pi)
    dL, dC = L2 - L1, C2p - C1p
    dh = h2 - h1
    dh = np.where(dh > np.pi, dh - 2 * np.pi, np.where(dh < -np.pi, dh + 2 * np.pi, dh))
    dh = np.where(C1p * C2p == 0, 0, dh)
    dH = 2 * np.sqrt(C1p * C2p) * np.sin(dh / 2)
    Lb, Cpb, hs = (L1 + L2) / 2, (C1p + C2p) / 2, h1 + h2
    hb = np.where(np.abs(h1 - h2) > np.pi, np.where(hs < 2 * np.pi, hs / 2 + np.pi, hs / 2 - np.pi), hs / 2)
    hb = np.where(C1p * C2p == 0, hs, hb)
    T = (1 - 0.17 * np.cos(hb - np.pi / 6) + 0.24 * np.cos(2 * hb) + 0.32 * np.cos(3 * hb + np.pi / 30)
         - 0.2 * np.cos(4 * hb - 63 * np.pi / 180))
    dth = np.pi / 6 * np.exp(-((hb * 180 / np.pi - 275) / 25) ** 2)
    Cpb7 = Cpb ** 7
    RT = -np.sin(2 * dth) * 2 * np.sqrt(Cpb7 / (Cpb7 + 25.0 ** 7))
    SL = 1 + 0.015 * (Lb - 50) ** 2 / np.sqrt(20 + (Lb - 50) ** 2)
    x, y, z = dL / SL, dC / (1 + 0.045 * Cpb), dH / (1 + 0.015 * Cpb * T)
    return np.sqrt(x * x + y * y + z * z + RT * y * z)


def s_l(m):
    return 1 + 0.015 * m * m / np.sqrt(20 + m * m)


def block_bounds(cellL, libL, B, linear):
    """[n][SEGS] lightness bound of each segment: sum over its blocks of |sum dL| / S_L at the block pair's worst mean lightness"""
    c = cellL.reshape(-1, B)
    l = libL.reshape(len(libL), -1, B)
    dsum = np.abs(l.sum(2) - c.sum(1)[None])
    lo = (l.min(2) + c.min(1)[None]) / 2 - 50
    hi = (l.max(2) + c.max(1)[None]) / 2 - 50
    m = np.maximum(np.abs(lo), np.abs(hi))
    b = dsum / ((1 + 0.015 * m) if linear else s_l(m))
    return b.reshape(len(libL), SEGS, -1).sum(2)


def executed(D, LB, tiles, inv):
    """share of (row, segment) work: pass 0 for all rows, candidate tiles completed, later passes only rows with a pair whose
    partial sum + bound of the segments not yet summed is <= T"""
    pre = np.cumsum(D, 1)
    full = pre[:, -1]
    rest = np.concatenate([LB[:, ::-1].cumsum(1)[:, ::-1][:, 1:], np.zeros((len(D), 1))], 1)  # rest[:, s] = bound after s
    M = int(1.25 * K) + 8
    cand = np.argsort(pre[:, 0] + rest[:, 0], kind="stable")[:M]
    T = np.sort(full[cand])[K - 1]
    assert T >= np.sort(full)[K - 1]
    work = np.ones(len(tiles))
    ct = np.unique(inv[cand] // 8)
    ct = ct[ct < len(tiles)]
    work[ct] = SEGS
    alive = np.ones(len(tiles), bool)
    alive[ct] = False
    for s in range(1, SEGS):
        a = ((pre[:, s - 1] + rest[:, s - 1])[tiles] <= T).any(1) & alive
        work[a] += 1
        alive = a
    return work.sum() / (len(tiles) * SEGS)


def main():
    lib = synthetic.make_library(NFULL, S, 1004)[::SUB]
    mainimg = synthetic.make_main_image(4320, 7680, 2004)
    libL = cv2.cvtColor(lib.reshape(-1, S, 3).astype(np.float32) / 255, cv2.COLOR_BGR2Lab).reshape(N, S, S, 3).astype(np.float64)
    mainL = cv2.cvtColor(mainimg.astype(np.float32) / 255, cv2.COLOR_BGR2Lab).astype(np.float64)
    means = libL.mean((1, 2))
    q = np.clip(((means - means.min(0)) / np.ptp(means, 0) * 1023).astype(np.int64), 0, 1023)
    code = np.zeros(N, np.int64)
    for b in range(10):
        for c in range(3):
            code |= ((q[:, c] >> b) & 1) << (3 * b + c)
    order = np.argsort(code, kind="stable")
    tiles = order[: N // 8 * 8].reshape(-1, 8)
    inv = np.empty(N, np.int64)
    inv[order] = np.arange(N)
    cols = ["partial <= T"] + ["B=%d %s" % (B, "lin" if lin else "exact") for B in BLOCKS for lin in (True, False)]
    res = []
    for cy, cx in CELLS:
        t = time.time()
        cell = mainL[cy * S:(cy + 1) * S, cx * S:(cx + 1) * S]
        D = np.empty((N, SEGS))
        for i in range(0, N, 25):
            l = libL[i:i + 25]
            e = ciede(cell[None, ..., 0], cell[None, ..., 1], cell[None, ..., 2], l[..., 0], l[..., 1], l[..., 2])
            D[i:i + 25] = e.reshape(-1, SEGS, S * S // SEGS).sum(2)
        row = [executed(D, np.zeros_like(D), tiles, inv)]
        ratio = []
        for B in BLOCKS:
            for lin in (True, False):
                LB = block_bounds(cell[..., 0].ravel(), libL[..., 0].reshape(N, -1), B, lin)
                assert (LB <= D * (1 + 1e-9)).all()
                row.append(executed(D, LB, tiles, inv))
                ratio.append((LB.sum(1) / D.sum(1)).mean())
        res.append(row)
        print((cy, cx), " ".join("%s %.3f" % kv for kv in zip(cols, row)),
              " bound/complete " + " ".join("%.2f" % r for r in ratio), "(%.0f s)" % (time.time() - t), flush=True)
    print("mean of %d cells, N = %d, K = %d:" % (len(CELLS), N, K))
    for c, v in zip(cols, np.mean(res, 0)):
        print("  %-16s executed share %.3f" % (c, v))


if __name__ == "__main__":
    main()
