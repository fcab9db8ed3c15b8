"""CPU checks of the usage limit (no device): the candidate bound K_s of DESIGN.md 4.4, the prefix scan of select_capped_kernel
restated in NumPy, and the new symbols of the C ABI and its mirrors.

With W = 2r^2 + 2r window cells and at most E images exhausted, at most O * (W + E) of the O * N slots are penalised or excluded, so
the capped winner (and, with report_margins, the runner-up) is among the K = min(O * N, O * (W + E) + 1) (+1) smallest (score, slot)
pairs of the unpenalised row."""
import ctypes
import os
import re

import numpy as np

from tests.helpers.usage_limit import full_row, k_bound, prefix_scan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _k_smallest(row, K):
    return set(np.lexsort((np.arange(row.size), row.astype(np.float64)))[:K].tolist())


def _random_case(rng):
    O = int(rng.choice([1, 2, 4]))
    N = int(rng.integers(2, 40))
    r = int(rng.integers(0, 3))
    W = 2 * r * r + 2 * r
    E = int(rng.integers(0, N))  # at most N - 1 exhausted: some image stays allowed
    A = float(rng.choice([0.0, 0.5, 3.0, 500.0]))
    row = rng.integers(0, 6, O * N).astype(np.float32) * float(rng.choice([1.0, 0.25]))  # coarse: many exact ties
    window = rng.integers(0, O * N, int(rng.integers(0, W + 1)))  # chosen slots of the window, any orientation
    counts = np.bincount(window % N, minlength=N)
    exhausted = rng.choice(N, int(rng.integers(0, E + 1)), replace=False)
    allowed_img = np.ones(N, bool)
    allowed_img[exhausted] = False
    return O, N, r, E, row, A * np.tile(counts, O).astype(np.float64), np.tile(allowed_img, O)


def test_capped_bound_is_exact_on_random_rows():
    rng = np.random.default_rng(4321)
    for trial in range(4000):
        O, N, r, E, row, pen, allowed = _random_case(rng)
        v = np.where(allowed, row.astype(np.float64) + pen, np.inf)
        order = np.lexsort((np.arange(v.size), v))  # penalised order over the allowed slots
        n_allowed = int(allowed.sum())
        assert int(order[0]) in _k_smallest(row, k_bound(O, N, r, E)), (trial, O, N, r, E)
        if n_allowed > 1:
            assert int(order[1]) in _k_smallest(row, k_bound(O, N, r, E, margins=True)), (trial, O, N, r, E)


def test_one_less_is_not_enough():
    """W window images and E exhausted images, all distinct, whose O * (W + E) slots hold the smallest scores: the winner is the
    smallest slot of the remaining images, ranked exactly O * (W + E) + 1, so K_s - 1 misses it."""
    for O in (1, 2, 4):
        for r, E in ((0, 3), (1, 2), (2, 5)):
            W = 2 * r * r + 2 * r
            N = W + E + 2
            row = np.empty(O * N, np.float32)
            for j in range(O):
                row[j * N: j * N + W + E] = np.arange(W + E) + j * (W + E)
                row[j * N + W + E:(j + 1) * N] = 1000.0 + j
            counts = np.bincount(np.arange(W), minlength=N)  # the window holds images 0..W-1 once each
            allowed_img = np.ones(N, bool)
            allowed_img[W:W + E] = False  # images W..W+E-1 are exhausted
            winner = full_row(row, np.tile(allowed_img, O), 1e4 * np.tile(counts, O))[0]
            K = k_bound(O, N, r, E)
            assert K == O * (W + E) + 1
            assert winner in _k_smallest(row, K)
            assert winner not in _k_smallest(row, K - 1)


def test_prefix_scan_equals_full_row_rule():
    """prefix + stop rule + fallback gives the full-row answer (and margins) whatever the prefix length, and the stop rule fires
    inside the prefix whenever the answer lies in it"""
    rng = np.random.default_rng(99)
    fell, stopped = 0, 0
    for trial in range(3000):
        O, N, r, E, row, pen, allowed = _random_case(rng)
        margins = bool(rng.integers(0, 2))
        k0 = int(rng.integers(1, O * N + 1))
        chunk = int(rng.choice([1, 4, 32]))
        want = full_row(row, allowed, pen, margins)
        got = prefix_scan(row, allowed, pen, k0, O * N, margins, chunk)
        assert got[0] == want[0] and got[1] == want[1], (trial, got, want)
        if margins and want[0] >= 0:
            assert got[2] == want[2], (trial, got, want)
        fell += got[3]
        stopped += not got[3] and k0 < O * N
    assert fell > 100 and stopped > 100  # both ways out of the prefix are exercised


def test_usage_limit_symbols_declared_and_bound():
    text = open(os.path.join(ROOT, "include", "mosaic_b200.h")).read()
    assert re.search(r"\bint mosaic_set_usage_limit\s*\(mosaic_generator \*g, int max_uses\)", text)
    from mosaicmagnifique_b200 import capi
    L = capi()
    assert L.mosaic_set_usage_limit.argtypes == [ctypes.c_void_p, ctypes.c_int]
    assert L.mosaic_set_usage_limit.restype == ctypes.c_int
    hpp = open(os.path.join(ROOT, "include", "mosaic_b200.hpp")).read()
    assert "void setUsageLimit(int maxUses)" in hpp
    from mosaicmagnifique_b200 import PhotomosaicGenerator
    assert hasattr(PhotomosaicGenerator, "setUsageLimit")
