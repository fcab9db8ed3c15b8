"""CPU checks of mirrored library tiles (no device): the grouped candidate bound of DESIGN.md 4.4 and the new C ABI symbols.

With O orientations of N images and repeats counted per source image, a window of W = 2r^2 + 2r cells penalises at most O * W of
the O * N slots, so the penalised winner (and, with report_margins, the runner-up) is among the K = min(O * N, O * W + 1) (+1)
smallest (score, slot) pairs of the unpenalised row."""
import ctypes
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _penalised_order(row, counts, O, A):
    """slots of one row by (penalised score, slot): repeats grouped, slot s pays A * counts[s mod N]"""
    pen = row.astype(np.float64) + A * np.tile(counts, O)
    return np.lexsort((np.arange(row.size), pen))


def _k_smallest(row, K):
    return set(np.lexsort((np.arange(row.size), row.astype(np.float64)))[:K].tolist())


def test_grouped_bound_is_exact_on_random_rows():
    rng = np.random.default_rng(1234)
    for trial in range(3000):
        O = int(rng.choice([1, 2, 4]))
        N = int(rng.integers(1, 40))
        r = int(rng.integers(0, 3))
        W = 2 * r * r + 2 * r
        A = float(rng.choice([0.5, 3.0, 500.0]))
        # coarse scores: plenty of exact ties between slots
        row = rng.integers(0, 6, O * N).astype(np.float32) * float(rng.choice([1.0, 0.25]))
        window = rng.integers(0, O * N, int(rng.integers(0, W + 1)))  # chosen slots of the window, any orientation
        counts = np.bincount(window % N, minlength=N)
        order = _penalised_order(row, counts, O, A)
        K = min(O * N, O * W + 1)
        assert int(order[0]) in _k_smallest(row, K), (trial, O, N, r)
        if O * N > 1:
            assert int(order[1]) in _k_smallest(row, min(O * N, O * W + 2)), (trial, O, N, r)


def test_one_less_is_not_enough():
    """A window of W distinct images whose O * W slots hold the smallest scores: every one of them is penalised, the winner is the
    smallest unpenalised slot, ranked exactly O * W + 1, and K = O * W is one short."""
    for O in (2, 4):
        r = 1
        W = 2 * r * r + 2 * r
        N = W + 2
        row = np.empty(O * N, np.float32)
        for j in range(O):
            row[j * N: j * N + W] = np.arange(W) + j * W  # the O * W slots of images 0..W-1: the smallest scores
            row[j * N + W:(j + 1) * N] = 1000.0 + j
        counts = np.bincount(np.arange(W), minlength=N)  # the window holds images 0..W-1 once each
        winner = int(_penalised_order(row, counts, O, 10000.0)[0])
        K = O * W + 1
        assert winner in _k_smallest(row, K)
        assert winner not in _k_smallest(row, K - 1)


def test_tile_flip_symbols_declared_and_bound():
    text = open(os.path.join(ROOT, "include", "mosaic_b200.h")).read()
    for name in ("mosaic_set_tile_flips", "mosaic_get_best_fit_flips"):
        assert re.search(r"\bint %s\s*\(" % name, text), name
    from mosaicmagnifique_b200 import capi
    L = capi()
    assert L.mosaic_set_tile_flips.argtypes == [ctypes.c_void_p, ctypes.c_int]
    assert "mosaic_get_best_fit_flips" in L._signatures
    hpp = open(os.path.join(ROOT, "include", "mosaic_b200.hpp")).read()
    assert "setTileFlips(bool horizontal, bool vertical)" in hpp and "getBestFitFlips()" in hpp
