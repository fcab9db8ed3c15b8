"""NumPy restatement of the usage limit (mosaic_set_usage_limit, DESIGN.md 4.4): the capped rule, its candidate bound K_s and the
prefix scan of select_capped_kernel. Shared by the CPU and GPU tests and tools/bench_usage_limit.py."""
import numpy as np

DBL_MAX = np.finfo(np.float64).max
PREFIX_MAX = 1024  # kernels.h kPrefixMax
CHUNK = 32         # entries select_capped_kernel examines between two checks of the stop rule


def exhausted_bound(cells_before, n_valid, max_uses):
    """E_s: the most images that can be exhausted before the last cell of a step"""
    return max(0, cells_before + n_valid - 1) // max_uses


def k_bound(O, N, rr, E, margins=False):
    """K_s = min(O * N, O * (W + E_s) + 1), + 1 with margins; W = 2r^2 + 2r"""
    return min(O * N, O * (2 * rr * rr + 2 * rr + E) + 1 + int(margins))


def window_counts(grid, x, y, rr, n_images):
    """calculateRepeats occurrence counts, orientations of an image pooled (slot s counts for image s mod N)"""
    rows, cols = grid.shape
    y0 = min(max(y - rr, 0), rows)
    x0 = min(max(x - rr, 0), cols)
    x1 = min(max(x + rr, 0), cols - 1)
    vals = np.concatenate([grid[y0:y, x0:x1 + 1].ravel(), grid[y, x0:x]])
    vals = vals[vals >= 0] % n_images
    return np.bincount(vals, minlength=n_images) if vals.size else np.zeros(n_images, np.int64)


def full_row(row, allowed, penalty, margins=False):
    """the capped rule on one row: lowest (D + penalty, slot) over the allowed slots -> (slot or -1, best, second)"""
    v = np.where(allowed, row.astype(np.float64) + penalty, np.inf)
    s = int(np.argmin(v))
    best = v[s]
    if not best < DBL_MAX:
        return -1, best, np.inf
    second = np.partition(v, 1)[1] if margins and v.size > 1 else np.inf
    return s, best, second


def prefix_scan(row, allowed, penalty, k0, row_len, margins=False, chunk=CHUNK):
    """select_capped_kernel on one cell: the sorted prefix (the k0 smallest (score, slot) pairs of the row) `chunk` entries at a
    time, stopping once the next entry's score is strictly above the best (with margins: second-best) allowed penalised value; a
    prefix that ends first falls back to the whole candidate row (row_len entries: the K list or the D row).
    Returns (slot or -1, best, second, fell_back)."""
    order = np.lexsort((np.arange(row.size), row.astype(np.float64)))[:k0]
    best, best_id, second = DBL_MAX, np.iinfo(np.int32).max, DBL_MAX
    for j0 in range(0, k0, chunk):
        if float(row[order[j0]]) > (second if margins else best):
            break
        for s in order[j0:j0 + chunk]:
            if allowed[s]:
                v = float(row[s]) + float(penalty[s])
                if v < best or (v == best and s < best_id):
                    best, best_id, second = v, int(s), min(best, second)
                else:
                    second = min(second, v)
    else:
        if k0 < row_len:
            s, b, sec = full_row(row, allowed, penalty, margins)
            return s, b, sec, True
    return (best_id if best < DBL_MAX else -1), best, (second if second < DBL_MAX else np.inf), False


def capped_rule(Ds, states, rr, ra, n_images, max_uses, scan=None):
    """The capped rule over all steps of one generate on the engine's D (f64), `used` carried across the steps.
    scan: None, or (list of (k0, row_len) per step, margins) to replay the prefix scan instead (counts the cells that fall back).
    Returns (grids, fallbacks)."""
    used = np.zeros(n_images, np.int64)
    grids, fallbacks = [], 0
    for step, (D, state) in enumerate(zip(Ds, states)):
        grid = np.where(np.asarray(state) >= 0, 0, -1).astype(np.int64)
        O = D.shape[1] // n_images if D.size else 1
        c = 0
        for y in range(grid.shape[0]):
            for x in range(grid.shape[1]):
                if grid[y, x] < 0:
                    continue
                pen = np.zeros(D.shape[1])
                if rr > 0 and ra:
                    pen = ra * np.tile(window_counts(grid, x, y, rr, n_images), O).astype(np.float64)
                allowed = np.tile(used < max_uses, O)
                if scan is None:
                    s = full_row(D[c], allowed, pen)[0]
                else:
                    (k0, row_len), margins = scan[0][step], scan[1]
                    s, _, _, fb = prefix_scan(D[c], allowed, pen, k0, row_len, margins)
                    fallbacks += fb
                grid[y, x] = s
                if s >= 0:
                    used[s % n_images] += 1
                c += 1
        grids.append(grid)
    return grids, fallbacks
