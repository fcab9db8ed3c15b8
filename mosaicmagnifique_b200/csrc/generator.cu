// Host orchestration + C ABI (include/mosaic_b200.h) of the B200 photomosaic best-fit engine.
//
// Mirrors the reference's generator object
//   PhotomosaicGeneratorBase   src/Photomosaic/PhotomosaicGeneratorBase.{h,cpp}
//   CUDAPhotomosaicGenerator   src/Photomosaic/CUDA/CUDAPhotomosaicGenerator.{h,cpp}
// but with a different execution plan: instead of ~3 * N_lib launches and 17 stream syncs PER CELL
// (CUDAPhotomosaicGenerator.cpp:231-292) a size step is a fixed handful of launches on one stream:
//   to_working_space (main) -> [area_u8] -> to_working_space (library) -> pack_library -> extract_cells
//   -> diff_sum (cells x library, one launch) -> [min_variants] -> [topk] -> select / keys_to_grid.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mosaic_b200.h"
#include "host_model.h"
#include "kernels.h"

extern "C" const int16_t mm_lab_lut_s16[];  // lab_lut.S

namespace {

using namespace mm;

struct Fail {
    int code;
    std::string msg;
};

#define CU(expr)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            throw Fail{e__ == cudaErrorMemoryAllocation ? MOSAIC_ERR_OUT_OF_MEMORY : MOSAIC_ERR_CUDA,          \
                       std::string(#expr) + ": " + cudaGetErrorString(e__)};                                  \
    } while (0)

// Stream-ordered device buffer that keeps its capacity: buffers live in the generator's workspace and are only
// re-allocated when a call needs more, so a steady-state generate() performs no device allocation at all
// (the reference allocates and frees everything per call, CUDAPhotomosaicGenerator.cpp:82, 356).
struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0, cap = 0;
    cudaStream_t stream = nullptr;
    void alloc(size_t n, cudaStream_t s)
    {
        if (p && cap >= n) {
            bytes = n;
            return;
        }
        release();
        stream = s;
        if (n == 0)
            return;
        CU(cudaMallocAsync(&p, n, s));
        bytes = cap = n;
    }
    void release()
    {
        if (p)
            cudaFreeAsync(p, stream);
        p = nullptr;
        bytes = cap = 0;
    }
    template <typename T>
    T *as() const { return reinterpret_cast<T *>(p); }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), bytes(o.bytes), cap(o.cap), stream(o.stream)
    {
        o.p = nullptr;
        o.bytes = o.cap = 0;
    }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            release();
            p = o.p;
            bytes = o.bytes;
            cap = o.cap;
            stream = o.stream;
            o.p = nullptr;
            o.bytes = o.cap = 0;
        }
        return *this;
    }
};

// segment passes of the CIEDE2000 difference sums (kernels.h: RowList): 8 passes over the pixel axis, work lists of columns of
// 256 cells (config 4: 16 chunks per segment, a column's hot set 10 MB of L2)
constexpr int kPruneSegments = 8;
constexpr int kColumnCells = 256;

// persistent device workspace of one generator (see DevBuf)
struct Workspace {
    DevBuf main_f32, main_var_u8, lib_small, lib_work, lib_half;
    DevBuf pix_list, masks4, descs, cells_packed, lib_packed, best_key;
    DevBuf grid, pos, next, prog, counts;
    DevBuf tab_start, tab_si, tab_alpha;  // fractional INTER_AREA table of the current step
    // segment passes over row work lists (kernels.h: RowList) and exact pruning
    DevBuf perm, inv_perm, order_scratch, row_cells, row_count, row_groups, list_scratch, row_state, listed, prune_score, prune_idx,
        threshold;
    DevBuf lib_stats, cell_stats, prune_rest, prune_rank;  // lightness bound of the segments not yet summed (launch_prune_bound)
    DevBuf prefix_score, prefix_idx;  // usage limit: sorted prefixes of D rows, or launch_topk's pick for a candidate list's prefix
};

struct StepPlan {
    int rows = 0, cols = 0;
    int S = 0, ds = 0, k = 1;          // normal size, detail size, integer reduction factor
    int n_active = 0, n_chunks = 0;    // compacted pixels of the detail mask (union of the 4 flips)
    std::vector<int> cell_pos;         // valid cells, raster order: y * cols + x (padded coordinates)
    std::vector<int> next_x;           // next valid column in the same row
    std::vector<int> row_first;        // per grid row: column of the first valid cell (cols if none)
    int64_t cell_begin = 0, cell_end = 0;  // this rank's block of valid cells
    int64_t per_rank = 0;                  // rows every rank owns in the all-gathered candidate buffer (multiple of the cell tile)
    double pixel_diffs = 0, pixel_diffs_nominal = 0;
};

// one size step's device products; they keep their buffers across generates (the vector is only rebuilt when the number of steps
// changes)
struct StepOut {
    DevBuf D;        // [n_local_cells_pad * V][n_lib_pad]
    DevBuf cand;     // candidate block: float scores [rows][K], then int32 slots [rows][K]
    DevBuf margins;  // [n_valid][2] when report_margins
    bool have_D = false, have_margins = false;
    int cand_k = 0;  // K of the block of mosaic_generate_candidates (0 after a generate)
};

// The generator's streams and its page-locked / device words. mosaic_generator derives from this, so `delete` destroys them after
// every DevBuf member: each buffer is freed, stream-ordered, before the stream it was allocated on goes away.
struct Handles {
    cudaStream_t stream = nullptr;
    // progress(int) while a launch runs: device counter of finished CTAs, polled over a second stream into pinned memory
    cudaStream_t poll_stream = nullptr;
    // cancel(): a flag in pinned host memory (what the host tests) mirrored into a word of DEVICE memory by a 4-byte DMA on the
    // poll stream; every CTA of the difference kernels reads the device word (an L2 hit) when it starts. (Reading mapped host
    // memory from every CTA was measured first: 296 CTAs polling one PCIe address cost 25 % of the kernel and made a cancelled
    // launch drain no faster than a complete one.)
    int *h_cancel = nullptr;
    int *d_cancel = nullptr;
    unsigned long long *h_progress = nullptr;  // [0] progress poll, [1] [2] row-list counts

    Handles() = default;
    Handles(const Handles &) = delete;
    Handles &operator=(const Handles &) = delete;
    ~Handles()
    {
        if (stream) {
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
        if (poll_stream)
            cudaStreamDestroy(poll_stream);
        if (h_cancel)
            cudaFreeHost(h_cancel);
        if (d_cancel)
            cudaFree(d_cancel);
        if (h_progress)
            cudaFreeHost(h_progress);
    }
};

}  // namespace

struct mosaic_generator : Handles {
    int device = 0;
    std::string error;
    int sm_count = 0;

    // inputs
    int img_rows = 0, img_cols = 0;
    int main_lo = 0, main_hi = 0;  // rows of the main image that are resident on the device (sharded handles upload a band)
    DevBuf d_main_u8;
    int64_t n_lib = 0;
    int lib_size = 0;
    DevBuf d_lib_u8;
    // sharded setLibrary (mosaic_set_library_shard): the library is stored at lib_stored_size -- the cell size, or already the
    // detail size of step 0 when detail != 100 % (each rank resized its own slice before the NVLink all-gather)
    int lib_stored_size = 0;
    int64_t lib_capacity = 0;
    int diff_type = MOSAIC_RGB_EUCLIDEAN;
    int scheme = MOSAIC_SCHEME_NONE;
    bool quirk_faithful = true;
    Group group;
    bool have_group = false;
    std::vector<GridStep> grid;  // state in, best fits out
    int repeat_range = 0, repeat_addition = 0;
    bool keep_D = false;
    bool report_margins = false;
    int rank = 0, world = 1;
    // mirrored library tiles (mosaic_set_tile_flips): the candidate set is the O * N oriented library, orientation-major
    int flips = 0;
    bool lib_sharded = false;      // the library came from mosaic_set_library_shard (stored at the detail size, filled by the caller)
    DevBuf d_lib_oriented;         // [O][N][size][size][3] 8U, built by launch_orient_library
    int lib_oriented_flips = 0;    // flips d_lib_oriented holds (0 = stale: rebuilt by the next generate)
    int fits_flips = -1;           // flips of the generate whose slots the grid holds (-1: no generate since the grid was set)
    int64_t n_slots = 0;           // candidate slots O * N of the last generate (columns of D)
    // usage limit (mosaic_set_usage_limit): each image is chosen at most max_uses times per generate (0 = unlimited)
    int max_uses = 0;
    int cand_max_uses = 0;         // max_uses of the last mosaic_generate_candidates: its K and sorted prefixes were built for it
    int cap_last_step = -1;        // sharded selection: last step selected since `used` was reset (-1: none)
    DevBuf d_used;                 // [N] choices per source image so far in this generate

    mosaic_progress_fn progress_fn = nullptr;
    void *progress_user = nullptr;
    bool cancel_pushed = false;  // the device word already holds 1 (generate thread only)
    DevBuf d_progress;

    bool is_cancelled() const { return h_cancel && __atomic_load_n(h_cancel, __ATOMIC_RELAXED) != 0; }

    // products
    DevBuf d_lut;
    Workspace ws;
    std::vector<StepPlan> plans;
    std::vector<StepOut> out;
    int V_eff = 1;
    mosaic_timings timings{};

    int fail(int code, const std::string &msg)
    {
        error = msg;
        return code;
    }
};

namespace {

using G = mosaic_generator;

template <typename Fn>
int guard(G *g, const char *what, Fn &&fn)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    try {
        cudaError_t e = cudaSetDevice(g->device);
        if (e != cudaSuccess)
            throw Fail{MOSAIC_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e)};
        fn();
        g->error.clear();
        return MOSAIC_OK;
    } catch (const Fail &f) {
        cudaGetLastError();
        return g->fail(f.code, std::string(what) + ": " + f.msg);
    } catch (const std::bad_alloc &) {
        return g->fail(MOSAIC_ERR_OUT_OF_MEMORY, std::string(what) + ": host allocation failed");
    } catch (const std::exception &e) {
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, std::string(what) + ": " + e.what());
    } catch (...) {
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, std::string(what) + ": unexpected failure");
    }
}

// a shape's parameters, and its mask if mask_out is given (mask_capacity bytes)
int shape_to_c(const Shape &s, mosaic_cell_shape &c, uint8_t *mask_out, size_t mask_capacity)
{
    c.size = s.size;
    c.row_spacing = s.row_spacing;
    c.col_spacing = s.col_spacing;
    c.alt_row_spacing = s.alt_row_spacing;
    c.alt_col_spacing = s.alt_col_spacing;
    c.alt_row_offset = s.alt_row_offset;
    c.alt_col_offset = s.alt_col_offset;
    c.alt_col_flip_h = s.alt_col_flip_h;
    c.alt_col_flip_v = s.alt_col_flip_v;
    c.alt_row_flip_h = s.alt_row_flip_h;
    c.alt_row_flip_v = s.alt_row_flip_v;
    if (mask_out) {
        if (mask_capacity < s.mask.size())
            return MOSAIC_ERR_INVALID_ARGUMENT;
        memcpy(mask_out, s.mask.data(), s.mask.size());
    }
    return MOSAIC_OK;
}

Shape shape_params_only(const mosaic_cell_shape &c)
{
    Shape s;
    s.size = c.size;
    s.row_spacing = c.row_spacing;
    s.col_spacing = c.col_spacing;
    s.alt_row_spacing = c.alt_row_spacing;
    s.alt_col_spacing = c.alt_col_spacing;
    s.alt_row_offset = c.alt_row_offset;
    s.alt_col_offset = c.alt_col_offset;
    s.alt_col_flip_h = c.alt_col_flip_h != 0;
    s.alt_col_flip_v = c.alt_col_flip_v != 0;
    s.alt_row_flip_h = c.alt_row_flip_h != 0;
    s.alt_row_flip_v = c.alt_row_flip_v != 0;
    return s;
}

Shape shape_from_c(const mosaic_cell_shape &c, const uint8_t *mask, bool mask_as_stored)
{
    Shape s = shape_params_only(c);
    if (mask_as_stored)
        s.set_mask_as_stored(mask, c.size);
    else
        s.set_mask(mask, c.size);
    return s;
}

// the cell group of a shape and mask, its top cell resized to cell_size (> 0): MOSAIC_ERR_UNSUPPORTED when that resize is not
// supported, MOSAIC_ERR_INVALID_ARGUMENT when the group cannot be built; err says why
int build_group(const mosaic_cell_shape &shape, const uint8_t *mask, bool mask_as_stored, int cell_size, int detail_percent, int size_steps,
                Group &grp, std::string &err)
{
    Shape top = shape_from_c(shape, mask, mask_as_stored);
    if (cell_size > 0 && cell_size != top.size) {
        Shape r;
        if (!top.resized(cell_size, r, err))
            return MOSAIC_ERR_UNSUPPORTED;
        top = r;
    }
    return grp.build(top, detail_percent, size_steps, err) ? MOSAIC_OK : MOSAIC_ERR_INVALID_ARGUMENT;
}

// orientations of a flips mask (mosaic_set_tile_flips): the enabled subset of the codes {0, 1 = H, 2 = V, 3 = HV}, in increasing code
int orient_count(int flips) { return 1 << __builtin_popcount((unsigned)flips & 3u); }
int orient_code(int flips, int j)
{
    for (int c = 0; c < 4; ++c)
        if ((c & ~flips) == 0 && j-- == 0)
            return c;
    return -1;
}

// Phase timing without host synchronisation inside the pipeline: every begin/end pair records two CUDA events on the
// launching stream; the sums are read after the call's final stream synchronise.
struct PhaseClock {
    cudaStream_t s;
    std::vector<cudaEvent_t> ev;  // start, stop, start, stop, ...
    std::vector<int> phase;
    explicit PhaseClock(cudaStream_t st) : s(st) {}
    ~PhaseClock()
    {
        for (cudaEvent_t e : ev)
            cudaEventDestroy(e);
    }
    void begin(int ph)
    {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        ev.push_back(a);
        ev.push_back(b);
        phase.push_back(ph);
        cudaEventRecord(a, s);
    }
    void end() { cudaEventRecord(ev.back(), s); }
    double sum(int ph)  // call after the stream has been synchronised
    {
        double t = 0;
        for (size_t i = 0; i < phase.size(); ++i)
            if (phase[i] == ph) {
                float m = 0;
                cudaEventElapsedTime(&m, ev[2 * i], ev[2 * i + 1]);
                t += m;
            }
        return t;
    }
};

// ------------------------------------------------------------------ cancel plumbing

// copies a raised host flag into the device word (once per generate call)
void push_cancel(G *g)
{
    if (!g->cancel_pushed && g->is_cancelled()) {
        cudaMemcpyAsync(g->d_cancel, g->h_cancel, sizeof(int), cudaMemcpyHostToDevice, g->poll_stream);
        g->cancel_pushed = true;
    }
}

// cudaStreamSynchronize that keeps an eye on cancel(): spins on the stream like the runtime's own wait does, and forwards a
// cancel raised meanwhile to the device so that the running kernel stops scheduling work
void wait_stream(G *g, cudaStream_t st)
{
    cudaError_t e;
    while ((e = cudaStreamQuery(st)) == cudaErrorNotReady)
        push_cancel(g);
    if (e != cudaSuccess)
        throw Fail{MOSAIC_ERR_CUDA, std::string("stream wait: ") + cudaGetErrorString(e)};
}

// ------------------------------------------------------------------ planning

void check_ready(G *g)
{
    if (g->img_rows == 0)
        throw Fail{MOSAIC_ERR_NOT_READY, "no main image set"};
    if (g->n_lib == 0)
        throw Fail{MOSAIC_ERR_NOT_READY, "no library set (the reference would find no best fit)"};
    if (!g->have_group)
        throw Fail{MOSAIC_ERR_NOT_READY, "no cell group set"};
    if (g->grid.empty())
        throw Fail{MOSAIC_ERR_NOT_READY, "no grid state set"};
    if ((int)g->grid.size() > g->group.size_steps + 1)
        throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "grid state has more steps than the cell group"};
    if (g->lib_size != g->group.cells[0].size)
        throw Fail{MOSAIC_ERR_INVALID_ARGUMENT,
                   "library images must be at the cell size (the reference resizes them before setLibrary, MainWindow.cpp:575-581)"};
}

// the shard split of one size step: rank r of `world` owns rows [begin, end) of the n valid cells (raster order); every rank owns
// per_rank rows of the padded list, a whole number of cell tiles of the colour difference's kernel
void shard_split(int64_t n, int diff_type, int rank, int world, int64_t &per_rank, int64_t &begin, int64_t &end)
{
    const int tcb = tile_geom(diff_type == MOSAIC_CIEDE2000 ? kLayoutCiede : kLayoutEuclid).tcb;
    const int64_t n_tiles = (n + tcb - 1) / tcb;
    per_rank = std::max<int64_t>(1, (n_tiles + world - 1) / world) * tcb;
    begin = std::min<int64_t>(n, (int64_t)rank * per_rank);
    end = std::min<int64_t>(n, (int64_t)(rank + 1) * per_rank);
}

void make_plans(G *g)
{
    const Group &grp = g->group;
    g->plans.assign(g->grid.size(), StepPlan());
    int lib_ds = 0;
    for (size_t s = 0; s < g->grid.size(); ++s) {
        StepPlan &p = g->plans[s];
        const GridStep &gs = g->grid[s];
        p.rows = gs.rows;
        p.cols = gs.cols;
        p.S = grp.cells[s].size;
        p.ds = grp.detail_cells[s].size;
        // library size at this step: round(detail size) at step 0, round(0.5 * previous) afterwards
        // (PhotomosaicGeneratorBase.cpp:262, ImageUtility.cpp:97-98); must agree with the detail mask (SURVEY Q4)
        if (s == 0)  // (before a library is set -- mosaic_get_shard_rows -- it is taken to be at the cell size, as check_ready demands)
            lib_ds = (grp.detail != 1.0) ? p.ds : (g->lib_size ? g->lib_size : grp.cells[0].size);
        else {
            if (lib_ds % 2 != 0)
                throw Fail{MOSAIC_ERR_UNSUPPORTED, "odd library size at a size step (the reference indexes out of range here)"};
            lib_ds /= 2;
        }
        if (lib_ds != p.ds)
            throw Fail{MOSAIC_ERR_UNSUPPORTED,
                       "library size and detail mask size disagree at step " + std::to_string(s) +
                           " (the reference reads out of range for this cell size / detail combination)"};
        // integer ratios take OpenCV's resizeAreaFast_ arithmetic, everything else its fractional resizeArea_ (k = 0)
        p.k = (p.S % p.ds == 0) ? p.S / p.ds : 0;

        int gx, gy;
        grid_size(grp.cells[s], g->img_cols, g->img_rows, kPadGrid, gx, gy);
        if (gx != gs.cols || gy != gs.rows)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "grid state of step " + std::to_string(s) + " is " + std::to_string(gs.rows) + "x" +
                                                        std::to_string(gs.cols) + " but the cell group needs " + std::to_string(gy) + "x" +
                                                        std::to_string(gx)};
        p.row_first.assign(gs.rows, gs.cols);
        for (int y = 0; y < gs.rows; ++y) {
            int prev = -1;
            for (int x = 0; x < gs.cols; ++x)
                if (gs.v[(size_t)y * gs.cols + x] >= 0) {
                    if (prev < 0)
                        p.row_first[y] = x;
                    else
                        p.next_x[prev] = x;
                    prev = (int)p.cell_pos.size();
                    p.cell_pos.push_back(y * gs.cols + x);
                    p.next_x.push_back(gs.cols);
                }
        }
        // rank's block of cells: a contiguous raster range of the step's valid cells, cut at cell granularity on whole cell
        // tiles. Every rank owns the same number of rows `per` of the padded list (the last ranks may own fewer real cells), so
        // that rank r's candidates land at row r * per of one all-gathered buffer without any size exchange.
        shard_split((int64_t)p.cell_pos.size(), g->diff_type, g->rank, g->world, p.per_rank, p.cell_begin, p.cell_end);
    }
}

// main-image rows [lo, hi) that this rank's cells (all size steps) read; whole rows, so that the hue rotation keeps OpenCV's
// per-row SIMD / tail split
void needed_rows(const G *g, int &row_lo, int &row_hi)
{
    row_lo = g->img_rows;
    row_hi = 0;
    for (size_t s = 0; s < g->plans.size(); ++s) {
        const StepPlan &p = g->plans[s];
        const Shape &normal = g->group.cells[s];
        for (int64_t c = p.cell_begin; c < p.cell_end; ++c) {
            const int pos = p.cell_pos[c];
            const Rect r = rect_at(normal, pos % p.cols - kPadGrid, pos / p.cols - kPadGrid);
            row_lo = std::min(row_lo, std::max(r.y, 0));
            row_hi = std::max(row_hi, std::min(r.y + r.h, g->img_rows));
        }
    }
    if (row_hi < row_lo)
        row_lo = row_hi = 0;
}

// usage limit: valid cells of all steps, and E_s = the most images that can be exhausted before the last cell of step s
int64_t total_valid_cells(const G *g)
{
    int64_t n = 0;
    for (const StepPlan &p : g->plans)
        n += (int64_t)p.cell_pos.size();
    return n;
}

int64_t exhausted_bound(const G *g, size_t step)
{
    int64_t before = 0;
    for (size_t t = 0; t < step; ++t)
        before += (int64_t)g->plans[t].cell_pos.size();
    return std::max<int64_t>(0, before + (int64_t)g->plans[step].cell_pos.size() - 1) / g->max_uses;
}

// a cap below the number of cells would leave cells without any allowed image: refused before any work
void check_usage_limit(const G *g)
{
    const int64_t cells = total_valid_cells(g);
    if (g->max_uses > 0 && (int64_t)g->max_uses * g->n_lib < cells)
        throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "usage limit " + std::to_string(g->max_uses) + " x " + std::to_string(g->n_lib) +
                                                    " images = " + std::to_string((int64_t)g->max_uses * g->n_lib) +
                                                    " placements is less than the " + std::to_string(cells) +
                                                    " valid cells of all size steps"};
}

// usage limit: sorted prefixes. The first k0 = min(K, kPrefixMax) smallest (score, slot) pairs of each of n_rows rows of src ([n_rows][n]
// at row_stride) in ascending order: in place at the front of a candidate list (list_i: its slots, n = K, launch_topk output), or, for
// D rows (list_i == nullptr), into ws.prefix_score / ws.prefix_idx
void sort_prefixes(G *g, float *src, int row_stride, int n, int n_rows, int K, int *list_i, mosaic_timings &tm)
{
    if (n_rows == 0)
        return;
    const int k0 = std::min(K, kPrefixMax);
    cudaStream_t st = g->stream;
    g->ws.prefix_score.alloc((size_t)n_rows * k0 * sizeof(float), st);
    g->ws.prefix_idx.alloc((size_t)n_rows * k0 * sizeof(int), st);
    CU(launch_topk(src, row_stride, n, n_rows, k0, g->ws.prefix_score.as<float>(), g->ws.prefix_idx.as<int>(), st));
    CU(launch_sort_prefix(g->ws.prefix_score.as<float>(), g->ws.prefix_idx.as<int>(), n_rows, k0, list_i ? src : nullptr, list_i, K, st));
    tm.kernel_launches += 2;
}

// ------------------------------------------------------------------ progress and cancel

// progress(int) and cancel() of one generate call.
// cancel() is polled by the host before every phase it enqueues and by every CTA of the difference kernels when it starts (the
// reference polls per step, row and cell, CPUPhotomosaicGenerator.cpp:52, 66, 73). Work already enqueued drains first.
// progress(int): the reference emits after every grid position, cumulative, with weight 4^(steps-1-step)
// (CPUPhotomosaicGenerator.cpp:55, 87-88). Here the host polls the device's count of finished difference rows / tiles while the
// step runs and emits base + weight * floor(positions * done / total): every emitted value is one the reference emits too, the
// sequence is increasing and each step ends on the reference's own step total. Only when a callback is installed -- otherwise the
// pipeline never waits on the host before its final synchronise.
struct Progress {
    G *g;
    unsigned long long *d_done = nullptr;  // device count of the running step's finished rows / tiles (with a callback)
    int base = 0, last = 0, weight = 0, positions = 0;
    unsigned long long total = 1;

    explicit Progress(G *gen) : g(gen)
    {
        check_cancel();  // sticky like m_wasCanceled: a cancelled handle does nothing until mosaic_reset_cancel
        g->cancel_pushed = false;
        CU(cudaStreamSynchronize(g->poll_stream));  // no stale flag copy may land after the reset below
        CU(cudaMemsetAsync(g->d_cancel, 0, sizeof(int), g->stream));
        if (g->progress_fn) {
            g->d_progress.alloc(sizeof(unsigned long long), g->stream);
            d_done = g->d_progress.as<unsigned long long>();
        }
    }

    void check_cancel()
    {
        if (g->is_cancelled()) {
            push_cancel(g);
            cudaStreamSynchronize(g->stream);
            throw Fail{MOSAIC_ERR_CANCELLED, "cancelled"};
        }
    }

    // the difference sums of step s are enqueued next; the device counts `work` rows / tiles for them
    void start_step(size_t s, unsigned long long work)
    {
        weight = (int)pow(4.0, (double)(g->grid.size() - 1 - s));
        positions = g->plans[s].rows * g->plans[s].cols;
        total = work;
        last = base;
        check_cancel();
        if (d_done)
            CU(cudaMemsetAsync(d_done, 0, sizeof(unsigned long long), g->stream));
    }

    // waits for the stream; with a callback the host polls the device's count meanwhile and emits base + weight * floor(positions *
    // done / total)
    void wait()
    {
        if (!g->progress_fn) {
            wait_stream(g, g->stream);
            check_cancel();
            return;
        }
        cudaEvent_t done;
        CU(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
        cudaEventRecord(done, g->stream);
        while (cudaEventQuery(done) == cudaErrorNotReady) {
            if (cudaMemcpyAsync(g->h_progress, d_done, sizeof(unsigned long long), cudaMemcpyDeviceToHost, g->poll_stream) == cudaSuccess &&
                cudaStreamSynchronize(g->poll_stream) == cudaSuccess && !g->is_cancelled()) {
                const unsigned long long dn = std::min(*g->h_progress, total);
                const int v = base + weight * (int)((unsigned long long)positions * dn / total);
                if (v > last && v < base + weight * positions) {
                    last = v;
                    g->progress_fn(v, g->progress_user);  // may call mosaic_cancel(): the running kernel then drains
                }
            }
            push_cancel(g);
            std::this_thread::sleep_for(std::chrono::microseconds(500));
        }
        cudaEventDestroy(done);
        cudaGetLastError();
        check_cancel();
    }

    // the step's own total: the value the reference reaches after the step's last grid position
    void end_step()
    {
        if (g->progress_fn) {
            wait_stream(g, g->stream);
            check_cancel();
            g->progress_fn(base + weight * positions, g->progress_user);
        }
        base += weight * positions;
    }

    void finish()
    {
        wait_stream(g, g->stream);
        check_cancel();
    }
};

// ------------------------------------------------------------------ the pipeline

AreaTab upload_area_table(G *g, int ssize, int dsize, mosaic_timings &tm)
{
    const AreaTable t = make_area_table(ssize, dsize);
    Workspace &w = g->ws;
    cudaStream_t st = g->stream;
    w.tab_start.alloc(t.start.size() * sizeof(int), st);
    w.tab_si.alloc(t.si.size() * sizeof(int), st);
    w.tab_alpha.alloc(t.alpha.size() * sizeof(float), st);
    CU(cudaMemcpyAsync(w.tab_start.p, t.start.data(), t.start.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(w.tab_si.p, t.si.data(), t.si.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(w.tab_alpha.p, t.alpha.data(), t.alpha.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += (double)((t.start.size() + t.si.size()) * sizeof(int) + t.alpha.size() * sizeof(float));
    return AreaTab{w.tab_start.as<int>(), w.tab_si.as<int>(), w.tab_alpha.as<float>()};
}

// what one generate call decides once for all of its size steps
struct Run {
    bool candidates_only = false;
    std::vector<float> rotations;  // hue rotation of each colour variant that is actually compared (0 = the image itself)
    int V = 1, O = 1;              // colour variants, tile orientations
    int64_t N = 0;                 // candidate slots: the O orientations of the library images, orientation-major (slot = j * n + i)
    PackLayout layout = kLayoutEuclid;
    TileGeom tg{};
    int n_lib_tiles = 0, n_lib_pad = 0;
    bool is_lab = false, penalise = false, capped = false, fused_argmin = false, row_passes = false;
};

// Colour-scheme variants (ColourScheme.cpp:36-177): original + hue rotations. Reference quirk Q1: getCellAt builds the V cell Mats
// over ONE shared buffer (PhotomosaicGeneratorBase.cpp:310-312), so every variant holds the LAST rotation and the original image is
// never compared. faithful mode reproduces that with a single variant.
std::vector<float> colour_variants(const G *g)
{
    static const float kRot[6][3] = {{0, 0, 0}, {180, 0, 0}, {120, 240, 0}, {150, 210, 0}, {90, 180, 270}, {30, 60, 90}};
    static const int kNumRot[6] = {0, 1, 2, 2, 3, 3};
    if (g->scheme == MOSAIC_SCHEME_NONE)
        return {0.0f};
    if (g->quirk_faithful)
        return {kRot[g->scheme][kNumRot[g->scheme] - 1]};
    std::vector<float> rotations = {0.0f};
    for (int i = 0; i < kNumRot[g->scheme]; ++i)
        rotations.push_back(kRot[g->scheme][i]);
    return rotations;
}

// main image -> working space, every colour variant (PhotomosaicGeneratorBase.cpp:223-252)
void main_to_working_space(G *g, const Run &r, mosaic_timings &tm)
{
    cudaStream_t st = g->stream;
    DevBuf &d_main_f32 = g->ws.main_f32;
    const size_t n_main_px = (size_t)g->img_rows * g->img_cols;
    d_main_f32.alloc((size_t)r.V * n_main_px * 3 * sizeof(float), st);
    // a sharded rank only reads the image rows its own cells cover: convert just those
    int row_lo, row_hi;
    needed_rows(g, row_lo, row_hi);
    if (row_lo < g->main_lo || row_hi > g->main_hi)
        throw Fail{MOSAIC_ERR_NOT_READY, "main image rows " + std::to_string(row_lo) + ".." + std::to_string(row_hi) +
                                             " are needed by this shard but only " + std::to_string(g->main_lo) + ".." +
                                             std::to_string(g->main_hi) + " were uploaded (mosaic_set_main_image_rows)"};
    const int n_rows_conv = row_hi - row_lo;
    const size_t row_off_px = (size_t)row_lo * g->img_cols;
    for (int v = 0; v < r.V && n_rows_conv > 0; ++v) {
        const uint8_t *src = g->d_main_u8.as<uint8_t>() + row_off_px * 3;
        if (r.rotations[v] != 0.0f) {
            g->ws.main_var_u8.alloc(n_main_px * 3, st);
            CU(launch_hue_rotate(src, g->ws.main_var_u8.as<uint8_t>() + row_off_px * 3, n_rows_conv, g->img_cols, r.rotations[v], st));
            tm.kernel_launches++;
            src = g->ws.main_var_u8.as<uint8_t>() + row_off_px * 3;
        }
        CU(launch_to_working_space(src, (size_t)g->img_cols * 3, n_rows_conv, g->img_cols,
                                   d_main_f32.as<float>() + ((size_t)v * n_main_px + row_off_px) * 3, r.is_lab, g->d_lut.as<short4>(),
                                   nullptr, st));
        tm.kernel_launches++;
    }
}

// the library as the packers read it (prepare_library)
struct LibSource {
    const uint8_t *oriented;  // 8U at the stored size, every candidate slot
    const uint8_t *u8;        // 8U source of the fused packers: at ds, or at ds * fused_k
    int ds, fused_k;          // detail size of step 0, integer reduction the fused packers apply on the fly
    bool fused;               // a single size step: the colour conversion is fused into the tile packing
};

// library preparation: orientation (rebuilt only when the library or the flips changed), resize to the detail size of step 0
// (PhotomosaicGeneratorBase.cpp:255-290) and, unless the packers convert on the fly, working space (ws.lib_work)
LibSource prepare_library(G *g, const Run &r, mosaic_timings &tm)
{
    cudaStream_t st = g->stream;
    const int64_t N = r.N;
    LibSource lib{g->d_lib_u8.as<uint8_t>(), nullptr, g->lib_size, 1, g->grid.size() == 1};
    if (r.O > 1) {
        if (g->lib_oriented_flips != g->flips) {
            g->lib_oriented_flips = 0;
            g->d_lib_oriented.alloc((size_t)N * g->lib_size * g->lib_size * 3, st);
            CU(launch_orient_library(lib.oriented, g->d_lib_oriented.as<uint8_t>(), g->n_lib, g->lib_size, g->flips, st));
            tm.kernel_launches++;
            g->lib_oriented_flips = g->flips;
        }
        lib.oriented = g->d_lib_oriented.as<uint8_t>();
    }
    lib.u8 = lib.oriented;
    if (g->group.detail != 1.0) {
        lib.ds = g->plans[0].ds;
        if (g->lib_stored_size != g->lib_size) {
            // sharded setLibrary already resized every slice to the detail size (mosaic_set_library_shard)
            if (g->lib_stored_size != lib.ds)
                throw Fail{MOSAIC_ERR_NOT_READY, "the library was uploaded for another detail size: call mosaic_set_library_shard "
                                                 "again after changing the cell group"};
        } else if (lib.fused && g->lib_size % lib.ds == 0) {
            // integer ratio and a single size step: the packers reduce on the fly, the resized 8U copy is never written
            lib.fused_k = g->lib_size / lib.ds;
        } else {
            DevBuf &small = g->ws.lib_small;
            small.alloc((size_t)N * lib.ds * lib.ds * 3, st);
            if (g->lib_size % lib.ds == 0) {
                CU(launch_area_u8(lib.oriented, small.as<uint8_t>(), N, g->lib_size, g->lib_size / lib.ds, st));
            } else {
                const AreaTab tab = upload_area_table(g, g->lib_size, lib.ds, tm);
                CU(launch_area_general_u8(lib.oriented, small.as<uint8_t>(), N, g->lib_size, lib.ds, tab, st));
            }
            tm.kernel_launches++;
            lib.u8 = small.as<uint8_t>();
        }
    } else if (g->lib_stored_size != g->lib_size) {
        throw Fail{MOSAIC_ERR_NOT_READY, "the library was uploaded at a detail size but the cell group now has detail 100 %"};
    }
    // a single size step: the colour conversion is fused into the tile-packing kernel (straight from the 8U library), the f32
    // working-space copy is only materialised when a later step has to halve it
    if (!lib.fused) {
        g->ws.lib_work.alloc((size_t)N * lib.ds * lib.ds * 3 * sizeof(float), st);
        // the library is one tall image of N * ds rows
        CU(launch_to_working_space(lib.u8, (size_t)lib.ds * 3, (int)std::min<int64_t>(N * lib.ds, INT32_MAX), lib.ds,
                                   g->ws.lib_work.as<float>(), r.is_lab, g->d_lut.as<short4>(), nullptr, st));
        tm.kernel_launches++;
    }
    return lib;
}

// one size step's sizes (prepare_step) and work plan (plan_step)
struct StepWork {
    int64_t n_local = 0, n_all = 0;                          // this rank's valid cells, all ranks' valid cells
    int n_rows_local = 0, n_cell_tiles = 0, n_rows_pad = 0;  // this rank's difference rows (cell x variant), in whole cell tiles
    bool need_D = false;
    int64_t k_need = 1;  // top-K count of the selection
    bool via_topk = false, prune = false;
    int M = 0;  // pruning: candidates of the first segment
    int n_segs = 1, seg_chunks = 0, col_cells = kColumnCells;
    unsigned long long prog_total = 1;  // rows / tiles the difference kernels count as done
};

// per step: the active pixel list, library packing, cell descriptors with pixel-diff counts, and cell extraction
void prepare_step(G *g, const Run &r, const LibSource &lib, size_t s, StepWork &w, mosaic_timings &tm)
{
    cudaStream_t st = g->stream;
    StepPlan &p = g->plans[s];
    const Shape &normal = g->group.cells[s];
    const Shape &dshape = g->group.detail_cells[s];
    const int ds = p.ds, P = ds * ds, V = r.V;
    const int64_t N = r.N;
    const TileGeom &tg = r.tg;
    Workspace &d = g->ws;
    if (s > 0) {
        // halve the working-space library (CPUPhotomosaicGenerator.cpp:95-99)
        d.lib_half.alloc((size_t)N * P * 3 * sizeof(float), st);
        CU(launch_area_f32(d.lib_work.as<float>(), d.lib_half.as<float>(), N, ds * 2, 2, st));
        tm.kernel_launches++;
        std::swap(d.lib_work, d.lib_half);
    }

    // active pixel list: union of the flipped detail masks THAT OCCUR among the step's valid cells (all ranks' cells, so that
    // every world size sums in the same order), raster order. A shape without flips (Puzzle.mcs) keeps its own 72 % of the
    // square instead of the ~100 % the union of all four flips would cover.
    const std::vector<uint8_t> m4 = dshape.masks4();
    bool flip_used[4] = {false, false, false, false};
    for (int pos : p.cell_pos)
        flip_used[flip_at(normal, pos % p.cols - kPadGrid, pos / p.cols - kPadGrid)] = true;
    std::vector<int> pix;
    pix.reserve(P);
    for (int i = 0; i < P; ++i) {
        bool on = false;
        for (int f = 0; f < 4; ++f)
            on = on || (flip_used[f] && m4[(size_t)f * P + i]);
        if (on)
            pix.push_back(i);
    }
    p.n_active = (int)pix.size();
    p.n_chunks = std::max(1, (p.n_active + tg.kp - 1) / tg.kp);
    d.pix_list.alloc(std::max<size_t>(pix.size(), 1) * sizeof(int), st);
    CU(cudaMemcpyAsync(d.pix_list.p, pix.data(), pix.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    d.masks4.alloc(m4.size(), st);
    CU(cudaMemcpyAsync(d.masks4.p, m4.data(), m4.size(), cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += (double)(pix.size() * sizeof(int) + m4.size());

    // library tiles
    d.lib_packed.alloc((size_t)r.n_lib_tiles * p.n_chunks * tg.lib_block, st);
    const int *perm = r.row_passes ? d.perm.as<int>() : nullptr;
    if (lib.fused && r.layout == kLayoutCiede)
        CU(launch_pack_library_ciede(lib.u8, true, d.lib_packed.p, N, P, d.pix_list.as<int>(), p.n_active, p.n_chunks, r.n_lib_tiles,
                                     g->d_lut.as<short4>(), st, ds * lib.fused_k, lib.fused_k, perm));
    else if (lib.fused)
        CU(launch_pack_library_euclid_u8(lib.u8, ds * lib.fused_k, lib.fused_k, r.is_lab, d.lib_packed.p, N, P, d.pix_list.as<int>(),
                                         p.n_active, p.n_chunks, r.n_lib_tiles, g->d_lut.as<short4>(), st));
    else
        CU(launch_pack_library(d.lib_work.as<float>(), d.lib_packed.p, N, P, d.pix_list.as<int>(), p.n_active, p.n_chunks, r.n_lib_tiles,
                               r.layout, st, perm));
    tm.kernel_launches++;

    // cell descriptors of this rank's cells (getCellAt, PhotomosaicGeneratorBase.cpp:293-329)
    w.n_local = p.cell_end - p.cell_begin;
    w.n_all = (int64_t)p.cell_pos.size();
    std::vector<CellDesc> descs((size_t)w.n_local * V);
    // mask pixel counts through integral images (for the pixel-diff statistics)
    std::vector<std::vector<int>> integ(4, std::vector<int>((size_t)(ds + 1) * (ds + 1), 0));
    for (int f = 0; f < 4; ++f)
        for (int y = 0; y < ds; ++y)
            for (int x = 0; x < ds; ++x)
                integ[f][(size_t)(y + 1) * (ds + 1) + x + 1] = (m4[((size_t)f * ds + y) * ds + x] != 0) + integ[f][(size_t)y * (ds + 1) + x + 1] +
                                                              integ[f][(size_t)(y + 1) * (ds + 1) + x] - integ[f][(size_t)y * (ds + 1) + x];
    for (int64_t c = 0; c < w.n_all; ++c) {
        const int pos = p.cell_pos[c];
        const int x = pos % p.cols - kPadGrid, y = pos / p.cols - kPadGrid;
        const Rect rc = rect_at(normal, x, y);
        const Rect b = detail_bound(normal, ds, g->group.detail, x, y, g->img_cols, g->img_rows);
        const int flip = flip_at(normal, x, y);
        const std::vector<int> &I = integ[flip];
        const int act = I[(size_t)(b.y + b.h) * (ds + 1) + b.x + b.w] - I[(size_t)b.y * (ds + 1) + b.x + b.w] -
                        I[(size_t)(b.y + b.h) * (ds + 1) + b.x] + I[(size_t)b.y * (ds + 1) + b.x];
        p.pixel_diffs += (double)act * N * V;
        p.pixel_diffs_nominal += (double)P * N * V;
        if (c >= p.cell_begin && c < p.cell_end)
            for (int v = 0; v < V; ++v)
                descs[(size_t)(c - p.cell_begin) * V + v] = CellDesc{rc.x, rc.y, b.x, b.y, b.w, b.h, flip, v};
    }
    tm.pixel_diffs += p.pixel_diffs;
    tm.pixel_diffs_nominal += p.pixel_diffs_nominal;

    w.n_rows_local = (int)(w.n_local * V);
    w.n_cell_tiles = (w.n_rows_local + tg.tcb - 1) / tg.tcb;
    w.n_rows_pad = w.n_cell_tiles * tg.tcb;
    d.descs.alloc(std::max<size_t>(descs.size(), 1) * sizeof(CellDesc), st);
    CU(cudaMemcpyAsync(d.descs.p, descs.data(), descs.size() * sizeof(CellDesc), cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += (double)(descs.size() * sizeof(CellDesc));
    d.cells_packed.alloc((size_t)std::max(w.n_cell_tiles, 1) * p.n_chunks * tg.cell_block, st);
    AreaTab cell_tab{nullptr, nullptr, nullptr};
    if (p.k == 0)
        cell_tab = upload_area_table(g, p.S, p.ds, tm);
    CU(launch_extract_cells(d.main_f32.as<float>(), g->img_rows, g->img_cols, d.descs.as<CellDesc>(), w.n_rows_local, p.S, p.ds, p.k,
                            cell_tab, d.masks4.as<uint8_t>(), d.pix_list.as<int>(), p.n_active, p.n_chunks, d.cells_packed.p, r.layout,
                            st));
    tm.kernel_launches++;
}

// the step's work plan: the top-K count of the selection, pruning, and the passes of the difference sums. MM_SPLITK (segments) and
// MM_SB_A (cell tiles per column) override the pass shapes for tuning.
void plan_step(const G *g, const Run &r, size_t s, StepWork &w)
{
    const StepPlan &p = g->plans[s];
    const int64_t N = r.N;
    w.need_D = !r.fused_argmin || g->keep_D;
    // top-K count of the selection; when D only feeds top-K (and need not be complete), pairs that cannot be among the k_need
    // smallest are pruned (launch_prune_threshold).
    // Grouped K: the window holds W = 2r^2 + 2r cells, so at most W distinct images and, as the O orientations of an image share
    // its count, at most O * W of the O * N slots carry a penalty. Among the O * W + 1 smallest (score, slot) pairs at least one
    // slot u is unpenalised. The penalised winner w has D[w] + A * count >= D[w] and must beat or tie u, so D[w] <= D[u], and at
    // D[w] == D[u] the lower slot wins: (D[w], w) <= (D[u], u), so w is among the O * W + 1 smallest. The runner-up is among the
    // O * W + 2 smallest by the same argument with two unpenalised slots. O = 1 is SURVEY.md 8e's bound.
    // With a usage limit at most E_s images are exhausted before the step's last cell, so O * E_s more slots may be excluded and
    // the same argument holds with O * (W + E_s) (DESIGN.md 4.4).
    const int64_t rr = g->repeat_range;
    const int64_t n_win = 2 * rr * rr + 2 * rr;
    const int64_t n_excl = r.capped ? r.O * exhausted_bound(g, s) : 0;
    w.k_need = r.candidates_only ? ((r.penalise || r.capped) ? std::min<int64_t>(N, r.O * n_win + n_excl + 1) : 1)
                                 : std::min<int64_t>(N, r.O * n_win + n_excl + 1 + (g->report_margins ? 1 : 0));
    w.via_topk = r.candidates_only || ((r.penalise || r.capped) && w.k_need * 4 <= N);
    w.M = (int)std::min<int64_t>(N, w.k_need + w.k_need / 4 + 8);  // candidates of the first segment: 1.25 k_need + 8
    w.prune = r.row_passes && w.via_topk && r.V == 1 && !g->keep_D && w.k_need * 4 <= N && w.M <= 4096 && w.n_rows_local > 0;
    // segments: 8 (or MM_SPLITK) passes over the pixel axis, chunk-aligned
    w.n_segs = 1;
    w.seg_chunks = p.n_chunks;
    if (r.row_passes) {
        const char *ev = getenv("MM_SPLITK");
        const int want = ev && atoi(ev) > 0 ? atoi(ev) : kPruneSegments;
        w.seg_chunks = (p.n_chunks + std::min(want, p.n_chunks) - 1) / std::min(want, p.n_chunks);
        w.n_segs = (p.n_chunks + w.seg_chunks - 1) / w.seg_chunks;
        if (const char *ea = getenv("MM_SB_A"))
            w.col_cells = std::max(32, std::min(1024, atoi(ea) * MM_TCB / 32 * 32));
    }
    w.prog_total = r.row_passes ? (unsigned long long)std::max(w.n_rows_local, 1) * r.n_lib_tiles * w.n_segs
                                : (unsigned long long)std::max(w.n_cell_tiles, 1) * r.n_lib_tiles;
}

// the difference sums of step s: segment passes over row work lists (with or without exact pruning), diff_sum, or diff_euclid.
// Returns the executed share of the step's (row, chunk) work.
double difference_sums(G *g, const Run &r, size_t s, const StepWork &w, Progress &prog, mosaic_timings &tm)
{
    cudaStream_t st = g->stream;
    const StepPlan &p = g->plans[s];
    Workspace &d = g->ws;
    StepOut &o = g->out[s];
    DevBuf &D = o.D;
    if (w.need_D) {
        D.alloc((size_t)std::max(w.n_rows_pad, 1) * r.n_lib_pad * sizeof(float), st);
        o.have_D = true;
    }
    if (r.fused_argmin) {
        d.best_key.alloc((size_t)std::max(w.n_rows_pad, 1) * sizeof(unsigned long long), st);
        CU(launch_fill_u64(d.best_key.as<unsigned long long>(), (size_t)std::max(w.n_rows_pad, 1), ~0ull, st));
        tm.kernel_launches++;
    }
    prog.start_step(s, w.prog_total);
    if (!r.row_passes || w.n_rows_local == 0) {
        float *Dp = w.need_D ? D.as<float>() : nullptr;
        unsigned long long *keys = r.fused_argmin ? d.best_key.as<unsigned long long>() : nullptr;
        if (r.layout == kLayoutCiede)
            CU(launch_diff_sum(MM_DIFF_CIEDE2000, d.cells_packed.p, d.lib_packed.p, Dp, keys, w.n_cell_tiles, r.n_lib_tiles, p.n_chunks,
                               (int)r.N, w.n_rows_local, st, g->d_cancel, prog.d_done));
        else
            CU(launch_diff_euclid(d.cells_packed.p, d.lib_packed.p, Dp, keys, w.n_cell_tiles, r.n_lib_tiles, p.n_chunks, (int)r.N,
                                  w.n_rows_local, st, g->d_cancel, prog.d_done));
        tm.kernel_launches += w.n_cell_tiles > 0;
        return 1.0;
    }

    CU(cudaMemsetAsync(D.p, 0, D.bytes, st));
    const int n_cols = (w.n_rows_local + w.col_cells - 1) / w.col_cells;
    RowList rows{nullptr, nullptr, nullptr, n_cols * r.n_lib_tiles, w.col_cells};
    d.row_cells.alloc((size_t)rows.n_buckets * w.col_cells * sizeof(int), st);
    d.row_count.alloc((size_t)rows.n_buckets * sizeof(int), st);
    d.row_groups.alloc((size_t)(rows.n_buckets + 1) * sizeof(int), st);
    d.list_scratch.alloc(list_rows_scratch_bytes(rows.n_buckets), st);
    d.listed.alloc(sizeof(unsigned long long), st);
    rows.cells = d.row_cells.as<int>();
    rows.count = d.row_count.as<int>();
    rows.groups = d.row_groups.as<int>();
    const int *perm = d.perm.as<int>();
    uint8_t *state = nullptr;
    if (w.prune) {
        d.row_state.alloc((size_t)w.n_rows_local * r.n_lib_tiles, st);
        CU(cudaMemsetAsync(d.row_state.p, kRowActive, d.row_state.bytes, st));
        state = d.row_state.as<uint8_t>();
    }
    double units = 0;  // rows x chunks evaluated
    int n_groups = 0;
    auto list = [&](uint8_t *st8, int want, const float *T, const float *R, int segs_left) {
        CU(cudaMemsetAsync(d.listed.p, 0, sizeof(unsigned long long), st));
        CU(launch_list_rows(D.as<float>(), r.n_lib_pad, (int)r.N, w.n_rows_local, r.n_lib_tiles, st8, want, T, R, perm, segs_left, rows,
                            d.list_scratch.p, d.list_scratch.bytes, d.listed.as<unsigned long long>(), prog.d_done, st));
        CU(cudaMemcpyAsync(g->h_progress + 1, rows.groups + rows.n_buckets, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(g->h_progress + 2, d.listed.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        tm.kernel_launches += 2;
        prog.wait();  // the pass size is needed on the host to size the next launch
        n_groups = (int)*reinterpret_cast<const int *>(g->h_progress + 1);
        return (double)g->h_progress[2];
    };
    auto pass = [&](int seg, double n_listed) {
        const int k0 = seg * w.seg_chunks, nk = std::min(p.n_chunks, k0 + w.seg_chunks) - k0;
        CU(launch_diff_rows(d.cells_packed.p, d.lib_packed.p, D.as<float>(), n_groups, r.n_lib_tiles, p.n_chunks, k0, nk, rows, perm, st,
                            g->d_cancel, prog.d_done));
        tm.kernel_launches += n_groups > 0;
        units += n_listed * nk;
    };
    double n_listed = list(nullptr, kRowActive, nullptr, nullptr, 0);  // every row
    if (!w.prune) {
        for (int seg = 0; seg < w.n_segs; ++seg)
            pass(seg, n_listed);
    } else {
        pass(0, n_listed);
        // R[s - 1][cell][slot]: lower bound of what segments s .. n_segs - 1 add to a pair (launch_prune_bound; its rounding argument
        // holds up to 168 segments), and the candidates' ranking D + R[0]
        const float *rank = D.as<float>();
        const float *rest = nullptr;
        const size_t plane = (size_t)w.n_rows_local * r.n_lib_pad;
        if (w.n_segs > 1 && w.n_segs <= 168) {
            const int n_blocks = p.n_chunks * (MM_KP / MM_BB);
            d.lib_stats.alloc((size_t)n_blocks * r.n_lib_pad * sizeof(float4), st);
            d.cell_stats.alloc((size_t)w.n_rows_local * n_blocks * sizeof(float4), st);
            d.prune_rest.alloc((w.n_segs - 1) * plane * sizeof(float), st);
            d.prune_rank.alloc(plane * sizeof(float), st);
            CU(launch_block_stats(d.lib_packed.p, r.n_lib_tiles, d.cells_packed.p, w.n_rows_local, p.n_chunks, d.lib_stats.as<float4>(),
                                  d.cell_stats.as<float4>(), st));
            CU(launch_prune_bound(d.lib_stats.as<float4>(), d.cell_stats.as<float4>(), w.n_rows_local, r.n_lib_pad, n_blocks,
                                  w.seg_chunks * (MM_KP / MM_BB), w.n_segs, d.prune_rest.as<float>(), D.as<float>(), perm,
                                  d.prune_rank.as<float>(), st));
            tm.kernel_launches += 2;
            rank = d.prune_rank.as<float>();
            rest = d.prune_rest.as<float>();
        }
        // candidates = the M smallest of pass 0's partial sum + R[0]; their tiles are completed first, T[cell] = the k_need-th
        // smallest of their complete sums, and every later pass lists only the rows that still have a pair with partial sum + the
        // bound of the segments not yet summed <= T
        d.prune_score.alloc((size_t)w.n_rows_local * w.M * sizeof(float), st);
        d.prune_idx.alloc((size_t)w.n_rows_local * w.M * sizeof(int), st);
        d.threshold.alloc((size_t)w.n_rows_local * sizeof(float), st);
        CU(launch_topk(rank, r.n_lib_pad, (int)r.N, w.n_rows_local, w.M, d.prune_score.as<float>(), d.prune_idx.as<int>(), st));
        CU(launch_prune_threshold(D.as<float>(), r.n_lib_pad, d.prune_idx.as<int>(), w.n_rows_local, w.M, (int)w.k_need,
                                  d.inv_perm.as<int>(), r.n_lib_tiles, state, nullptr, true, st));
        tm.kernel_launches += 2;
        if (w.n_segs > 1) {
            n_listed = list(state, kRowComplete, nullptr, nullptr, 0);
            for (int seg = 1; seg < w.n_segs; ++seg)
                pass(seg, n_listed);
        }
        CU(launch_prune_threshold(D.as<float>(), r.n_lib_pad, d.prune_idx.as<int>(), w.n_rows_local, w.M, (int)w.k_need,
                                  d.inv_perm.as<int>(), r.n_lib_tiles, state, d.threshold.as<float>(), false, st));
        tm.kernel_launches++;
        for (int seg = 1; seg < w.n_segs; ++seg) {
            n_listed = list(state, kRowActive, d.threshold.as<float>(), rest ? rest + (size_t)(seg - 1) * plane : nullptr, w.n_segs - seg);
            pass(seg, n_listed);
        }
    }
    return units / ((double)w.n_rows_local * r.n_lib_tiles * p.n_chunks);
}

// the candidate source of select_step: every cell's full row -- its D row (idx == nullptr: entry j is slot j) or its top-K list --
// and, for the capped selection, its sorted prefix of k0 entries; rows_per_block > 0 addresses all-gathered per-rank blocks
// (kernels.h: launch_select)
struct Candidates {
    const float *scores = nullptr;
    const int *idx = nullptr;
    int M = 0, M_stride = 0;
    const float *pscores = nullptr;
    const int *pidx = nullptr;
    int k0 = 0, p_stride = 0;
    long long rows_per_block = 0, block_stride = 0;
};

// selection of step s, for mosaic_generate and the sharded selection alike: uploads the selection state, resets `used` when a capped
// generate starts (it carries across the generate's steps), selects every valid cell and enqueues the copy of the grid back to the
// host. The cells take the fused argmin's best keys, or select / select_capped scans the Candidates that candidates() enqueues
// after the uploads (so that the host's pageable copies overlap its launches). launch_clock, if given, times the selection launch
// alone.
template <typename Source>
void select_step(G *g, size_t s, const unsigned long long *keys, Source &&candidates, int max_uses, bool restart_used, float *margins,
                 PhaseClock *launch_clock, mosaic_timings &tm)
{
    const StepPlan &p = g->plans[s];
    GridStep &gs = g->grid[s];
    Workspace &w = g->ws;
    cudaStream_t st = g->stream;
    const int n_all = (int)p.cell_pos.size();
    w.grid.alloc(gs.v.size() * sizeof(long long), st);
    CU(cudaMemcpyAsync(w.grid.p, gs.v.data(), gs.v.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    w.pos.alloc(std::max<size_t>(p.cell_pos.size(), 1) * sizeof(int), st);
    CU(cudaMemcpyAsync(w.pos.p, p.cell_pos.data(), p.cell_pos.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += (double)(gs.v.size() * sizeof(long long) + p.cell_pos.size() * sizeof(int));
    if (keys) {
        CU(launch_keys_to_grid(keys, w.pos.as<int>(), w.grid.as<long long>(), n_all, nullptr, st));
    } else {
        w.next.alloc(std::max<size_t>(p.next_x.size(), 1) * sizeof(int), st);
        CU(cudaMemcpyAsync(w.next.p, p.next_x.data(), p.next_x.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        w.prog.alloc((size_t)p.rows * sizeof(int), st);
        CU(cudaMemcpyAsync(w.prog.p, p.row_first.data(), (size_t)p.rows * sizeof(int), cudaMemcpyHostToDevice, st));
        const int n_ctas = std::max(1, std::min(n_all, select_max_ctas(g->device)));
        w.counts.alloc((size_t)n_ctas * g->n_lib * sizeof(int), st);  // per source image: candidates are slots of g->flips
        CU(cudaMemsetAsync(w.counts.p, 0, w.counts.bytes, st));
        const Candidates c = candidates();
        if (max_uses > 0 && restart_used) {
            g->d_used.alloc((size_t)g->n_lib * sizeof(int), st);
            CU(cudaMemsetAsync(g->d_used.p, 0, g->d_used.bytes, st));
        }
        if (launch_clock)
            launch_clock->begin(0);
        if (max_uses > 0)
            CU(launch_select_capped(w.grid.as<long long>(), w.pos.as<int>(), n_all, p.rows, p.cols, c.scores, c.idx, c.M, c.M_stride,
                                    c.pscores, c.pidx, c.k0, c.p_stride, (int)g->n_lib, g->repeat_range, g->repeat_addition, max_uses,
                                    w.counts.as<int>(), g->d_used.as<int>(), margins, st, c.rows_per_block, c.block_stride));
        else
            CU(launch_select(w.grid.as<long long>(), w.pos.as<int>(), w.next.as<int>(), n_all, p.rows, p.cols, c.scores, c.idx, c.M,
                             c.M_stride, (int)g->n_lib, g->repeat_range, g->repeat_addition, w.prog.as<int>(), w.counts.as<int>(), n_ctas,
                             margins, st, c.rows_per_block, c.block_stride));
        if (launch_clock)
            launch_clock->end();
    }
    tm.kernel_launches += n_all > 0;
    CU(cudaMemcpyAsync(gs.v.data(), w.grid.p, gs.v.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
    tm.d2h_bytes += (double)(gs.v.size() * sizeof(long long));
}

// the K smallest (score, slot) pairs of n_rows rows of D into the step's candidate block of `rows` rows; under a usage limit every
// row's first min(K, kPrefixMax) entries become its sorted prefix. Returns the block's slots.
int *fill_candidates(G *g, StepOut &o, float *D, int row_stride, int N, int64_t rows, int64_t n_rows, int K, bool capped,
                     mosaic_timings &tm)
{
    const size_t half = (size_t)std::max<int64_t>(rows, 1) * K;
    o.cand.alloc(half * (sizeof(float) + sizeof(int)), g->stream);
    float *cs = o.cand.as<float>();
    int *ci = reinterpret_cast<int *>(cs + half);
    CU(launch_topk(D, row_stride, N, (int)n_rows, K, cs, ci, g->stream));
    tm.kernel_launches += n_rows > 0;
    if (capped)  // the capped selection reads every row's sorted prefix first
        sort_prefixes(g, cs, K, K, (int)n_rows, K, ci, tm);
    return ci;
}

// ---- Repeats + FindLowest: the candidate block of this rank's cells (mosaic_generate_candidates), or the step's best fits
void select_phase(G *g, const Run &r, size_t s, const StepWork &w, mosaic_timings &tm)
{
    const StepPlan &p = g->plans[s];
    StepOut &o = g->out[s];
    float *D = o.D.as<float>();
    const int D_stride = r.V * r.n_lib_pad, K = (int)w.k_need;
    if (r.V > 1 && w.need_D) {
        CU(launch_min_variants(D, (int)w.n_local, r.V, r.n_lib_pad, g->stream));
        tm.kernel_launches++;
    }
    if (r.candidates_only) {
        // one block per rank, per_rank rows: every rank's block has the same size, so ONE all-gather assembles the candidates of
        // the whole step (rank r's rows start at r * per_rank)
        o.cand_k = K;
        fill_candidates(g, o, D, D_stride, (int)r.N, p.per_rank, w.n_local, K, r.capped, tm);
        return;
    }
    float *margins = nullptr;
    if (g->report_margins && !r.fused_argmin) {
        o.margins.alloc(std::max<size_t>((size_t)w.n_all, 1) * 2 * sizeof(float), g->stream);
        margins = o.margins.as<float>();
        o.have_margins = true;
    }
    auto candidates = [&] {
        Candidates c;
        c.scores = D;
        c.M = (int)r.N;
        c.M_stride = D_stride;
        // With a penalty the winner (and the runner-up) lies among the K (+1) smallest unpenalised scores (SURVEY.md 8e), so the
        // selection scans candidate lists instead of whole D rows when that is shorter.
        if (w.via_topk) {
            c.idx = fill_candidates(g, o, D, D_stride, (int)r.N, w.n_all, w.n_all, K, r.capped, tm);
            tm.kernel_launches += w.n_all == 0;  // a generate counts its top-K launch even for a step without cells
            c.scores = o.cand.as<float>();
            c.M = c.M_stride = K;
        } else if (r.capped) {
            sort_prefixes(g, D, D_stride, (int)r.N, (int)w.n_all, K, nullptr, tm);
        }
        if (r.capped) {
            // sequential capped selection: every cell's sorted prefix first, its full row (K list or D row) as the fallback
            c.k0 = std::min(K, kPrefixMax);
            c.pscores = w.via_topk ? c.scores : g->ws.prefix_score.as<float>();
            c.pidx = w.via_topk ? c.idx : g->ws.prefix_idx.as<int>();
            c.p_stride = w.via_topk ? K : c.k0;
        }
        return c;
    };
    select_step(g, s, r.fused_argmin ? g->ws.best_key.as<unsigned long long>() : nullptr, candidates, g->max_uses, s == 0, margins,
                nullptr, tm);
}

void run_pipeline(G *g, bool candidates_only)
{
    check_ready(g);
    if (g->is_cancelled())  // sticky like m_wasCanceled (never reset by the reference): nothing runs until mosaic_reset_cancel
        throw Fail{MOSAIC_ERR_CANCELLED, "cancelled"};
    make_plans(g);
    check_usage_limit(g);
    cudaStream_t st = g->stream;
    const auto t_host0 = std::chrono::steady_clock::now();
    g->timings = mosaic_timings{};
    mosaic_timings &tm = g->timings;
    const size_t n_steps = g->grid.size();
    Run r;
    r.candidates_only = candidates_only;
    r.rotations = colour_variants(g);
    r.V = g->V_eff = (int)r.rotations.size();
    // candidate slots: the O orientations of the N library images, orientation-major (slot = j * N + i); every stage up to D runs
    // on the oriented library as if it were the library itself
    r.O = orient_count(g->flips);
    if (r.O > 1 && g->lib_sharded)
        throw Fail{MOSAIC_ERR_UNSUPPORTED, "tile flips need the library from mosaic_set_library: a library stored at the detail size "
                                           "cannot be re-oriented exactly"};
    r.N = g->n_lib * r.O;
    if (r.N * g->lib_size > INT32_MAX)
        throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large with tile flips (orientations * n * size must fit 31 bits)"};
    g->n_slots = r.N;
    if (!candidates_only)
        g->fits_flips = g->flips;
    r.is_lab = g->diff_type != MOSAIC_RGB_EUCLIDEAN;
    r.layout = g->diff_type == MOSAIC_CIEDE2000 ? kLayoutCiede : kLayoutEuclid;
    r.tg = tile_geom(r.layout);
    r.n_lib_tiles = (int)((r.N + r.tg.tnb - 1) / r.tg.tnb);
    r.n_lib_pad = r.n_lib_tiles * r.tg.tnb;
    r.penalise = g->repeat_range > 0 && g->repeat_addition != 0;
    r.capped = g->max_uses > 0;
    r.fused_argmin = !r.penalise && !r.capped && r.V == 1 && !candidates_only && g->world == 1 && !g->report_margins;
    // CIEDE2000 steps that need D run as segment passes over row work lists; the library tiles then hold the library in colour
    // order (kernels.h: RowList), which is what lets exact pruning drop whole tiles of a cell
    r.row_passes = r.layout == kLayoutCiede && !r.fused_argmin;
    PhaseClock clock(st);
    enum { kPre = 0, kDiff = 1, kSel = 2 };

    if (!g->d_lut.p) {
        const std::vector<int16_t> lut4 = expand_lab_lut(mm_lab_lut_s16);
        g->d_lut.alloc(lut4.size() * sizeof(int16_t), st);
        CU(cudaMemcpyAsync(g->d_lut.p, lut4.data(), g->d_lut.bytes, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));  // lut4 is a local
        tm.h2d_bytes += (double)g->d_lut.bytes;
    }

    clock.begin(kPre);
    main_to_working_space(g, r, tm);
    const LibSource lib = prepare_library(g, r, tm);
    clock.end();

    if (g->out.size() != n_steps) {
        g->out.clear();
        g->out.resize(n_steps);
    }
    for (StepOut &o : g->out) {
        o.have_D = o.have_margins = false;
        o.cand_k = 0;
    }
    if (candidates_only) {
        g->cand_max_uses = g->max_uses;
        g->cap_last_step = -1;
    }
    if (r.row_passes) {
        g->ws.perm.alloc((size_t)r.n_lib_pad * sizeof(int), st);
        g->ws.inv_perm.alloc((size_t)r.n_lib_pad * sizeof(int), st);
        g->ws.order_scratch.alloc(library_order_scratch_bytes(r.N), st);
        CU(launch_library_order(lib.oriented, g->lib_stored_size, r.N, r.n_lib_pad, g->ws.perm.as<int>(), g->ws.inv_perm.as<int>(),
                                g->ws.order_scratch.p, g->ws.order_scratch.bytes, st));
        tm.kernel_launches += 3;
    }
    Progress prog(g);
    for (size_t s = 0; s < n_steps; ++s) {
        prog.check_cancel();
        StepWork w;
        clock.begin(kPre);
        prepare_step(g, r, lib, s, w, tm);
        clock.end();
        plan_step(g, r, s, w);

        clock.begin(kDiff);
        const double evaluated = difference_sums(g, r, s, w, prog, tm);
        tm.evaluated_pixel_diffs += g->plans[s].pixel_diffs * evaluated;
        clock.end();
        if (g->progress_fn)
            prog.wait();  // the host watches the launch from here (before anything that could block it, e.g. the pageable D2H copy)

        clock.begin(kSel);
        select_phase(g, r, s, w, tm);
        clock.end();
        prog.end_step();
    }
    prog.finish();
    tm.preprocess_ms = clock.sum(kPre);
    tm.diff_ms = clock.sum(kDiff);
    tm.select_ms = clock.sum(kSel);
    tm.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
}

}  // namespace

// =============================================================================== C ABI

extern "C" {

const char *mosaic_version(void) { return "mosaicmagnifique_b200 0.1 (sm_100a)"; }

int mosaic_create(int device, mosaic_generator **out)
{
    if (!out)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return MOSAIC_ERR_CUDA;  // no CPU fallback by design
    }
    mosaic_generator *g = new (std::nothrow) mosaic_generator();
    if (!g)
        return MOSAIC_ERR_OUT_OF_MEMORY;
    g->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&g->poll_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaHostAlloc((void **)&g->h_cancel, sizeof(int), cudaHostAllocDefault) != cudaSuccess ||
        cudaMalloc((void **)&g->d_cancel, 256) != cudaSuccess || cudaMemset(g->d_cancel, 0, 256) != cudaSuccess ||
        cudaHostAlloc((void **)&g->h_progress, 4 * sizeof(unsigned long long), cudaHostAllocDefault) != cudaSuccess) {
        mosaic_destroy(g);
        return MOSAIC_ERR_CUDA;
    }
    *g->h_cancel = 0;
    *g->h_progress = 0;
    cudaDeviceGetAttribute(&g->sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;  // keep freed blocks cached between generate() calls
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = g;
    return MOSAIC_OK;
}

void mosaic_destroy(mosaic_generator *g)
{
    if (!g)
        return;
    cudaSetDevice(g->device);
    if (g->stream)
        cudaStreamSynchronize(g->stream);
    delete g;  // the device buffers first, then the streams and pinned words they were allocated with (Handles)
}

const char *mosaic_last_error(const mosaic_generator *g) { return g ? g->error.c_str() : "null generator"; }

int mosaic_set_main_image(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride)
{
    return guard(g, "setMainImage", [&] {
        if (!bgr || rows <= 0 || cols <= 0 || row_stride < (size_t)cols * 3)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "main image must be a non-empty 8U BGR image"};
        g->d_main_u8.alloc((size_t)rows * cols * 3, g->stream);
        // host or device pointer (unified addressing): cudaMemcpyDefault lets the driver pick the direction
        CU(cudaMemcpy2DAsync(g->d_main_u8.p, (size_t)cols * 3, bgr, row_stride, (size_t)cols * 3, rows, cudaMemcpyDefault, g->stream));
        CU(cudaStreamSynchronize(g->stream));

        g->img_rows = rows;
        g->img_cols = cols;
        g->main_lo = 0;
        g->main_hi = rows;
    });
}

int mosaic_get_shard_rows(mosaic_generator *g, int rows, int cols, int *row_lo, int *row_hi)
{
    return guard(g, "getShardRows", [&] {
        if (rows <= 0 || cols <= 0 || !row_lo || !row_hi)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "image size and output pointers are required"};
        if (!g->have_group || g->grid.empty())
            throw Fail{MOSAIC_ERR_NOT_READY, "cell group and grid state must be set first"};
        if (rows != g->img_rows || cols != g->img_cols) {
            g->img_rows = rows;  // the image is declared; no row is resident yet
            g->img_cols = cols;
            g->main_lo = g->main_hi = 0;
        }
        make_plans(g);
        needed_rows(g, *row_lo, *row_hi);
    });
}

int mosaic_set_main_image_rows(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride, int row_lo, int row_hi)
{
    return guard(g, "setMainImageRows", [&] {
        if (!bgr || rows <= 0 || cols <= 0 || row_stride < (size_t)cols * 3 || row_lo < 0 || row_hi > rows || row_lo > row_hi)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "main image must be a non-empty 8U BGR image and 0 <= row_lo <= row_hi <= rows"};
        g->d_main_u8.alloc((size_t)rows * cols * 3, g->stream);  // full-size buffer: row indices stay global
        if (row_hi > row_lo)
            CU(cudaMemcpy2DAsync(g->d_main_u8.as<uint8_t>() + (size_t)row_lo * cols * 3, (size_t)cols * 3, bgr + (size_t)row_lo * row_stride,
                                 row_stride, (size_t)cols * 3, (size_t)(row_hi - row_lo), cudaMemcpyDefault, g->stream));
        CU(cudaStreamSynchronize(g->stream));
        g->img_rows = rows;
        g->img_cols = cols;
        g->main_lo = row_lo;
        g->main_hi = row_hi;
    });
}

int mosaic_set_library(mosaic_generator *g, const uint8_t *bgr, int64_t n, int size)
{
    return guard(g, "setLibrary", [&] {
        if (!bgr || n <= 0 || size <= 0)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "library must hold n > 0 square 8U BGR images"};
        if (n * size > INT32_MAX)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large (n * size must fit 31 bits)"};
        g->d_lib_u8.alloc((size_t)n * size * size * 3, g->stream);
        CU(cudaMemcpyAsync(g->d_lib_u8.p, bgr, g->d_lib_u8.bytes, cudaMemcpyDefault, g->stream));  // host or device pointer
        CU(cudaStreamSynchronize(g->stream));
        g->n_lib = n;
        g->lib_size = size;
        g->lib_stored_size = size;
        g->lib_capacity = n;
        g->lib_sharded = false;
        g->lib_oriented_flips = 0;
    });
}

int mosaic_set_library_shard(mosaic_generator *g, const uint8_t *bgr_slice, int64_t first, int64_t count, int64_t n_total, int size,
                             int64_t capacity_images)
{
    return guard(g, "setLibraryShard", [&] {
        if (n_total <= 0 || size <= 0 || first < 0 || count < 0 || first + count > n_total || capacity_images < n_total ||
            (count > 0 && !bgr_slice))
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "need 0 <= first, first + count <= n_total <= capacity and a slice pointer"};
        if (n_total * size > INT32_MAX)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large (n * size must fit 31 bits)"};
        if (g->flips != 0)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "tile flips are set: a library stored at the detail size cannot be re-oriented exactly "
                                               "(use mosaic_set_library, or mosaic_set_tile_flips(g, 0))"};
        if (!g->have_group)
            throw Fail{MOSAIC_ERR_NOT_READY, "the cell group must be set first (its detail level decides the stored size)"};
        if (size != g->group.cells[0].size)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "library images must be at the cell size"};
        cudaStream_t st = g->stream;
        // stored size: the detail size of step 0 when the generator would resize anyway (PhotomosaicGeneratorBase.cpp:262-270)
        const int ds = g->group.detail != 1.0 ? g->group.detail_cells[0].size : size;
        const size_t stored_img = (size_t)ds * ds * 3, full_img = (size_t)size * size * 3;
        g->d_lib_u8.alloc((size_t)capacity_images * stored_img, st);
        uint8_t *dst = g->d_lib_u8.as<uint8_t>() + (size_t)first * stored_img;
        if (count > 0) {
            if (ds == size) {
                CU(cudaMemcpyAsync(dst, bgr_slice, (size_t)count * full_img, cudaMemcpyDefault, st));
            } else {
                DevBuf &stage = g->ws.lib_small;  // full-size slice, resized on the GPU into its place
                stage.alloc((size_t)count * full_img, st);
                CU(cudaMemcpyAsync(stage.p, bgr_slice, (size_t)count * full_img, cudaMemcpyDefault, st));
                if (size % ds == 0) {
                    CU(launch_area_u8(stage.as<uint8_t>(), dst, count, size, size / ds, st));
                } else {
                    mosaic_timings scratch{};
                    const AreaTab tab = upload_area_table(g, size, ds, scratch);
                    CU(launch_area_general_u8(stage.as<uint8_t>(), dst, count, size, ds, tab, st));
                }
            }
        }
        CU(cudaStreamSynchronize(st));
        g->n_lib = n_total;
        g->lib_size = size;
        g->lib_stored_size = ds;
        g->lib_capacity = capacity_images;
        g->lib_sharded = true;
        g->lib_oriented_flips = 0;
    });
}

int mosaic_get_library_device(const mosaic_generator *g, void **ptr, int *stored_size, int64_t *capacity_images)
{
    if (!g || !g->d_lib_u8.p)
        return MOSAIC_ERR_NOT_READY;
    if (ptr)
        *ptr = g->d_lib_u8.p;
    if (stored_size)
        *stored_size = g->lib_stored_size;
    if (capacity_images)
        *capacity_images = g->lib_capacity;
    return MOSAIC_OK;
}

int mosaic_set_colour_difference(mosaic_generator *g, int type)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (type < 0 || type > 2)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setColourDifference: no function for given type");  // ColourDifference.cpp:23
    g->diff_type = type;
    return MOSAIC_OK;
}

int mosaic_set_colour_scheme(mosaic_generator *g, int type)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (type < 0 || type > 5)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setColourScheme: no function for given type");  // ColourScheme.cpp:30
    g->scheme = type;
    return MOSAIC_OK;
}

int mosaic_set_variant_quirk(mosaic_generator *g, int faithful)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    g->quirk_faithful = faithful != 0;
    return MOSAIC_OK;
}

int mosaic_set_cell_group(mosaic_generator *g, const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size, int detail_percent,
                          int size_steps)
{
    return mosaic_set_cell_group_ex(g, shape, mask, cell_size, detail_percent, size_steps, 0);
}

int mosaic_set_cell_group_ex(mosaic_generator *g, const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size, int detail_percent,
                             int size_steps, int mask_as_stored)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (!shape || !mask || shape->size <= 0)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setCellGroup: missing shape or mask");
    try {
        Group grp;
        std::string err;
        if (const int rc = build_group(*shape, mask, mask_as_stored != 0, cell_size, detail_percent, size_steps, grp, err))
            return g->fail(rc, "setCellGroup: " + err);
        g->group = grp;
        g->have_group = true;
        g->grid.clear();
        g->fits_flips = -1;
        return MOSAIC_OK;
    } catch (const std::bad_alloc &) {
        return g->fail(MOSAIC_ERR_OUT_OF_MEMORY, "setCellGroup: host allocation failed");
    } catch (...) {
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setCellGroup: unexpected failure");
    }
}

int mosaic_host_cell_group_cell(const mosaic_cell_shape *shape, const uint8_t *mask, int mask_as_stored, int cell_size, int detail_percent,
                                int size_steps, int step, int detail, mosaic_cell_shape *out, uint8_t *mask_out, size_t mask_capacity)
{
    if (!shape || !mask || !out || shape->size <= 0 || step < 0 || step > size_steps)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    try {
        Group grp;
        std::string err;
        if (const int rc = build_group(*shape, mask, mask_as_stored != 0, cell_size, detail_percent, size_steps, grp, err))
            return rc;
        return shape_to_c(detail ? grp.detail_cells[step] : grp.cells[step], *out, mask_out, mask_capacity);
    } catch (const std::bad_alloc &) {
        return MOSAIC_ERR_OUT_OF_MEMORY;
    } catch (...) {
        return MOSAIC_ERR_INVALID_ARGUMENT;
    }
}

int mosaic_get_cell_shape(const mosaic_generator *g, int step, int detail, mosaic_cell_shape *out, uint8_t *mask_out, size_t mask_capacity)
{
    if (!g || !out || !g->have_group || step < 0 || step > g->group.size_steps)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    return shape_to_c(detail ? g->group.detail_cells[step] : g->group.cells[step], *out, mask_out, mask_capacity);
}

int mosaic_set_grid_state(mosaic_generator *g, int step, int rows, int cols, const uint8_t *valid)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (!valid || step < 0 || rows <= 0 || cols <= 0 || step > (int)g->grid.size())
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setGridState: steps must be set in order with a rows x cols validity map");
    // no exception may cross the C ABI: the grid vectors are the only host allocation whose size the caller controls
    if ((int64_t)rows * cols > ((int64_t)1 << 28))
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setGridState: rows * cols is implausibly large (> 2^28 cells)");
    try {
        if (step == (int)g->grid.size())
            g->grid.emplace_back();
        GridStep &gs = g->grid[step];
        gs.rows = rows;
        gs.cols = cols;
        gs.v.resize((size_t)rows * cols);
        for (size_t i = 0; i < gs.v.size(); ++i)
            gs.v[i] = valid[i] ? 0 : -1;  // valid cells start as 0 (GridGenerator.cpp:192)
        g->grid.resize(step + 1);
        g->fits_flips = -1;
    } catch (...) {
        g->grid.clear();
        return g->fail(MOSAIC_ERR_OUT_OF_MEMORY, "setGridState: host allocation failed");
    }
    return MOSAIC_OK;
}

int mosaic_compute_grid_state(mosaic_generator *g)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (!g->have_group || g->img_rows == 0)
        return g->fail(MOSAIC_ERR_NOT_READY, "getGridState: main image and cell group must be set");
    std::string err;
    // GridGenerator::getGridState with the entropy rule evaluated on the GPU (grid_kernels.cu), one batch per size step
    EntropyEvaluator gpu_eval = [g](int step, const std::vector<EntropyCandidate> &cand, std::vector<uint8_t> &split,
                                    std::string &e) -> bool {
        try {
            if (cudaSetDevice(g->device) != cudaSuccess)
                throw Fail{MOSAIC_ERR_CUDA, "cudaSetDevice failed"};
            if (g->main_lo != 0 || g->main_hi != g->img_rows)
                throw Fail{MOSAIC_ERR_NOT_READY, "the entropy rule needs the whole main image on the device (only a band of rows was uploaded)"};
            cudaStream_t st = g->stream;
            const Shape &dshape = g->group.detail_cells[step];
            const std::vector<uint8_t> m4 = dshape.masks4();
            std::vector<GridCandidate> gc(cand.size());
            for (size_t i = 0; i < cand.size(); ++i)
                gc[i] = GridCandidate{cand[i].cg.x, cand[i].cg.y, cand[i].cg.w, cand[i].cg.h, cand[i].db.x, cand[i].db.y,
                                      cand[i].db.w, cand[i].db.h, cand[i].flip};
            Workspace &w = g->ws;
            w.masks4.alloc(m4.size(), st);
            w.descs.alloc(gc.size() * sizeof(GridCandidate), st);
            w.prog.alloc(gc.size(), st);
            CU(cudaMemcpyAsync(w.masks4.p, m4.data(), m4.size(), cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(w.descs.p, gc.data(), gc.size() * sizeof(GridCandidate), cudaMemcpyHostToDevice, st));
            CU(launch_grid_entropy(g->d_main_u8.as<uint8_t>(), g->img_cols, w.descs.as<GridCandidate>(), (int)gc.size(),
                                   w.masks4.as<uint8_t>(), dshape.size, 8.0 * 0.7, w.prog.as<uint8_t>(), st));
            CU(cudaMemcpyAsync(split.data(), w.prog.p, gc.size(), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            return true;
        } catch (const Fail &f) {
            cudaGetLastError();
            e = f.msg;
            return false;
        }
    };
    g->fits_flips = -1;
    if (!compute_grid_state(g->group, g->img_rows, g->img_cols, gpu_eval, g->grid, err))
        return g->fail(MOSAIC_ERR_UNSUPPORTED, "getGridState: " + err);
    return MOSAIC_OK;
}

int mosaic_get_grid_steps(const mosaic_generator *g) { return g ? (int)g->grid.size() : MOSAIC_ERR_INVALID_ARGUMENT; }

int mosaic_get_grid_size(const mosaic_generator *g, int step, int *rows, int *cols)
{
    if (!g || step < 0 || step >= (int)g->grid.size() || !rows || !cols)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    *rows = g->grid[step].rows;
    *cols = g->grid[step].cols;
    return MOSAIC_OK;
}

int mosaic_set_repeat(mosaic_generator *g, int range, int addition)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (range < 0 || addition < 0)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setRepeat: range and addition must be >= 0");
    g->repeat_range = range;
    g->repeat_addition = addition;
    return MOSAIC_OK;
}

int mosaic_generate(mosaic_generator *g)
{
    if (g && g->world != 1)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "generateBestFits: sharded handles use mosaic_generate_candidates + mosaic_select_from_candidates");
    // m_wasCanceled is never reset by the reference (PhotomosaicGeneratorBase.cpp:35, 219): a cancel() issued before the call
    // makes it return at once; mosaic_reset_cancel() re-arms the handle
    return guard(g, "generateBestFits", [&] { run_pipeline(g, false); });
}

int mosaic_get_best_fits(const mosaic_generator *g, int step, int64_t *out, int rows, int cols)
{
    if (!g || !out || step < 0 || step >= (int)g->grid.size())
        return MOSAIC_ERR_INVALID_ARGUMENT;
    const GridStep &gs = g->grid[step];
    if (rows != gs.rows || cols != gs.cols)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (g->fits_flips > 0) {  // the grid holds slots j * N + i: report the image i
        for (size_t i = 0; i < gs.v.size(); ++i)
            out[i] = gs.v[i] >= 0 ? gs.v[i] % g->n_lib : gs.v[i];
    } else {
        memcpy(out, gs.v.data(), gs.v.size() * sizeof(int64_t));
    }
    return MOSAIC_OK;
}

int mosaic_set_tile_flips(mosaic_generator *g, int flips)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (flips < 0 || flips > 3)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setTileFlips: flips is a mask of 1 (horizontal) and 2 (vertical)");
    g->flips = flips;
    return MOSAIC_OK;
}

int mosaic_set_usage_limit(mosaic_generator *g, int max_uses)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (max_uses < 0)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setUsageLimit: max_uses must be >= 0 (0 = unlimited)");
    g->max_uses = max_uses;
    return MOSAIC_OK;
}

int mosaic_get_best_fit_flips(const mosaic_generator *g, int step, int8_t *out, int rows, int cols)
{
    if (!g || !out || step < 0 || step >= (int)g->grid.size())
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (g->fits_flips < 0)
        return MOSAIC_ERR_NOT_READY;
    const GridStep &gs = g->grid[step];
    if (rows != gs.rows || cols != gs.cols)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    for (size_t i = 0; i < gs.v.size(); ++i)
        out[i] = (int8_t)(gs.v[i] >= 0 ? orient_code(g->fits_flips, (int)(gs.v[i] / g->n_lib)) : -1);
    return MOSAIC_OK;
}

int mosaic_get_max_progress(const mosaic_generator *g)
{
    if (!g || g->grid.empty())
        return 0;
    // PhotomosaicGeneratorBase.cpp:210-214
    return (int)(pow(4.0, (double)g->grid.size() - 1) * (double)g->grid.size() * g->grid[0].cols * g->grid[0].rows);
}

void mosaic_set_progress_callback(mosaic_generator *g, mosaic_progress_fn fn, void *user)
{
    if (!g)
        return;
    g->progress_fn = fn;
    g->progress_user = user;
}

void mosaic_cancel(mosaic_generator *g)
{
    if (!g || !g->h_cancel)
        return;
    __atomic_store_n(g->h_cancel, 1, __ATOMIC_RELAXED);
    // mirror it into the device word right away (the generate thread does the same from its wait loops, so a failure here --
    // e.g. a calling thread that cannot touch the device -- only delays the kernel's reaction by one poll)
    int prev = -1;
    if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(g->device) == cudaSuccess) {
        cudaMemcpyAsync(g->d_cancel, g->h_cancel, sizeof(int), cudaMemcpyHostToDevice, g->poll_stream);
        if (prev >= 0 && prev != g->device)
            cudaSetDevice(prev);
    }
    cudaGetLastError();
}

void mosaic_reset_cancel(mosaic_generator *g)
{
    if (g && g->h_cancel)
        __atomic_store_n(g->h_cancel, 0, __ATOMIC_RELAXED);
}

int mosaic_set_keep_differences(mosaic_generator *g, int keep)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    g->keep_D = keep != 0;
    return MOSAIC_OK;
}

int64_t mosaic_get_valid_cell_count(const mosaic_generator *g, int step)
{
    if (!g || step < 0 || step >= (int)g->grid.size())
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (step < (int)g->plans.size())
        return (int64_t)g->plans[step].cell_pos.size();
    int64_t n = 0;
    for (int64_t v : g->grid[step].v)
        n += v >= 0;
    return n;
}

int mosaic_get_differences(const mosaic_generator *g, int step, float *out, int64_t n_cells, int64_t n_lib)
{
    if (!g || !out || step < 0 || step >= (int)g->out.size() || !g->out[step].have_D)
        return MOSAIC_ERR_NOT_READY;
    const StepPlan &p = g->plans[step];
    const int64_t n_local = p.cell_end - p.cell_begin;
    if (n_cells != n_local || n_lib != g->n_slots)  // n_slots = O * N: D has a column per slot
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (n_local == 0)
        return MOSAIC_OK;
    const int tnb = tile_geom(g->diff_type == MOSAIC_CIEDE2000 ? kLayoutCiede : kLayoutEuclid).tnb;
    const int n_lib_pad = (int)((g->n_slots + tnb - 1) / tnb) * tnb;
    cudaSetDevice(g->device);
    cudaError_t e = cudaMemcpy2D(out, (size_t)n_lib * sizeof(float), g->out[step].D.p, (size_t)g->V_eff * n_lib_pad * sizeof(float),
                                 (size_t)n_lib * sizeof(float), (size_t)n_local, cudaMemcpyDeviceToHost);
    return e == cudaSuccess ? MOSAIC_OK : MOSAIC_ERR_CUDA;
}

int mosaic_set_report_margins(mosaic_generator *g, int report)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    g->report_margins = report != 0;
    return MOSAIC_OK;
}

int mosaic_get_margins(const mosaic_generator *g, int step, float *best, float *second, int64_t n_cells)
{
    if (!g || !best || !second || step < 0 || step >= (int)g->out.size() || !g->out[step].have_margins)
        return MOSAIC_ERR_NOT_READY;
    if (n_cells != (int64_t)g->plans[step].cell_pos.size())
        return MOSAIC_ERR_INVALID_ARGUMENT;
    std::vector<float> m((size_t)n_cells * 2);
    cudaSetDevice(g->device);
    if (n_cells && cudaMemcpy(m.data(), g->out[step].margins.p, m.size() * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return MOSAIC_ERR_CUDA;
    }
    for (int64_t i = 0; i < n_cells; ++i) {
        best[i] = m[2 * i];
        second[i] = m[2 * i + 1];
    }
    return MOSAIC_OK;
}

int mosaic_get_timings(const mosaic_generator *g, mosaic_timings *out)
{
    if (!g || !out)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    *out = g->timings;
    return MOSAIC_OK;
}

// ---- buildPhotomosaic (PhotomosaicGeneratorBase.cpp:110-207)

int mosaic_build_photomosaic(mosaic_generator *g, const uint8_t background_bgra[4], uint8_t *out_bgra, int rows, int cols, size_t row_stride)
{
    return guard(g, "buildPhotomosaic", [&] {
        if (!background_bgra || !out_bgra || rows != g->img_rows || cols != g->img_cols || row_stride < (size_t)cols * 4 || row_stride % 4 != 0)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "output must be a rows x cols BGRA buffer of the main image's size"};
        if (g->grid.empty() || !g->have_group || g->n_lib == 0)
            throw Fail{MOSAIC_ERR_NOT_READY, "no best fits to build from"};
        if (g->lib_size != g->group.cells[0].size)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "library images must be at the cell size"};
        if (g->lib_stored_size != g->lib_size)
            throw Fail{MOSAIC_ERR_NOT_READY, "buildPhotomosaic needs the library at the cell size (it was uploaded at the detail size "
                                             "by mosaic_set_library_shard)"};
        cudaStream_t st = g->stream;
        const int H = g->img_rows, W = g->img_cols, n_steps = (int)g->grid.size();
        const int64_t N = g->n_lib;
        // the grid holds slots j * N + i of the generate's orientations: image i, placed mirrored by orientation j
        const int fl = std::max(g->fits_flips, 0), O = orient_count(fl);
        DevBuf owner, out, d_steps;
        std::vector<DevBuf> libs(n_steps), cells(n_steps), masks(n_steps);
        std::vector<BuildStep> hsteps(n_steps);
        owner.alloc((size_t)H * W * sizeof(unsigned long long), st);
        CU(cudaMemsetAsync(owner.p, 0, owner.bytes, st));
        const uint8_t *lib_prev = g->d_lib_u8.as<uint8_t>();
        int S_prev = g->lib_size;
        for (int s = 0; s < n_steps; ++s) {
            const Shape &shape = g->group.cells[s];
            const GridStep &gs = g->grid[s];
            // library at this step: halved like batchResizeMat(libImg) (8U INTER_AREA, round(0.5 * size))
            const uint8_t *lib_s = lib_prev;
            int S = S_prev;
            if (s > 0) {
                S = (int)lround(0.5 * S_prev);
                // the 2 x 2 halving is exact in integers and commutes with mirroring; the fractional table of an odd size need not
                if (O > 1 && S_prev % 2 != 0)
                    throw Fail{MOSAIC_ERR_UNSUPPORTED, "mirrored tiles at an odd cell size (" + std::to_string(S_prev) + ") of step " +
                                                           std::to_string(s - 1) + ": halving it does not commute with mirroring"};
                libs[s].alloc((size_t)N * S * S * 3, st);
                if (S_prev % 2 == 0) {
                    CU(launch_area_u8(lib_prev, libs[s].as<uint8_t>(), N, S_prev, 2, st));
                } else {
                    mosaic_timings scratch{};
                    const AreaTab tab = upload_area_table(g, S_prev, S, scratch);
                    CU(launch_area_general_u8(lib_prev, libs[s].as<uint8_t>(), N, S_prev, S, tab, st));
                }
                lib_s = libs[s].as<uint8_t>();
            }
            if (S != shape.size)
                throw Fail{MOSAIC_ERR_UNSUPPORTED, "library and cell size disagree at step " + std::to_string(s) +
                                                       " (the reference copies out of range here)"};
            std::vector<BuildCell> hc;
            for (int y = 0; y < gs.rows; ++y)
                for (int x = 0; x < gs.cols; ++x) {
                    const int64_t v = gs.v[(size_t)y * gs.cols + x];
                    if (v < 0)
                        continue;
                    if (v >= O * N)
                        throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "best fit index outside the library"};
                    const Rect r = rect_at(shape, x - kPadGrid, y - kPadGrid);
                    hc.push_back(BuildCell{r.x, r.y, flip_at(shape, x - kPadGrid, y - kPadGrid), (int)hc.size() + 1, (int)(v % N),
                                           orient_code(fl, (int)(v / N))});
                }
            const std::vector<uint8_t> m4 = shape.masks4();
            masks[s].alloc(m4.size(), st);
            CU(cudaMemcpyAsync(masks[s].p, m4.data(), m4.size(), cudaMemcpyHostToDevice, st));
            cells[s].alloc(std::max<size_t>(hc.size(), 1) * sizeof(BuildCell), st);
            CU(cudaMemcpyAsync(cells[s].p, hc.data(), hc.size() * sizeof(BuildCell), cudaMemcpyHostToDevice, st));
            CU(launch_build_scatter(cells[s].as<BuildCell>(), (int)hc.size(), S, masks[s].as<uint8_t>(), H, W, s, n_steps,
                                    owner.as<unsigned long long>(), st));
            hsteps[s] = BuildStep{cells[s].as<BuildCell>(), lib_s, S};
            lib_prev = lib_s;
            S_prev = S;
        }
        d_steps.alloc(hsteps.size() * sizeof(BuildStep), st);
        CU(cudaMemcpyAsync(d_steps.p, hsteps.data(), d_steps.bytes, cudaMemcpyHostToDevice, st));
        out.alloc((size_t)H * W * 4, st);
        CU(launch_build_gather(owner.as<unsigned long long>(), H, W, n_steps, d_steps.as<BuildStep>(), background_bgra, out.as<uint8_t>(),
                               (size_t)W, st));
        CU(cudaMemcpy2DAsync(out_bgra, row_stride, out.p, (size_t)W * 4, (size_t)W * 4, H, cudaMemcpyDefault, st));
        CU(cudaStreamSynchronize(st));
    });
}

// ---- sharding

int mosaic_set_shard(mosaic_generator *g, int rank, int world)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (world < 1 || rank < 0 || rank >= world)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setShard: need 0 <= rank < world");
    g->rank = rank;
    g->world = world;
    return MOSAIC_OK;
}

int mosaic_host_shard_split(int64_t n_valid_cells, int colour_difference, int rank, int world, int64_t *rows_per_rank, int64_t *first_cell,
                            int64_t *n_cells)
{
    if (n_valid_cells < 0 || colour_difference < 0 || colour_difference > 2 || world < 1 || rank < 0 || rank >= world)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    int64_t per = 0, b = 0, e = 0;
    shard_split(n_valid_cells, colour_difference, rank, world, per, b, e);
    if (rows_per_rank)
        *rows_per_rank = per;
    if (first_cell)
        *first_cell = b;
    if (n_cells)
        *n_cells = e - b;
    return MOSAIC_OK;
}

int mosaic_generate_candidates(mosaic_generator *g)
{
    return guard(g, "generateCandidates", [&] { run_pipeline(g, true); });
}

int mosaic_get_candidate_count(const mosaic_generator *g, int step, int64_t *first_cell, int64_t *n_cells, int *k)
{
    if (!g || step < 0 || step >= (int)g->plans.size() || step >= (int)g->out.size())
        return MOSAIC_ERR_NOT_READY;
    if (first_cell)
        *first_cell = g->plans[step].cell_begin;
    if (n_cells)
        *n_cells = g->plans[step].cell_end - g->plans[step].cell_begin;
    if (k)
        *k = g->out[step].cand_k;
    return MOSAIC_OK;
}

int mosaic_get_candidates_device(const mosaic_generator *g, int step, void **scores, void **indices)
{
    if (!g || step < 0 || step >= (int)g->out.size() || step >= (int)g->plans.size() || !scores || !indices)
        return MOSAIC_ERR_NOT_READY;
    float *cs = g->out[step].cand.as<float>();
    *scores = cs;
    *indices = cs ? (void *)(cs + (size_t)g->plans[step].per_rank * g->out[step].cand_k) : nullptr;
    return MOSAIC_OK;
}

int mosaic_get_candidate_block(const mosaic_generator *g, int step, void **block, int64_t *rows_per_rank, int *k, size_t *block_bytes)
{
    if (!g || step < 0 || step >= (int)g->out.size() || step >= (int)g->plans.size())
        return MOSAIC_ERR_NOT_READY;
    const StepOut &o = g->out[step];
    if (block)
        *block = o.cand.p;
    if (rows_per_rank)
        *rows_per_rank = g->plans[step].per_rank;
    if (k)
        *k = o.cand_k;
    if (block_bytes)
        *block_bytes = (size_t)g->plans[step].per_rank * o.cand_k * (sizeof(float) + sizeof(int));
    return MOSAIC_OK;
}

namespace {
// selection over the candidates of ALL cells of a step. rows_per_block == 0: scores / indices are plain [n_valid][k] arrays;
// otherwise `scores` is the all-gathered buffer of per-rank blocks {float [rows_per_block][k], int32 [rows_per_block][k]}.
int select_impl(mosaic_generator *g, int step, const void *scores, const void *indices, int k, int64_t rows_per_block)
{
    return guard(g, "selectFromCandidates", [&] {
        if (step < 0 || step >= (int)g->plans.size() || !scores || (!indices && rows_per_block == 0) || k < 1)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "bad step or candidate buffers"};
        for (auto &v : g->grid[step].v)
            v = v >= 0 ? 0 : -1;
        g->fits_flips = g->flips;
        Candidates c;
        c.scores = (const float *)scores;
        c.idx = (const int *)indices;
        c.M = c.M_stride = k;
        if (rows_per_block > 0) {
            c.idx = reinterpret_cast<const int *>(c.scores + (size_t)rows_per_block * k);  // indices follow the scores inside every block
            c.rows_per_block = rows_per_block;
            c.block_stride = 2 * rows_per_block * k;  // in 4-byte elements
        }
        bool restart_used = false;
        if (g->cand_max_uses > 0) {
            // `used` carries across the steps of one generate: selecting a step at or below the last one starts a new generate, and
            // every earlier step with cells must have been selected since
            if (step <= g->cap_last_step)
                g->cap_last_step = -1;
            for (int s = g->cap_last_step + 1; s < step; ++s)
                if (!g->plans[s].cell_pos.empty())
                    throw Fail{MOSAIC_ERR_NOT_READY, "usage limit: step " + std::to_string(s) + " must be selected before step " +
                                                         std::to_string(step) + " (image uses carry across the steps in order)"};
            restart_used = g->cap_last_step < 0;
            // the blocks were sorted by mosaic_generate_candidates: every row's prefix is its own front
            c.pscores = c.scores;
            c.pidx = c.idx;
            c.k0 = std::min(k, kPrefixMax);
            c.p_stride = k;
        }
        PhaseClock clock(g->stream);
        mosaic_timings t{};
        select_step(g, step, nullptr, [&] { return c; }, g->cand_max_uses, restart_used, nullptr, &clock, t);
        if (g->cand_max_uses > 0)
            g->cap_last_step = step;
        CU(cudaStreamSynchronize(g->stream));
        // added to the timings of mosaic_generate_candidates: the selection launch, its time and the grid's copy back
        g->timings.select_ms += clock.sum(0);
        g->timings.kernel_launches += t.kernel_launches;
        g->timings.d2h_bytes += t.d2h_bytes;
    });
}
}  // namespace

int mosaic_select_from_candidates(mosaic_generator *g, int step, const void *scores, const void *indices, int k)
{
    return select_impl(g, step, scores, indices, k, 0);
}

int mosaic_select_from_gathered(mosaic_generator *g, int step, const void *gathered_blocks, int k, int64_t rows_per_rank)
{
    if (g && rows_per_rank <= 0)
        return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "selectFromGathered: rows_per_rank must be positive");
    return select_impl(g, step, gathered_blocks, nullptr, k, rows_per_rank);
}

// ---- host geometry

void mosaic_grid_size(const mosaic_cell_shape *shape, int image_w, int image_h, int pad, int *grid_w, int *grid_h)
{
    if (!shape || !grid_w || !grid_h)
        return;
    int gx = 0, gy = 0;
    grid_size(shape_params_only(*shape), image_w, image_h, pad, gx, gy);
    *grid_w = gx;
    *grid_h = gy;
}

void mosaic_rect_at(const mosaic_cell_shape *shape, int x, int y, int rect_xywh[4])
{
    if (!shape || !rect_xywh)
        return;
    const Rect r = rect_at(shape_params_only(*shape), x, y);
    rect_xywh[0] = r.x;
    rect_xywh[1] = r.y;
    rect_xywh[2] = r.w;
    rect_xywh[3] = r.h;
}

int mosaic_flip_at(const mosaic_cell_shape *shape, int x, int y)
{
    return shape ? flip_at(shape_params_only(*shape), x, y) : MOSAIC_ERR_INVALID_ARGUMENT;
}

int mosaic_host_grid_state(const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size, int detail_percent, int size_steps,
                           const uint8_t *bgr, int rows, int cols, size_t row_stride, int max_steps, int *n_steps, int *step_rows,
                           int *step_cols, int64_t *out, size_t out_capacity)
{
    if (!shape || !mask || !n_steps || !step_rows || !step_cols || !out || rows <= 0 || cols <= 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    try {
        Group grp;
        std::string err;
        if (const int rc = build_group(*shape, mask, false, cell_size, detail_percent, size_steps, grp, err))
            return rc;
        std::vector<GridStep> grid;
        const EntropyEvaluator eval = bgr ? host_entropy_evaluator(grp, bgr, row_stride) : EntropyEvaluator();
        if (!compute_grid_state(grp, rows, cols, eval, grid, err))
            return MOSAIC_ERR_UNSUPPORTED;
        if ((int)grid.size() > max_steps)
            return MOSAIC_ERR_INVALID_ARGUMENT;
        size_t used = 0;
        for (size_t s = 0; s < grid.size(); ++s) {
            if (used + grid[s].v.size() > out_capacity)
                return MOSAIC_ERR_INVALID_ARGUMENT;
            step_rows[s] = grid[s].rows;
            step_cols[s] = grid[s].cols;
            memcpy(out + used, grid[s].v.data(), grid[s].v.size() * sizeof(int64_t));
            used += grid[s].v.size();
        }
        *n_steps = (int)grid.size();
        return MOSAIC_OK;
    } catch (const std::bad_alloc &) {
        return MOSAIC_ERR_OUT_OF_MEMORY;
    } catch (...) {
        return MOSAIC_ERR_INVALID_ARGUMENT;
    }
}

int mosaic_host_resize_area_u8(const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w)
{
    if (!src || !dst || cn < 1 || cn > 4)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    return resize_area_u8(src, src_h, src_w, cn, dst, dst_h, dst_w) ? MOSAIC_OK : MOSAIC_ERR_UNSUPPORTED;
}

}  // extern "C"
