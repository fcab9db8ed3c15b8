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

}  // namespace

struct mosaic_generator {
    int device = 0;
    cudaStream_t stream = nullptr;
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
    // cancel(): a flag in pinned host memory (what the host tests) mirrored into a word of DEVICE memory by a 4-byte DMA on the
    // poll stream; every CTA of the difference kernels reads the device word (an L2 hit) when it starts. (Reading mapped host
    // memory from every CTA was measured first: 296 CTAs polling one PCIe address cost 25 % of the kernel and made a cancelled
    // launch drain no faster than a complete one.)
    int *h_cancel = nullptr;
    int *d_cancel = nullptr;
    bool cancel_pushed = false;  // the device word already holds 1 (generate thread only)
    // progress(int) while a launch runs: device counter of finished CTAs, polled over a second stream into pinned memory
    cudaStream_t poll_stream = nullptr;
    DevBuf d_progress;
    unsigned long long *h_progress = nullptr;  // [0] progress poll, [1] [2] row-list counts

    bool is_cancelled() const { return h_cancel && __atomic_load_n(h_cancel, __ATOMIC_RELAXED) != 0; }

    // products
    DevBuf d_lut;
    Workspace ws;
    std::vector<bool> have_D;
    std::vector<StepPlan> plans;
    std::vector<DevBuf> d_D;            // per step [n_local_cells_pad * V][n_lib_pad]
    std::vector<DevBuf> d_cand_score, d_cand_idx;
    std::vector<DevBuf> d_margins;      // per step [n_valid][2] when report_margins
    std::vector<bool> have_margins;
    std::vector<int> cand_k;
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

int guard(G *g, const char *what, void (*fn)(G *, void *), void *arg)
{
    if (!g)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    try {
        cudaError_t e = cudaSetDevice(g->device);
        if (e != cudaSuccess)
            throw Fail{MOSAIC_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e)};
        fn(g, arg);
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

void shape_from_c(const mosaic_cell_shape &c, const uint8_t *mask, Shape &s, bool mask_as_stored = false)
{
    if (mask_as_stored)
        s.set_mask_as_stored(mask, c.size);
    else
        s.set_mask(mask, c.size);
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
}

void shape_to_c(const Shape &s, mosaic_cell_shape &c)
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

struct Timer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s;
    explicit Timer(cudaStream_t st) : s(st)
    {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
    }
    ~Timer()
    {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
    void start() { cudaEventRecord(a, s); }
    void stop() { cudaEventRecord(b, s); }
    double ms()
    {
        float m = 0;
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&m, a, b);
        return m;
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

// sorted prefixes of candidate lists [n_rows][K] (launch_topk output), in place: the first min(K, kPrefixMax) entries of every row
// become its smallest (score, slot) pairs in ascending order
void sort_list_prefixes(G *g, float *cs, int *ci, int n_rows, int K, mosaic_timings &tm)
{
    if (n_rows == 0)
        return;
    const int k0 = std::min(K, kPrefixMax);
    cudaStream_t st = g->stream;
    g->ws.prefix_score.alloc((size_t)n_rows * k0 * sizeof(float), st);
    g->ws.prefix_idx.alloc((size_t)n_rows * k0 * sizeof(int), st);
    CU(launch_topk(cs, K, K, n_rows, k0, g->ws.prefix_score.as<float>(), g->ws.prefix_idx.as<int>(), st));
    CU(launch_sort_prefix(g->ws.prefix_score.as<float>(), g->ws.prefix_idx.as<int>(), n_rows, k0, cs, ci, K, st));
    tm.kernel_launches += 2;
}

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
    const bool is_lab = g->diff_type != MOSAIC_RGB_EUCLIDEAN;
    const PackLayout layout = g->diff_type == MOSAIC_CIEDE2000 ? kLayoutCiede : kLayoutEuclid;
    const TileGeom tg = tile_geom(layout);
    // Colour-scheme variants (ColourScheme.cpp:36-177): original + hue rotations. Reference quirk Q1: getCellAt builds the
    // V cell Mats over ONE shared buffer (PhotomosaicGeneratorBase.cpp:310-312), so every variant holds the LAST rotation
    // and the original image is never compared. faithful mode reproduces that with a single variant.
    static const float kRot[6][3] = {{0, 0, 0}, {180, 0, 0}, {120, 240, 0}, {150, 210, 0}, {90, 180, 270}, {30, 60, 90}};
    static const int kNumRot[6] = {0, 1, 2, 2, 3, 3};
    std::vector<float> rotations;  // rotation of each variant that is actually compared (0 = the image itself)
    if (g->scheme == MOSAIC_SCHEME_NONE)
        rotations = {0.0f};
    else if (g->quirk_faithful)
        rotations = {kRot[g->scheme][kNumRot[g->scheme] - 1]};
    else {
        rotations = {0.0f};
        for (int i = 0; i < kNumRot[g->scheme]; ++i)
            rotations.push_back(kRot[g->scheme][i]);
    }
    const int V = (int)rotations.size();
    g->V_eff = V;
    // candidate slots: the O orientations of the N library images, orientation-major (slot = j * N + i); every stage up to D runs
    // on the oriented library as if it were the library itself
    const int O = orient_count(g->flips);
    if (O > 1 && g->lib_sharded)
        throw Fail{MOSAIC_ERR_UNSUPPORTED, "tile flips need the library from mosaic_set_library: a library stored at the detail size "
                                           "cannot be re-oriented exactly"};
    const int64_t N = g->n_lib * O;
    if (N * g->lib_size > INT32_MAX)
        throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large with tile flips (orientations * n * size must fit 31 bits)"};
    g->n_slots = N;
    if (!candidates_only)
        g->fits_flips = g->flips;
    const int n_lib_tiles = (int)((N + tg.tnb - 1) / tg.tnb);
    const int n_lib_pad = n_lib_tiles * tg.tnb;
    const size_t n_steps = g->grid.size();
    PhaseClock clock(st);
    enum { kPre = 0, kDiff = 1, kSel = 2 };

    if (!g->d_lut.p) {
        const std::vector<int16_t> lut4 = expand_lab_lut(mm_lab_lut_s16);
        g->d_lut.alloc(lut4.size() * sizeof(int16_t), st);
        CU(cudaMemcpyAsync(g->d_lut.p, lut4.data(), g->d_lut.bytes, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));  // lut4 is a local
        tm.h2d_bytes += (double)g->d_lut.bytes;
    }

    // ---- Preprocess: main image -> working space (PhotomosaicGeneratorBase.cpp:223-252)
    clock.begin(kPre);
    DevBuf &d_main_f32 = g->ws.main_f32;
    const size_t n_main_px = (size_t)g->img_rows * g->img_cols;
    d_main_f32.alloc((size_t)V * n_main_px * 3 * sizeof(float), st);
    // a sharded rank only reads the image rows its own cells cover: convert just those
    int row_lo, row_hi;
    needed_rows(g, row_lo, row_hi);
    if (row_lo < g->main_lo || row_hi > g->main_hi)
        throw Fail{MOSAIC_ERR_NOT_READY, "main image rows " + std::to_string(row_lo) + ".." + std::to_string(row_hi) +
                                             " are needed by this shard but only " + std::to_string(g->main_lo) + ".." +
                                             std::to_string(g->main_hi) + " were uploaded (mosaic_set_main_image_rows)"};
    const int n_rows_conv = row_hi - row_lo;
    const size_t row_off_px = (size_t)row_lo * g->img_cols;
    for (int v = 0; v < V && n_rows_conv > 0; ++v) {
        const uint8_t *src = g->d_main_u8.as<uint8_t>() + row_off_px * 3;
        if (rotations[v] != 0.0f) {
            g->ws.main_var_u8.alloc(n_main_px * 3, st);
            CU(launch_hue_rotate(src, g->ws.main_var_u8.as<uint8_t>() + row_off_px * 3, n_rows_conv, g->img_cols, rotations[v], st));
            tm.kernel_launches++;
            src = g->ws.main_var_u8.as<uint8_t>() + row_off_px * 3;
        }
        CU(launch_to_working_space(src, (size_t)g->img_cols * 3, n_rows_conv, g->img_cols,
                                   d_main_f32.as<float>() + ((size_t)v * n_main_px + row_off_px) * 3, is_lab, g->d_lut.as<short4>(),
                                   nullptr, st));
        tm.kernel_launches++;
    }

    // ---- Preprocess: oriented library (rebuilt only when the library or the flips changed)
    const uint8_t *lib_src = g->d_lib_u8.as<uint8_t>();
    if (O > 1) {
        if (g->lib_oriented_flips != g->flips) {
            g->lib_oriented_flips = 0;
            g->d_lib_oriented.alloc((size_t)N * g->lib_size * g->lib_size * 3, st);
            CU(launch_orient_library(lib_src, g->d_lib_oriented.as<uint8_t>(), g->n_lib, g->lib_size, g->flips, st));
            tm.kernel_launches++;
            g->lib_oriented_flips = g->flips;
        }
        lib_src = g->d_lib_oriented.as<uint8_t>();
    }

    // ---- Preprocess: library -> working space at the detail size of step 0 (:255-290)
    DevBuf &d_lib_work = g->ws.lib_work, &d_lib_small = g->ws.lib_small;
    int lib_ds = g->lib_size;
    const uint8_t *lib_u8_at_ds = nullptr;  // 8U source of the fused packers: at lib_ds, or at lib_ds * fused_k
    bool fuse_lib_conversion = false;
    int fused_k = 1;
    {
        const uint8_t *src = lib_src;
        if (g->group.detail != 1.0) {
            lib_ds = g->plans[0].ds;
            if (g->lib_stored_size != g->lib_size) {
                // sharded setLibrary already resized every slice to the detail size (mosaic_set_library_shard)
                if (g->lib_stored_size != lib_ds)
                    throw Fail{MOSAIC_ERR_NOT_READY, "the library was uploaded for another detail size: call mosaic_set_library_shard "
                                                     "again after changing the cell group"};
            } else if (n_steps == 1 && g->lib_size % lib_ds == 0) {
                // integer ratio and a single size step: the packers below reduce on the fly, the resized 8U copy is never written
                fused_k = g->lib_size / lib_ds;
            } else {
                d_lib_small.alloc((size_t)N * lib_ds * lib_ds * 3, st);
                if (g->lib_size % lib_ds == 0) {
                    CU(launch_area_u8(src, d_lib_small.as<uint8_t>(), N, g->lib_size, g->lib_size / lib_ds, st));
                } else {
                    const AreaTab tab = upload_area_table(g, g->lib_size, lib_ds, tm);
                    CU(launch_area_general_u8(src, d_lib_small.as<uint8_t>(), N, g->lib_size, lib_ds, tab, st));
                }
                tm.kernel_launches++;
                src = d_lib_small.as<uint8_t>();
            }
        } else if (g->lib_stored_size != g->lib_size) {
            throw Fail{MOSAIC_ERR_NOT_READY, "the library was uploaded at a detail size but the cell group now has detail 100 %"};
        }
        // a single size step: the colour conversion is fused into the tile-packing kernel below (straight from the 8U
        // library), the f32 working-space copy is only materialised when a later step has to halve it
        lib_u8_at_ds = src;
        fuse_lib_conversion = n_steps == 1;
        if (!fuse_lib_conversion) {
            d_lib_work.alloc((size_t)N * lib_ds * lib_ds * 3 * sizeof(float), st);
            // the library is one tall image of N * ds rows
            CU(launch_to_working_space(src, (size_t)lib_ds * 3, (int)std::min<int64_t>(N * lib_ds, INT32_MAX), lib_ds,
                                       d_lib_work.as<float>(), is_lab, g->d_lut.as<short4>(), nullptr, st));
            tm.kernel_launches++;
        }
    }
    clock.end();

    if (g->d_D.size() != n_steps) {
        g->d_D.clear();
        g->d_D.resize(n_steps);
        g->d_cand_score.clear();
        g->d_cand_score.resize(n_steps);
        g->d_cand_idx.clear();
        g->d_cand_idx.resize(n_steps);
    }
    g->have_D.assign(n_steps, false);
    if (g->d_margins.size() != n_steps) {
        g->d_margins.clear();
        g->d_margins.resize(n_steps);
    }
    g->have_margins.assign(n_steps, false);
    g->cand_k.assign(n_steps, 0);

    const bool penalise = g->repeat_range > 0 && g->repeat_addition != 0;
    const bool capped = g->max_uses > 0;
    const bool fused_argmin = !penalise && !capped && V == 1 && !candidates_only && g->world == 1 && !g->report_margins;
    if (candidates_only) {
        g->cand_max_uses = g->max_uses;
        g->cap_last_step = -1;
    } else if (capped) {  // `used` starts at 0 for every generate and carries across its steps
        g->d_used.alloc((size_t)g->n_lib * sizeof(int), st);
        CU(cudaMemsetAsync(g->d_used.p, 0, g->d_used.bytes, st));
    }
    // CIEDE2000 steps that need D run as segment passes over row work lists; the library tiles then hold the library in colour
    // order (kernels.h: RowList), which is what lets exact pruning drop whole tiles of a cell
    const bool row_passes = layout == kLayoutCiede && !fused_argmin;
    if (row_passes) {
        g->ws.perm.alloc((size_t)n_lib_pad * sizeof(int), st);
        g->ws.inv_perm.alloc((size_t)n_lib_pad * sizeof(int), st);
        g->ws.order_scratch.alloc(library_order_scratch_bytes(N), st);
        CU(launch_library_order(lib_src, g->lib_stored_size, N, n_lib_pad, g->ws.perm.as<int>(), g->ws.inv_perm.as<int>(), g->ws.order_scratch.p,
                                g->ws.order_scratch.bytes, st));
        tm.kernel_launches += 3;
    }
    int progress = 0;
    // cancel(): polled by the host before every phase it enqueues and by every CTA of the difference kernels when it starts
    // (the reference polls per step, row and cell, CPUPhotomosaicGenerator.cpp:52, 66, 73). Work already enqueued drains first.
    auto check_cancel = [&]() {
        if (g->is_cancelled()) {
            push_cancel(g);
            cudaStreamSynchronize(st);
            throw Fail{MOSAIC_ERR_CANCELLED, "cancelled"};
        }
    };
    check_cancel();  // sticky like m_wasCanceled: a cancelled handle does nothing until mosaic_reset_cancel
    g->cancel_pushed = false;
    CU(cudaStreamSynchronize(g->poll_stream));                     // no stale flag copy may land after the reset below
    CU(cudaMemsetAsync(g->d_cancel, 0, sizeof(int), st));
    unsigned long long *d_tiles_done = nullptr;
    if (g->progress_fn) {
        g->d_progress.alloc(sizeof(unsigned long long), st);
        d_tiles_done = g->d_progress.as<unsigned long long>();
    }

    for (size_t s = 0; s < n_steps; ++s) {
        check_cancel();
        StepPlan &p = g->plans[s];
        const Shape &normal = g->group.cells[s];
        const Shape &dshape = g->group.detail_cells[s];
        GridStep &gs = g->grid[s];
        const int ds = p.ds, P = ds * ds;
        Workspace &d = g->ws;

        clock.begin(kPre);
        if (s > 0) {
            // halve the working-space library (CPUPhotomosaicGenerator.cpp:95-99)
            DevBuf &half = g->ws.lib_half;
            half.alloc((size_t)N * P * 3 * sizeof(float), st);
            CU(launch_area_f32(d_lib_work.as<float>(), half.as<float>(), N, ds * 2, 2, st));
            tm.kernel_launches++;
            std::swap(d_lib_work, half);
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
        d.lib_packed.alloc((size_t)n_lib_tiles * p.n_chunks * tg.lib_block, st);
        const int *perm = row_passes ? d.perm.as<int>() : nullptr;
        if (fuse_lib_conversion && layout == kLayoutCiede)
            CU(launch_pack_library_ciede(lib_u8_at_ds, true, d.lib_packed.p, N, P, d.pix_list.as<int>(), p.n_active, p.n_chunks,
                                         n_lib_tiles, g->d_lut.as<short4>(), st, ds * fused_k, fused_k, perm));
        else if (fuse_lib_conversion)
            CU(launch_pack_library_euclid_u8(lib_u8_at_ds, ds * fused_k, fused_k, is_lab, d.lib_packed.p, N, P, d.pix_list.as<int>(),
                                             p.n_active, p.n_chunks, n_lib_tiles, g->d_lut.as<short4>(), st));
        else
            CU(launch_pack_library(d_lib_work.as<float>(), d.lib_packed.p, N, P, d.pix_list.as<int>(), p.n_active, p.n_chunks,
                                   n_lib_tiles, layout, st, perm));
        tm.kernel_launches++;

        // cell descriptors of this rank's cells (getCellAt, PhotomosaicGeneratorBase.cpp:293-329)
        const int64_t n_local = p.cell_end - p.cell_begin;
        const int64_t n_all = (int64_t)p.cell_pos.size();
        std::vector<CellDesc> descs((size_t)n_local * V);
        // mask pixel counts through integral images (for the pixel-diff statistics)
        std::vector<std::vector<int>> integ(4, std::vector<int>((size_t)(ds + 1) * (ds + 1), 0));
        for (int f = 0; f < 4; ++f)
            for (int y = 0; y < ds; ++y)
                for (int x = 0; x < ds; ++x)
                    integ[f][(size_t)(y + 1) * (ds + 1) + x + 1] = (m4[((size_t)f * ds + y) * ds + x] != 0) + integ[f][(size_t)y * (ds + 1) + x + 1] +
                                                                  integ[f][(size_t)(y + 1) * (ds + 1) + x] - integ[f][(size_t)y * (ds + 1) + x];
        for (int64_t c = 0; c < n_all; ++c) {
            const int pos = p.cell_pos[c];
            const int x = pos % p.cols - kPadGrid, y = pos / p.cols - kPadGrid;
            const Rect r = rect_at(normal, x, y);
            const Rect b = detail_bound(normal, ds, g->group.detail, x, y, g->img_cols, g->img_rows);
            const int flip = flip_at(normal, x, y);
            const std::vector<int> &I = integ[flip];
            const int act = I[(size_t)(b.y + b.h) * (ds + 1) + b.x + b.w] - I[(size_t)b.y * (ds + 1) + b.x + b.w] -
                            I[(size_t)(b.y + b.h) * (ds + 1) + b.x] + I[(size_t)b.y * (ds + 1) + b.x];
            p.pixel_diffs += (double)act * N * V;
            p.pixel_diffs_nominal += (double)P * N * V;
            if (c >= p.cell_begin && c < p.cell_end)
                for (int v = 0; v < V; ++v)
                    descs[(size_t)(c - p.cell_begin) * V + v] = CellDesc{r.x, r.y, b.x, b.y, b.w, b.h, flip, v};
        }
        tm.pixel_diffs += p.pixel_diffs;
        tm.pixel_diffs_nominal += p.pixel_diffs_nominal;

        const int n_rows_local = (int)(n_local * V);
        const int n_cell_tiles = (n_rows_local + tg.tcb - 1) / tg.tcb;
        const int n_rows_pad = n_cell_tiles * tg.tcb;
        d.descs.alloc(std::max<size_t>(descs.size(), 1) * sizeof(CellDesc), st);
        CU(cudaMemcpyAsync(d.descs.p, descs.data(), descs.size() * sizeof(CellDesc), cudaMemcpyHostToDevice, st));
        tm.h2d_bytes += (double)(descs.size() * sizeof(CellDesc));
        d.cells_packed.alloc((size_t)std::max(n_cell_tiles, 1) * p.n_chunks * tg.cell_block, st);
        AreaTab cell_tab{nullptr, nullptr, nullptr};
        if (p.k == 0)
            cell_tab = upload_area_table(g, p.S, p.ds, tm);
        CU(launch_extract_cells(d_main_f32.as<float>(), g->img_rows, g->img_cols, d.descs.as<CellDesc>(), n_rows_local, p.S, p.ds,
                                p.k, cell_tab, d.masks4.as<uint8_t>(), d.pix_list.as<int>(), p.n_active, p.n_chunks,
                                d.cells_packed.p, layout, st));
        tm.kernel_launches++;
        clock.end();

        // ---- DiffReduce
        clock.begin(kDiff);
        const bool need_D = !fused_argmin || g->keep_D;
        DevBuf &D = g->d_D[s];
        if (need_D) {
            D.alloc((size_t)std::max(n_rows_pad, 1) * n_lib_pad * sizeof(float), st);
            g->have_D[s] = true;
        }
        if (fused_argmin) {
            d.best_key.alloc((size_t)std::max(n_rows_pad, 1) * sizeof(unsigned long long), st);
            CU(launch_fill_u64(d.best_key.as<unsigned long long>(), (size_t)std::max(n_rows_pad, 1), ~0ull, st));
            tm.kernel_launches++;
        }
        // top-K count of the selection below; when D only feeds top-K (and need not be complete), pairs that cannot be among the
        // k_need smallest are pruned (launch_prune_threshold).
        // Grouped K: the window holds W = 2r^2 + 2r cells, so at most W distinct images and, as the O orientations of an image share
        // its count, at most O * W of the O * N slots carry a penalty. Among the O * W + 1 smallest (score, slot) pairs at least one
        // slot u is unpenalised. The penalised winner w has D[w] + A * count >= D[w] and must beat or tie u, so D[w] <= D[u], and at
        // D[w] == D[u] the lower slot wins: (D[w], w) <= (D[u], u), so w is among the O * W + 1 smallest. The runner-up is among the
        // O * W + 2 smallest by the same argument with two unpenalised slots. O = 1 is SURVEY.md 8e's bound.
        // With a usage limit at most E_s images are exhausted before the step's last cell, so O * E_s more slots may be excluded and
        // the same argument holds with O * (W + E_s) (DESIGN.md 4.4).
        const int64_t rr = g->repeat_range;
        const int64_t n_win = 2 * rr * rr + 2 * rr;
        const int64_t n_excl = capped ? O * exhausted_bound(g, s) : 0;
        const int64_t k_need = candidates_only ? ((penalise || capped) ? std::min<int64_t>(N, O * n_win + n_excl + 1) : 1)
                                               : std::min<int64_t>(N, O * n_win + n_excl + 1 + (g->report_margins ? 1 : 0));
        const bool via_topk = candidates_only || ((penalise || capped) && k_need * 4 <= N);
        const int M = (int)std::min<int64_t>(N, k_need + k_need / 4 + 8);  // candidates of the first segment: 1.25 k_need + 8
        const bool prune = row_passes && via_topk && V == 1 && !g->keep_D && k_need * 4 <= N && M <= 4096 && n_rows_local > 0;
        // segments: 8 (or MM_SPLITK) passes over the pixel axis, chunk-aligned
        int n_segs = 1, seg_chunks = p.n_chunks;
        if (row_passes) {
            const char *ev = getenv("MM_SPLITK");
            const int want = ev && atoi(ev) > 0 ? atoi(ev) : kPruneSegments;
            seg_chunks = (p.n_chunks + std::min(want, p.n_chunks) - 1) / std::min(want, p.n_chunks);
            n_segs = (p.n_chunks + seg_chunks - 1) / seg_chunks;
        }
        const unsigned long long prog_total = row_passes ? (unsigned long long)std::max(n_rows_local, 1) * n_lib_tiles * n_segs
                                                         : (unsigned long long)std::max(n_cell_tiles, 1) * n_lib_tiles;
        const int step_weight = (int)pow(4.0, (double)(n_steps - 1 - s));
        const int positions = p.rows * p.cols;
        int last = progress;
        // waits for the stream; with a callback the host polls the device's count of finished rows / tiles meanwhile and emits
        // base + weight * floor(positions * done / total) (see the end of the step)
        auto watch = [&]() {
            if (!g->progress_fn) {
                wait_stream(g, st);
                check_cancel();
                return;
            }
            cudaEvent_t done;
            CU(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
            cudaEventRecord(done, st);
            while (cudaEventQuery(done) == cudaErrorNotReady) {
                if (cudaMemcpyAsync(g->h_progress, d_tiles_done, sizeof(unsigned long long), cudaMemcpyDeviceToHost, g->poll_stream) == cudaSuccess &&
                    cudaStreamSynchronize(g->poll_stream) == cudaSuccess && !g->is_cancelled()) {
                    const unsigned long long dn = std::min(*g->h_progress, prog_total);
                    const int v = progress + step_weight * (int)((unsigned long long)positions * dn / prog_total);
                    if (v > last && v < progress + step_weight * positions) {
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
        };
        check_cancel();
        if (d_tiles_done)
            CU(cudaMemsetAsync(d_tiles_done, 0, sizeof(unsigned long long), st));
        double evaluated = 1.0;  // executed share of the step's (row, chunk) work
        if (row_passes && n_rows_local > 0) {
            CU(cudaMemsetAsync(D.p, 0, D.bytes, st));
            int col_cells = kColumnCells;
            if (const char *ev = getenv("MM_SB_A"))
                col_cells = std::max(32, std::min(1024, atoi(ev) * MM_TCB / 32 * 32));
            const int n_cols = (n_rows_local + col_cells - 1) / col_cells;
            RowList rows{nullptr, nullptr, nullptr, n_cols * n_lib_tiles, col_cells};
            d.row_cells.alloc((size_t)rows.n_buckets * col_cells * sizeof(int), st);
            d.row_count.alloc((size_t)rows.n_buckets * sizeof(int), st);
            d.row_groups.alloc((size_t)(rows.n_buckets + 1) * sizeof(int), st);
            d.list_scratch.alloc(list_rows_scratch_bytes(rows.n_buckets), st);
            d.listed.alloc(sizeof(unsigned long long), st);
            rows.cells = d.row_cells.as<int>();
            rows.count = d.row_count.as<int>();
            rows.groups = d.row_groups.as<int>();
            const int *perm = d.perm.as<int>();
            uint8_t *state = nullptr;
            if (prune) {
                d.row_state.alloc((size_t)n_rows_local * n_lib_tiles, st);
                CU(cudaMemsetAsync(d.row_state.p, kRowActive, d.row_state.bytes, st));
                state = d.row_state.as<uint8_t>();
            }
            double units = 0;  // rows x chunks evaluated
            int n_groups = 0;
            auto list = [&](uint8_t *st8, int want, const float *T, int segs_left) {
                CU(cudaMemsetAsync(d.listed.p, 0, sizeof(unsigned long long), st));
                CU(launch_list_rows(D.as<float>(), n_lib_pad, (int)N, n_rows_local, n_lib_tiles, st8, want, T, perm, segs_left, rows,
                                    d.list_scratch.p, d.list_scratch.bytes, d.listed.as<unsigned long long>(), d_tiles_done, st));
                CU(cudaMemcpyAsync(g->h_progress + 1, rows.groups + rows.n_buckets, sizeof(int), cudaMemcpyDeviceToHost, st));
                CU(cudaMemcpyAsync(g->h_progress + 2, d.listed.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
                tm.kernel_launches += 2;
                watch();  // the pass size is needed on the host to size the next launch
                n_groups = (int)*reinterpret_cast<const int *>(g->h_progress + 1);
                return (double)g->h_progress[2];
            };
            auto pass = [&](int seg, double n_listed) {
                const int k0 = seg * seg_chunks, nk = std::min(p.n_chunks, k0 + seg_chunks) - k0;
                CU(launch_diff_rows(d.cells_packed.p, d.lib_packed.p, D.as<float>(), n_groups, n_lib_tiles, p.n_chunks, k0, nk, rows, perm,
                                    st, g->d_cancel, d_tiles_done));
                tm.kernel_launches += n_groups > 0;
                units += n_listed * nk;
            };
            double n_listed = list(nullptr, kRowActive, nullptr, 0);  // every row
            if (!prune) {
                for (int seg = 0; seg < n_segs; ++seg)
                    pass(seg, n_listed);
            } else {
                pass(0, n_listed);
                // candidates = the M smallest partial sums of segment 0; their tiles are completed first, T[cell] = the k_need-th
                // smallest of their complete sums, and every later pass lists only the rows that still have a pair <= T
                d.prune_score.alloc((size_t)n_rows_local * M * sizeof(float), st);
                d.prune_idx.alloc((size_t)n_rows_local * M * sizeof(int), st);
                d.threshold.alloc((size_t)n_rows_local * sizeof(float), st);
                CU(launch_topk(D.as<float>(), n_lib_pad, (int)N, n_rows_local, M, d.prune_score.as<float>(), d.prune_idx.as<int>(), st));
                CU(launch_prune_threshold(D.as<float>(), n_lib_pad, d.prune_idx.as<int>(), n_rows_local, M, (int)k_need,
                                          d.inv_perm.as<int>(), n_lib_tiles, state, nullptr, true, st));
                tm.kernel_launches += 2;
                if (n_segs > 1) {
                    n_listed = list(state, kRowComplete, nullptr, 0);
                    for (int seg = 1; seg < n_segs; ++seg)
                        pass(seg, n_listed);
                }
                CU(launch_prune_threshold(D.as<float>(), n_lib_pad, d.prune_idx.as<int>(), n_rows_local, M, (int)k_need,
                                          d.inv_perm.as<int>(), n_lib_tiles, state, d.threshold.as<float>(), false, st));
                tm.kernel_launches++;
                for (int seg = 1; seg < n_segs; ++seg) {
                    n_listed = list(state, kRowActive, d.threshold.as<float>(), n_segs - seg);
                    pass(seg, n_listed);
                }
            }
            evaluated = units / ((double)n_rows_local * n_lib_tiles * p.n_chunks);
        } else if (layout == kLayoutCiede) {
            CU(launch_diff_sum(MM_DIFF_CIEDE2000, d.cells_packed.p, d.lib_packed.p, need_D ? D.as<float>() : nullptr,
                               fused_argmin ? d.best_key.as<unsigned long long>() : nullptr, n_cell_tiles, n_lib_tiles, p.n_chunks,
                               (int)N, n_rows_local, st, g->d_cancel, d_tiles_done));
            tm.kernel_launches += n_cell_tiles > 0;
        } else {
            CU(launch_diff_euclid(d.cells_packed.p, d.lib_packed.p, need_D ? D.as<float>() : nullptr,
                                  fused_argmin ? d.best_key.as<unsigned long long>() : nullptr, n_cell_tiles, n_lib_tiles, p.n_chunks,
                                  (int)N, n_rows_local, st, g->d_cancel, d_tiles_done));
            tm.kernel_launches += n_cell_tiles > 0;
        }
        tm.evaluated_pixel_diffs += p.pixel_diffs * evaluated;
        clock.end();
        if (g->progress_fn)
            watch();  // the host watches the launch from here (before anything that could block it, e.g. the pageable D2H copy)

        // ---- Repeats + FindLowest
        clock.begin(kSel);
        if (V > 1 && need_D) {
            CU(launch_min_variants(D.as<float>(), (int)n_local, V, n_lib_pad, st));
            tm.kernel_launches++;
        }
        if (candidates_only) {
            // K = min(O * N, O * (2r^2 + 2r) + 1) smallest entries always contain the penalised winner (k_need above)
            const int K = (int)k_need;
            g->cand_k[s] = K;
            // one block per rank: float scores [per_rank][K] followed by int32 indices [per_rank][K]; every rank's block has the
            // same size, so ONE all-gather assembles the candidates of the whole step (rank r's rows start at r * per_rank)
            const size_t half = (size_t)p.per_rank * K;
            g->d_cand_score[s].alloc(half * (sizeof(float) + sizeof(int)), st);
            float *cs = g->d_cand_score[s].as<float>();
            int *ci = reinterpret_cast<int *>(cs + half);
            CU(launch_topk(D.as<float>(), V * n_lib_pad, (int)N, (int)n_local, K, cs, ci, st));
            if (n_local > 0)
                tm.kernel_launches++;
            if (capped)  // the capped selection on the gathered blocks reads every row's sorted prefix first
                sort_list_prefixes(g, cs, ci, (int)n_local, K, tm);
        } else {
            DevBuf &d_grid = d.grid, &d_pos = d.pos, &d_next = d.next, &d_prog = d.prog, &d_counts = d.counts;
            d_grid.alloc(gs.v.size() * sizeof(long long), st);
            CU(cudaMemcpyAsync(d_grid.p, gs.v.data(), gs.v.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
            d_pos.alloc(std::max<size_t>(p.cell_pos.size(), 1) * sizeof(int), st);
            CU(cudaMemcpyAsync(d_pos.p, p.cell_pos.data(), p.cell_pos.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            tm.h2d_bytes += (double)(gs.v.size() * sizeof(long long) + p.cell_pos.size() * sizeof(int));
            if (fused_argmin) {
                CU(launch_keys_to_grid(d.best_key.as<unsigned long long>(), d_pos.as<int>(), d_grid.as<long long>(), (int)n_all,
                                       nullptr, st));
                if (n_all > 0)
                    tm.kernel_launches++;
            } else {
                d_next.alloc(std::max<size_t>(p.next_x.size(), 1) * sizeof(int), st);
                CU(cudaMemcpyAsync(d_next.p, p.next_x.data(), p.next_x.size() * sizeof(int), cudaMemcpyHostToDevice, st));
                d_prog.alloc((size_t)p.rows * sizeof(int), st);
                CU(cudaMemcpyAsync(d_prog.p, p.row_first.data(), (size_t)p.rows * sizeof(int), cudaMemcpyHostToDevice, st));
                const int n_ctas = (int)std::max<int64_t>(1, std::min<int64_t>(n_all, select_max_ctas(g->device)));
                d_counts.alloc((size_t)n_ctas * g->n_lib * sizeof(int), st);  // per source image
                CU(cudaMemsetAsync(d_counts.p, 0, d_counts.bytes, st));
                float *margins = nullptr;
                if (g->report_margins) {
                    g->d_margins[s].alloc(std::max<size_t>((size_t)n_all, 1) * 2 * sizeof(float), st);
                    margins = g->d_margins[s].as<float>();
                    g->have_margins[s] = true;
                }
                // With a penalty the winner (and the runner-up) lies among the K (+1) smallest unpenalised scores
                // (SURVEY.md 8e), so the wavefront scans candidate lists instead of whole D rows when that is shorter.
                if (capped) {
                    // sequential capped selection: every cell's sorted prefix first, its full row (K list or D row) as the fallback
                    const int k0 = (int)std::min<int64_t>(k_need, kPrefixMax);
                    const float *row_s = D.as<float>(), *ps;
                    const int *row_i = nullptr, *pi;
                    int row_n = (int)N, row_stride = V * n_lib_pad, p_stride = k0;
                    if (via_topk) {
                        const int K = (int)k_need;
                        g->d_cand_score[s].alloc((size_t)std::max<int64_t>(n_all, 1) * K * sizeof(float), st);
                        g->d_cand_idx[s].alloc((size_t)std::max<int64_t>(n_all, 1) * K * sizeof(int), st);
                        CU(launch_topk(D.as<float>(), V * n_lib_pad, (int)N, (int)n_all, K, g->d_cand_score[s].as<float>(),
                                       g->d_cand_idx[s].as<int>(), st));
                        tm.kernel_launches++;
                        sort_list_prefixes(g, g->d_cand_score[s].as<float>(), g->d_cand_idx[s].as<int>(), (int)n_all, K, tm);
                        row_s = ps = g->d_cand_score[s].as<float>();
                        row_i = pi = g->d_cand_idx[s].as<int>();
                        row_n = row_stride = p_stride = K;
                    } else {
                        d.prefix_score.alloc((size_t)std::max<int64_t>(n_all, 1) * k0 * sizeof(float), st);
                        d.prefix_idx.alloc((size_t)std::max<int64_t>(n_all, 1) * k0 * sizeof(int), st);
                        CU(launch_topk(D.as<float>(), V * n_lib_pad, (int)N, (int)n_all, k0, d.prefix_score.as<float>(),
                                       d.prefix_idx.as<int>(), st));
                        CU(launch_sort_prefix(d.prefix_score.as<float>(), d.prefix_idx.as<int>(), (int)n_all, k0, nullptr, nullptr, 0, st));
                        tm.kernel_launches += n_all > 0 ? 2 : 0;
                        ps = d.prefix_score.as<float>();
                        pi = d.prefix_idx.as<int>();
                    }
                    CU(launch_select_capped(d_grid.as<long long>(), d_pos.as<int>(), (int)n_all, p.rows, p.cols, row_s, row_i, row_n,
                                            row_stride, ps, pi, k0, p_stride, (int)g->n_lib, g->repeat_range, g->repeat_addition,
                                            g->max_uses, d_counts.as<int>(), g->d_used.as<int>(), margins, st));
                } else if (via_topk) {
                    const int K = (int)k_need;
                    g->d_cand_score[s].alloc((size_t)std::max<int64_t>(n_all, 1) * K * sizeof(float), st);
                    g->d_cand_idx[s].alloc((size_t)std::max<int64_t>(n_all, 1) * K * sizeof(int), st);
                    CU(launch_topk(D.as<float>(), V * n_lib_pad, (int)N, (int)n_all, K, g->d_cand_score[s].as<float>(),
                                   g->d_cand_idx[s].as<int>(), st));
                    tm.kernel_launches++;
                    CU(launch_select(d_grid.as<long long>(), d_pos.as<int>(), d_next.as<int>(), (int)n_all, p.rows, p.cols,
                                     g->d_cand_score[s].as<float>(), g->d_cand_idx[s].as<int>(), K, K, (int)g->n_lib, g->repeat_range,
                                     g->repeat_addition, d_prog.as<int>(), d_counts.as<int>(), n_ctas, margins, st));
                } else {
                    CU(launch_select(d_grid.as<long long>(), d_pos.as<int>(), d_next.as<int>(), (int)n_all, p.rows, p.cols,
                                     D.as<float>(), nullptr, (int)N, V * n_lib_pad, (int)g->n_lib, g->repeat_range, g->repeat_addition,
                                     d_prog.as<int>(), d_counts.as<int>(), n_ctas, margins, st));
                }
                if (n_all > 0)
                    tm.kernel_launches++;
            }
            CU(cudaMemcpyAsync(gs.v.data(), d_grid.p, gs.v.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
            tm.d2h_bytes += (double)(gs.v.size() * sizeof(long long));
        }
        clock.end();
        // progress(int): the reference emits after every grid position, cumulative, with weight 4^(steps-1-step)
        // (CPUPhotomosaicGenerator.cpp:55, 87-88). Here the host polls the device's count of finished difference tiles while the
        // step runs and emits base + weight * floor(positions * done / total): every emitted value is one the reference emits too,
        // the sequence is increasing and each step ends on the reference's own step total. Only when a callback is installed --
        // otherwise the pipeline never waits on the host before its final synchronise.
        if (g->progress_fn) {  // the step's own total: the value the reference reaches after the step's last grid position
            wait_stream(g, st);
            check_cancel();
            g->progress_fn(progress + step_weight * positions, g->progress_user);
        }
        progress += step_weight * positions;
    }
    wait_stream(g, st);
    check_cancel();
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
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete g;
        return MOSAIC_ERR_CUDA;
    }
    if (cudaStreamCreateWithFlags(&g->poll_stream, cudaStreamNonBlocking) != cudaSuccess ||
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
    g->d_main_u8.release();
    g->d_lib_u8.release();
    g->d_lib_oriented.release();
    g->d_used.release();
    g->d_lut.release();
    g->ws = Workspace();
    g->d_D.clear();
    g->d_cand_score.clear();
    g->d_cand_idx.clear();
    g->d_margins.clear();
    g->d_progress.release();
    if (g->stream) {
        cudaStreamSynchronize(g->stream);
        cudaStreamDestroy(g->stream);
    }
    if (g->poll_stream)
        cudaStreamDestroy(g->poll_stream);
    if (g->h_cancel)
        cudaFreeHost(g->h_cancel);
    if (g->d_cancel)
        cudaFree(g->d_cancel);
    if (g->h_progress)
        cudaFreeHost(g->h_progress);
    delete g;
}

const char *mosaic_last_error(const mosaic_generator *g) { return g ? g->error.c_str() : "null generator"; }

int mosaic_set_main_image(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride)
{
    struct A {
        const uint8_t *bgr;
        int rows, cols;
        size_t stride;
    } a{bgr, rows, cols, row_stride};
    return guard(g, "setMainImage", [](G *g, void *p) {
        A &a = *(A *)p;
        if (!a.bgr || a.rows <= 0 || a.cols <= 0 || a.stride < (size_t)a.cols * 3)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "main image must be a non-empty 8U BGR image"};
        g->d_main_u8.alloc((size_t)a.rows * a.cols * 3, g->stream);
        // host or device pointer (unified addressing): cudaMemcpyDefault lets the driver pick the direction
        CU(cudaMemcpy2DAsync(g->d_main_u8.p, (size_t)a.cols * 3, a.bgr, a.stride, (size_t)a.cols * 3, a.rows, cudaMemcpyDefault,
                             g->stream));
        CU(cudaStreamSynchronize(g->stream));

        g->img_rows = a.rows;
        g->img_cols = a.cols;
        g->main_lo = 0;
        g->main_hi = a.rows;
    }, &a);
}

int mosaic_get_shard_rows(mosaic_generator *g, int rows, int cols, int *row_lo, int *row_hi)
{
    struct A {
        int rows, cols, *lo, *hi;
    } a{rows, cols, row_lo, row_hi};
    return guard(g, "getShardRows", [](G *g, void *p) {
        A &a = *(A *)p;
        if (a.rows <= 0 || a.cols <= 0 || !a.lo || !a.hi)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "image size and output pointers are required"};
        if (!g->have_group || g->grid.empty())
            throw Fail{MOSAIC_ERR_NOT_READY, "cell group and grid state must be set first"};
        if (a.rows != g->img_rows || a.cols != g->img_cols) {
            g->img_rows = a.rows;  // the image is declared; no row is resident yet
            g->img_cols = a.cols;
            g->main_lo = g->main_hi = 0;
        }
        make_plans(g);
        needed_rows(g, *a.lo, *a.hi);
    }, &a);
}

int mosaic_set_main_image_rows(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride, int row_lo, int row_hi)
{
    struct A {
        const uint8_t *bgr;
        int rows, cols;
        size_t stride;
        int lo, hi;
    } a{bgr, rows, cols, row_stride, row_lo, row_hi};
    return guard(g, "setMainImageRows", [](G *g, void *p) {
        A &a = *(A *)p;
        if (!a.bgr || a.rows <= 0 || a.cols <= 0 || a.stride < (size_t)a.cols * 3 || a.lo < 0 || a.hi > a.rows || a.lo > a.hi)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "main image must be a non-empty 8U BGR image and 0 <= row_lo <= row_hi <= rows"};
        g->d_main_u8.alloc((size_t)a.rows * a.cols * 3, g->stream);  // full-size buffer: row indices stay global
        if (a.hi > a.lo)
            CU(cudaMemcpy2DAsync(g->d_main_u8.as<uint8_t>() + (size_t)a.lo * a.cols * 3, (size_t)a.cols * 3, a.bgr + (size_t)a.lo * a.stride,
                                 a.stride, (size_t)a.cols * 3, (size_t)(a.hi - a.lo), cudaMemcpyDefault, g->stream));
        CU(cudaStreamSynchronize(g->stream));
        g->img_rows = a.rows;
        g->img_cols = a.cols;
        g->main_lo = a.lo;
        g->main_hi = a.hi;
    }, &a);
}

int mosaic_set_library(mosaic_generator *g, const uint8_t *bgr, int64_t n, int size)
{
    struct A {
        const uint8_t *bgr;
        int64_t n;
        int size;
    } a{bgr, n, size};
    return guard(g, "setLibrary", [](G *g, void *p) {
        A &a = *(A *)p;
        if (!a.bgr || a.n <= 0 || a.size <= 0)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "library must hold n > 0 square 8U BGR images"};
        if (a.n * a.size > INT32_MAX)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large (n * size must fit 31 bits)"};
        g->d_lib_u8.alloc((size_t)a.n * a.size * a.size * 3, g->stream);
        CU(cudaMemcpyAsync(g->d_lib_u8.p, a.bgr, g->d_lib_u8.bytes, cudaMemcpyDefault, g->stream));  // host or device pointer
        CU(cudaStreamSynchronize(g->stream));
        g->n_lib = a.n;
        g->lib_size = a.size;
        g->lib_stored_size = a.size;
        g->lib_capacity = a.n;
        g->lib_sharded = false;
        g->lib_oriented_flips = 0;
    }, &a);
}

int mosaic_set_library_shard(mosaic_generator *g, const uint8_t *bgr_slice, int64_t first, int64_t count, int64_t n_total, int size,
                             int64_t capacity_images)
{
    struct A {
        const uint8_t *bgr;
        int64_t first, count, n, cap;
        int size;
    } a{bgr_slice, first, count, n_total, capacity_images, size};
    return guard(g, "setLibraryShard", [](G *g, void *p) {
        A &a = *(A *)p;
        if (a.n <= 0 || a.size <= 0 || a.first < 0 || a.count < 0 || a.first + a.count > a.n || a.cap < a.n || (a.count > 0 && !a.bgr))
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "need 0 <= first, first + count <= n_total <= capacity and a slice pointer"};
        if (a.n * a.size > INT32_MAX)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "library too large (n * size must fit 31 bits)"};
        if (g->flips != 0)
            throw Fail{MOSAIC_ERR_UNSUPPORTED, "tile flips are set: a library stored at the detail size cannot be re-oriented exactly "
                                               "(use mosaic_set_library, or mosaic_set_tile_flips(g, 0))"};
        if (!g->have_group)
            throw Fail{MOSAIC_ERR_NOT_READY, "the cell group must be set first (its detail level decides the stored size)"};
        if (a.size != g->group.cells[0].size)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "library images must be at the cell size"};
        cudaStream_t st = g->stream;
        // stored size: the detail size of step 0 when the generator would resize anyway (PhotomosaicGeneratorBase.cpp:262-270)
        const int ds = g->group.detail != 1.0 ? g->group.detail_cells[0].size : a.size;
        const size_t stored_img = (size_t)ds * ds * 3, full_img = (size_t)a.size * a.size * 3;
        g->d_lib_u8.alloc((size_t)a.cap * stored_img, st);
        uint8_t *dst = g->d_lib_u8.as<uint8_t>() + (size_t)a.first * stored_img;
        if (a.count > 0) {
            if (ds == a.size) {
                CU(cudaMemcpyAsync(dst, a.bgr, (size_t)a.count * full_img, cudaMemcpyDefault, st));
            } else {
                DevBuf &stage = g->ws.lib_small;  // full-size slice, resized on the GPU into its place
                stage.alloc((size_t)a.count * full_img, st);
                CU(cudaMemcpyAsync(stage.p, a.bgr, (size_t)a.count * full_img, cudaMemcpyDefault, st));
                if (a.size % ds == 0) {
                    CU(launch_area_u8(stage.as<uint8_t>(), dst, a.count, a.size, a.size / ds, st));
                } else {
                    mosaic_timings scratch{};
                    const AreaTab tab = upload_area_table(g, a.size, ds, scratch);
                    CU(launch_area_general_u8(stage.as<uint8_t>(), dst, a.count, a.size, ds, tab, st));
                }
            }
        }
        CU(cudaStreamSynchronize(st));
        g->n_lib = a.n;
        g->lib_size = a.size;
        g->lib_stored_size = ds;
        g->lib_capacity = a.cap;
        g->lib_sharded = true;
        g->lib_oriented_flips = 0;
    }, &a);
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
        Shape top;
        shape_from_c(*shape, mask, top, mask_as_stored != 0);
        std::string err;
        if (cell_size > 0 && cell_size != top.size) {
            Shape r;
            if (!top.resized(cell_size, r, err))
                return g->fail(MOSAIC_ERR_UNSUPPORTED, "setCellGroup: " + err);
            top = r;
        }
        Group grp;
        if (!grp.build(top, detail_percent, size_steps, err))
            return g->fail(MOSAIC_ERR_INVALID_ARGUMENT, "setCellGroup: " + err);
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
        Shape top;
        shape_from_c(*shape, mask, top, mask_as_stored != 0);
        std::string err;
        if (cell_size > 0 && cell_size != top.size) {
            Shape r;
            if (!top.resized(cell_size, r, err))
                return MOSAIC_ERR_UNSUPPORTED;
            top = r;
        }
        Group grp;
        if (!grp.build(top, detail_percent, size_steps, err))
            return MOSAIC_ERR_INVALID_ARGUMENT;
        const Shape &s = detail ? grp.detail_cells[step] : grp.cells[step];
        shape_to_c(s, *out);
        if (mask_out) {
            if (mask_capacity < s.mask.size())
                return MOSAIC_ERR_INVALID_ARGUMENT;
            memcpy(mask_out, s.mask.data(), s.mask.size());
        }
        return MOSAIC_OK;
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
    const Shape &s = detail ? g->group.detail_cells[step] : g->group.cells[step];
    shape_to_c(s, *out);
    if (mask_out) {
        if (mask_capacity < s.mask.size())
            return MOSAIC_ERR_INVALID_ARGUMENT;
        memcpy(mask_out, s.mask.data(), s.mask.size());
    }
    return MOSAIC_OK;
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
    return guard(g, "generateBestFits", [](G *g, void *) { run_pipeline(g, false); }, nullptr);
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
    if (!g || !out || step < 0 || step >= (int)g->d_D.size() || step >= (int)g->have_D.size() || !g->have_D[step])
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
    cudaError_t e = cudaMemcpy2D(out, (size_t)n_lib * sizeof(float), g->d_D[step].p, (size_t)g->V_eff * n_lib_pad * sizeof(float),
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
    if (!g || !best || !second || step < 0 || step >= (int)g->have_margins.size() || !g->have_margins[step])
        return MOSAIC_ERR_NOT_READY;
    if (n_cells != (int64_t)g->plans[step].cell_pos.size())
        return MOSAIC_ERR_INVALID_ARGUMENT;
    std::vector<float> m((size_t)n_cells * 2);
    cudaSetDevice(g->device);
    if (n_cells && cudaMemcpy(m.data(), g->d_margins[step].p, m.size() * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess) {
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
    struct A {
        const uint8_t *bg;
        uint8_t *out;
        int rows, cols;
        size_t stride;
    } a{background_bgra, out_bgra, rows, cols, row_stride};
    return guard(g, "buildPhotomosaic", [](G *g, void *ap) {
        A &a = *(A *)ap;
        if (!a.bg || !a.out || a.rows != g->img_rows || a.cols != g->img_cols || a.stride < (size_t)a.cols * 4 || a.stride % 4 != 0)
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
                    const AreaTable t = make_area_table(S_prev, S);
                    DevBuf ts, tsi, ta;
                    ts.alloc(t.start.size() * sizeof(int), st);
                    tsi.alloc(t.si.size() * sizeof(int), st);
                    ta.alloc(t.alpha.size() * sizeof(float), st);
                    CU(cudaMemcpyAsync(ts.p, t.start.data(), ts.bytes, cudaMemcpyHostToDevice, st));
                    CU(cudaMemcpyAsync(tsi.p, t.si.data(), tsi.bytes, cudaMemcpyHostToDevice, st));
                    CU(cudaMemcpyAsync(ta.p, t.alpha.data(), ta.bytes, cudaMemcpyHostToDevice, st));
                    CU(launch_area_general_u8(lib_prev, libs[s].as<uint8_t>(), N, S_prev, S, AreaTab{ts.as<int>(), tsi.as<int>(), ta.as<float>()}, st));
                    CU(cudaStreamSynchronize(st));
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
        CU(launch_build_gather(owner.as<unsigned long long>(), H, W, n_steps, d_steps.as<BuildStep>(), a.bg, out.as<uint8_t>(), (size_t)W, st));
        CU(cudaMemcpy2DAsync(a.out, a.stride, out.p, (size_t)W * 4, (size_t)W * 4, H, cudaMemcpyDefault, st));
        CU(cudaStreamSynchronize(st));
    }, &a);
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
    return guard(g, "generateCandidates", [](G *g, void *) { run_pipeline(g, true); }, nullptr);
}

int mosaic_get_candidate_count(const mosaic_generator *g, int step, int64_t *first_cell, int64_t *n_cells, int *k)
{
    if (!g || step < 0 || step >= (int)g->plans.size() || step >= (int)g->cand_k.size())
        return MOSAIC_ERR_NOT_READY;
    if (first_cell)
        *first_cell = g->plans[step].cell_begin;
    if (n_cells)
        *n_cells = g->plans[step].cell_end - g->plans[step].cell_begin;
    if (k)
        *k = g->cand_k[step];
    return MOSAIC_OK;
}

int mosaic_get_candidates_device(const mosaic_generator *g, int step, void **scores, void **indices)
{
    if (!g || step < 0 || step >= (int)g->d_cand_score.size() || step >= (int)g->plans.size() || step >= (int)g->cand_k.size() ||
        !scores || !indices)
        return MOSAIC_ERR_NOT_READY;
    float *cs = g->d_cand_score[step].as<float>();
    *scores = cs;
    *indices = cs ? (void *)(cs + (size_t)g->plans[step].per_rank * g->cand_k[step]) : nullptr;
    return MOSAIC_OK;
}

int mosaic_get_candidate_block(const mosaic_generator *g, int step, void **block, int64_t *rows_per_rank, int *k, size_t *block_bytes)
{
    if (!g || step < 0 || step >= (int)g->d_cand_score.size() || step >= (int)g->plans.size() || step >= (int)g->cand_k.size())
        return MOSAIC_ERR_NOT_READY;
    if (block)
        *block = g->d_cand_score[step].p;
    if (rows_per_rank)
        *rows_per_rank = g->plans[step].per_rank;
    if (k)
        *k = g->cand_k[step];
    if (block_bytes)
        *block_bytes = (size_t)g->plans[step].per_rank * g->cand_k[step] * (sizeof(float) + sizeof(int));
    return MOSAIC_OK;
}

namespace {
// selection over the candidates of ALL cells of a step. rows_per_block == 0: scores / indices are plain [n_valid][k] arrays;
// otherwise `scores` is the all-gathered buffer of per-rank blocks {float [rows_per_block][k], int32 [rows_per_block][k]}.
int select_impl(mosaic_generator *g, int step, const void *scores, const void *indices, int k, int64_t rows_per_block)
{
    struct A {
        int step;
        const void *scores, *indices;
        int k;
        int64_t rpb;
    } a{step, scores, indices, k, rows_per_block};
    return guard(g, "selectFromCandidates", [](G *g, void *ap) {
        A &a = *(A *)ap;
        if (a.step < 0 || a.step >= (int)g->plans.size() || !a.scores || (!a.indices && a.rpb == 0) || a.k < 1)
            throw Fail{MOSAIC_ERR_INVALID_ARGUMENT, "bad step or candidate buffers"};
        StepPlan &p = g->plans[a.step];
        GridStep &gs = g->grid[a.step];
        cudaStream_t st = g->stream;
        const int64_t n_all = (int64_t)p.cell_pos.size();
        for (auto &v : gs.v)
            v = v >= 0 ? 0 : -1;
        DevBuf &d_grid = g->ws.grid, &d_pos = g->ws.pos, &d_next = g->ws.next, &d_prog = g->ws.prog, &d_counts = g->ws.counts;
        d_grid.alloc(gs.v.size() * sizeof(long long), st);
        CU(cudaMemcpyAsync(d_grid.p, gs.v.data(), gs.v.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
        d_pos.alloc(std::max<size_t>(p.cell_pos.size(), 1) * sizeof(int), st);
        CU(cudaMemcpyAsync(d_pos.p, p.cell_pos.data(), p.cell_pos.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        d_next.alloc(std::max<size_t>(p.next_x.size(), 1) * sizeof(int), st);
        CU(cudaMemcpyAsync(d_next.p, p.next_x.data(), p.next_x.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        d_prog.alloc((size_t)p.rows * sizeof(int), st);
        CU(cudaMemcpyAsync(d_prog.p, p.row_first.data(), (size_t)p.rows * sizeof(int), cudaMemcpyHostToDevice, st));
        const int n_ctas = (int)std::max<int64_t>(1, std::min<int64_t>(n_all, select_max_ctas(g->device)));
        d_counts.alloc((size_t)n_ctas * g->n_lib * sizeof(int), st);  // per source image: candidates are slots of g->flips
        CU(cudaMemsetAsync(d_counts.p, 0, d_counts.bytes, st));
        g->fits_flips = g->flips;
        const float *sc = (const float *)a.scores;
        const int *ix = (const int *)a.indices;
        int64_t block_stride = 0;
        if (a.rpb > 0) {
            ix = reinterpret_cast<const int *>(sc + (size_t)a.rpb * a.k);  // indices follow the scores inside every block
            block_stride = 2 * a.rpb * a.k;                                 // in 4-byte elements
        }
        Timer t(st);
        if (g->cand_max_uses > 0) {
            // `used` carries across the steps of one generate: selecting a step at or below the last one starts a new generate, and
            // every earlier step with cells must have been selected since
            if (a.step <= g->cap_last_step)
                g->cap_last_step = -1;
            for (int s = g->cap_last_step + 1; s < a.step; ++s)
                if (!g->plans[s].cell_pos.empty())
                    throw Fail{MOSAIC_ERR_NOT_READY, "usage limit: step " + std::to_string(s) + " must be selected before step " +
                                                         std::to_string(a.step) + " (image uses carry across the steps in order)"};
            if (g->cap_last_step < 0) {
                g->d_used.alloc((size_t)g->n_lib * sizeof(int), st);
                CU(cudaMemsetAsync(g->d_used.p, 0, g->d_used.bytes, st));
            }
            t.start();
            CU(launch_select_capped(d_grid.as<long long>(), d_pos.as<int>(), (int)n_all, p.rows, p.cols, sc, ix, a.k, a.k, sc, ix,
                                    std::min(a.k, kPrefixMax), a.k, (int)g->n_lib, g->repeat_range, g->repeat_addition, g->cand_max_uses,
                                    d_counts.as<int>(), g->d_used.as<int>(), nullptr, st, a.rpb, block_stride));
            t.stop();
            g->cap_last_step = a.step;
        } else {
            t.start();
            CU(launch_select(d_grid.as<long long>(), d_pos.as<int>(), d_next.as<int>(), (int)n_all, p.rows, p.cols, sc, ix, a.k, a.k,
                             (int)g->n_lib, g->repeat_range, g->repeat_addition, d_prog.as<int>(), d_counts.as<int>(), n_ctas, nullptr,
                             st, a.rpb, block_stride));
            t.stop();
        }
        CU(cudaMemcpyAsync(gs.v.data(), d_grid.p, gs.v.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        g->timings.select_ms += t.ms();
        g->timings.kernel_launches += n_all > 0;
        g->timings.d2h_bytes += (double)(gs.v.size() * sizeof(long long));
    }, &a);
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
        Shape top;
        shape_from_c(*shape, mask, top);
        std::string err;
        if (cell_size > 0 && cell_size != top.size) {
            Shape r;
            if (!top.resized(cell_size, r, err))
                return MOSAIC_ERR_UNSUPPORTED;
            top = r;
        }
        Group grp;
        if (!grp.build(top, detail_percent, size_steps, err))
            return MOSAIC_ERR_INVALID_ARGUMENT;
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
