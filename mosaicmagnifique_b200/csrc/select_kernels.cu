// Selection stage: repeat-penalised argmin in the reference's raster order, as a GPU wavefront.
//
// Replaces the reference's serial <<<1,1>>> kernels
//   calculateRepeats  src/Photomosaic/CUDA/PhotomosaicGenerator.cu:127-172
//   findLowestKernel  src/Photomosaic/CUDA/PhotomosaicGenerator.cu:175-196
// with the CPU generator's semantics (CPUPhotomosaicGenerator.cpp:137-169, 185-225):
//   best(x,y) = argmin_i ( A * #{already chosen cells in the window with value i} + D[cell, i] ),
//   strict <, lowest index wins; window = rows y-r..y-1 x columns x-r..x+r, plus row y columns x-r..x-1.
//
// Wavefront: valid cells are dealt to the CTAs of one co-resident (cooperative) grid in raster order.
// A cell may start once every valid cell left of it in its row is final and rows y-r..y-1 are final up
// to column x+r; rows publish "final up to column" counters (release/acquire through L2). All
// dependencies point backwards in raster order, so the earliest unfinished cell can always run.
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include <algorithm>

#include "kernels.h"

namespace mm {

__global__ void fill_u64_kernel(unsigned long long *p, size_t n, unsigned long long v)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = v;
}

cudaError_t launch_fill_u64(unsigned long long *p, size_t n, unsigned long long v, cudaStream_t stream)
{
    if (n == 0)
        return cudaSuccess;
    fill_u64_kernel<<<(unsigned)((n + 255) / 256 > 1024 ? 1024 : (n + 255) / 256), 256, 0, stream>>>(p, n, v);
    return cudaGetLastError();
}

// rows are laid out cell-major: row(cell, v) = cell * V + v; the minimum lands in row(cell, 0)
__global__ void min_variants_kernel(float *D, int n_cells, int V, int n_lib_pad)
{
    const size_t total = (size_t)n_cells * n_lib_pad;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / n_lib_pad, l = i - c * n_lib_pad;
        float *row = D + c * V * (size_t)n_lib_pad + l;
        float m = row[0];
        for (int v = 1; v < V; ++v)
            m = fminf(m, row[(size_t)v * n_lib_pad]);
        row[0] = m;
    }
}

cudaError_t launch_min_variants(float *D, int n_cells, int V, int n_lib_pad, cudaStream_t stream)
{
    const size_t total = (size_t)n_cells * n_lib_pad;
    if (total == 0 || V <= 1)
        return cudaSuccess;
    min_variants_kernel<<<(unsigned)((total + 255) / 256 > 4736 ? 4736 : (total + 255) / 256), 256, 0, stream>>>(D, n_cells, V,
                                                                                                                  n_lib_pad);
    return cudaGetLastError();
}

__global__ void keys_to_grid_kernel(const unsigned long long *best_key, const int *cell_pos, long long *grid, int n_cells,
                                    float *best_score)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells)
        return;
    const unsigned long long k = best_key[c];
    // an untouched key means no library image produced a finite sum: the reference's "should never
    // happen" nullopt (CPUPhotomosaicGenerator.cpp:174-178)
    grid[cell_pos[c]] = (k == ~0ull) ? -1ll : (long long)(k & 0xffffffffull);
    if (best_score)
        best_score[c] = __uint_as_float((unsigned)(k >> 32));
}

cudaError_t launch_keys_to_grid(const unsigned long long *best_key, const int *cell_pos, long long *grid, int n_cells,
                                float *best_score, cudaStream_t stream)
{
    if (n_cells == 0)
        return cudaSuccess;
    keys_to_grid_kernel<<<(n_cells + 255) / 256, 256, 0, stream>>>(best_key, cell_pos, grid, n_cells, best_score);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ top-K candidates per cell

constexpr int kTopkThreads = 256;

// K smallest entries of one row by (score bits, index): 4-pass radix select for the K-th value, then an
// index-ordered compaction so that ties at the threshold keep the lowest indices (the CPU's tie rule).
__global__ void __launch_bounds__(kTopkThreads)
topk_kernel(const float *__restrict__ D, int row_stride, int n_lib, int K, float *__restrict__ cand_score,
            int *__restrict__ cand_idx)
{
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix, s_remaining, s_base;
    __shared__ unsigned scan[kTopkThreads];
    const float *row = D + (size_t)blockIdx.x * row_stride;
    const int tid = threadIdx.x;

    unsigned prefix = 0, remaining = (unsigned)K;  // looking for the remaining-th smallest among keys matching prefix
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        hist[tid] = 0;
        __syncthreads();
        const unsigned mask_hi = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
        for (int i = tid; i < n_lib; i += kTopkThreads) {
            const unsigned b = __float_as_uint(row[i]);
            if ((b & mask_hi) == prefix)
                atomicAdd(&hist[(b >> shift) & 255], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned acc = 0, d = 0;
            for (; d < 256; ++d) {
                if (acc + hist[d] >= remaining)
                    break;
                acc += hist[d];
            }
            s_prefix = prefix | (d << shift);
            s_remaining = remaining - acc;
        }
        __syncthreads();
        prefix = s_prefix;
        remaining = s_remaining;
        __syncthreads();
    }
    // prefix = bits of the K-th smallest value; `remaining` of the entries equal to it are taken (lowest indices)
    const unsigned thr = prefix;
    if (tid == 0)
        s_base = 0;
    unsigned eq_taken = 0;  // uniform across the block: equal-to-threshold entries accepted so far
    float *out_s = cand_score + (size_t)blockIdx.x * K;
    int *out_i = cand_idx + (size_t)blockIdx.x * K;
    __syncthreads();
    for (int base = 0; base < n_lib; base += kTopkThreads) {
        const int i = base + tid;
        unsigned b = 0xffffffffu;
        if (i < n_lib)
            b = __float_as_uint(row[i]);
        const bool less = i < n_lib && b < thr;
        const bool eq = i < n_lib && b == thr;
        // inclusive scans of both predicates (packed: low 16 bits = less, high 16 bits = eq)
        unsigned v = (less ? 1u : 0u) | (eq ? 0x10000u : 0u);
        scan[tid] = v;
        __syncthreads();
        for (int o = 1; o < kTopkThreads; o <<= 1) {
            const unsigned t = tid >= o ? scan[tid - o] : 0u;
            __syncthreads();
            scan[tid] += t;
            __syncthreads();
        }
        const unsigned incl = scan[tid];
        const unsigned total = scan[kTopkThreads - 1];
        const unsigned eq_before = eq_taken + (incl >> 16) - (eq ? 1u : 0u);
        const bool take_eq = eq && eq_before < remaining;
        // number of accepted entries before this one inside the chunk
        const unsigned less_before = (incl & 0xffffu) - (less ? 1u : 0u);
        const unsigned eq_acc_before = min(eq_before, remaining) - min(eq_taken, remaining);
        if (less || take_eq) {
            const unsigned pos = s_base + less_before + eq_acc_before;
            out_s[pos] = __uint_as_float(b);
            out_i[pos] = i;
        }
        __syncthreads();
        const unsigned eq_total = total >> 16;
        const unsigned eq_acc_total = min(eq_taken + eq_total, remaining) - min(eq_taken, remaining);
        if (tid == 0)
            s_base += (total & 0xffffu) + eq_acc_total;
        eq_taken += eq_total;
        __syncthreads();
    }
}

cudaError_t launch_topk(const float *D, int row_stride, int n_lib, int n_cells, int K, float *cand_score, int *cand_idx,
                        cudaStream_t stream)
{
    if (n_cells == 0 || K <= 0)
        return cudaSuccess;
    if (K > n_lib)
        return cudaErrorInvalidValue;
    topk_kernel<<<n_cells, kTopkThreads, 0, stream>>>(D, row_stride, n_lib, K, cand_score, cand_idx);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ pruning threshold

// After pass 0 the M smallest partial sums of a cell name its candidates; their library tiles are completed before anything is
// pruned. Marking: state[cell][tile of the candidate] = kRowComplete.
__global__ void mark_candidates_kernel(const int *__restrict__ cand_idx, int M, int n_rows, const int *__restrict__ inv_perm, int n_lib_tiles,
                                       uint8_t *__restrict__ state)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)n_rows * M; i += (size_t)gridDim.x * blockDim.x) {
        const size_t cell = i / M;
        state[cell * n_lib_tiles + inv_perm[cand_idx[i]] / MM_TNB] = kRowComplete;
    }
}

// T[cell] = k-th smallest complete sum among the cell's M candidates: at least k complete sums are <= T, so the k-th smallest
// sum of the whole row is <= T, and a pair whose (monotone) partial sum is already > T cannot be among the k smallest.
__global__ void threshold_kernel(const float *__restrict__ D, int row_stride, const int *__restrict__ cand_idx, int M, int k,
                                 float *__restrict__ T)
{
    const float *row = D + (size_t)blockIdx.x * row_stride;
    const int *idx = cand_idx + (size_t)blockIdx.x * M;
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
        const float v = row[idx[j]];
        int lt = 0, le = 0;
        for (int i = 0; i < M; ++i) {
            const float u = row[idx[i]];
            lt += u < v;
            le += u <= v;
        }
        if (lt < k && k <= le)
            T[blockIdx.x] = v;  // every thread that writes holds the same value
    }
}

cudaError_t launch_prune_threshold(const float *D, int row_stride, const int *cand_idx, int n_rows, int M, int k, const int *inv_perm,
                                   int n_lib_tiles, uint8_t *state, float *T, bool mark, cudaStream_t stream)
{
    if (n_rows <= 0)
        return cudaSuccess;
    if (k < 1 || k > M)
        return cudaErrorInvalidValue;
    if (mark)
        mark_candidates_kernel<<<(unsigned)std::min<size_t>(((size_t)n_rows * M + 255) / 256, 4096), 256, 0, stream>>>(
            cand_idx, M, n_rows, inv_perm, n_lib_tiles, state);
    else
        threshold_kernel<<<(unsigned)n_rows, 128, 0, stream>>>(D, row_stride, cand_idx, M, k, T);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ wavefront selection

constexpr int kSelThreads = 256;

struct SelArgs {
    long long *grid;
    const int *cell_pos;   // [n_cells] y * cols + x of each valid cell, raster order
    const int *next_x;     // [n_cells] column of the next valid cell in the same row (cols if none)
    int n_cells, rows, cols;
    const float *scores;   // per cell M entries, row stride M_stride
    const int *idx;        // per cell M entries (stride M) or nullptr: entry j is library image j
    int M, M_stride;
    int n_images;          // library images: entry id v is slot v of an orientation-major candidate set, image v % n_images
    int range, addition;
    int *row_progress;     // [rows], initialised to the column of the first valid cell (cols if none)
    int *counts;           // [gridDim.x][n_images] zeroed scratch: occurrences of each library image in the window
    float *margins;        // optional [n_cells][2]: best and second-best PENALISED score (tie-band reporting)
    // all-gathered candidate blocks (multi-GPU): cell c lives in block c / rows_per_block at row c % rows_per_block; blocks are
    // block_stride 4-byte elements apart (scores and indices alike). rows_per_block == 0: one plain array.
    long long rows_per_block, block_stride;
};

__device__ __forceinline__ int ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// (best, id, second) of the union of two disjoint candidate sets: lexicographic (value, slot) minimum, second-best value
__device__ __forceinline__ void merge_best(double &best, int &id, double &second, double ob, int oid, double os)
{
    if (ob < best || (ob == best && oid < id)) {
        second = fmin(best, os);
        best = ob;
        id = oid;
    } else {
        second = fmin(second, ob);
    }
}

__device__ __forceinline__ void warp_best(double &best, int &id, double &second)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oid = __shfl_xor_sync(0xffffffffu, id, o);
        const double os = __shfl_xor_sync(0xffffffffu, second, o);
        merge_best(best, id, second, ob, oid, os);
    }
}

// clamped repeat window of the cell at (y, x) (CPUPhotomosaicGenerator.cpp:188-192): rows y0..y-1 over columns x0..x1, then row y
// over columns x0..x-1; n entries (0 without a penalty)
struct Window {
    int y, y0, x0, x1, ww, n_above, n;
    __device__ Window(int y_, int x, int rows, int cols, int range, bool penalise)
        : y(y_), y0(min(max(y_ - range, 0), rows)), x0(min(max(x - range, 0), cols)), x1(min(max(x + range, 0), cols - 1)),
          ww(x1 - x0 + 1), n_above((y_ - y0) * ww), n(penalise ? n_above + (x - x0) : 0)
    {
    }
    // grid offset of window entry j, raster order
    __device__ size_t cell(int j, int cols) const
    {
        const int ry = j < n_above ? y0 + j / ww : y, rx = j < n_above ? x0 + j % ww : x0 + (j - n_above);
        return (size_t)ry * cols + rx;
    }
};

// offset of cell c's candidate row: row c of a plain array, or row c % rows_per_block of block c / rows_per_block of the all-gathered
// candidate blocks (block_stride 4-byte elements apart)
__device__ __forceinline__ size_t cand_row(int c, size_t stride, long long rows_per_block, long long block_stride)
{
    if (rows_per_block == 0)
        return (size_t)c * stride;
    return (size_t)(c / rows_per_block) * (size_t)block_stride + (size_t)(c % rows_per_block) * stride;
}

__global__ void __launch_bounds__(kSelThreads) select_kernel(SelArgs a)
{
    __shared__ double s_val[kSelThreads / 32];
    __shared__ int s_id[kSelThreads / 32];
    __shared__ double s_second[kSelThreads / 32];
    // repeats count per source image: every orientation of image i shares cnt[i] (kernels.h: launch_select)
    int *cnt = a.counts + (size_t)blockIdx.x * a.n_images;
    const int tid = threadIdx.x;

    for (int c = blockIdx.x; c < a.n_cells; c += gridDim.x) {
        const int pos = a.cell_pos[c];
        const int y = pos / a.cols, x = pos - y * a.cols;
        const bool penalise = a.range > 0 && a.addition != 0;
        const Window win(y, x, a.rows, a.cols, a.range, penalise);

        // ---- wait for the dependencies
        if (penalise) {
            // row y final up to x (exclusive); rows y0..y-1 final up to x1 (inclusive)
            for (int ry = win.y0 + tid; ry <= y; ry += kSelThreads) {
                const int need = ry == y ? x : win.x1 + 1;
                while (ld_acquire(a.row_progress + ry) < need)
                    __nanosleep(64);
            }
        }
        __syncthreads();

        // ---- count the window's library images
        for (int j = tid; j < win.n; j += kSelThreads) {
            const long long v = __ldcg(a.grid + win.cell(j, a.cols));
            if (v >= 0)
                atomicAdd(cnt + v % a.n_images, 1);
        }
        __syncthreads();

        // ---- penalised argmin over this cell's entries
        const float *sc = a.scores + cand_row(c, a.M_stride, a.rows_per_block, a.block_stride);
        const int *ids = a.idx ? a.idx + cand_row(c, a.M, a.rows_per_block, a.block_stride) : nullptr;
        double best = DBL_MAX, second = DBL_MAX;
        int best_id = 0x7fffffff;
        for (int j = tid; j < a.M; j += kSelThreads) {
            const int id = ids ? ids[j] : j;
            const int k = penalise ? __ldcg(cnt + id % a.n_images) : 0;
            merge_best(best, best_id, second, (double)sc[j] + (double)a.addition * (double)k, id, DBL_MAX);
        }
        warp_best(best, best_id, second);
        if ((tid & 31) == 0) {
            s_val[tid >> 5] = best;
            s_id[tid >> 5] = best_id;
            s_second[tid >> 5] = second;
        }
        __syncthreads();

        // ---- undo the counts (every thread revisits its own window entries)
        for (int j = tid; j < win.n; j += kSelThreads) {
            const long long v = __ldcg(a.grid + win.cell(j, a.cols));
            if (v >= 0)
                cnt[v % a.n_images] = 0;
        }

        if (tid == 0) {
            for (int w = 1; w < kSelThreads / 32; ++w)
                merge_best(best, best_id, second, s_val[w], s_id[w], s_second[w]);
            // DBL_MAX start + strict < as in the reference: NaN / inf rows leave the cell unset (nullopt)
            const long long result = (best < DBL_MAX && best_id != 0x7fffffff) ? (long long)best_id : -1ll;
            __stcg(a.grid + pos, result);
            if (a.margins) {
                a.margins[2 * c] = (float)best;
                a.margins[2 * c + 1] = (float)second;
            }
        }
        __syncthreads();  // count resets and the result are complete before the row counter moves
        if (tid == 0) {
            __threadfence();
            st_release(a.row_progress + y, a.next_x[c]);
        }
    }
}

cudaError_t launch_select(long long *grid, const int *cell_pos, const int *next_x, int n_cells, int rows, int cols,
                          const float *scores, const int *idx, int M, int M_stride, int n_images, int repeat_range,
                          int repeat_addition, int *row_progress, int *counts, int n_ctas, float *margins,
                          cudaStream_t stream, long long rows_per_block, long long block_stride)
{
    if (n_cells == 0)
        return cudaSuccess;
    if (n_images < 1)
        return cudaErrorInvalidValue;
    SelArgs a{grid, cell_pos, next_x, n_cells, rows, cols, scores, idx, M, M_stride, n_images, repeat_range, repeat_addition,
              row_progress, counts, margins, rows_per_block, block_stride};
    void *args[] = {&a};
    // cooperative launch: fails instead of deadlocking if the CTAs could not all be resident
    return cudaLaunchCooperativeKernel((void *)select_kernel, dim3(n_ctas), dim3(kSelThreads), args, 0, stream);
}

int select_max_ctas(int device)
{
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, select_kernel, kSelThreads, 0);
    return sms * (per_sm > 0 ? 1 : 0);
}

// ------------------------------------------------------------------ usage limit: sorted candidate prefixes

constexpr int kSortThreads = 512;

// One CTA per row. sel_s / sel_pos hold the k0 smallest entries of the row's source by (score bits, position), positions ascending
// (launch_topk). Without a list the source is a D row (position = slot) and sel_s / sel_pos are sorted in place by (score, slot).
// With a list (a top-K candidate row of K entries, slots ascending, so position order is slot order) the k0 entries move to the
// front of the list, sorted; the list entries they displace take the positions the k0 entries left, so the row keeps its K entries.
__global__ void __launch_bounds__(kSortThreads)
sort_prefix_kernel(float *__restrict__ sel_s, int *__restrict__ sel_pos, int k0, float *__restrict__ list_s, int *__restrict__ list_i, int K)
{
    __shared__ unsigned long long key[kPrefixMax];
    __shared__ unsigned char in_front[kPrefixMax];  // list position < k0 holds one of the k0 entries
    __shared__ int word_base[kPrefixMax / 32];
    const int tid = threadIdx.x, lane = tid & 31;
    float *ss = sel_s + (size_t)blockIdx.x * k0;
    int *sp = sel_pos + (size_t)blockIdx.x * k0;
    float *ls = list_s ? list_s + (size_t)blockIdx.x * K : nullptr;
    int *li = list_s ? list_i + (size_t)blockIdx.x * K : nullptr;
    int n2 = 1;
    while (n2 < k0)
        n2 <<= 1;
    for (int j = tid; j < kPrefixMax; j += kSortThreads) {
        unsigned long long k = ~0ull;
        if (j < k0) {
            const int p = sp[j];
            k = (unsigned long long)__float_as_uint(ss[j]) << 32 | (unsigned)(ls ? li[p] : p);
        }
        key[j] = k;
        in_front[j] = 0;
    }
    __syncthreads();
    // bitonic sort of the n2 keys (scores are sums of non-negative terms, +inf when pruned: their bits order like the values)
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n2; i += kSortThreads) {
                const int o = i ^ j;
                if (o > i) {
                    const unsigned long long a = key[i], b = key[o];
                    if ((a > b) == ((i & k) == 0)) {
                        key[i] = b;
                        key[o] = a;
                    }
                }
            }
            __syncthreads();
        }
    if (!ls) {
        for (int j = tid; j < k0; j += kSortThreads) {
            ss[j] = __uint_as_float((unsigned)(key[j] >> 32));
            sp[j] = (int)(key[j] & 0xffffffffu);
        }
        return;
    }
    // t of the k0 entries already sit in front; the other k0 - t (sel_pos[t..k0), ascending) sit behind it. They swap places with
    // the k0 - t front entries that are not among them, paired in position order.
    for (int j = tid; j < k0; j += kSortThreads)
        if (sp[j] < k0)
            in_front[sp[j]] = 1;
    __syncthreads();
    unsigned m[kPrefixMax / kSortThreads];
    for (int r = 0; r < kPrefixMax / kSortThreads; ++r) {
        const int a = tid + r * kSortThreads;
        m[r] = __ballot_sync(0xffffffffu, a < k0 && !in_front[a]);
        if (lane == 0)
            word_base[a >> 5] = __popc(m[r]);
    }
    __shared__ int s_leaving;
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int w = 0; w < kPrefixMax / 32; ++w) {
            const int c = word_base[w];
            word_base[w] = acc;
            acc += c;
        }
        s_leaving = acc;
    }
    __syncthreads();
    const int t = k0 - s_leaving;
    float out_s[kPrefixMax / kSortThreads];
    int out_i[kPrefixMax / kSortThreads], out_to[kPrefixMax / kSortThreads];
    for (int r = 0; r < kPrefixMax / kSortThreads; ++r) {
        const int a = tid + r * kSortThreads;
        out_to[r] = -1;
        if (m[r] >> lane & 1u) {  // the rank-th front entry that leaves goes to sel_pos[t + rank]
            out_to[r] = sp[t + word_base[a >> 5] + __popc(m[r] & ((1u << lane) - 1u))];
            out_s[r] = ls[a];
            out_i[r] = li[a];
        }
    }
    __syncthreads();  // every displaced entry is read before the front is overwritten
    for (int r = 0; r < kPrefixMax / kSortThreads; ++r)
        if (out_to[r] >= 0) {
            ls[out_to[r]] = out_s[r];
            li[out_to[r]] = out_i[r];
        }
    for (int j = tid; j < k0; j += kSortThreads) {
        ls[j] = __uint_as_float((unsigned)(key[j] >> 32));
        li[j] = (int)(key[j] & 0xffffffffu);
    }
}

cudaError_t launch_sort_prefix(float *sel_s, int *sel_pos, int n_rows, int k0, float *list_s, int *list_i, int K, cudaStream_t stream)
{
    if (n_rows == 0)
        return cudaSuccess;
    if (k0 < 1 || k0 > kPrefixMax || (list_s && (!list_i || K < k0)))
        return cudaErrorInvalidValue;
    sort_prefix_kernel<<<n_rows, kSortThreads, 0, stream>>>(sel_s, sel_pos, k0, list_s, list_i, K);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ usage limit: sequential capped selection

constexpr int kCapThreads = 256;

struct CapArgs {
    long long *grid;
    const int *cell_pos;
    int n_cells, rows, cols;
    const float *scores;   // full candidate row of every cell (M entries, stride M_stride): the fallback
    const int *idx;        // nullptr: entry j is slot j (a D row)
    int M, M_stride;
    const float *pscores;  // sorted prefix of every cell: the k0 smallest (score, slot), stride p_stride
    const int *pidx;
    int k0, p_stride;
    int n_images, range, addition, max_uses;
    int *counts;           // [n_images] zeroed scratch: window occurrences
    int *used;             // [n_images] choices so far in this generate
    float *margins;
    long long rows_per_block, block_stride;  // all-gathered candidate blocks, as SelArgs (prefix and row share them)
};

// One CTA walks the step's valid cells in raster order (every choice depends on all earlier ones through `used`). Per cell: window
// counts as select_kernel; warp 0 scans the sorted prefix 32 entries at a time and stops once the next entry's unpenalised score is
// strictly above the best (with margins: second-best) allowed penalised score -- every later entry scores at least that much, and
// an equal one can only win on a lower slot if it is unpenalised, so it is still examined. A prefix that ends first means the
// answer may lie behind it: the whole block then scans the cell's full row.
__global__ void __launch_bounds__(kCapThreads) select_capped_kernel(CapArgs a)
{
    __shared__ double s_val[kCapThreads / 32], s_second[kCapThreads / 32];
    __shared__ int s_id[kCapThreads / 32];
    __shared__ int s_fallback;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool penalise = a.range > 0 && a.addition != 0;
    const bool margins = a.margins != nullptr;

    for (int c = 0; c < a.n_cells; ++c) {
        const int pos = a.cell_pos[c];
        const int y = pos / a.cols, x = pos - y * a.cols;
        const Window win(y, x, a.rows, a.cols, a.range, penalise);
        for (int j = tid; j < win.n; j += kCapThreads) {
            const long long v = a.grid[win.cell(j, a.cols)];
            if (v >= 0)
                atomicAdd(a.counts + v % a.n_images, 1);
        }
        __syncthreads();

        if (warp == 0) {
            const size_t prow = cand_row(c, a.p_stride, a.rows_per_block, a.block_stride);
            const float *ps = a.pscores + prow;
            const int *pi = a.pidx + prow;
            double best = DBL_MAX, second = DBL_MAX;
            int best_id = 0x7fffffff;
            bool stopped = false;
            float s = lane < a.k0 ? ps[lane] : 0.0f;
            int id = lane < a.k0 ? pi[lane] : 0;
            for (int j0 = 0; j0 < a.k0; j0 += 32) {
                const float first = __shfl_sync(0xffffffffu, s, 0);
                if ((double)first > (margins ? second : best)) {
                    stopped = true;
                    break;
                }
                const bool have = j0 + lane < a.k0;
                const float cs = s;
                const int cid = id;
                if (j0 + 32 + lane < a.k0) {  // next chunk's loads overlap this chunk's reduction
                    s = ps[j0 + 32 + lane];
                    id = pi[j0 + 32 + lane];
                }
                double v = DBL_MAX;
                int vid = 0x7fffffff;
                if (have) {
                    const int img = cid % a.n_images;
                    if (a.used[img] < a.max_uses) {
                        v = (double)cs + (double)a.addition * (double)(penalise ? __ldcg(a.counts + img) : 0);
                        vid = cid;
                    }
                }
                double vs = DBL_MAX;
                warp_best(v, vid, vs);
                merge_best(best, best_id, second, v, vid, vs);
            }
            if (lane == 0) {
                s_val[0] = best;
                s_id[0] = best_id;
                s_second[0] = second;
                s_fallback = !stopped && a.k0 < a.M;
            }
        }
        __syncthreads();

        if (s_fallback) {  // uniform: the block scans the full row
            const float *sc = a.scores + cand_row(c, a.M_stride, a.rows_per_block, a.block_stride);
            const int *ids = a.idx ? a.idx + cand_row(c, a.M, a.rows_per_block, a.block_stride) : nullptr;
            double best = DBL_MAX, second = DBL_MAX;
            int best_id = 0x7fffffff;
            for (int j = tid; j < a.M; j += kCapThreads) {
                const int id = ids ? ids[j] : j;
                const int img = id % a.n_images;
                if (a.used[img] < a.max_uses)
                    merge_best(best, best_id, second, (double)sc[j] + (double)a.addition * (double)(penalise ? __ldcg(a.counts + img) : 0), id,
                               DBL_MAX);
            }
            warp_best(best, best_id, second);
            if (lane == 0) {
                s_val[warp] = best;
                s_id[warp] = best_id;
                s_second[warp] = second;
            }
            __syncthreads();
            if (tid == 0)
                for (int w = 1; w < kCapThreads / 32; ++w)
                    merge_best(s_val[0], s_id[0], s_second[0], s_val[w], s_id[w], s_second[w]);
        }

        // undo the window counts (every thread revisits its own window entries); then the choice
        for (int j = tid; j < win.n; j += kCapThreads) {
            const long long v = a.grid[win.cell(j, a.cols)];
            if (v >= 0)
                a.counts[v % a.n_images] = 0;
        }
        if (tid == 0) {
            const double best = s_val[0];
            const int best_id = s_id[0];
            const long long result = (best < DBL_MAX && best_id != 0x7fffffff) ? (long long)best_id : -1ll;
            a.grid[pos] = result;
            if (result >= 0)
                a.used[best_id % a.n_images] += 1;
            if (margins) {
                a.margins[2 * c] = (float)best;
                a.margins[2 * c + 1] = (float)s_second[0];
            }
        }
        __syncthreads();  // counts reset, grid and used updated before the next cell reads them
    }
}

cudaError_t launch_select_capped(long long *grid, const int *cell_pos, int n_cells, int rows, int cols, const float *scores, const int *idx,
                                 int M, int M_stride, const float *pscores, const int *pidx, int k0, int p_stride, int n_images,
                                 int repeat_range, int repeat_addition, int max_uses, int *counts, int *used, float *margins,
                                 cudaStream_t stream, long long rows_per_block, long long block_stride)
{
    if (n_cells == 0)
        return cudaSuccess;
    if (n_images < 1 || max_uses < 1 || k0 < 1 || k0 > M)
        return cudaErrorInvalidValue;
    CapArgs a{grid, cell_pos, n_cells, rows, cols, scores, idx, M, M_stride, pscores, pidx, k0, p_stride, n_images, repeat_range,
              repeat_addition, max_uses, counts, used, margins, rows_per_block, block_stride};
    select_capped_kernel<<<1, kCapThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mm
