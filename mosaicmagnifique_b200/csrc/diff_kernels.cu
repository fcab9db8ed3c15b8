// Fused masked difference-sum kernel: D[cell, lib] = sum_p w[cell,p] * diff(cell[p], lib[p]).
//
// Replaces, in ONE launch per size step, the reference's per-(cell, library image) chain
//   imageDifference / imageDifferenceEdge  src/Photomosaic/CUDA/PhotomosaicGenerator.cu:35-72
//   reduceAdd tree + D2D copies            src/Photomosaic/CUDA/Reduction.cu:24-211
//   flattenKernel                          src/Photomosaic/CUDA/PhotomosaicGenerator.cu:201-209
// and, when no repeat penalty is active, findLowestKernel (:175-189) through the argmin epilogue.
// CPU semantics followed: CPUPhotomosaicGenerator.cpp:137-169 (masked, bounded sum; strict <,
// lowest index wins).
//
// Data layout (built by prep_kernels.cu):
//   lib  : float4 (x0,x1,x2,-)  [lib_tile][chunk][TNB][KP]   one contiguous 16 KB block per (tile, chunk)
//          CIEDE2000: stored-scale channels (L/2-25, a/50, b/50, C/50), w = 50, and image PAIRS interleaved for the packed
//          FP32 path: [lib_tile][chunk][TNB/2][2][KP] float4 = (L0,L1,a0,a1) then (b0,b1,C0,C1)
//   cell : float4 (x0,x1,x2,C)  [cell_tile][chunk][TCB][KP]  followed by float w[TCB][KP] -> 20 KB block
//   w = 1 where the (flipped) detail mask is set and the pixel lies inside the cell's detail-space bound,
//   else 0; pixels are stored in the compacted order of the step's active-pixel list, padded with w = 0.
//
// Kernel shape: one CTA = 8 consumer warps + 1 producer warp. The producer lane streams (cell block,
// lib block) pairs into a 3-stage shared-memory ring with cp.async.bulk (TMA bulk copy, UBLKCP in SASS)
// completing on "full" mbarriers; consumers release stages through "empty" mbarriers. Consumer warp w
// owns cell w of the tile, its 32 lanes stride the chunk's pixels (conflict-free LDS.128), and every lane
// keeps TNB running sums, reduced with warp shuffles at the end. Roofline: FP32 + MUFU issue (DESIGN.md).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>
#include <cub/device/device_scan.cuh>

#include "colour_math.cuh"
#include "kernels.h"

namespace mm {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

#ifndef MM_PIXEL_UNROLL
#define MM_PIXEL_UNROLL 1
#endif
constexpr int kPixelUnroll = MM_PIXEL_UNROLL;
constexpr int kStages = MM_STAGES;
constexpr int kConsumerWarps = MM_TCB;
constexpr int kThreads = (kConsumerWarps + 1) * 32;
constexpr uint32_t kLibBlockBytes = MM_TNB * MM_KP * 16;
constexpr uint32_t kCellBlockBytes = MM_TCB * MM_KP * 20;
constexpr uint32_t kStageBytes = kLibBlockBytes + kCellBlockBytes;

// Consumer side of the ring: warp `warp` walks nk chunks of its cell slot against the 8 library images of the stage and leaves,
// per lane, the TNB running sums of the pixels it strode over. Shared by both kernels below, so that a pair's arithmetic (and the
// measured loop body, DESIGN.md 4.1) is the same whichever launch computes it.
template <int DIFF>
__device__ __forceinline__ void consume_ring(const unsigned char *smem, uint64_t *full_bar, uint64_t *empty_bar, int nk, int warp,
                                             int lane, float (&acc)[MM_TNB])
{
#pragma unroll
    for (int i = 0; i < MM_TNB; ++i)
        acc[i] = 0.0f;

    for (int k = 0; k < nk; ++k) {
        const int s = k % kStages;
        mbar_wait(&full_bar[s], (k / kStages) & 1);
        if (MM_STRESS_SKEW)
            __nanosleep((unsigned)((warp * 97 + k * 29 + blockIdx.x * 7) % 400));
        const float4 *lib_s = reinterpret_cast<const float4 *>(smem + (size_t)s * kStageBytes);
        const float4 *cell_s = reinterpret_cast<const float4 *>(smem + (size_t)s * kStageBytes + kLibBlockBytes) + warp * MM_KP;
        const float *w_s = reinterpret_cast<const float *>(smem + (size_t)s * kStageBytes + kLibBlockBytes + MM_TCB * MM_KP * 16) + warp * MM_KP;
#pragma unroll kPixelUnroll
        for (int j = 0; j < MM_KP / 32; ++j) {
            const int p = j * 32 + lane;
            const float4 c = cell_s[p];
            const float w = w_s[p];
            if (DIFF == MM_DIFF_CIEDE2000) {
                // packed FP32: two library images per lane vector. The tile stores image pairs interleaved:
                // [pair][0][p] = (L0, L1, a0, a1), [pair][1][p] = (b0, b1, C0, C1)  (prep_kernels.cu)
#pragma unroll
                for (int i = 0; i < MM_TNB / 2; ++i) {
                    const float4 la = lib_s[(i * 2 + 0) * MM_KP + p];
                    const float4 lb = lib_s[(i * 2 + 1) * MM_KP + p];
                    const mm_f2 d = mm_ciede2000_stored_v<mm_f2>(c.x, c.y, c.z, c.w, mm_f2{la.x, la.y}, mm_f2{la.z, la.w},
                                                               mm_f2{lb.x, lb.y}, mm_f2{lb.z, lb.w});
                    const mm_f2 a2 = v_fma(mm_f2{w, w}, d, mm_f2{acc[2 * i], acc[2 * i + 1]});
                    acc[2 * i] = a2.x;
                    acc[2 * i + 1] = a2.y;
                }
            } else {
#pragma unroll
                for (int i = 0; i < MM_TNB; ++i) {
                    const float4 l = lib_s[i * MM_KP + p];
                    acc[i] = fmaf(w, mm_euclid(c.x, c.y, c.z, l.x, l.y, l.z), acc[i]);
                }
            }
        }
        __syncwarp();
        if (lane == 0)
            mbar_arrive(&empty_bar[s]);
    }
}

template <int DIFF>
__global__ void __launch_bounds__(kThreads, MM_MIN_CTAS)
diff_sum_kernel(const unsigned char *__restrict__ cells, const unsigned char *__restrict__ lib, float *__restrict__ D,
                unsigned long long *__restrict__ best_key, int n_chunks, int n_lib, int n_lib_pad, int n_cells,
                int n_cell_tiles, int n_lib_tiles, const int *__restrict__ cancel, unsigned long long *__restrict__ progress,
                int nk, int sb_a, int sb_b)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full_bar[kStages];
    __shared__ uint64_t empty_bar[kStages];
    __shared__ int s_cancelled;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int cell_tile, lib_tile;
    {
        // super-block raster (kernels.h: Raster): keep a column of sb_a cell tiles and sweep the library in bands of sb_b tiles
        const unsigned id = blockIdx.x;
        const unsigned col_all = (unsigned)sb_a * (unsigned)n_lib_tiles;
        const unsigned cb = id / col_all;
        const unsigned r = id - cb * col_all;
        const int cw = min(sb_a, n_cell_tiles - (int)cb * sb_a);
        const unsigned band_ctas = (unsigned)cw * (unsigned)sb_b;
        const unsigned band = r / band_ctas;
        const unsigned r2 = r - band * band_ctas;
        cell_tile = (int)cb * sb_a + (int)(r2 % cw);
        lib_tile = (int)band * sb_b + (int)(r2 / cw);
    }

    if (threadIdx.x == 0) {
        const int cancelled = cancel ? load_cancel_flag(cancel) : 0;  // device word (L2 hit), in flight during the barrier set-up
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kConsumerWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_cancelled = cancelled;
    }
    __syncthreads();
    if (s_cancelled)
        return;  // cancel(): nothing has been issued yet, the whole CTA leaves

    if (warp == kConsumerWarps) {
        // ---------------- producer warp: one elected lane drives the TMA ring
        if (lane == 0) {
            const unsigned char *cell_src = cells + (size_t)cell_tile * n_chunks * kCellBlockBytes;
            const unsigned char *lib_src = lib + (size_t)lib_tile * n_chunks * kLibBlockBytes;
            for (int k = 0; k < nk; ++k) {
                const int s = k % kStages;
                if (k >= kStages)
                    mbar_wait(&empty_bar[s], ((k / kStages) - 1) & 1);
                unsigned char *dst = smem + (size_t)s * kStageBytes;
                if (MM_STRESS_SKEW)
                    __nanosleep((unsigned)((k * 131 + blockIdx.x * 17) % 300));
                mbar_expect_tx(&full_bar[s], kStageBytes);
                bulk_g2s(dst, lib_src + (size_t)k * kLibBlockBytes, kLibBlockBytes, &full_bar[s]);
                bulk_g2s(dst + kLibBlockBytes, cell_src + (size_t)k * kCellBlockBytes, kCellBlockBytes, &full_bar[s]);
            }
        }
        return;
    }

    // ---------------- consumer warps: warp = cell within the tile, lanes stride pixels
    float acc[MM_TNB];
    consume_ring<DIFF>(smem, full_bar, empty_bar, nk, warp, lane, acc);

    // ---------------- epilogue: warp-shuffle reduction, D store, fused argmin
#pragma unroll
    for (int i = 0; i < MM_TNB; ++i) {
        float v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            v += __shfl_xor_sync(0xffffffffu, v, o);
        acc[i] = v;
    }
    const int cell = cell_tile * MM_TCB + warp;
    if (lane < MM_TNB) {
        float v = 0.0f;
#pragma unroll
        for (int i = 0; i < MM_TNB; ++i)
            v = (lane == i) ? acc[i] : v;
        const int li = lib_tile * MM_TNB + lane;
        if (D)
            D[(size_t)cell * n_lib_pad + li] = v;
        if (best_key && li < n_lib && cell < n_cells) {
            // non-negative floats order like their bit patterns; low word = index -> lowest index wins ties
            const unsigned long long key = ((unsigned long long)__float_as_uint(v) << 32) | (unsigned)li;
            atomicMin(best_key + cell, key);
        }
    }
    if (progress && threadIdx.x == 0)
        atomicAdd(progress, 1ull);  // consumer warp 0 has stored its results; an approximate "tiles done" count is all that is needed
}

template <int DIFF>
static cudaError_t launch(const void *cells, const void *lib, float *D, unsigned long long *best_key, int n_cell_tiles,
                          int n_lib_tiles, int n_chunks, int n_lib, int n_cells, cudaStream_t stream, const int *cancel,
                          unsigned long long *progress, Raster raster)
{
    const size_t smem = (size_t)kStages * kStageBytes;
    // per device (context) attribute: set on every launch, it is cheap
    cudaError_t e = cudaFuncSetAttribute(diff_sum_kernel<DIFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess)
        return e;
    const unsigned grid = (unsigned)n_cell_tiles * (unsigned)n_lib_tiles;  // 1-D, super-block rasterisation (kernels.h)
    diff_sum_kernel<DIFF><<<grid, kThreads, smem, stream>>>((const unsigned char *)cells, (const unsigned char *)lib, D, best_key, n_chunks,
                                                            n_lib, n_lib_tiles * MM_TNB, n_cells, n_cell_tiles, n_lib_tiles, cancel,
                                                            progress, n_chunks, raster.sb_a, raster.sb_b);
    return cudaGetLastError();
}

cudaError_t launch_diff_sum(int diff_type, const void *cells, const void *lib, float *D, unsigned long long *best_key,
                            int n_cell_tiles, int n_lib_tiles, int n_chunks, int n_lib, int n_cells, cudaStream_t stream,
                            const int *cancel, unsigned long long *progress)
{
    if (n_cell_tiles <= 0 || n_lib_tiles <= 0 || n_chunks <= 0)
        return cudaSuccess;
    if (diff_type != MM_DIFF_CIEDE2000)
        return cudaErrorInvalidValue;  // RGB Euclidean / CIE76 run diff_euclid_kernel (diff_euclid.cu)
    auto env = [](const char *name) -> int {
        const char *v = getenv(name);
        return v ? atoi(v) : 0;
    };
    // Measured on config 4 (ncu dram__bytes_read, profiles/r2_raster_sweep.txt): whole cells per CTA, 16 x 16 super-blocks:
    // 47.4 GB at the kernel's compute-bound time. MM_SB_A / MM_SB_B in the environment override the shape (tuning).
    Raster r{std::min(kSuperTiles, n_cell_tiles), std::min(kSuperTiles, n_lib_tiles)};
    if (env("MM_SB_A") > 0)
        r.sb_a = std::min(env("MM_SB_A"), n_cell_tiles);
    if (env("MM_SB_B") > 0)
        r.sb_b = std::min(env("MM_SB_B"), n_lib_tiles);
    return launch<MM_DIFF_CIEDE2000>(cells, lib, D, best_key, n_cell_tiles, n_lib_tiles, n_chunks, n_lib, n_cells, stream, cancel, progress,
                                     r);
}

// ---------------------------------------------------------------- row work lists (segment passes, exact pruning)

// One CTA = one group of up to 8 rows (cell x library tile) that share a library tile. Bucket b = column * n_lib_tiles + lib_tile
// holds the bucket's listed cells (in cell order) at cells[b * col_cells ...]; groups[] is the exclusive scan of its group counts.
// The producer streams the tile's 16 KB library block and, per warp, that cell's 2 KB pixel slice + 512 B weight slice of its cell
// block: the shared-memory stage has exactly the layout of diff_sum_kernel's, so the consumer loop is the same code. A group with
// fewer than 8 rows repeats its first cell in the empty warps and does not store them.
__global__ void __launch_bounds__(kThreads, MM_MIN_CTAS)
diff_rows_kernel(const unsigned char *__restrict__ cells, const unsigned char *__restrict__ lib, float *__restrict__ D, int n_chunks,
                 int nk, int n_lib_pad, int n_lib_tiles, RowList rows, const int *__restrict__ perm, const int *cancel,
                 unsigned long long *__restrict__ progress)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full_bar[kStages];
    __shared__ uint64_t empty_bar[kStages];
    __shared__ int s_cancelled, s_cell[kConsumerWarps], s_lib_tile, s_n_rows;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        const int cancelled = cancel ? load_cancel_flag(cancel) : 0;  // device word (L2 hit), in flight during the set-up
        // bucket of this group: last b with groups[b] <= blockIdx.x (groups is non-decreasing, groups[0] = 0)
        int lo = 0, hi = rows.n_buckets;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (rows.groups[mid] <= (int)blockIdx.x)
                lo = mid;
            else
                hi = mid;
        }
        const int g = (int)blockIdx.x - rows.groups[lo];
        const int n_in = min(kConsumerWarps, rows.count[lo] - g * kConsumerWarps);
        const int *list = rows.cells + (size_t)lo * rows.col_cells + g * kConsumerWarps;
        for (int w = 0; w < kConsumerWarps; ++w)
            s_cell[w] = list[w < n_in ? w : 0];
        s_lib_tile = lo % n_lib_tiles;
        s_n_rows = n_in;
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kConsumerWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_cancelled = cancelled;
    }
    __syncthreads();
    if (s_cancelled)
        return;  // cancel(): nothing has been issued yet, the whole CTA leaves
    const int lib_tile = s_lib_tile;

    if (warp == kConsumerWarps) {
        if (lane == 0) {
            const unsigned char *lib_src = lib + (size_t)lib_tile * n_chunks * kLibBlockBytes;
            constexpr uint32_t kSlice = MM_KP * 16, kWSlice = MM_KP * 4;
            for (int k = 0; k < nk; ++k) {
                const int s = k % kStages;
                if (k >= kStages)
                    mbar_wait(&empty_bar[s], ((k / kStages) - 1) & 1);
                unsigned char *dst = smem + (size_t)s * kStageBytes;
                if (MM_STRESS_SKEW)
                    __nanosleep((unsigned)((k * 131 + blockIdx.x * 17) % 300));
                mbar_expect_tx(&full_bar[s], kLibBlockBytes + kConsumerWarps * (kSlice + kWSlice));
                bulk_g2s(dst, lib_src + (size_t)k * kLibBlockBytes, kLibBlockBytes, &full_bar[s]);
                for (int w = 0; w < kConsumerWarps; ++w) {
                    const int c = s_cell[w];
                    const unsigned char *blk = cells + ((size_t)(c / MM_TCB) * n_chunks + k) * kCellBlockBytes;
                    const int slot = c % MM_TCB;
                    bulk_g2s(dst + kLibBlockBytes + w * kSlice, blk + slot * kSlice, kSlice, &full_bar[s]);
                    bulk_g2s(dst + kLibBlockBytes + MM_TCB * kSlice + w * kWSlice, blk + MM_TCB * kSlice + slot * kWSlice, kWSlice,
                             &full_bar[s]);
                }
            }
        }
        return;
    }

    float acc[MM_TNB];
    consume_ring<MM_DIFF_CIEDE2000>(smem, full_bar, empty_bar, nk, warp, lane, acc);
#pragma unroll
    for (int i = 0; i < MM_TNB; ++i) {
        float v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            v += __shfl_xor_sync(0xffffffffu, v, o);
        acc[i] = v;
    }
    if (warp < s_n_rows && lane < MM_TNB) {
        float v = 0.0f;
#pragma unroll
        for (int i = 0; i < MM_TNB; ++i)
            v = (lane == i) ? acc[i] : v;
        // segments are added in pass order, one pass at a time: D = ((seg 0 + seg 1) + seg 2) + ... for every pair
        float *d = D + (size_t)s_cell[warp] * n_lib_pad + perm[lib_tile * MM_TNB + lane];
        *d += v;
    }
    if (progress && threadIdx.x == 0)
        atomicAdd(progress, (unsigned long long)s_n_rows);
}

cudaError_t launch_diff_rows(const void *cells, const void *lib, float *D, int n_groups, int n_lib_tiles, int n_chunks, int k0, int nk,
                             RowList rows, const int *perm, cudaStream_t stream, const int *cancel, unsigned long long *progress)
{
    if (n_groups <= 0 || nk <= 0)
        return cudaSuccess;
    const size_t smem = (size_t)kStages * kStageBytes;
    cudaError_t e = cudaFuncSetAttribute(diff_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess)
        return e;
    // the kernel gets its tensors pre-offset to the segment's first chunk; the tile stride inside them stays n_chunks
    diff_rows_kernel<<<(unsigned)n_groups, kThreads, smem, stream>>>(
        (const unsigned char *)cells + (size_t)k0 * kCellBlockBytes, (const unsigned char *)lib + (size_t)k0 * kLibBlockBytes, D, n_chunks, nk,
        n_lib_tiles * MM_TNB, n_lib_tiles, rows, perm, cancel, progress);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- lightness bound of the segments not yet summed (DESIGN.md 4.1)

// Per pixel the kernel's value is sqrt(N) / den25 with N = X^2 + Y (Y + R_T Z) + Z^2 (colour_math.cuh). For |R_T| < 2 the part
// after X^2 is a positive semi-definite form, so N >= X^2 and dE/50 >= |X| / den25 = |dLh| / sl25, sl25 = 25 S_L(lm), lm = Lbar - 50
// = Lh_cell + Lh_lib. S_L = 1 + 0.015 lm^2 / sqrt(20 + lm^2) <= 1 + 0.015 |lm| because sqrt(20 + lm^2) >= |lm|, and S_L grows with
// |lm|. Over a block of MM_BB compacted pixels where every cell weight is w, the triangle inequality gives
//     sum_p w |dLh_p| / sl25_p  >=  w |sum_p Lh_lib,p - sum_p Lh_cell,p| / (25 + 0.375 m),   m = max(|lo|, |hi|),
// with lo = min Lh_cell + min Lh_lib <= lm_p <= max Lh_cell + max Lh_lib = hi. A block whose weights differ contributes 0.
//
// Rounding. The block sums are FP32 sums of 16 values |Lh| <= 25: each is within 15 * 2^-24 * 400 < 3.6e-4 of its exact value and
// their difference adds < 4.8e-5, so kSumErr = 2^-10 is subtracted from every |difference| (this also covers pixels whose |dLh| <
// 1e-19 flush to a zero N under ftz). What remains is relative: the kernel's per-pixel value is within ~1e-5 of the formula
// (rsqrt.approx / sqrt.approx, colour_math.cuh; the tiny terms only raise t and leave rsq(N den^2 + tiny) within 1e-18 of
// rsq(N den^2) since N >= 1e-12 whenever dLh != 0), a pair's FP32 sums of at most 16,384 non-negative terms lose < 1e-3 -- all
// in the direction that could put a computed sum below its exact value -- and this kernel's own rcp.approx and FP32 sums of
// non-negative terms lose < 3e-4. kSlack = 1 - 2^-8 covers all of it: R stays below what the kernels will sum. The dropped dTheta
// Gaussian and the R_T polynomial enter only through R_T, and the bound holds for any |R_T| < 2.
constexpr int kBoundThreads = 128, kBoundRows = 8;
constexpr float kSumErr = 0x1p-10f, kSlack = 1.0f - 0x1p-8f;

// One thread per library slot (coalesced over lib_stats and R) and kBoundRows cell rows (their statistics are warp-uniform loads).
// Segments are walked from the last, so that every R[s] is the running suffix sum.
__global__ void __launch_bounds__(kBoundThreads)
prune_bound_kernel(const float4 *__restrict__ lib_stats, const float4 *__restrict__ cell_stats, int n_rows, int n_lib_pad, int n_blocks,
                   int seg_blocks, int n_segs, float *__restrict__ R, const float *__restrict__ D, const int *__restrict__ perm,
                   float *__restrict__ score)
{
    const int slot = blockIdx.x * kBoundThreads + threadIdx.x;
    const int row0 = blockIdx.y * kBoundRows;
    if (slot >= n_lib_pad)
        return;
    const int nr = min(kBoundRows, n_rows - row0);
    const size_t plane = (size_t)n_rows * n_lib_pad;
    float suffix[kBoundRows];
#pragma unroll
    for (int r = 0; r < kBoundRows; ++r)
        suffix[r] = 0.0f;
    for (int seg = n_segs - 1; seg >= 1; --seg) {
        float acc[kBoundRows];
#pragma unroll
        for (int r = 0; r < kBoundRows; ++r)
            acc[r] = 0.0f;
        const int b1 = min(n_blocks, (seg + 1) * seg_blocks);
        for (int b = seg * seg_blocks; b < b1; ++b) {
            const float4 l = lib_stats[(size_t)b * n_lib_pad + slot];
#pragma unroll
            for (int r = 0; r < kBoundRows; ++r) {
                const float4 c = cell_stats[(size_t)min(row0 + r, n_rows - 1) * n_blocks + b];  // (sum, min, max, w)
                const float d = fmaxf(fabsf(l.x - c.x) - kSumErr, 0.0f);
                const float m = fmaxf(fabsf(l.y + c.y), fabsf(l.z + c.z));
                acc[r] = fmaf(c.w * d, mm_rcp(fmaf(25.0f * 0.015f, m, 25.0f)), acc[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < kBoundRows; ++r) {
            suffix[r] += acc[r];
            if (r < nr)
                R[(size_t)(seg - 1) * plane + (size_t)(row0 + r) * n_lib_pad + slot] = suffix[r] * kSlack;
        }
    }
    if (score) {
        const int j = perm[slot];
#pragma unroll
        for (int r = 0; r < kBoundRows; ++r)
            if (r < nr) {
                const size_t e = (size_t)(row0 + r) * n_lib_pad + j;
                score[e] = D[e] + suffix[r] * kSlack;
            }
    }
}

cudaError_t launch_prune_bound(const float4 *lib_stats, const float4 *cell_stats, int n_rows, int n_lib_pad, int n_blocks, int seg_blocks,
                               int n_segs, float *R, const float *D, const int *perm, float *score, cudaStream_t stream)
{
    if (n_rows <= 0 || n_lib_pad <= 0 || n_segs < 2)
        return cudaSuccess;
    if (seg_blocks <= 0 || (score && (!D || !perm)))
        return cudaErrorInvalidValue;
    const dim3 grid((unsigned)((n_lib_pad + kBoundThreads - 1) / kBoundThreads), (unsigned)((n_rows + kBoundRows - 1) / kBoundRows));
    prune_bound_kernel<<<grid, kBoundThreads, 0, stream>>>(lib_stats, cell_stats, n_rows, n_lib_pad, n_blocks, seg_blocks, n_segs, R, D, perm,
                                                           score);
    return cudaGetLastError();
}

// One CTA per bucket (column of col_cells cells x one library tile), one thread per cell. A cell is listed when its row is in
// state `want`; with a threshold T (pruning) an active row is listed only while one of its pairs still has a partial sum plus R,
// the bound of the segments not yet summed, <= T[cell] -- otherwise it dies: its pairs become +inf (their complete sums are > T,
// top-K can never take them) and its remaining segments count as done. Listing keeps cell order, so the lists do not depend on
// scheduling.
//
// Why a pair with fl(P + R) > T has a complete sum C > T (P = partial sum, C its continuation in FP32): the later segments'
// computed sums add up to at least R (1 - 1.01e-3) / ((1 - 2^-8)(1 + 3e-4)) > R (1 + 2.6e-3) (kSlack above), and C and fl(P + R)
// round each of their n <= n_segs additions of non-negative terms by <= 2^-24 of the result, so C - fl(P + R) >= 2.6e-3 R -
// n 2^-24 (P + R) > 0 whenever R >= 2^-8 P and n <= 168. A smaller R is not used (the test is then the plain P > T, exact because
// partial sums only grow); at under 1/256 of the partial sum it would prune next to nothing anyway.
__global__ void __launch_bounds__(1024)
list_rows_kernel(float *__restrict__ D, int n_lib_pad, int n_lib, int n_rows, int n_lib_tiles, uint8_t *__restrict__ state, int want,
                 const float *__restrict__ T, const float *__restrict__ R, const int *__restrict__ perm, int segs_left, RowList rows,
                 int *__restrict__ group_count, unsigned long long *__restrict__ listed, unsigned long long *__restrict__ progress)
{
    __shared__ int warp_sum[32];
    const int lib_tile = blockIdx.x, col = blockIdx.y;
    const int b = col * n_lib_tiles + lib_tile;
    const int cell = col * rows.col_cells + threadIdx.x;
    bool on = false;
    if (threadIdx.x < rows.col_cells && cell < n_rows) {
        uint8_t *st = state ? state + (size_t)cell * n_lib_tiles + lib_tile : nullptr;
        on = !st || *st == want;
        if (on && T) {
            const float t = T[cell];
            float *row = D + (size_t)cell * n_lib_pad;
            const float *rest = R ? R + (size_t)cell * n_lib_pad + lib_tile * MM_TNB : nullptr;
            bool alive = false;
            for (int i = 0; i < MM_TNB; ++i) {
                const int j = perm[lib_tile * MM_TNB + i];
                if (j < n_lib) {
                    const float p = row[j], r = rest ? rest[i] : 0.0f;
                    alive = alive || p + (r >= p * 0x1p-8f ? r : 0.0f) <= t;
                }
            }
            if (!alive) {
                for (int i = 0; i < MM_TNB; ++i)
                    row[perm[lib_tile * MM_TNB + i]] = __int_as_float(0x7f800000);
                *st = kRowDead;
                if (progress)
                    atomicAdd(progress, (unsigned long long)segs_left);
                on = false;
            }
        }
    }
    // block-wide exclusive rank of the listed cells, in thread (= cell) order
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned ballot = __ballot_sync(0xffffffffu, on);
    if (lane == 0)
        warp_sum[warp] = __popc(ballot);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
        before += w < warp ? warp_sum[w] : 0;
        total += warp_sum[w];
    }
    if (on)
        rows.cells[(size_t)b * rows.col_cells + before + __popc(ballot & ((1u << lane) - 1u))] = cell;
    if (threadIdx.x == 0) {
        rows.count[b] = total;
        group_count[b] = (total + MM_TCB - 1) / MM_TCB;
        if (total)
            atomicAdd(listed, (unsigned long long)total);
    }
}

size_t list_rows_scratch_bytes(int n_buckets)
{
    size_t temp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, temp, (const int *)nullptr, (int *)nullptr, n_buckets + 1);
    return ((size_t)(n_buckets + 1) * sizeof(int) + 255 & ~(size_t)255) + temp;
}

cudaError_t launch_list_rows(float *D, int n_lib_pad, int n_lib, int n_rows, int n_lib_tiles, uint8_t *state, int want, const float *T,
                             const float *R, const int *perm, int segs_left, RowList rows, void *scratch, size_t scratch_bytes,
                             unsigned long long *listed, unsigned long long *progress, cudaStream_t stream)
{
    const int n_cols = (n_rows + rows.col_cells - 1) / rows.col_cells;
    if (n_cols <= 0 || n_lib_tiles <= 0)
        return cudaSuccess;
    if (rows.col_cells > 1024 || rows.col_cells % 32 || rows.n_buckets != n_cols * n_lib_tiles)
        return cudaErrorInvalidValue;
    // group counts in scratch[0 .. n_buckets], the last one stays 0 so that the scan's last entry is the total
    int *group_count = (int *)scratch;
    const size_t head = (size_t)(rows.n_buckets + 1) * sizeof(int) + 255 & ~(size_t)255;
    cudaError_t e = cudaMemsetAsync(group_count + rows.n_buckets, 0, sizeof(int), stream);
    if (e != cudaSuccess)
        return e;
    list_rows_kernel<<<dim3((unsigned)n_lib_tiles, (unsigned)n_cols), rows.col_cells, 0, stream>>>(
        D, n_lib_pad, n_lib, n_rows, n_lib_tiles, state, want, T, R, perm, segs_left, rows, group_count, listed, progress);
    if ((e = cudaGetLastError()) != cudaSuccess)
        return e;
    size_t temp = scratch_bytes - head;
    return cub::DeviceScan::ExclusiveSum((unsigned char *)scratch + head, temp, group_count, rows.groups, rows.n_buckets + 1, stream);
}

}  // namespace mm
