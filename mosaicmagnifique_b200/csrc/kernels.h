// Internal interface between the host generator (generator.cpp) and the CUDA kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

// colour difference types (values of the reference enum, src/Photomosaic/ColourDifference.h:13-19)
#define MM_DIFF_RGB_EUCLIDEAN 0
#define MM_DIFF_CIE76 1
#define MM_DIFF_CIEDE2000 2
#define MM_DIFF_EUCLID 0  // kernel family used for both RGB_EUCLIDEAN and CIE76

// tile geometry of the packed tensors (see diff_kernels.cu)
#define MM_TCB 8    // cells per cell tile (= consumer warps per CTA)
#define MM_TNB 8    // library images per library tile
#ifndef MM_KP
#define MM_KP 128   // pixels per chunk
#endif
#ifndef MM_STAGES
#define MM_STAGES 3  // shared-memory ring depth of the difference kernel
#endif
#ifndef MM_ESTAGES
#define MM_ESTAGES 3  // ring depth of the Euclidean kernel
#endif
// MM_STRESS_SKEW=1 (stress build only, `make stress`): consumer warps and the producer lane sleep pseudo-random amounts per
// chunk, so that the warps of a CTA drift apart by more than the ring depth would allow if the full/empty protocol had a hole
#ifndef MM_STRESS_SKEW
#define MM_STRESS_SKEW 0
#endif
#ifndef MM_MIN_CTAS
#define MM_MIN_CTAS 2  // __launch_bounds__ residency target of the difference kernel
#endif

// tile geometry of the Euclidean / CIE76 kernel (see diff_euclid.cu)
#define MM_ETC 64   // cells per cell tile
#define MM_ETN 64   // library images per library tile
#define MM_EKP 16   // pixels per chunk

namespace mm {

// CTA rasterisation of the CIEDE2000 kernel: a 1-D grid walks the (cell tile, library tile) plane of one pixel segment in
// super-blocks of sb_a cell tiles x sb_b library tiles (cell tile fastest inside a super-block), so that the ~296 co-resident
// CTAs (2 per SM) form one super-block and stream its chunks roughly in step:
//   * inside a super-block every library chunk is fetched from HBM once for sb_a CTAs and every cell chunk once for sb_b CTAs
//     (L2 serves the rest);
//   * consecutive super-blocks keep the SAME column of sb_a cell tiles and move along the library axis, so the column's cell
//     chunks (sb_a x seg_chunks x 20 KB) stay hot in the 126 MB L2 for the whole sweep: the library is streamed from HBM once per
//     cell column, the cells once.
// Config 4 history (ncu dram__bytes_read): plain order 842 GB; round 1 (16 x 16 super-blocks, library band kept, whole cells per
// CTA) 124-132 GB = 40 x the 3.3 GB the launch needs; cell column kept instead 47.4 GB (profiles/r2_raster_sweep.txt). Launches
// that write D run as row work lists instead (RowList).
struct Raster {
    int sb_a, sb_b;  // super-block: cell tiles x library tiles
};
constexpr int kSuperTiles = 16;
#if defined(__CUDACC__)
// strong system-scope load of the cancel word: it is written by the copy engine while the kernel runs, so it must come from L2
// (the point of coherence for device memory), never from a stale L1 line
__device__ __forceinline__ int load_cancel_flag(const int *p)
{
    int v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Euclidean kernel: 16 x 16 super-blocks, a band of library tiles kept (cell tile fastest inside a super-block, super-blocks along
// the cell axis first) -- round 1's order; its operand traffic per pixel pair is 10 x smaller than the CIEDE2000 kernel's
__device__ __forceinline__ void tile_of_block(unsigned id, int n_ct, int n_lt, int &cell_tile, int &lib_tile)
{
    const unsigned band_ctas = (unsigned)n_ct * kSuperTiles;  // CTAs of one full band of kSuperTiles library tiles
    const unsigned band = id / band_ctas;
    const unsigned r = id - band * band_ctas;
    const int band_h = min(kSuperTiles, n_lt - (int)band * kSuperTiles);
    const unsigned col_ctas = (unsigned)kSuperTiles * band_h;  // CTAs of one full column block inside the band
    const unsigned cb = r / col_ctas;
    const unsigned r2 = r - cb * col_ctas;
    const int cw = min(kSuperTiles, n_ct - (int)cb * kSuperTiles);
    cell_tile = (int)cb * kSuperTiles + (int)(r2 % cw);
    lib_tile = (int)band * kSuperTiles + (int)(r2 / cw);
}
#endif

// which packed layout the prep kernels produce
enum PackLayout { kLayoutCiede = 0, kLayoutEuclid = 1 };
struct TileGeom {
    int tcb, tnb, kp;
    size_t cell_block, lib_block;  // bytes of one (tile, chunk) block
};
inline TileGeom tile_geom(PackLayout l)
{
    return l == kLayoutEuclid ? TileGeom{MM_ETC, MM_ETN, MM_EKP, (size_t)MM_EKP * 4 * MM_ETC * 4, (size_t)MM_EKP * 3 * MM_ETN * 4}
                              : TileGeom{MM_TCB, MM_TNB, MM_KP, (size_t)MM_TCB * MM_KP * 20, (size_t)MM_TNB * MM_KP * 16};
}

// ---- diff_euclid.cu
// cancel   : optional flag word in device memory (the host mirrors cancel() into it by DMA); a CTA that finds it set at its start returns at once, so a
//            cancelled launch drains in the time the remaining CTAs take to be scheduled (CPUPhotomosaicGenerator.cpp:52-73 polls
//            m_wasCanceled per cell)
// progress : optional device counter, +1 per finished CTA (progress(int) reporting while the launch runs)
cudaError_t launch_diff_euclid(const void *cells, const void *lib, float *D, unsigned long long *best_key, int n_cell_tiles,
                               int n_lib_tiles, int n_chunks, int n_lib, int n_cells, cudaStream_t stream,
                               const int *cancel = nullptr, unsigned long long *progress = nullptr);

// ---- diff_kernels.cu
// Fused argmin launch (best_key, no D) or a complete D: whole cells per CTA, super-block raster (above).
cudaError_t launch_diff_sum(int diff_type, const void *cells, const void *lib, float *D, unsigned long long *best_key,
                            int n_cell_tiles, int n_lib_tiles, int n_chunks, int n_lib, int n_cells, cudaStream_t stream,
                            const int *cancel = nullptr, unsigned long long *progress = nullptr);

// CIEDE2000 launches that write D run the pixel axis as segment passes over row work lists. A row = one cell x one library tile
// of 8 images (tile slot i holds image perm[i], the library's colour order). Each pass adds the segment's sum of every listed pair
// into D[cell][perm[slot]] -- D stays in library index order and holds, for every pair, ((seg 0 + seg 1) + seg 2) + ... whichever
// launches computed it. Buckets = columns of col_cells consecutive cells x library tiles, column-major, so a column's cells
// stay hot in L2 while the library sweeps past them.
struct RowList {
    int *cells;        // [n_buckets][col_cells] listed cells of each bucket, cell order
    int *count;        // [n_buckets] listed cells
    int *groups;       // [n_buckets + 1] exclusive scan of the groups of <= 8 rows per bucket (one CTA each)
    int n_buckets, col_cells;
};
// row states (uint8 [n_rows][n_lib_tiles]): still summing / candidate tile, completed before the threshold / pruned
enum : uint8_t { kRowActive = 0, kRowComplete = 1, kRowDead = 2 };
// one segment pass: chunks [k0, k0 + nk) of the n_groups groups of `rows`; progress += rows stored
cudaError_t launch_diff_rows(const void *cells, const void *lib, float *D, int n_groups, int n_lib_tiles, int n_chunks, int k0, int nk,
                             RowList rows, const int *perm, cudaStream_t stream, const int *cancel = nullptr,
                             unsigned long long *progress = nullptr);
// lists the rows in state `want` (state null: every row) into rows.cells / rows.count / rows.groups (rows.groups[n_buckets] = groups
// in all); with T: active rows whose pairs all have partial sum + R > T die (pairs -> +inf, progress += segs_left); listed += rows
// listed. R (optional, [n_rows][n_lib_pad] in SLOT order): launch_prune_bound's lower bound of the segments not yet summed.
size_t list_rows_scratch_bytes(int n_buckets);
cudaError_t launch_list_rows(float *D, int n_lib_pad, int n_lib, int n_rows, int n_lib_tiles, uint8_t *state, int want, const float *T,
                             const float *R, const int *perm, int segs_left, RowList rows, void *scratch, size_t scratch_bytes,
                             unsigned long long *listed, unsigned long long *progress, cudaStream_t stream);
// Lightness lower bound of the CIEDE2000 segments not yet summed (DESIGN.md 4.1), from launch_block_stats' statistics.
// R [n_segs - 1][n_rows][n_lib_pad], slot order: R[s - 1][row][slot] <= the sum that segments s .. n_segs - 1 will add to the pair
// (row, image perm[slot]), s = 1 .. n_segs - 1. score (optional, [n_rows][n_lib_pad], image order): D + R[0], pass 0's partial
// sum plus the bound of the rest, which ranks the pruning candidates.
cudaError_t launch_prune_bound(const float4 *lib_stats, const float4 *cell_stats, int n_rows, int n_lib_pad, int n_blocks, int seg_blocks,
                               int n_segs, float *R, const float *D, const int *perm, float *score, cudaStream_t stream);

// ---- prep_kernels.cu
// u8 BGR -> working space f32 AoS [pixel][3]: Lab through the OpenCV-compatible LUT (is_lab) or a plain cast.
// lab_lut: the 33^3 OpenCV-compatible table expanded to 8-byte entries (L, a, b, 0) by expand_lab_lut
cudaError_t launch_to_working_space(const uint8_t *bgr, size_t row_stride, int rows, int cols, float *out, bool is_lab,
                                    const short4 *lab_lut, const int *c8, cudaStream_t stream);
constexpr size_t kLabLutEntries = 33 * 33 * 33;
// 3 x int16 per entry (lab_lut.S, data/lab_lut_s16.bin) -> 4 x int16 per entry, so that a cube corner is one 8-byte load
inline std::vector<int16_t> expand_lab_lut(const int16_t *lut3)
{
    std::vector<int16_t> out(kLabLutEntries * 4, 0);
    for (size_t i = 0; i < kLabLutEntries; ++i)
        for (int c = 0; c < 3; ++c)
            out[i * 4 + c] = lut3[i * 3 + c];
    return out;
}
// hue-rotated 8U copy of an 8U BGR image (ColourScheme.cpp:36-177, OpenCV float HSV_FULL round trip)
cudaError_t launch_hue_rotate(const uint8_t *in, uint8_t *out, int rows, int cols, float rot, cudaStream_t stream);
// INTER_AREA for integer ratios, 8U 3-channel, batch of n square images (src size s -> dst size s / k)
cudaError_t launch_area_u8(const uint8_t *src, uint8_t *dst, int64_t n, int src_size, int k, cudaStream_t stream);
// oriented 8U BGR library for mosaic_set_tile_flips: dst [O][n][S][S][3], orientation-major, the enabled subset of the codes
// {0 none, 1 = H (columns mirrored), 2 = V (rows mirrored), 3 = HV} of `flips` in increasing code (O = 1, 2, 2 or 4)
cudaError_t launch_orient_library(const uint8_t *src, uint8_t *dst, int64_t n, int S, int flips, cudaStream_t stream);
// INTER_AREA for integer ratios, f32 3-channel, batch of n square images
cudaError_t launch_area_f32(const float *src, float *dst, int64_t n, int src_size, int k, cudaStream_t stream);
// INTER_AREA for any down-scaling ratio (OpenCV's resizeArea_): device CSR table of host_model's make_area_table
struct AreaTab {
    const int *start;    // [dst_size + 1]
    const int *si;       // source sample of each tap
    const float *alpha;  // weight of each tap
};
cudaError_t launch_area_general_u8(const uint8_t *src, uint8_t *dst, int64_t n, int src_size, int dst_size, AreaTab tab,
                                   cudaStream_t stream);
cudaError_t launch_area_general_f32(const float *src, float *dst, int64_t n, int src_size, int dst_size, AreaTab tab,
                                    cudaStream_t stream);
// INTER_CUBIC for 8U, cn channels, one image (library ingest, mask growth): device copies of host_model's CubicTable
struct CubicTab {
    const int *idx;        // [dst_size][4] clamped source indices
    const int16_t *coef;   // [dst_size][4] 11-bit fixed-point coefficients
};
cudaError_t launch_cubic_u8(const uint8_t *src, int sh, int sw, int cn, uint8_t *dst, int dh, int dw, CubicTab xt, CubicTab yt,
                            cudaStream_t stream);
// working f32 AoS library [n][P][3] -> packed float4 tiles (compacted pixel order, chroma in .w)
// perm (CIEDE2000 layout only, optional): tile slot i holds image perm[i] (launch_library_order)
cudaError_t launch_pack_library(const float *lib, void *packed, int64_t n, int P, const int *pix_list, int n_active,
                                int n_chunks, int n_lib_tiles, PackLayout layout, cudaStream_t stream, const int *perm = nullptr);
// colour order of an 8U library of n S x S images: perm[n_pad] (slot -> image; padding slots -> themselves) and its inverse
size_t library_order_scratch_bytes(int64_t n);
cudaError_t launch_library_order(const uint8_t *lib, int S, int64_t n, int n_pad, int *perm, int *inv_perm, void *scratch,
                                 size_t scratch_bytes, cudaStream_t stream);

// CIEDE2000 layout straight from the 8U BGR library at the detail size (Lab conversion fused, no f32 intermediate) or from
// the f32 working-space library; padding slots are written by the same pass
// src_is_u8: src_size x src_size images reduced k-fold on the fly (8U INTER_AREA, integer ratio; src_size 0 = already P pixels)
cudaError_t launch_pack_library_ciede(const void *src, bool src_is_u8, void *packed, int64_t n, int P, const int *pix_list,
                                      int n_active, int n_chunks, int n_lib_tiles, const short4 *lab_lut, cudaStream_t stream,
                                      int src_size = 0, int k = 1, const int *perm = nullptr);

// Euclidean layout straight from the 8U BGR library (src_size x src_size images, reduced k-fold on the fly by the 8U INTER_AREA
// arithmetic; plain cast, or the Lab conversion for CIE76, fused); padding slots are written by the same pass
cudaError_t launch_pack_library_euclid_u8(const uint8_t *lib, int src_size, int k, bool is_lab, void *packed, int64_t n, int P,
                                          const int *pix_list, int n_active, int n_chunks, int n_lib_tiles, const short4 *lab_lut,
                                          cudaStream_t stream);

// Block statistics of the packed CIEDE2000 tiles for the pruning bound (launch_prune_bound): a block is a run of MM_BB compacted
// pixels inside a chunk, n_blocks = n_chunks * MM_KP / MM_BB. Stored lightness Lh = L/2 - 25.
//   lib_stats  [n_blocks][n_lib_tiles * MM_TNB] (sum Lh, min Lh, max Lh, 0) per library slot
//   cell_stats [n_rows][n_blocks]             (sum Lh, min Lh, max Lh, w) per cell row; w = the weight every pixel of the block has,
//                                              0 when the weights differ (clipped edges, flipped masks, detail-space bounds)
#define MM_BB 16
cudaError_t launch_block_stats(const void *lib_packed, int n_lib_tiles, const void *cells_packed, int n_rows, int n_chunks,
                               float4 *lib_stats, float4 *cell_stats, cudaStream_t stream);

struct CellDesc {
    int x0, y0;          // top-left of the (unclipped) cell rect in main-image space
    int bx, by, bw, bh;  // detail-space bound
    int flip;            // mask index: flip_h + 2 * flip_v
    int variant;         // main-image variant this row compares against
};
// main f32 AoS [V][H][W][3] -> packed cell tiles with weights (cell size S -> detail size ds = S / k)
// k > 0: integer ratio S / ds = k; k == 0: fractional ratio through `tab` (detail size ds)
cudaError_t launch_extract_cells(const float *mains, int H, int W, const CellDesc *cells, int n_cells, int S, int ds, int k,
                                 AreaTab tab, const uint8_t *masks4, const int *pix_list, int n_active, int n_chunks,
                                 void *packed, PackLayout layout, cudaStream_t stream);

// ---- grid_kernels.cu: entropy rule of GridGenerator::findCellState for a batch of candidate cells
struct GridCandidate {
    int cx, cy, cw, ch;  // cell rect clamped to the image
    int bx, by, bw, bh;  // detail-space bound (resize target and mask window)
    int flip;
};
cudaError_t launch_grid_entropy(const uint8_t *main_bgr, int W, const GridCandidate *cand, int n_cand, const uint8_t *masks4, int ds,
                                double threshold, uint8_t *split, cudaStream_t stream);

// ---- build_kernels.cu: buildPhotomosaic compositing
struct BuildCell {
    int x0, y0;      // top-left of the (unclipped) cell rect
    int flip;        // mask index
    int raster;      // 1-based raster index of the cell inside its step (0 = "no cell" in the owner map)
    int lib_index;   // chosen library image
    int orient;      // mirroring of the tile (mosaic_set_tile_flips): flip_h + 2 * flip_v
};
struct BuildStep {
    const BuildCell *cells;  // indexed by raster - 1
    const uint8_t *lib;      // 8U BGR (render) library of this step, [N][side][side][3]
    int side;                // k * S_s: the step's cell size at the output scale k
};
cudaError_t launch_build_scatter(const BuildCell *cells, int n_cells, int S, const uint8_t *masks4, int H, int W, int step, int n_steps,
                                 unsigned long long *owner, cudaStream_t stream);
// rows [y_begin, y_end) of the BGRA mosaic at k times the owner map's size (cols = k * W) into out, row y_begin first, out_stride
// bytes per row; bytes past cols * 4 in a row are not written. out and out_stride must be multiples of 4 bytes.
cudaError_t launch_build_gather(const unsigned long long *owner, int W, int k, int n_steps, const BuildStep *steps, const uint8_t bgra[4],
                                int y_begin, int y_end, int cols, uint8_t *out, size_t out_stride, cudaStream_t stream);

// ---- select_kernels.cu
cudaError_t launch_fill_u64(unsigned long long *p, size_t n, unsigned long long v, cudaStream_t stream);
// D rows of V variants -> element-wise minimum into the first variant's rows
cudaError_t launch_min_variants(float *D, int n_cells, int V, int n_lib_pad, cudaStream_t stream);
// K smallest (score, index) per row, unsorted. cand_score/cand_idx: [n_cells][K]
cudaError_t launch_topk(const float *D, int row_stride, int n_lib, int n_cells, int K, float *cand_score, int *cand_idx,
                        cudaStream_t stream);
// exact pruning: mark = true sets the rows of the candidates' tiles to kRowComplete; mark = false writes T[cell], the k-th smallest
// of the candidates' (by then complete) sums
cudaError_t launch_prune_threshold(const float *D, int row_stride, const int *cand_idx, int n_rows, int M, int k, const int *inv_perm,
                                   int n_lib_tiles, uint8_t *state, float *T, bool mark, cudaStream_t stream);
// Repeat-penalised selection in raster order (CPUPhotomosaicGenerator.cpp:81-82, 137-169, 185-225).
//   grid         : rows x cols int64, in: -1 invalid / >= 0 valid, out: best fit per valid cell
//   cell_pos     : [n_cells] y * cols + x of each valid cell in raster order (= row order of the scores)
//   next_x       : [n_cells] column of the next valid cell in the same grid row (cols if none)
//   scores / idx : per cell M entries; idx == nullptr means "entry j is slot j" (rows of D, stride M_stride)
//   n_images     : library images N. Slots are orientation-major (slot = j * N + i for orientation j of image i, mosaic_set_tile_flips)
//                  and repeats count per source image: the penalty of slot s is addition * count[s % N], and a chosen slot s in the
//                  window adds to count[s % N]. With one orientation slot = image and this is the reference's rule.
//   row_progress : [rows] initialised to the column of the first valid cell of each row (cols if none)
//   counts       : [n_ctas][n_images] zero-filled scratch
//   margins      : optional [n_cells][2] best / second-best penalised score of every cell
//   rows_per_block / block_stride : candidate lists all-gathered from several GPUs (see SelArgs); 0 = one plain array
cudaError_t launch_select(long long *grid, const int *cell_pos, const int *next_x, int n_cells, int rows, int cols,
                          const float *scores, const int *idx, int M, int M_stride, int n_images, int repeat_range,
                          int repeat_addition, int *row_progress, int *counts, int n_ctas, float *margins,
                          cudaStream_t stream, long long rows_per_block = 0, long long block_stride = 0);
int select_max_ctas(int device);
// Usage limit (mosaic_set_usage_limit, DESIGN.md 4.4). Sorted prefixes: every cell's k0 = min(K, kPrefixMax) smallest (score, slot)
// pairs in ascending order, the part of its candidates the capped selection scans first.
constexpr int kPrefixMax = 1024;
// sel_s / sel_pos [n_rows][k0]: launch_topk's k0 smallest of each row's source. list_s == nullptr: the source is a D row and
// sel_s / sel_pos become its sorted prefix (score, slot). Otherwise the source is the candidate list list_s / list_i [n_rows][K]
// (launch_topk output, slots ascending) and its first k0 entries become the sorted prefix; the row keeps its K entries.
cudaError_t launch_sort_prefix(float *sel_s, int *sel_pos, int n_rows, int k0, float *list_s, int *list_i, int K, cudaStream_t stream);
// Capped selection in raster order, one CTA: a cell takes the lowest (D[s] + A * count[s % N], s) over the slots s whose image
// s % N has used[s % N] < max_uses, then used[s % N] += 1. scores / idx: the full candidate row of each cell as launch_select's
// (M entries, stride M_stride; idx nullptr = D rows); pscores / pidx: its sorted prefix of k0 entries, stride p_stride. All-gathered
// blocks address prefix and row alike (rows_per_block, block_stride as launch_select). counts: [n_images] zeroed scratch;
// used: [n_images], carried across the steps of one generate. margins: best / second-best ALLOWED penalised score.
cudaError_t launch_select_capped(long long *grid, const int *cell_pos, int n_cells, int rows, int cols, const float *scores, const int *idx,
                                 int M, int M_stride, const float *pscores, const int *pidx, int k0, int p_stride, int n_images,
                                 int repeat_range, int repeat_addition, int max_uses, int *counts, int *used, float *margins,
                                 cudaStream_t stream, long long rows_per_block = 0, long long block_stride = 0);
// best_key (from the diff epilogue) -> grid
cudaError_t launch_keys_to_grid(const unsigned long long *best_key, const int *cell_pos, long long *grid, int n_cells,
                                float *best_score, cudaStream_t stream);

// ---- microbench.cu
// out[0..]: FFMA lane-ops/s, packed FFMA2 lane-ops/s, MUFU rsq ops/s, MUFU ex2 ops/s, sm clock used (Hz, from clock64)
cudaError_t run_microbench(double *out, int n_out, cudaStream_t stream);

}  // namespace mm
