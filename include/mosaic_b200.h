/*
 * mosaic_b200.h -- C ABI of the B200-native photomosaic best-fit engine (libmosaic_b200.so).
 *
 * Drop-in boundary for the reference's generator API (MorganGrundy/MosaicMagnifique):
 *   class PhotomosaicGeneratorBase        src/Photomosaic/PhotomosaicGeneratorBase.h:32-112
 *   CPUPhotomosaicGenerator::generateBestFits   src/Photomosaic/CPUPhotomosaicGenerator.cpp:33-112
 *   CUDAPhotomosaicGenerator::generateBestFits  src/Photomosaic/CUDA/CUDAPhotomosaicGenerator.cpp:40-370
 * Every entry point names the reference interface it replaces. Qt-free, OpenCV-free: plain pointers and
 * sizes, no exceptions across the boundary, the caller owns every host buffer (inputs are copied).
 * One handle = one generator object = one in-flight generate; a handle is bound to one CUDA device.
 *
 * The C++ mirror of the reference class (same method names) is include/mosaic_b200.hpp; the Python mirror
 * is mosaicmagnifique_b200/generator.py; INTEGRATION.md shows the reference-side binding.
 *
 * All functions return MOSAIC_OK (0) or a negative mosaic_status; mosaic_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device mosaic_create fails with MOSAIC_ERR_CUDA.
 */
#ifndef MOSAIC_B200_H
#define MOSAIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden; this header is its export list */
#endif

typedef struct mosaic_generator mosaic_generator;

typedef enum mosaic_status {
    MOSAIC_OK = 0,
    MOSAIC_ERR_INVALID_ARGUMENT = -1, /* std::invalid_argument in the reference (ColourDifference.cpp:23) */
    MOSAIC_ERR_CUDA = -2,             /* any CUDA error: the reference returns false (CUDAPhotomosaicGenerator.cpp:367) */
    MOSAIC_ERR_OUT_OF_MEMORY = -3,    /* reference: cudaMemGetInfo pre-check (CUDAPhotomosaicGenerator.cpp:409-430) */
    MOSAIC_ERR_NOT_READY = -4,        /* a required input has not been set */
    MOSAIC_ERR_UNSUPPORTED = -5,      /* configuration the engine does not implement yet (text says which) */
    MOSAIC_ERR_CANCELLED = -6         /* cancel() was called: the reference returns false (CPUPhotomosaicGenerator.cpp:111) */
} mosaic_status;

/* ColourDifference::Type, src/Photomosaic/ColourDifference.h:13-19 */
enum { MOSAIC_RGB_EUCLIDEAN = 0, MOSAIC_CIE76 = 1, MOSAIC_CIEDE2000 = 2 };
/* ColourScheme::Type, src/Photomosaic/ColourScheme.h:10-19 */
enum {
    MOSAIC_SCHEME_NONE = 0, MOSAIC_SCHEME_COMPLEMENTARY = 1, MOSAIC_SCHEME_TRIADIC = 2,
    MOSAIC_SCHEME_COMPOUND = 3, MOSAIC_SCHEME_TETRADIC = 4, MOSAIC_SCHEME_ANALAGOUS = 5
};

/* CellShape tiling parameters, src/CellShape/CellShape.h:98-109 */
typedef struct mosaic_cell_shape {
    int32_t size;                 /* mask is size x size, 8U, non-zero = active (thresholded at >127 like setCellMask) */
    int32_t row_spacing, col_spacing;
    int32_t alt_row_spacing, alt_col_spacing;
    int32_t alt_row_offset, alt_col_offset;
    int32_t alt_col_flip_h, alt_col_flip_v, alt_row_flip_h, alt_row_flip_v;
} mosaic_cell_shape;

/* Phase timings of the last generate(), milliseconds. Names follow the reference's TimingLogger scopes
 * (CPUPhotomosaicGenerator.cpp:38-105, CUDAPhotomosaicGenerator.cpp:47-360). */
typedef struct mosaic_timings {
    double preprocess_ms;   /* "Preprocess": colour conversion, library resize/pack, cell extraction (GPU time) */
    double diff_ms;         /* "DiffReduce": fused difference-sum kernel(s) */
    double select_ms;       /* "Repeats" + "FindLowest": top-K / wavefront / argmin */
    double total_ms;        /* "generateBestFits": host wall time of the call incl. H2D / D2H */
    double h2d_bytes, d2h_bytes;
    double pixel_diffs;         /* active, in-bound mask pixels x library images x variants, all steps */
    double pixel_diffs_nominal; /* bounding-box pixels (detail size squared) x library x variants x valid cells */
    int64_t kernel_launches;    /* kernels this library launched inside the call */
    double evaluated_pixel_diffs; /* pixel_diffs scaled by the share of the difference work actually executed: below pixel_diffs
                                   * when exact pruning skipped pairs that cannot be selected */
} mosaic_timings;

typedef void (*mosaic_progress_fn)(int progress, void *user); /* signal progress(int), PhotomosaicGeneratorBase.h:78 */

/* ---- lifetime: CUDAPhotomosaicGenerator(const int device), CUDAPhotomosaicGenerator.h:31 */
int mosaic_create(int device, mosaic_generator **out);
void mosaic_destroy(mosaic_generator *g);
const char *mosaic_last_error(const mosaic_generator *g); /* replaces the modal message boxes, CUDAUtility.h:34-62 */
const char *mosaic_version(void);

/* ---- setters: PhotomosaicGeneratorBase.h:40-66, .cpp:45-93 */
/* setMainImage(const cv::Mat&): 8U BGR, rows x cols, row_stride in bytes (>= cols*3). Host OR device pointer (unified addressing). */
int mosaic_set_main_image(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride);
/* setLibrary(const std::vector<cv::Mat>&): n square 8U BGR images of size x size, contiguous.
 * As in the reference the images must already be at the cell size (MainWindow.cpp:575-581). Host OR device pointer. */
int mosaic_set_library(mosaic_generator *g, const uint8_t *bgr, int64_t n, int size);
int mosaic_set_colour_difference(mosaic_generator *g, int type); /* setColourDifference */
int mosaic_set_colour_scheme(mosaic_generator *g, int type);     /* setColourScheme */
/* setCellGroup(const CellGroup&): the group is described by its top-level shape, detail and size steps;
 * the per-step normal/detail cells are derived as CellGroup does (CellGroup.cpp:65-128). If cell_size > 0 and
 * differs from shape->size the shape is first resized like CellShape::resized (CellShape.cpp:281-312). */
int mosaic_set_cell_group(mosaic_generator *g, const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size,
                          int detail_percent, int size_steps);
/* The same for a shape that came from CellShape::loadFromFile (mosaic_mcs_load): with mask_as_stored != 0 the mask is taken as the
 * file holds it -- loadFromFile does not threshold (CellShape.cpp:405-410), non-zero = active everywhere downstream
 * (CPUPhotomosaicGenerator.cpp:150), and only RESIZED masks are binarised (CellShape::resized -> setCellMask). Identical to
 * mosaic_set_cell_group for the binary masks the reference itself writes. */
int mosaic_set_cell_group_ex(mosaic_generator *g, const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size,
                             int detail_percent, int size_steps, int mask_as_stored);
/* getCellGroup(): geometry of the normal (detail = 0) or detail (detail = 1) cell of one step */
int mosaic_get_cell_shape(const mosaic_generator *g, int step, int detail, mosaic_cell_shape *out, uint8_t *mask_out,
                          size_t mask_capacity);
/* setGridState(const MosaicBestFit&): one call per step; valid[r*cols+c] != 0 <=> has_value() */
int mosaic_set_grid_state(mosaic_generator *g, int step, int rows, int cols, const uint8_t *valid);
/* GridGenerator::getGridState (Grid/GridGenerator.cpp:29-110) on the current main image and cell group */
int mosaic_compute_grid_state(mosaic_generator *g);
int mosaic_get_grid_steps(const mosaic_generator *g);
int mosaic_get_grid_size(const mosaic_generator *g, int step, int *rows, int *cols);
int mosaic_set_repeat(mosaic_generator *g, int range, int addition); /* setRepeat */
/* Reference quirk Q1 (SURVEY.md section 8a): with a colour scheme every cell variant aliases ONE buffer, so only the
 * last hue rotation is compared. faithful = 1 (default) reproduces that, 0 compares all variants (min over them). */
int mosaic_set_variant_quirk(mosaic_generator *g, int faithful);

/* ---- run: generateBestFits() / getBestFits() / getMaxProgress() / cancel() / progress(int) */
int mosaic_generate(mosaic_generator *g);
/* out[r*cols+c] = library index, -1 = std::nullopt */
int mosaic_get_best_fits(const mosaic_generator *g, int step, int64_t *out, int rows, int cols);
/* buildPhotomosaic(const cv::Scalar &background) (PhotomosaicGeneratorBase.cpp:110-207): composites the chosen library images
 * through the (flipped) cell masks into an 8U BGRA image of the main image's size, on the GPU. out: host or device pointer. */
int mosaic_build_photomosaic(mosaic_generator *g, const uint8_t background_bgra[4], uint8_t *out_bgra, int rows, int cols,
                             size_t row_stride);
int mosaic_get_max_progress(const mosaic_generator *g);
void mosaic_set_progress_callback(mosaic_generator *g, mosaic_progress_fn fn, void *user);
/* cancel() (PhotomosaicGeneratorBase.cpp:217-220): callable from any thread and from inside the progress callback. The running
 * difference kernel stops scheduling work (every CTA checks the flag when it starts), generate returns MOSAIC_ERR_CANCELLED within
 * milliseconds. Like m_wasCanceled the flag is sticky: later generate calls return MOSAIC_ERR_CANCELLED until mosaic_reset_cancel. */
void mosaic_cancel(mosaic_generator *g);
void mosaic_reset_cancel(mosaic_generator *g);

/* ---- mirrored library tiles (no reference counterpart: the reference mirrors cell masks, CellShape alternate*Flip*, never the
 * tile placed in a cell). flips is a mask: 1 = horizontal (columns mirrored, cv::flip code 1), 2 = vertical (rows mirrored, code 0);
 * 0 (the default) compares the library as it is. The candidates of a cell are then the O = 1, 2, 2 or 4 enabled orientations
 * {0 none, 1 H, 2 V, 3 HV} (in increasing code) of every image: O * N slots, orientation-major, slot = j * N + i for the j-th
 * orientation of image i -- exactly a library given as [lib, flip_1(lib), ...]. Everything up to the difference matrix is that run's;
 * ties go to the lowest slot, so an image that is its own mirror image is placed unflipped. Repeats count per source image: all
 * orientations of image i share one count and the penalty of slot s is addition * count[s mod N]. mosaic_get_best_fits keeps
 * returning image indices in [0, N); mosaic_get_best_fit_flips gives the orientation; mosaic_get_differences has O * N columns in
 * slot order; pixel_diffs count the O * N work; buildPhotomosaic places each tile mirrored by its orientation.
 * MOSAIC_ERR_INVALID_ARGUMENT outside 0..3. A library from mosaic_set_library_shard cannot be combined with flips
 * (MOSAIC_ERR_UNSUPPORTED): it is stored at the detail size, where mirroring is no longer exact. */
int mosaic_set_tile_flips(mosaic_generator *g, int flips);
/* out[r*cols+c] = orientation of the tile chosen for the cell (flip_h + 2 * flip_v, as mosaic_flip_at), -1 = std::nullopt;
 * MOSAIC_ERR_NOT_READY before a generate on the current grid state */
int mosaic_get_best_fit_flips(const mosaic_generator *g, int step, int8_t *out, int rows, int cols);

/* ---- usage limit (no reference counterpart: the reference limits repetition only through the windowed penalty of setRepeat).
 * max_uses = M >= 1 lets each library image be chosen at most M times in one generate, over all size steps (M = 1: no duplicates);
 * 0 (the default) is unlimited and changes nothing. Cells are decided in the engine's order -- size step 0, 1, ..., and inside a
 * step the reference's raster order over valid cells -- and a cell takes the lowest (D[s] + addition * count[s mod N], s) over the
 * slots s whose image s mod N has been chosen fewer than M times so far in this generate (ties to the lowest slot, the value in
 * f64 as without the limit; the window penalty is unchanged). With tile flips all orientations of an image share one use count.
 * If M * N is less than the number of valid cells of all steps, generate fails with MOSAIC_ERR_INVALID_ARGUMENT before any work
 * (the text gives both numbers); otherwise every cell has an allowed image, so the limit never leaves a cell without a fit.
 * mosaic_get_best_fits, mosaic_get_best_fit_flips and mosaic_get_differences keep their meaning; margins are the best and
 * second-best ALLOWED penalised scores. Sharded handles: mosaic_generate_candidates uses the limit set at that call; the steps
 * must then be selected in increasing order (steps without cells may be skipped) -- use counts restart when a step at or below
 * the last selected one is selected, and selecting a step before an earlier step with cells gives MOSAIC_ERR_NOT_READY.
 * Candidates handed to mosaic_select_from_candidates / _gathered must be the engine's own (their rows start with a sorted prefix).
 * MOSAIC_ERR_INVALID_ARGUMENT for M < 0. */
int mosaic_set_usage_limit(mosaic_generator *g, int max_uses);

/* ---- scaled compositing (no reference counterpart: the reference composites at the main image's size, from the library it
 * matched with). Print wants tiles with far more pixels than matching needs; these two calls build the mosaic at k times the main
 * image's size without matching at that size.
 * mosaic_set_render_library: the render library -- the SAME n images as the library, in the same index order, square 8U BGR at
 *   side size = R, contiguous, host OR device pointer. It is copied to the device and stays resident until replaced; n = 0 clears it.
 *   The copy runs on the handle's own stream, which does not wait for work on other streams: device data must be complete when the
 *   call is made (e.g. torch.cuda.synchronize() after the kernels that wrote it).
 *   Nothing is checked against the cell group here (it may be set later), and the plain build never uses it.
 *   MOSAIC_ERR_INVALID_ARGUMENT for n < 0, size < 1, or bgr == NULL with n > 0.
 * mosaic_build_photomosaic_scaled: with S the cell size of step 0 and k = R / S, writes a (k * H) x (k * W) 8U BGRA image (rows, cols)
 *   that is exactly what buildPhotomosaic (PhotomosaicGeneratorBase.cpp:110-207) produces from
 *     - a main image of k * H x k * W, the render library and the same best fits (slots with tile flips) and background;
 *     - the k-scaled cell group: per step the normal cell with size, row / col spacing, alternate spacings and alternate offsets
 *       times k (flip flags unchanged) and its mask upsampled by nearest neighbour (every mask pixel a k x k block).
 *   So each cell's rect is k times its rect at scale 1 and the output pixel (Y, X) comes from the tile of the cell that owns base
 *   pixel (Y / k, X / k), at (Y - k * y0, X - k * x0) of the render tile. The render tiles of size step s are the step s - 1 tiles
 *   halved with 8U INTER_AREA (side k * S_s); a step after an odd cell size gives MOSAIC_ERR_UNSUPPORTED, as the plain build does.
 *   With tile flips slot j * N + i places render image i mirrored by orientation j. Tile pixels get alpha 255, uncovered pixels the
 *   background. k = 1 with the render library equal to the library is byte-identical to mosaic_build_photomosaic.
 *   The library at the cell size is not needed, so a handle loaded with mosaic_set_library_shard can build (after
 *   mosaic_select_from_gathered). out: 4-byte aligned device memory of the handle's GPU is written in place; any other pointer
 *   (pinned or pageable host memory, an unaligned address) is filled through device bands of about 256 MB. Bytes past cols * 4 in
 *   each row are left untouched.
 *   MOSAIC_ERR_NOT_READY: no render library, or no best fits on the current grid state. MOSAIC_ERR_INVALID_ARGUMENT (the text gives
 *   the numbers): render n != the library's N (n_total of a sharded handle), R not a multiple of S, rows != k * H or cols != k * W,
 *   k * H or k * W above INT_MAX, row_stride < cols * 4 or not a multiple of 4. */
int mosaic_set_render_library(mosaic_generator *g, const uint8_t *bgr, int64_t n, int size);
int mosaic_build_photomosaic_scaled(mosaic_generator *g, const uint8_t background_bgra[4], uint8_t *out_bgra, int rows, int cols,
                                    size_t row_stride);

/* ---- parity / measurement taps (no reference counterpart; used by tests and bench.py) */
/* keep the full difference matrix of every step on the device so it can be read back */
int mosaic_set_keep_differences(mosaic_generator *g, int keep);
int64_t mosaic_get_valid_cell_count(const mosaic_generator *g, int step);
/* D[cell][lib] = min over variants of the masked difference sum (no repeat penalty), cells in raster order; with tile flips the
 * columns are the O * N slots and n_lib must equal O * N */
int mosaic_get_differences(const mosaic_generator *g, int step, float *out, int64_t n_cells, int64_t n_lib);
/* Tie-band reporting (BASELINE.json: cells whose best two candidates differ by less than the FP32 tolerance): when switched
 * on, generate() records for every valid cell the best and the second-best PENALISED score it compared (the fused-argmin
 * shortcut is bypassed). Raster order of the step's valid cells; unsharded handles only. */
int mosaic_set_report_margins(mosaic_generator *g, int report);
int mosaic_get_margins(const mosaic_generator *g, int step, float *best, float *second, int64_t n_cells);
int mosaic_get_timings(const mosaic_generator *g, mosaic_timings *out);

/* ---- multi-GPU sharding (no reference counterpart; SURVEY.md section 8e). One process per GPU:
 * rank r of world computes the differences of its block of grid rows only and exposes the K best
 * (score, index) candidates per cell; the caller all-gathers them (NCCL) and every rank runs the
 * order-dependent selection on the gathered candidates. */
int mosaic_set_shard(mosaic_generator *g, int rank, int world);
/* the split mosaic_set_shard implies for a step with n_valid_cells valid cells (host arithmetic, no device needed): rank r owns the
 * cells [first_cell, first_cell + n_cells) of the raster order and rows_per_rank rows of the all-gathered candidate buffer */
int mosaic_host_shard_split(int64_t n_valid_cells, int colour_difference, int rank, int world, int64_t *rows_per_rank, int64_t *first_cell,
                            int64_t *n_cells);
/* preprocessing + difference sums + top-K for this rank's cells of every step */
int mosaic_generate_candidates(mosaic_generator *g);
int mosaic_get_candidate_count(const mosaic_generator *g, int step, int64_t *first_cell, int64_t *n_cells, int *k);
/* device pointers (float scores [n_cells][k], int32 indices [n_cells][k]) of this rank's candidates */
int mosaic_get_candidates_device(const mosaic_generator *g, int step, void **scores, void **indices);
/* selection over candidates of ALL cells of a step (device pointers, [n_valid][k]) -> best fits */
int mosaic_select_from_candidates(mosaic_generator *g, int step, const void *scores, const void *indices, int k);
/* The same exchange as ONE collective: every rank's candidates of a step are one device block of identical size
 * {float scores [rows_per_rank][k], int32 indices [rows_per_rank][k]} (rank r owns the valid cells r * rows_per_rank ... of the
 * step's raster order, a split every rank computes by itself); the blocks are all-gathered in rank order into one buffer
 * (world * block_bytes) and handed to mosaic_select_from_gathered. No sizes are exchanged and nothing is read back. */
int mosaic_get_candidate_block(const mosaic_generator *g, int step, void **block, int64_t *rows_per_rank, int *k, size_t *block_bytes);
int mosaic_select_from_gathered(mosaic_generator *g, int step, const void *gathered_blocks, int k, int64_t rows_per_rank);
/* Sharded inputs (end-to-end path of a multi-GPU run): a rank uploads only what it computes on.
 * mosaic_get_shard_rows: main-image rows [row_lo, row_hi) that this handle's cells read (cell group, grid state and shard must
 *   be set; rows x cols declares the image size). mosaic_set_main_image_rows: setMainImage from a pointer to row 0 of the FULL
 *   image, copying only rows [row_lo, row_hi); generate fails with MOSAIC_ERR_NOT_READY if a needed row is missing.
 * mosaic_set_library_shard: this rank's slice [first, first + count) of an n_total-image library at the cell size; it is stored
 *   at the detail size of step 0 when detail != 100 % (resized on the GPU, PhotomosaicGeneratorBase.cpp:262-270) so that the
 *   remaining slices, delivered by the caller into the buffer of mosaic_get_library_device (NCCL all-gather over NVLink, images
 *   back to back at *stored_size, room for capacity_images >= n_total), cross the wire at the small size. */
int mosaic_get_shard_rows(mosaic_generator *g, int rows, int cols, int *row_lo, int *row_hi);
int mosaic_set_main_image_rows(mosaic_generator *g, const uint8_t *bgr, int rows, int cols, size_t row_stride, int row_lo, int row_hi);
int mosaic_set_library_shard(mosaic_generator *g, const uint8_t *bgr_slice, int64_t first, int64_t count, int64_t n_total, int size,
                             int64_t capacity_images);
int mosaic_get_library_device(const mosaic_generator *g, void **ptr, int *stored_size, int64_t *capacity_images);

/* ---- kernel-level entry points, mirroring the wrapper functions the reference's kernel tests call
 * (src/Photomosaic/CUDA/PhotomosaicGenerator.cuh:6-43, Reduction.cuh:23; test/tst_ColourDifference.h:233-543,
 * test/tst_CUDAKernel.h:16-272). Host pointers in, host pointers out. */
/* out[i] = diff(a[i], b[i]) for n pixels (3 floats each) -- euclideanDifference / CIEDE2000Difference with size = 1 */
int mosaic_kernel_colour_difference(int device, int type, const float *a, const float *b, int64_t n, float *out);
/* one cell x n_lib images: out[i] = sum over mask != 0 and inside target_area (row0,row1,col0,col1; NULL = all)
 * of diff(cell[p], lib[i][p]) -- imageDifference(+Edge) + reduceAdd + flatten */
int mosaic_kernel_image_difference_sum(int device, int type, const float *cell, const float *lib, int64_t n_lib,
                                       const uint8_t *mask, int size, const int32_t *target_area, float *out);
/* CIEDE2000 pruning bound (no reference counterpart): n_cells cells against n_lib images, pixel axis cut into segments of
   seg_chunks 128-pixel chunks of the compacted mask; out [n_segs - 1][n_cells][n_lib] = R[s - 1], a lower bound of what
   segments s .. n_segs - 1 add to the pair's difference sum */
int mosaic_kernel_prune_bound(int device, const float *cells, int n_cells, const float *lib, int64_t n_lib, const uint8_t *mask,
                              int size, const int32_t *target_area, int seg_chunks, float *out);
/* calculateRepeats + findLowest over a whole grid: scores [n_valid][n_lib] (raster order of valid cells) */
int mosaic_kernel_select(int device, const float *scores, int64_t n_lib, int64_t *grid, int rows, int cols,
                         int repeat_range, int repeat_addition);
/* K smallest (score, index) of each row */
int mosaic_kernel_topk(int device, const float *scores, int64_t n_rows, int64_t n_lib, int k, float *out_scores,
                       int32_t *out_indices);
/* OpenCV-compatible preprocessing pieces */
int mosaic_kernel_bgr_to_lab(int device, const uint8_t *bgr, int64_t n_pixels, float *lab_out);
/* one hue-rotated colour-scheme variant: 8U BGR -> HSV_FULL (f32) -> H = fmod(H + rotation, 360) -> BGR -> 8U (ColourScheme.cpp:36-177) */
int mosaic_kernel_hue_rotate(int device, const uint8_t *bgr, int rows, int cols, float rotation_degrees, uint8_t *out);
int mosaic_kernel_resize_area_u8(int device, const uint8_t *src, int64_t n, int size, int k, uint8_t *dst);
int mosaic_kernel_resize_area_f32(int device, const float *src, int64_t n, int size, int k, float *dst);
int mosaic_kernel_resize_cubic_u8(int device, const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w);
/* The packed inputs of the difference kernels at size step `step`, as a generate on this handle would build them (test tap of the
 * preprocessing): main image variants, library preparation and colour order, and the packing of steps 0 .. step (the working
 * library is halved step by step). No difference or selection kernel runs and the handle's results are kept.
 * info always; cells / lib (cell_bytes / lib_bytes, raw tile layout of csrc/diff_kernels.cu or csrc/diff_euclid.cu),
 * pix_list (n_active compacted pixel indices) and perm (n_lib_tiles * slots_per_tile slot -> image, only when has_perm) when
 * non-NULL. Call with NULL buffers first to size them (the preprocessing runs either way); MOSAIC_ERR_INVALID_ARGUMENT when
 * cells_cap or lib_cap is too small. */
typedef struct mosaic_step_inputs {
    int layout;       /* 0: CIEDE2000 tiles (csrc/diff_kernels.cu), 1: Euclidean tiles (csrc/diff_euclid.cu) */
    int n_variants;   /* difference rows per cell (colour-scheme variants compared) */
    int n_active, n_chunks;
    int n_rows;       /* this handle's rows: its valid cells x n_variants, raster order, variant fastest */
    int n_cell_tiles;
    int64_t n_slots;  /* library slots: orientations x images, orientation-major */
    int n_lib_tiles;
    int cells_per_tile, slots_per_tile, pixels_per_chunk;
    size_t cell_bytes, lib_bytes;
    int fused;        /* one size step: the library packer reads the 8U library and converts on the fly */
    int fused_k;      /* integer reduction the fused packer applies to the stored library (1: none) */
    int has_perm;     /* library tiles in colour order (CIEDE2000 row passes): slot i holds image perm[i] */
} mosaic_step_inputs;
int mosaic_debug_step_inputs(mosaic_generator *g, int step, mosaic_step_inputs *info, void *cells, size_t cells_cap, void *lib,
                             size_t lib_cap, int32_t *pix_list, int32_t *perm);

/* ---- on-disk containers of the reference (Qt-free, OpenCV-free: QDataStream layout and PNG codec inside the library).
 * A file the reference would reject with std::invalid_argument gives MOSAIC_ERR_INVALID_ARGUMENT; mosaic_io_last_error() has
 * the text (thread-local). Strings are UTF-8.
 * .mcs = CellShape::loadFromFile / saveToFile (CellShape/CellShape.cpp:321-434): tiling parameters + the mask as stored.
 *   mask_out may be NULL to query shape->size first; name_out may be NULL. */
int mosaic_mcs_load(const char *path, mosaic_cell_shape *shape, uint8_t *mask_out, size_t mask_capacity, char *name_out,
                    size_t name_capacity);
int mosaic_mcs_save(const char *path, const mosaic_cell_shape *shape, const uint8_t *mask, const char *name_utf8);
/* .mil = ImageLibrary::loadFromFile / saveToFile (ImageLibrary/ImageLibrary.cpp:117-236): n images of image_size^2 x 3 (BGR) and
 * their names. mosaic_mil_info sizes the buffers (names_bytes = all names, each NUL-terminated, back to back). */
int mosaic_mil_info(const char *path, int64_t *n_images, int *image_size, size_t *names_bytes);
int mosaic_mil_load(const char *path, uint8_t *images_out, size_t images_capacity, char *names_out, size_t names_capacity);
int mosaic_mil_save(const char *path, const uint8_t *images, int64_t n_images, int image_size, const char *names_nul_separated);
const char *mosaic_io_last_error(void);

/* ---- library ingest: ImageLibrary::addImage (ImageLibrary/ImageLibrary.cpp:62-86) minus the container bookkeeping.
 * Centre crop to a square (ImageUtility::imageToSquare CROP, Other/ImageUtility.cpp:249-267), then
 * ImageUtility::resizeImage EXACT to image_size (Other/ImageUtility.cpp:34-62: INTER_AREA when shrinking, INTER_CUBIC when
 * growing, a plain copy when the side already matches) -- crop upload, resize and download on the GPU.
 * bgr: 8U BGR rows x cols with row_stride bytes per row; out: image_size x image_size x 3, contiguous.
 * MOSAIC_ERR_INVALID_ARGUMENT for an empty image (std::invalid_argument in the reference, ImageLibrary.cpp:65-66). */
int mosaic_library_ingest(int device, const uint8_t *bgr, int rows, int cols, size_t row_stride, int image_size, uint8_t *out);
/* FP32 / MUFU pipe-rate micro-benchmark (roofline denominators): out[0] FFMA lane-ops/s, [1] FFMA2 lane-ops/s,
 * [2] MUFU.RSQ ops/s, [3] MUFU.EX2 ops/s, [4] SM count, [5] cycles per 16-FFMA loop iteration, and (n_out >= 9) the rate of a
 * synthetic loop in the CIEDE2000 kernel's instruction proportions, in "pixel pairs"/s: [6] 40 FFMA2 + 9 MUFU + 5 ALU,
 * [7] 40 FFMA2 + 9 MUFU, [8] 40 FFMA2; (n_out >= 11) FP32 lane-ops/s of a loop mixing packed and scalar FMAs:
 * [9] 8 FFMA2 + 8 FFMA, [10] 8 FFMA2 + 16 FFMA per iteration */
int mosaic_kernel_microbench(int device, double *out, int n_out);

/* ---- host-side geometry (no GPU needed): GridUtility.cpp:25-52, 86-132; CellShape::resized */
void mosaic_grid_size(const mosaic_cell_shape *shape, int image_w, int image_h, int pad, int *grid_w, int *grid_h);
void mosaic_rect_at(const mosaic_cell_shape *shape, int x, int y, int rect_xywh[4]);
int mosaic_flip_at(const mosaic_cell_shape *shape, int x, int y); /* flip_h + 2 * flip_v */
/* CellGroup::getCell(step, detail) (CellShape/CellGroup.cpp:65-145) of the group mosaic_set_cell_group[_ex] would build, computed on
 * the host without a generator handle (what the CPU tests compare with the reference's own CellGroup.cpp object code) */
int mosaic_host_cell_group_cell(const mosaic_cell_shape *shape, const uint8_t *mask, int mask_as_stored, int cell_size,
                                int detail_percent, int size_steps, int step, int detail, mosaic_cell_shape *out, uint8_t *mask_out,
                                size_t mask_capacity);
/* GridGenerator::getGridState (Grid/GridGenerator.cpp:29-193) with the reference's HOST arithmetic (the generator object
 * evaluates the same rule on the GPU, mosaic_compute_grid_state). Steps are written back to back into out:
 * step s holds step_rows[s] x step_cols[s] values, -1 = nullopt, 0 = valid. bgr may be NULL (no entropy rule). */
int mosaic_host_grid_state(const mosaic_cell_shape *shape, const uint8_t *mask, int cell_size, int detail_percent, int size_steps,
                           const uint8_t *bgr, int rows, int cols, size_t row_stride, int max_steps, int *n_steps, int *step_rows,
                           int *step_cols, int64_t *out, size_t out_capacity);
/* GridBounds::addBound x n + mergeBounds (Grid/GridBounds.cpp:26-104): rects are x, y, w, h quadruples; returns the number of
 * merged bounds (the first min(count, out_capacity) are written to out), or a negative status */
int mosaic_host_merge_bounds(const int *rects_xywh, int n, int *out_xywh, int out_capacity);
/* cv::resize(INTER_AREA) for 8U images with cn channels (OpenCV-compatible, any down-scaling ratio) */
int mosaic_host_resize_area_u8(const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w);
/* cv::resize(INTER_CUBIC) for 8U images with cn channels, as OpenCV's own (non-IPP) code computes it: what
 * ImageUtility::resizeImage uses when growing (Other/ImageUtility.cpp:50-51); CellShape::resized mask growth goes through it */
int mosaic_host_resize_cubic_u8(const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MOSAIC_B200_H */
