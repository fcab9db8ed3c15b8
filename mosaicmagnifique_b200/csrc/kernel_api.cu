// Kernel-level C entry points (include/mosaic_b200.h, "kernel-level entry points"): the counterparts of the
// wrapper functions the reference's kernel tests drive
//   euclideanDifferenceKernelWrapper / CIEDE2000DifferenceKernelWrapper   CUDA/PhotomosaicGenerator.cuh:6-43
//   reduceAddKernelWrapper                                                CUDA/Reduction.cuh:23
//   calculateRepeatsKernelWrapper / findLowestKernelWrapper / flattenKernelWrapper
// Host pointers in, host pointers out; each call runs the SAME kernels the generator uses.
#include <cuda_runtime.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <string>
#include <vector>

#include "../../include/mosaic_b200.h"
#include "containers.h"
#include "host_model.h"
#include "kernels.h"

extern "C" const int16_t mm_lab_lut_s16[];

namespace {

using namespace mm;

struct Dev {
    void *p = nullptr;
    ~Dev()
    {
        if (p)
            cudaFree(p);
    }
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, std::max<size_t>(n, 16)); }
    template <typename T>
    T *as() { return (T *)p; }
};

#define KCHECK(expr)                  \
    do {                              \
        cudaError_t e__ = (expr);     \
        if (e__ != cudaSuccess) {     \
            cudaGetLastError();       \
            return MOSAIC_ERR_CUDA;   \
        }                             \
    } while (0)

int use_device(int device)
{
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return MOSAIC_ERR_CUDA;
    }
    return cudaSetDevice(device) == cudaSuccess ? MOSAIC_OK : MOSAIC_ERR_CUDA;
}

// cells: n_cells images [size*size][3] f32 treated as "main images" of their own; lib: n_lib images
// seg_chunks > 0 (CIEDE2000): instead of the sums, the pruning bound R of segments of seg_chunks chunks (launch_prune_bound) goes to
// out [n_segs - 1][n_cells][n_lib]
int difference_sums(int type, const float *cells, int n_cells, const float *lib, int64_t n_lib, const uint8_t *mask, int size,
                    const int32_t *target_area, float *out /* [n_cells][n_lib] */, int seg_chunks = 0)
{
    const int P = size * size;
    std::vector<int> pix;
    for (int i = 0; i < P; ++i)
        if (mask[i])
            pix.push_back(i);
    const int n_active = (int)pix.size();
    const bool chroma = type == MOSAIC_CIEDE2000;
    const PackLayout layout = chroma ? kLayoutCiede : kLayoutEuclid;
    const TileGeom tg = tile_geom(layout);
    const int n_chunks = std::max(1, (n_active + tg.kp - 1) / tg.kp);
    const int n_lib_tiles = (int)((n_lib + tg.tnb - 1) / tg.tnb), n_lib_pad = n_lib_tiles * tg.tnb;
    const int n_cell_tiles = (n_cells + tg.tcb - 1) / tg.tcb, n_cells_pad = n_cell_tiles * tg.tcb;
    std::vector<uint8_t> m4((size_t)4 * P, 0);
    for (int i = 0; i < P; ++i)
        m4[i] = mask[i] ? 255 : 0;
    std::vector<CellDesc> descs(n_cells);
    for (int c = 0; c < n_cells; ++c) {
        CellDesc d{0, c * size, 0, 0, size, size, 0, 0};
        if (target_area) {  // rows [ta0, ta1), cols [ta2, ta3) as in imageDifferenceEdge (PhotomosaicGenerator.cu:53-72)
            d.by = target_area[0];
            d.bh = target_area[1] - target_area[0];
            d.bx = target_area[2];
            d.bw = target_area[3] - target_area[2];
        }
        descs[c] = d;
    }
    Dev d_cells, d_lib, d_pix, d_m4, d_desc, d_cp, d_lp, d_D;
    KCHECK(d_cells.alloc((size_t)n_cells * P * 3 * sizeof(float)));
    KCHECK(d_lib.alloc((size_t)n_lib * P * 3 * sizeof(float)));
    KCHECK(d_pix.alloc(pix.size() * sizeof(int)));
    KCHECK(d_m4.alloc(m4.size()));
    KCHECK(d_desc.alloc(descs.size() * sizeof(CellDesc)));
    KCHECK(d_cp.alloc((size_t)n_cell_tiles * n_chunks * tg.cell_block));
    KCHECK(d_lp.alloc((size_t)n_lib_tiles * n_chunks * tg.lib_block));
    KCHECK(d_D.alloc((size_t)n_cells_pad * n_lib_pad * sizeof(float)));
    KCHECK(cudaMemcpy(d_cells.p, cells, (size_t)n_cells * P * 3 * sizeof(float), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_lib.p, lib, (size_t)n_lib * P * 3 * sizeof(float), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_pix.p, pix.data(), pix.size() * sizeof(int), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_m4.p, m4.data(), m4.size(), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_desc.p, descs.data(), descs.size() * sizeof(CellDesc), cudaMemcpyHostToDevice));
    KCHECK(launch_pack_library(d_lib.as<float>(), d_lp.p, n_lib, P, d_pix.as<int>(), n_active, n_chunks, n_lib_tiles, layout, 0));
    // the cells stacked vertically form one "main image" of n_cells*size rows; cell c sits at y0 = c*size; the bound
    // is relative to the cell, so descs carry by/bx in cell space (extract_cells tests bounds in detail space, k = 1)
    for (int c = 0; c < n_cells; ++c)
        descs[c].y0 = c * size;
    KCHECK(launch_extract_cells(d_cells.as<float>(), n_cells * size, size, d_desc.as<CellDesc>(), n_cells, size, size, 1,
                                AreaTab{nullptr, nullptr, nullptr}, d_m4.as<uint8_t>(), d_pix.as<int>(), n_active, n_chunks, d_cp.p,
                                layout, 0));
    if (chroma && seg_chunks > 0) {
        const int n_blocks = n_chunks * (MM_KP / MM_BB), n_segs = (n_chunks + seg_chunks - 1) / seg_chunks;
        if (n_segs < 2)
            return MOSAIC_ERR_INVALID_ARGUMENT;
        Dev d_ls, d_cs, d_R;
        KCHECK(d_ls.alloc((size_t)n_blocks * n_lib_pad * sizeof(float4)));
        KCHECK(d_cs.alloc((size_t)n_cells * n_blocks * sizeof(float4)));
        KCHECK(d_R.alloc((size_t)(n_segs - 1) * n_cells * n_lib_pad * sizeof(float)));
        KCHECK(launch_block_stats(d_lp.p, n_lib_tiles, d_cp.p, n_cells, n_chunks, d_ls.as<float4>(), d_cs.as<float4>(), 0));
        KCHECK(launch_prune_bound(d_ls.as<float4>(), d_cs.as<float4>(), n_cells, n_lib_pad, n_blocks, seg_chunks * (MM_KP / MM_BB), n_segs,
                                  d_R.as<float>(), nullptr, nullptr, nullptr, 0));
        KCHECK(cudaMemcpy2D(out, (size_t)n_lib * sizeof(float), d_R.p, (size_t)n_lib_pad * sizeof(float), (size_t)n_lib * sizeof(float),
                            (size_t)(n_segs - 1) * n_cells, cudaMemcpyDeviceToHost));
        return MOSAIC_OK;
    }
    if (chroma)
        KCHECK(launch_diff_sum(MM_DIFF_CIEDE2000, d_cp.p, d_lp.p, d_D.as<float>(), nullptr, n_cell_tiles, n_lib_tiles, n_chunks, (int)n_lib,
                               n_cells, 0));
    else
        KCHECK(launch_diff_euclid(d_cp.p, d_lp.p, d_D.as<float>(), nullptr, n_cell_tiles, n_lib_tiles, n_chunks, (int)n_lib, n_cells, 0));
    KCHECK(cudaMemcpy2D(out, (size_t)n_lib * sizeof(float), d_D.p, (size_t)n_lib_pad * sizeof(float), (size_t)n_lib * sizeof(float),
                        n_cells, cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

}  // namespace

extern "C" {

int mosaic_kernel_image_difference_sum(int device, int type, const float *cell, const float *lib, int64_t n_lib, const uint8_t *mask,
                                       int size, const int32_t *target_area, float *out)
{
    if (!cell || !lib || !mask || !out || n_lib <= 0 || size <= 0 || type < 0 || type > 2)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    return difference_sums(type, cell, 1, lib, n_lib, mask, size, target_area, out);
}

int mosaic_kernel_prune_bound(int device, const float *cells, int n_cells, const float *lib, int64_t n_lib, const uint8_t *mask, int size,
                              const int32_t *target_area, int seg_chunks, float *out)
{
    if (!cells || !lib || !mask || !out || n_cells <= 0 || n_lib <= 0 || size <= 0 || seg_chunks <= 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    return difference_sums(MOSAIC_CIEDE2000, cells, n_cells, lib, n_lib, mask, size, target_area, out, seg_chunks);
}

int mosaic_kernel_colour_difference(int device, int type, const float *a, const float *b, int64_t n, float *out)
{
    // per-pixel differences = difference sums of 1x1 "images" (the reference's tests call its kernels with size = 1,
    // tst_ColourDifference.h:233-309): pixel i of a is a cell, pixel i of b its library image.
    if (!a || !b || !out || n < 0 || type < 0 || type > 2)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (n == 0)
        return MOSAIC_OK;
    if (int rc = use_device(device))
        return rc;
    const uint8_t mask1 = 255;
    const int64_t slab = 2048;  // pixels per launch: D is slab x slab floats (16 MB), only its diagonal is kept
    std::vector<float> D((size_t)slab * slab);
    for (int64_t s0 = 0; s0 < n; s0 += slab) {
        const int64_t m = std::min(slab, n - s0);
        const int rc = difference_sums(type, a + 3 * s0, (int)m, b + 3 * s0, m, &mask1, 1, nullptr, D.data());
        if (rc)
            return rc;
        for (int64_t i = 0; i < m; ++i)
            out[s0 + i] = D[(size_t)i * m + i];
    }
    return MOSAIC_OK;
}

int mosaic_kernel_select(int device, const float *scores, int64_t n_lib, int64_t *grid, int rows, int cols, int repeat_range,
                         int repeat_addition)
{
    if (!scores || !grid || n_lib <= 0 || rows <= 0 || cols <= 0 || repeat_range < 0 || repeat_addition < 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    std::vector<int> pos, next, first(rows, cols);
    std::vector<long long> g((size_t)rows * cols);
    for (int y = 0; y < rows; ++y) {
        int prev = -1;
        for (int x = 0; x < cols; ++x) {
            g[(size_t)y * cols + x] = grid[(size_t)y * cols + x] >= 0 ? 0 : -1;
            if (grid[(size_t)y * cols + x] >= 0) {
                if (prev < 0)
                    first[y] = x;
                else
                    next[prev] = x;
                prev = (int)pos.size();
                pos.push_back(y * cols + x);
                next.push_back(cols);
            }
        }
    }
    const int n_cells = (int)pos.size();
    if (n_cells == 0)
        return MOSAIC_OK;
    const int n_ctas = std::max(1, std::min(n_cells, select_max_ctas(device)));
    Dev d_s, d_g, d_pos, d_next, d_prog, d_cnt;
    KCHECK(d_s.alloc((size_t)n_cells * n_lib * sizeof(float)));
    KCHECK(d_g.alloc(g.size() * sizeof(long long)));
    KCHECK(d_pos.alloc(pos.size() * sizeof(int)));
    KCHECK(d_next.alloc(next.size() * sizeof(int)));
    KCHECK(d_prog.alloc((size_t)rows * sizeof(int)));
    KCHECK(d_cnt.alloc((size_t)n_ctas * n_lib * sizeof(int)));
    KCHECK(cudaMemcpy(d_s.p, scores, (size_t)n_cells * n_lib * sizeof(float), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_g.p, g.data(), g.size() * sizeof(long long), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_pos.p, pos.data(), pos.size() * sizeof(int), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_next.p, next.data(), next.size() * sizeof(int), cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_prog.p, first.data(), (size_t)rows * sizeof(int), cudaMemcpyHostToDevice));
    KCHECK(cudaMemset(d_cnt.p, 0, (size_t)n_ctas * n_lib * sizeof(int)));
    KCHECK(launch_select(d_g.as<long long>(), d_pos.as<int>(), d_next.as<int>(), n_cells, rows, cols, d_s.as<float>(), nullptr, (int)n_lib,
                         (int)n_lib, (int)n_lib, repeat_range, repeat_addition, d_prog.as<int>(), d_cnt.as<int>(), n_ctas, nullptr, 0));
    KCHECK(cudaMemcpy(g.data(), d_g.p, g.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < g.size(); ++i)
        grid[i] = g[i];
    return MOSAIC_OK;
}

int mosaic_kernel_topk(int device, const float *scores, int64_t n_rows, int64_t n_lib, int k, float *out_scores, int32_t *out_indices)
{
    if (!scores || !out_scores || !out_indices || n_rows <= 0 || n_lib <= 0 || k <= 0 || k > n_lib)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    Dev d_s, d_os, d_oi;
    KCHECK(d_s.alloc((size_t)n_rows * n_lib * sizeof(float)));
    KCHECK(d_os.alloc((size_t)n_rows * k * sizeof(float)));
    KCHECK(d_oi.alloc((size_t)n_rows * k * sizeof(int)));
    KCHECK(cudaMemcpy(d_s.p, scores, (size_t)n_rows * n_lib * sizeof(float), cudaMemcpyHostToDevice));
    KCHECK(launch_topk(d_s.as<float>(), (int)n_lib, (int)n_lib, (int)n_rows, k, d_os.as<float>(), d_oi.as<int>(), 0));
    KCHECK(cudaMemcpy(out_scores, d_os.p, (size_t)n_rows * k * sizeof(float), cudaMemcpyDeviceToHost));
    KCHECK(cudaMemcpy(out_indices, d_oi.p, (size_t)n_rows * k * sizeof(int), cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

int mosaic_kernel_bgr_to_lab(int device, const uint8_t *bgr, int64_t n_pixels, float *lab_out)
{
    if (!bgr || !lab_out || n_pixels <= 0 || n_pixels > INT32_MAX)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    Dev d_in, d_out, d_lut;
    KCHECK(d_in.alloc((size_t)n_pixels * 3));
    KCHECK(d_out.alloc((size_t)n_pixels * 3 * sizeof(float)));
    const std::vector<int16_t> lut4 = expand_lab_lut(mm_lab_lut_s16);
    KCHECK(d_lut.alloc(lut4.size() * sizeof(int16_t)));
    KCHECK(cudaMemcpy(d_in.p, bgr, (size_t)n_pixels * 3, cudaMemcpyHostToDevice));
    KCHECK(cudaMemcpy(d_lut.p, lut4.data(), lut4.size() * sizeof(int16_t), cudaMemcpyHostToDevice));
    KCHECK(launch_to_working_space(d_in.as<uint8_t>(), (size_t)n_pixels * 3, 1, (int)n_pixels, d_out.as<float>(), true, d_lut.as<short4>(),
                                   nullptr, 0));
    KCHECK(cudaMemcpy(lab_out, d_out.p, (size_t)n_pixels * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

int mosaic_kernel_hue_rotate(int device, const uint8_t *bgr, int rows, int cols, float rotation_degrees, uint8_t *out)
{
    const int64_t n_pixels = (int64_t)rows * cols;
    if (!bgr || !out || rows <= 0 || cols <= 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    Dev d_in, d_out;
    KCHECK(d_in.alloc((size_t)n_pixels * 3));
    KCHECK(d_out.alloc((size_t)n_pixels * 3));
    KCHECK(cudaMemcpy(d_in.p, bgr, (size_t)n_pixels * 3, cudaMemcpyHostToDevice));
    KCHECK(launch_hue_rotate(d_in.as<uint8_t>(), d_out.as<uint8_t>(), rows, cols, rotation_degrees, 0));
    KCHECK(cudaMemcpy(out, d_out.p, (size_t)n_pixels * 3, cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

int mosaic_kernel_resize_area_u8(int device, const uint8_t *src, int64_t n, int size, int k, uint8_t *dst)
{
    if (!src || !dst || n <= 0 || size <= 0 || k < 1 || size % k != 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    const int ds = size / k;
    Dev d_in, d_out;
    KCHECK(d_in.alloc((size_t)n * size * size * 3));
    KCHECK(d_out.alloc((size_t)n * ds * ds * 3));
    KCHECK(cudaMemcpy(d_in.p, src, (size_t)n * size * size * 3, cudaMemcpyHostToDevice));
    KCHECK(launch_area_u8(d_in.as<uint8_t>(), d_out.as<uint8_t>(), n, size, k, 0));
    KCHECK(cudaMemcpy(dst, d_out.p, (size_t)n * ds * ds * 3, cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

int mosaic_kernel_resize_area_f32(int device, const float *src, int64_t n, int size, int k, float *dst)
{
    if (!src || !dst || n <= 0 || size <= 0 || k < 1 || size % k != 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    const int ds = size / k;
    Dev d_in, d_out;
    KCHECK(d_in.alloc((size_t)n * size * size * 3 * sizeof(float)));
    KCHECK(d_out.alloc((size_t)n * ds * ds * 3 * sizeof(float)));
    KCHECK(cudaMemcpy(d_in.p, src, (size_t)n * size * size * 3 * sizeof(float), cudaMemcpyHostToDevice));
    KCHECK(launch_area_f32(d_in.as<float>(), d_out.as<float>(), n, size, k, 0));
    KCHECK(cudaMemcpy(dst, d_out.p, (size_t)n * ds * ds * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

namespace {
struct CubicDev {
    Dev idx, coef;
    CubicTab tab{};
    cudaError_t upload(const CubicTable &t)
    {
        cudaError_t e = idx.alloc(t.idx.size() * sizeof(int));
        if (e == cudaSuccess)
            e = coef.alloc(t.coef.size() * sizeof(int16_t));
        if (e == cudaSuccess)
            e = cudaMemcpy(idx.p, t.idx.data(), t.idx.size() * sizeof(int), cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
            e = cudaMemcpy(coef.p, t.coef.data(), t.coef.size() * sizeof(int16_t), cudaMemcpyHostToDevice);
        tab = CubicTab{idx.as<int>(), coef.as<int16_t>()};
        return e;
    }
};

// device image (contiguous, cn channels) -> device image of another size with the reference's choice of filter
// (ImageUtility::resizeImage: INTER_AREA when shrinking, INTER_CUBIC when growing); square, 3 channels for INTER_AREA
int resize_like_reference(const uint8_t *d_src, int side, uint8_t *d_dst, int new_side)
{
    if (new_side < side) {
        if (side % new_side == 0) {
            KCHECK(launch_area_u8(d_src, d_dst, 1, side, side / new_side, 0));
        } else {
            const AreaTable t = make_area_table(side, new_side);
            Dev ts, tsi, ta;
            KCHECK(ts.alloc(t.start.size() * sizeof(int)));
            KCHECK(tsi.alloc(t.si.size() * sizeof(int)));
            KCHECK(ta.alloc(t.alpha.size() * sizeof(float)));
            KCHECK(cudaMemcpy(ts.p, t.start.data(), t.start.size() * sizeof(int), cudaMemcpyHostToDevice));
            KCHECK(cudaMemcpy(tsi.p, t.si.data(), t.si.size() * sizeof(int), cudaMemcpyHostToDevice));
            KCHECK(cudaMemcpy(ta.p, t.alpha.data(), t.alpha.size() * sizeof(float), cudaMemcpyHostToDevice));
            KCHECK(launch_area_general_u8(d_src, d_dst, 1, side, new_side, AreaTab{ts.as<int>(), tsi.as<int>(), ta.as<float>()}, 0));
            KCHECK(cudaDeviceSynchronize());  // the tables die with this scope
        }
    } else {
        CubicDev xt;
        KCHECK(xt.upload(make_cubic_table(side, new_side)));
        KCHECK(launch_cubic_u8(d_src, side, side, 3, d_dst, new_side, new_side, xt.tab, xt.tab, 0));
        KCHECK(cudaDeviceSynchronize());
    }
    return MOSAIC_OK;
}
}  // namespace

int mosaic_kernel_resize_cubic_u8(int device, const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w)
{
    if (!src || !dst || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0 || cn <= 0)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    Dev d_in, d_out;
    CubicDev xt, yt;
    KCHECK(d_in.alloc((size_t)src_h * src_w * cn));
    KCHECK(d_out.alloc((size_t)dst_h * dst_w * cn));
    KCHECK(cudaMemcpy(d_in.p, src, (size_t)src_h * src_w * cn, cudaMemcpyHostToDevice));
    KCHECK(xt.upload(make_cubic_table(src_w, dst_w)));
    KCHECK(yt.upload(make_cubic_table(src_h, dst_h)));
    KCHECK(launch_cubic_u8(d_in.as<uint8_t>(), src_h, src_w, cn, d_out.as<uint8_t>(), dst_h, dst_w, xt.tab, yt.tab, 0));
    KCHECK(cudaMemcpy(dst, d_out.p, (size_t)dst_h * dst_w * cn, cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

// ---------------------------------------------------------------------------------------- containers (.mcs / .mil)
namespace {
thread_local std::string g_io_error;
int io_fail(const std::string &err)
{
    g_io_error = err;
    return MOSAIC_ERR_INVALID_ARGUMENT;
}
// nothing may throw across the C ABI (a multi-gigabyte file can make a vector allocation fail)
int io_guard(const std::function<int()> &body)
{
    try {
        return body();
    } catch (const std::bad_alloc &) {
        return io_fail("out of host memory");
    } catch (const std::exception &e) {
        return io_fail(e.what());
    }
}
void copy_text(const std::string &s, char *out, size_t cap)
{
    if (!out || !cap)
        return;
    const size_t n = std::min(cap - 1, s.size());
    memcpy(out, s.data(), n);
    out[n] = 0;
}
}  // namespace

const char *mosaic_io_last_error(void) { return g_io_error.c_str(); }

int mosaic_mcs_load(const char *path, mosaic_cell_shape *shape, uint8_t *mask_out, size_t mask_capacity, char *name_out,
                    size_t name_capacity)
{
    return io_guard([&]() -> int {
        if (!path || !shape)
            return io_fail("null argument");
        McsFile f;
        std::string err;
        if (!load_mcs(path, f, err))
            return io_fail(err);
        const Shape &s = f.shape;
        *shape = mosaic_cell_shape{s.size, s.row_spacing, s.col_spacing, s.alt_row_spacing, s.alt_col_spacing, s.alt_row_offset,
                                   s.alt_col_offset, s.alt_col_flip_h, s.alt_col_flip_v, s.alt_row_flip_h, s.alt_row_flip_v};
        if (mask_out) {
            if (mask_capacity < s.mask.size())
                return io_fail("mask buffer too small");
            memcpy(mask_out, s.mask.data(), s.mask.size());
        }
        copy_text(f.name, name_out, name_capacity);
        return MOSAIC_OK;
    });
}

int mosaic_mcs_save(const char *path, const mosaic_cell_shape *shape, const uint8_t *mask, const char *name_utf8)
{
    return io_guard([&]() -> int {
        if (!path || !shape || !mask || shape->size <= 0)
            return io_fail("null argument");
        McsFile f;
        f.name = name_utf8 ? name_utf8 : "";
        Shape &s = f.shape;
        s.size = shape->size;
        s.mask.assign(mask, mask + (size_t)shape->size * shape->size);
        s.row_spacing = shape->row_spacing; s.col_spacing = shape->col_spacing;
        s.alt_row_spacing = shape->alt_row_spacing; s.alt_col_spacing = shape->alt_col_spacing;
        s.alt_row_offset = shape->alt_row_offset; s.alt_col_offset = shape->alt_col_offset;
        s.alt_col_flip_h = shape->alt_col_flip_h != 0; s.alt_col_flip_v = shape->alt_col_flip_v != 0;
        s.alt_row_flip_h = shape->alt_row_flip_h != 0; s.alt_row_flip_v = shape->alt_row_flip_v != 0;
        std::string err;
        return save_mcs(path, f, err) ? MOSAIC_OK : io_fail(err);
    });
}

int mosaic_mil_info(const char *path, int64_t *n_images, int *image_size, size_t *names_bytes)
{
    return io_guard([&]() -> int {
        if (!path)
            return io_fail("null argument");
        MilFile f;
        std::string err;
        if (!load_mil(path, f, err))
            return io_fail(err);
        if (n_images)
            *n_images = (int64_t)f.names.size();
        if (image_size)
            *image_size = f.image_size;
        if (names_bytes) {
            *names_bytes = 0;
            for (const std::string &n : f.names)
                *names_bytes += n.size() + 1;
        }
        return MOSAIC_OK;
    });
}

int mosaic_mil_load(const char *path, uint8_t *images_out, size_t images_capacity, char *names_out, size_t names_capacity)
{
    return io_guard([&]() -> int {
        if (!path)
            return io_fail("null argument");
        MilFile f;
        std::string err;
        if (!load_mil(path, f, err))
            return io_fail(err);
        if (images_out) {
            if (images_capacity < f.images.size())
                return io_fail("image buffer too small");
            memcpy(images_out, f.images.data(), f.images.size());
        }
        if (names_out) {
            size_t off = 0;
            for (const std::string &n : f.names) {
                if (off + n.size() + 1 > names_capacity)
                    return io_fail("name buffer too small");
                memcpy(names_out + off, n.c_str(), n.size() + 1);
                off += n.size() + 1;
            }
        }
        return MOSAIC_OK;
    });
}

int mosaic_mil_save(const char *path, const uint8_t *images, int64_t n_images, int image_size, const char *names_nul_separated)
{
    return io_guard([&]() -> int {
        if (!path || n_images < 0 || image_size < 0 || (n_images > 0 && !images))
            return io_fail("null argument");
        MilFile f;
        f.image_size = image_size;
        f.images.assign(images, images + (size_t)n_images * image_size * image_size * 3);
        const char *p = names_nul_separated;
        for (int64_t i = 0; i < n_images; ++i) {
            f.names.push_back(p ? std::string(p) : std::string());
            if (p)
                p += f.names.back().size() + 1;
        }
        std::string err;
        return save_mil(path, f, err) ? MOSAIC_OK : io_fail(err);
    });
}

int mosaic_host_merge_bounds(const int *rects_xywh, int n, int *out_xywh, int out_capacity)
{
    if (n < 0 || (n > 0 && !rects_xywh) || out_capacity < 0 || (out_capacity > 0 && !out_xywh))
        return MOSAIC_ERR_INVALID_ARGUMENT;
    std::vector<Rect> b((size_t)n);
    for (int i = 0; i < n; ++i) {
        b[i].x = rects_xywh[4 * i];
        b[i].y = rects_xywh[4 * i + 1];
        b[i].w = rects_xywh[4 * i + 2];
        b[i].h = rects_xywh[4 * i + 3];
    }
    if (!b.empty())
        merge_bounds(b);
    for (size_t i = 0; i < b.size() && (int)i < out_capacity; ++i) {
        out_xywh[4 * i] = b[i].x;
        out_xywh[4 * i + 1] = b[i].y;
        out_xywh[4 * i + 2] = b[i].w;
        out_xywh[4 * i + 3] = b[i].h;
    }
    return (int)b.size();
}

int mosaic_host_resize_cubic_u8(const uint8_t *src, int src_h, int src_w, int cn, uint8_t *dst, int dst_h, int dst_w)
{
    if (!src || !dst)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    return resize_cubic_u8(src, src_h, src_w, cn, dst, dst_h, dst_w) ? MOSAIC_OK : MOSAIC_ERR_INVALID_ARGUMENT;
}

int mosaic_library_ingest(int device, const uint8_t *bgr, int rows, int cols, size_t row_stride, int image_size, uint8_t *out)
{
    if (!bgr || !out || rows <= 0 || cols <= 0 || image_size <= 0 || row_stride < (size_t)cols * 3)
        return MOSAIC_ERR_INVALID_ARGUMENT;  // empty image: std::invalid_argument, ImageLibrary.cpp:65-66
    if (int rc = use_device(device))
        return rc;
    // ImageUtility::imageToSquare, CROP (ImageUtility.cpp:255-267): keep the centre square, offset = (long - short) / 2
    const int side = std::min(rows, cols);
    const int y0 = cols < rows ? (rows - cols) / 2 : 0, x0 = cols > rows ? (cols - rows) / 2 : 0;
    const uint8_t *crop = bgr + (size_t)y0 * row_stride + (size_t)x0 * 3;
    Dev d_in, d_out;
    KCHECK(d_in.alloc((size_t)side * side * 3));
    KCHECK(cudaMemcpy2D(d_in.p, (size_t)side * 3, crop, row_stride, (size_t)side * 3, side, cudaMemcpyHostToDevice));
    if (side == image_size) {  // resizeFactor == 1: the image itself (ImageUtility.cpp:47-48)
        KCHECK(cudaMemcpy(out, d_in.p, (size_t)side * side * 3, cudaMemcpyDeviceToHost));
        return MOSAIC_OK;
    }
    KCHECK(d_out.alloc((size_t)image_size * image_size * 3));
    if (int rc = resize_like_reference(d_in.as<uint8_t>(), side, d_out.as<uint8_t>(), image_size))
        return rc;
    KCHECK(cudaMemcpy(out, d_out.p, (size_t)image_size * image_size * 3, cudaMemcpyDeviceToHost));
    return MOSAIC_OK;
}

int mosaic_kernel_microbench(int device, double *out, int n_out)
{
    if (!out || n_out < 6)
        return MOSAIC_ERR_INVALID_ARGUMENT;
    if (int rc = use_device(device))
        return rc;
    KCHECK(run_microbench(out, n_out, 0));
    return MOSAIC_OK;
}

}  // extern "C"
