// GPU preprocessing: colour-space conversion, INTER_AREA resizing, cell extraction and packing.
//
// Replaces the OpenCV calls of the reference's preprocessing
//   preprocessMainImage      src/Photomosaic/PhotomosaicGeneratorBase.cpp:223-252
//   preprocessLibraryImages  src/Photomosaic/PhotomosaicGeneratorBase.cpp:255-290
//   getCellAt                src/Photomosaic/PhotomosaicGeneratorBase.cpp:293-329
//   batchResizeMat(lib, .5)  src/Other/ImageUtility.cpp:91-101 (CPUPhotomosaicGenerator.cpp:95-99)
// bit-exactly with OpenCV's own arithmetic (probed against cv2 4.13, tests/test_prep_parity.py):
//   * cvtColor(f32, BGR2Lab) is a 33^3 int16 LUT with 4-bit trilinear weights, not the analytic formula;
//   * INTER_AREA with an integer ratio k sums each k x k block in groups of four in row-major order and
//     multiplies by float(1/k^2); the 8U version rounds (s+2)>>2 for k == 2 and to nearest-even otherwise.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>

#include "colour_math.cuh"
#include "host_model.h"
#include "kernels.h"

namespace mm {

// ------------------------------------------------------------------ BGR8 -> working space

__device__ __forceinline__ int lab_coord(unsigned char v)
{
    // convertTo(CV_32F, 1/255.0) multiplies in f32 by float(1/255.0); cvRound(x * LAB_BASE), LAB_BASE = 1 << 14
    const float f = __fmul_rn((float)v, 0.003921568859368563f);
    return __float2int_rn(__fmul_rn(f, 16384.0f));
}

__device__ __forceinline__ void lab_from_bgr8(unsigned char b8, unsigned char g8, unsigned char r8,
                                              const short4 *__restrict__ lut, float &L, float &a, float &b)
{
    const int cb = lab_coord(b8), cg = lab_coord(g8), cr = lab_coord(r8);
    const int tb = cb >> 9, tg = cg >> 9, tr = cr >> 9;
    const int wb = (cb >> 5) & 15, wg = (cg >> 5) & 15, wr = (cr >> 5) & 15;
    int sL = 0, sa = 0, sb = 0;
#pragma unroll
    for (int db = 0; db < 2; ++db)
#pragma unroll
        for (int dg = 0; dg < 2; ++dg)
#pragma unroll
            for (int dr = 0; dr < 2; ++dr) {
                const int w = (db ? wb : 16 - wb) * (dg ? wg : 16 - wg) * (dr ? wr : 16 - wr);
                const int ib = min(tb + db, 32), ig = min(tg + dg, 32), ir = min(tr + dr, 32);
                const short4 e = lut[(ib * 33 + ig) * 33 + ir];  // (L, a, b, -): one 8-byte load per cube corner
                sL += w * e.x;
                sa += w * e.y;
                sb += w * e.z;
            }
    const int iL = (sL + 2048) >> 12, ia = (sa + 2048) >> 12, ib2 = (sb + 2048) >> 12;
    L = __fmul_rn((float)iL * (1.0f / 16384.0f), 100.0f);
    a = __fadd_rn(__fmul_rn((float)ia * (1.0f / 16384.0f), 256.0f), -128.0f);
    b = __fadd_rn(__fmul_rn((float)ib2 * (1.0f / 16384.0f), 256.0f), -128.0f);
}

__global__ void to_working_space_kernel(const uint8_t *__restrict__ bgr, size_t row_stride, int rows, int cols,
                                        float *__restrict__ out, bool is_lab, const short4 *__restrict__ lut)
{
    const size_t n = (size_t)rows * cols;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t y = i / cols, x = i - y * cols;
        const uint8_t *p = bgr + y * row_stride + x * 3;
        float v0, v1, v2;
        if (is_lab) {
            lab_from_bgr8(p[0], p[1], p[2], lut, v0, v1, v2);
        } else {
            v0 = (float)p[0];
            v1 = (float)p[1];
            v2 = (float)p[2];
        }
        out[i * 3 + 0] = v0;
        out[i * 3 + 1] = v1;
        out[i * 3 + 2] = v2;
    }
}

static int grid_for(size_t n, int block)
{
    size_t g = (n + block - 1) / block;
    const size_t cap = 148 * 32;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

cudaError_t launch_to_working_space(const uint8_t *bgr, size_t row_stride, int rows, int cols, float *out, bool is_lab,
                                    const short4 *lab_lut, const int *, cudaStream_t stream)
{
    const size_t n = (size_t)rows * cols;
    if (n == 0)
        return cudaSuccess;
    to_working_space_kernel<<<grid_for(n, 256), 256, 0, stream>>>(bgr, row_stride, rows, cols, out, is_lab, lab_lut);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ colour-scheme variants (hue rotation)
// ColourScheme::getColourScheme* (src/Photomosaic/ColourScheme.cpp:36-177): 8U BGR -> f32 -> cvtColor(BGR2HSV_FULL)
// -> H = fmod(H + rot, 360) -> cvtColor(HSV2BGR_FULL) -> convertTo(8U). OpenCV's float HSV code contracts a few
// operations into FMAs (probed against cv2 4.13, bit-exact with the forms below):
//   H = fma(c1 - c2, 60/(diff + eps), offset), offset in {0 or 360, 120, 240};  tab2 = V * fma(-S, f, 1);  tab3 = V * fma(-S, 1 - f, 1)
// OpenCV converts rows in blocks of 8 pixels (8-lane float SIMD); the < 8 pixels left at the end of a row go through its
// scalar code, where a negative red-sector hue gets "+ 360" as a separate rounded addition (`scalar_tail`).
__device__ __forceinline__ void hue_rotate_pixel(const uint8_t *in, uint8_t *out, float rot, bool scalar_tail)
{
    const float b = (float)in[0], g = (float)in[1], r = (float)in[2];
    const float eps = 1.1920928955078125e-07f;  // FLT_EPSILON
    const float v = fmaxf(fmaxf(r, g), b), vmin = fminf(fminf(r, g), b);
    const float diff = __fsub_rn(v, vmin);
    const float s = __fdiv_rn(diff, __fadd_rn(fabsf(v), eps));
    const float d = __fdiv_rn(60.0f, __fadd_rn(diff, eps));
    float h;
    if (v == r) {
        if (scalar_tail) {
            h = __fmul_rn(__fsub_rn(g, b), d);
            if (h < 0.0f)
                h = __fadd_rn(h, 360.0f);
        } else {
            h = __fmaf_rn(__fsub_rn(g, b), d, g < b ? 360.0f : 0.0f);
        }
    }
    else if (v == g)
        h = __fmaf_rn(__fsub_rn(b, r), d, 120.0f);
    else
        h = __fmaf_rn(__fsub_rn(r, g), d, 240.0f);
    h = fmodf(__fadd_rn(h, rot), 360.0f);  // ColourScheme.cpp:52 etc.
    // HSV2BGR_FULL
    const float hs = __fmul_rn(h, 6.0f / 360.0f);
    const float pre = truncf(hs);
    const float f = __fsub_rn(hs, pre);
    float tab[4];
    tab[0] = v;
    tab[1] = __fmul_rn(v, __fsub_rn(1.0f, s));
    tab[2] = __fmul_rn(v, __fmaf_rn(-s, f, 1.0f));
    tab[3] = __fmul_rn(v, __fmaf_rn(-s, __fsub_rn(1.0f, f), 1.0f));
    int sector = (int)__fsub_rn(pre, __fmul_rn(truncf(__fmul_rn(pre, 1.0f / 6.0f)), 6.0f));
    sector = min(max(sector, 0), 5);
    const int sd[6][3] = {{1, 3, 0}, {1, 0, 2}, {3, 0, 1}, {0, 2, 1}, {0, 1, 3}, {2, 1, 0}};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float t = tab[0];
#pragma unroll
        for (int k = 1; k < 4; ++k)
            t = (sd[sector][c] == k) ? tab[k] : t;
        out[c] = (uint8_t)min(max(__float2int_rn(t), 0), 255);  // convertTo(8U): saturate_cast(cvRound)
    }
}

__global__ void hue_rotate_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, size_t n, float rot, int cols)
{
    const int tail_from = cols - cols % 8;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        hue_rotate_pixel(in + i * 3, out + i * 3, rot, (int)(i % cols) >= tail_from);
}

cudaError_t launch_hue_rotate(const uint8_t *in, uint8_t *out, int rows, int cols, float rot, cudaStream_t stream)
{
    const size_t n_pixels = (size_t)rows * cols;
    if (n_pixels == 0)
        return cudaSuccess;
    hue_rotate_kernel<<<grid_for(n_pixels, 256), 256, 0, stream>>>(in, out, n_pixels, rot, cols);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ INTER_AREA, integer ratio

__global__ void area_u8_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int64_t n, int S, int k)
{
    const int ds = S / k;
    const size_t total = (size_t)n * ds * ds * 3;
    const float scale = 1.0f / (float)(k * k);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i % 3);
        size_t t = i / 3;
        const int dx = (int)(t % ds);
        t /= ds;
        const int dy = (int)(t % ds);
        const size_t im = t / ds;
        const uint8_t *s = src + (im * S * S + (size_t)(dy * k) * S + (size_t)dx * k) * 3 + ch;
        int sum = 0;
        for (int yy = 0; yy < k; ++yy)
            for (int xx = 0; xx < k; ++xx)
                sum += s[((size_t)yy * S + xx) * 3];
        int v;
        if (k == 2)
            v = (sum + 2) >> 2;  // OpenCV's SIMD 2x2 path
        else
            v = __float2int_rn(__fmul_rn((float)sum, scale));  // saturate_cast<uchar>(sum * scale): cvRound, ties to even
        dst[i] = (uint8_t)min(max(v, 0), 255);
    }
}

cudaError_t launch_area_u8(const uint8_t *src, uint8_t *dst, int64_t n, int src_size, int k, cudaStream_t stream)
{
    const size_t total = (size_t)n * (src_size / k) * (src_size / k) * 3;
    if (total == 0)
        return cudaSuccess;
    area_u8_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, n, src_size, k);
    return cudaGetLastError();
}

// Oriented library: dst[j][i] = source image i mirrored by the j-th orientation of `codes` (2 bits each, code = flip_h + 2 * flip_v;
// flip_h mirrors the columns like cv::flip code 1, flip_v the rows like code 0). One thread per output pixel of 3 bytes.
__global__ void orient_library_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int64_t n, int S, int n_orient,
                                      unsigned codes)
{
    const size_t img_px = (size_t)S * S;
    const size_t total = (size_t)n_orient * n * img_px;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t im = i / img_px;  // output image = j * n + source image
        const int p = (int)(i - im * img_px);
        const int j = (int)(im / n);
        const size_t si = im - (size_t)j * n;
        const unsigned code = (codes >> (2 * j)) & 3u;
        int y = p / S, x = p - (p / S) * S;
        if (code & 1u)
            x = S - 1 - x;
        if (code & 2u)
            y = S - 1 - y;
        const uint8_t *s = src + (si * img_px + (size_t)y * S + x) * 3;
        uint8_t *d = dst + i * 3;
        d[0] = s[0];
        d[1] = s[1];
        d[2] = s[2];
    }
}

cudaError_t launch_orient_library(const uint8_t *src, uint8_t *dst, int64_t n, int S, int flips, cudaStream_t stream)
{
    if (flips < 0 || flips > 3)
        return cudaErrorInvalidValue;
    int n_orient = 0;
    unsigned codes = 0;
    for (int c = 0; c < 4; ++c)
        if ((c & ~flips) == 0)
            codes |= (unsigned)c << (2 * n_orient++);
    const size_t total = (size_t)n_orient * n * S * S;
    if (total == 0)
        return cudaSuccess;
    orient_library_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, n, S, n_orient, codes);
    return cudaGetLastError();
}

// One output pixel of the same 8U INTER_AREA (integer ratio k) straight from the source image: what the fused library packers read
// when the resize to the detail size has not been materialised (k == 1: the pixel itself)
__device__ __forceinline__ void area_pixel_u8(const uint8_t *__restrict__ img, int S, int k, int py, int px, int out[3])
{
    const uint8_t *s = img + ((size_t)(py * k) * S + (size_t)px * k) * 3;
    if (k == 1) {
        out[0] = s[0];
        out[1] = s[1];
        out[2] = s[2];
        return;
    }
    int sum[3] = {0, 0, 0};
    for (int yy = 0; yy < k; ++yy)
        for (int xx = 0; xx < k; ++xx) {
            const uint8_t *t = s + ((size_t)yy * S + xx) * 3;
            sum[0] += t[0];
            sum[1] += t[1];
            sum[2] += t[2];
        }
    const float scale = 1.0f / (float)(k * k);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int v = (k == 2) ? (sum[c] + 2) >> 2 : __float2int_rn(__fmul_rn((float)sum[c], scale));
        out[c] = min(max(v, 0), 255);
    }
}

// sum of a k x k block in OpenCV's order: groups of four taps (row-major inside the block) are added
// left to right and each group total is added to the running sum; the remainder tap by tap.
template <typename F>
__device__ __forceinline__ float area_block_f32(int k, F tap)
{
    const int area = k * k;
    float sum = 0.0f;
    int t = 0;
    for (; t + 4 <= area; t += 4) {
        const float g = __fadd_rn(__fadd_rn(__fadd_rn(tap(t), tap(t + 1)), tap(t + 2)), tap(t + 3));
        sum = __fadd_rn(sum, g);
    }
    for (; t < area; ++t)
        sum = __fadd_rn(sum, tap(t));
    return __fmul_rn(sum, 1.0f / (float)area);
}

__global__ void area_f32_kernel(const float *__restrict__ src, float *__restrict__ dst, int64_t n, int S, int k)
{
    const int ds = S / k;
    const size_t total = (size_t)n * ds * ds * 3;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i % 3);
        size_t t = i / 3;
        const int dx = (int)(t % ds);
        t /= ds;
        const int dy = (int)(t % ds);
        const size_t im = t / ds;
        const float *s = src + (im * S * S + (size_t)(dy * k) * S + (size_t)dx * k) * 3 + ch;
        dst[i] = area_block_f32(k, [&](int tp) { return s[((size_t)(tp / k) * S + (tp % k)) * 3]; });
    }
}

cudaError_t launch_area_f32(const float *src, float *dst, int64_t n, int src_size, int k, cudaStream_t stream)
{
    const size_t total = (size_t)n * (src_size / k) * (src_size / k) * 3;
    if (total == 0)
        return cudaSuccess;
    area_f32_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, n, src_size, k);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ INTER_AREA, any down-scaling ratio
// OpenCV's resizeArea_: per source row of the destination row's span, buf = sum_k S[sx_k] * alpha_k accumulated in
// table order from 0; rows are combined as sum = beta_0 * buf_0, sum += beta_j * buf_j. No FMA contraction.
template <typename F>
__device__ __forceinline__ float area_general(const AreaTab &t, int dy, int dx, F tap)
{
    float sum = 0.0f;
    const int y0 = t.start[dy], y1 = t.start[dy + 1];
    const int x0 = t.start[dx], x1 = t.start[dx + 1];
    for (int j = y0; j < y1; ++j) {
        const int sy = t.si[j];
        float buf = 0.0f;
        for (int k = x0; k < x1; ++k)
            buf = __fadd_rn(buf, __fmul_rn(tap(sy, t.si[k]), t.alpha[k]));
        const float term = __fmul_rn(t.alpha[j], buf);
        sum = (j == y0) ? term : __fadd_rn(sum, term);
    }
    return sum;
}

__global__ void area_general_u8_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int64_t n, int S, int ds, AreaTab tab)
{
    const size_t total = (size_t)n * ds * ds * 3;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i % 3);
        size_t t = i / 3;
        const int dx = (int)(t % ds);
        t /= ds;
        const int dy = (int)(t % ds);
        const uint8_t *s = src + (t / ds) * (size_t)S * S * 3 + ch;
        const float v = area_general(tab, dy, dx, [&](int sy, int sx) { return (float)s[((size_t)sy * S + sx) * 3]; });
        dst[i] = (uint8_t)min(max(__float2int_rn(v), 0), 255);  // saturate_cast<uchar>: cvRound, ties to even
    }
}

__global__ void area_general_f32_kernel(const float *__restrict__ src, float *__restrict__ dst, int64_t n, int S, int ds, AreaTab tab)
{
    const size_t total = (size_t)n * ds * ds * 3;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i % 3);
        size_t t = i / 3;
        const int dx = (int)(t % ds);
        t /= ds;
        const int dy = (int)(t % ds);
        const float *s = src + (t / ds) * (size_t)S * S * 3 + ch;
        dst[i] = area_general(tab, dy, dx, [&](int sy, int sx) { return s[((size_t)sy * S + sx) * 3]; });
    }
}

cudaError_t launch_area_general_u8(const uint8_t *src, uint8_t *dst, int64_t n, int src_size, int dst_size, AreaTab tab,
                                   cudaStream_t stream)
{
    const size_t total = (size_t)n * dst_size * dst_size * 3;
    if (total == 0)
        return cudaSuccess;
    area_general_u8_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, n, src_size, dst_size, tab);
    return cudaGetLastError();
}

cudaError_t launch_area_general_f32(const float *src, float *dst, int64_t n, int src_size, int dst_size, AreaTab tab,
                                    cudaStream_t stream)
{
    const size_t total = (size_t)n * dst_size * dst_size * 3;
    if (total == 0)
        return cudaSuccess;
    area_general_f32_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, n, src_size, dst_size, tab);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ INTER_CUBIC (8U), library ingest / mask growth
//
// cv::resize(..., INTER_CUBIC) as OpenCV's own code computes it (host_model.cpp: make_cubic_table / resize_cubic_u8):
// one thread per destination element, 16 taps; the vertical pass is host_model.h's cubic_vertical_u8, shared with the host.
__global__ void cubic_u8_kernel(const uint8_t *__restrict__ src, int sw, int cn, uint8_t *__restrict__ dst, int dh, int dw,
                                CubicTab xt, CubicTab yt)
{
    const int row = dw * cn, n_vec = row / 8 * 8;
    const size_t total = (size_t)dh * row;
    const float scale = 1.0f / (2048.0f * 2048.0f);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int e = (int)(i % row), y = (int)(i / row);
        const int x = e / cn, c = e % cn;
        int h[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint8_t *S = src + (size_t)yt.idx[y * 4 + r] * sw * cn + c;
            int v = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                v += (int)S[(size_t)xt.idx[x * 4 + k] * cn] * (int)xt.coef[x * 4 + k];
            h[r] = v;
        }
        const int16_t b[4] = {yt.coef[y * 4], yt.coef[y * 4 + 1], yt.coef[y * 4 + 2], yt.coef[y * 4 + 3]};
        dst[i] = cubic_vertical_u8(h[0], h[1], h[2], h[3], b, scale, e < n_vec);
    }
}

cudaError_t launch_cubic_u8(const uint8_t *src, int sh, int sw, int cn, uint8_t *dst, int dh, int dw, CubicTab xt, CubicTab yt,
                            cudaStream_t stream)
{
    (void)sh;
    const size_t total = (size_t)dh * dw * cn;
    if (total == 0)
        return cudaSuccess;
    cubic_u8_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, sw, cn, dst, dh, dw, xt, yt);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ packing

__device__ __forceinline__ float chroma_of(float a, float b)
{
    // ColourDifference.cpp:48-49 evaluates sqrt(a*a + b*b) in f64 on the f32 pixel values
    return (float)sqrt((double)a * (double)a + (double)b * (double)b);
}

// CIEDE2000 channels as colour_math.cuh wants them: (L/2 - 25, a/50, b/50, C/50)
__device__ __forceinline__ float4 half_scale_lab(float L, float a, float b)
{
    return make_float4(fmaf(0.5f, L, -25.0f), MM_CIEDE_AB_SCALE * a, MM_CIEDE_AB_SCALE * b, MM_CIEDE_AB_SCALE * chroma_of(a, b));
}

// Euclidean layout (diff_euclid.cu): pixel-major, NEGATED: [lib_tile][chunk][pixel][x0,x1,x2][64 images]; one thread per
// (image, active pixel), padding comes from the memset in launch_pack_library
__global__ void pack_library_euclid_kernel(const float *__restrict__ lib, unsigned char *__restrict__ packed, int64_t n, int P,
                                           const int *__restrict__ pix_list, int n_active, int n_chunks)
{
    const size_t total = (size_t)n * n_active;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int q = (int)(i % n_active);
        const size_t im = i / n_active;
        const float *s = lib + (im * P + pix_list[q]) * 3;
        const size_t tile = im / MM_ETN, ti = im % MM_ETN;
        const int chunk = q / MM_EKP, pi = q % MM_EKP;
        float *f = reinterpret_cast<float *>(packed + (tile * n_chunks + chunk) * (size_t)(MM_EKP * 3 * MM_ETN * 4));
        f[(pi * 3 + 0) * MM_ETN + ti] = -s[0];
        f[(pi * 3 + 1) * MM_ETN + ti] = -s[1];
        f[(pi * 3 + 2) * MM_ETN + ti] = -s[2];
    }
}

// Euclidean layout straight from the 8U BGR library at the detail size: one CTA per (library tile, chunk) block of
// 16 pixels x 64 images. Loads run along the pixels of one image (pix_list is raster order, so 16 slots are mostly 48 contiguous
// bytes), the conversion (plain cast for RGB, OpenCV's Lab LUT for CIE76 -- lab_from_bgr8, same arithmetic as
// to_working_space_kernel) is fused in, the block is transposed through shared memory and leaves as one coalesced 12 KB write with
// its padding slots zeroed: the f32 working-space copy of the library (0.98 GB written and read again at config 5) and the memset
// of the packed tensor are gone. Used when there is a single size step (with size steps the f32 copy feeds the per-step halving).
constexpr int kEuclidRow = 3 * MM_ETN + 1;  // padded pixel stride of the staging tile (bank spread of the transposing writes)
template <bool kLab>
__global__ void __launch_bounds__(256)
pack_library_euclid_u8_kernel(const uint8_t *__restrict__ lib, int S, int k, unsigned char *__restrict__ packed, int64_t n, int P,
                              const int *__restrict__ pix_list, int n_active, int n_chunks, size_t n_blocks,
                              const short4 *__restrict__ lut)
{
    __shared__ float s[MM_EKP * kEuclidRow];
    for (size_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const size_t tile = blk / n_chunks;
        const int chunk = (int)(blk - tile * n_chunks);
        for (int item = threadIdx.x; item < MM_EKP * MM_ETN; item += 256) {
            const int pi = item % MM_EKP, ti = item / MM_EKP;
            const int q = chunk * MM_EKP + pi;
            const int64_t im = (int64_t)tile * MM_ETN + ti;
            float v0 = 0.0f, v1 = 0.0f, v2 = 0.0f;
            if (q < n_active && im < n) {
                const int ds = S / k, p = pix_list[q];
                int c8[3];
                area_pixel_u8(lib + (size_t)im * S * S * 3, S, k, p / ds, p % ds, c8);
                if (kLab) {
                    lab_from_bgr8((unsigned char)c8[0], (unsigned char)c8[1], (unsigned char)c8[2], lut, v0, v1, v2);
                } else {
                    v0 = (float)c8[0];
                    v1 = (float)c8[1];
                    v2 = (float)c8[2];
                }
            }
            float *d = s + pi * kEuclidRow + ti;  // library values are stored NEGATED (cell - lib becomes a packed add)
            d[0] = -v0;
            d[MM_ETN] = -v1;
            d[2 * MM_ETN] = -v2;
        }
        __syncthreads();
        float *out = reinterpret_cast<float *>(packed + blk * (size_t)(MM_EKP * 3 * MM_ETN * 4));
        for (int j = threadIdx.x; j < MM_EKP * 3 * MM_ETN; j += 256)
            out[j] = s[(j / (3 * MM_ETN)) * kEuclidRow + j % (3 * MM_ETN)];
        __syncthreads();
    }
}

cudaError_t launch_pack_library_euclid_u8(const uint8_t *lib, int src_size, int k, bool is_lab, void *packed, int64_t n, int P,
                                          const int *pix_list, int n_active, int n_chunks, int n_lib_tiles, const short4 *lab_lut,
                                          cudaStream_t stream)
{
    if (k < 1 || src_size % k != 0 || (src_size / k) * (src_size / k) != P)
        return cudaErrorInvalidValue;
    const size_t n_blocks = (size_t)n_lib_tiles * n_chunks;
    if (n_blocks == 0)
        return cudaSuccess;
    const int grid = (int)(n_blocks < 148 * 16 ? n_blocks : 148 * 16);
    if (is_lab)
        pack_library_euclid_u8_kernel<true><<<grid, 256, 0, stream>>>(lib, src_size, k, (unsigned char *)packed, n, P, pix_list, n_active,
                                                                      n_chunks, n_blocks, lab_lut);
    else
        pack_library_euclid_u8_kernel<false><<<grid, 256, 0, stream>>>(lib, src_size, k, (unsigned char *)packed, n, P, pix_list, n_active,
                                                                       n_chunks, n_blocks, lab_lut);
    return cudaGetLastError();
}

// CIEDE2000 layout, one thread per (image PAIR slot, pixel slot) of the padded tile grid: two complete float4 stores per
// thread (consecutive threads = consecutive pixels -> fully coalesced), padding slots written as zeros by the same pass
// (no separate memset of the 2.6 GB tensor). kFromU8: the source is the 8U BGR library at the detail size and the Lab
// conversion (lab_from_bgr8, same arithmetic as to_working_space_kernel) is fused in -- the f32 working-space copy of the
// library (1.97 GB written and read again at config 4) is never materialised. Used when there is a single size step;
// with size steps the f32 copy is needed for the per-step halving (CPUPhotomosaicGenerator.cpp:95-99).
template <bool kFromU8>
__global__ void pack_library_ciede_kernel(const void *__restrict__ src, int S, int k, unsigned char *__restrict__ packed, int64_t n, int P,
                                          const int *__restrict__ pix_list, int n_active, int n_chunks, int64_t n_pair_slots,
                                          const short4 *__restrict__ lut, const int *__restrict__ perm)
{
    const int slots_per_image = n_chunks * MM_KP;
    const size_t total = (size_t)n_pair_slots * slots_per_image;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int q = (int)(i % slots_per_image);
        const int64_t pr = (int64_t)(i / slots_per_image);
        float4 v[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
        if (q < n_active) {
            const int px = pix_list[q];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int64_t slot = pr * 2 + j;
                if (slot >= n)
                    continue;
                const int64_t im = perm ? perm[slot] : slot;
                float L, a, b;
                if (kFromU8) {
                    // S x S source, reduced k-fold on the fly (8U INTER_AREA as area_u8_kernel computes it; k == 1: a plain read)
                    const int ds = S / k;
                    int c8[3];
                    area_pixel_u8(reinterpret_cast<const uint8_t *>(src) + (size_t)im * S * S * 3, S, k, px / ds, px % ds, c8);
                    lab_from_bgr8((unsigned char)c8[0], (unsigned char)c8[1], (unsigned char)c8[2], lut, L, a, b);
                } else {
                    const float *sf = reinterpret_cast<const float *>(src) + ((size_t)im * P + px) * 3;
                    L = sf[0];
                    a = sf[1];
                    b = sf[2];
                }
                v[j] = half_scale_lab(L, a, b);
            }
        }
        const int64_t tile = pr / (MM_TNB / 2);
        const int tp = (int)(pr % (MM_TNB / 2)), chunk = q / MM_KP, pi = q % MM_KP;
        float4 *blk = reinterpret_cast<float4 *>(packed + ((size_t)tile * n_chunks + chunk) * (size_t)(MM_TNB * MM_KP * 16));
        // [pair][0][p] = (L0, L1, a0, a1), [pair][1][p] = (b0, b1, C0, C1)
        blk[(tp * 2 + 0) * MM_KP + pi] = make_float4(v[0].x, v[1].x, v[0].y, v[1].y);
        blk[(tp * 2 + 1) * MM_KP + pi] = make_float4(v[0].z, v[1].z, v[0].w, v[1].w);
    }
}

cudaError_t launch_pack_library_ciede(const void *src, bool src_is_u8, void *packed, int64_t n, int P, const int *pix_list,
                                      int n_active, int n_chunks, int n_lib_tiles, const short4 *lab_lut, cudaStream_t stream,
                                      int src_size, int k, const int *perm)
{
    if (src_is_u8 && src_size == 0) {  // source already at the detail size
        src_size = 1;
        while (src_size * src_size < P)
            ++src_size;
        k = 1;
    }
    if (src_is_u8 && (k < 1 || src_size % k != 0 || (src_size / k) * (src_size / k) != P))
        return cudaErrorInvalidValue;
    const int64_t n_pair_slots = (int64_t)n_lib_tiles * (MM_TNB / 2);
    const size_t total = (size_t)n_pair_slots * n_chunks * MM_KP;
    if (total == 0)
        return cudaSuccess;
    if (src_is_u8)
        pack_library_ciede_kernel<true><<<grid_for(total, 256), 256, 0, stream>>>(src, src_size, k, (unsigned char *)packed, n, P, pix_list,
                                                                                  n_active, n_chunks, n_pair_slots, lab_lut, perm);
    else
        pack_library_ciede_kernel<false><<<grid_for(total, 256), 256, 0, stream>>>(src, 0, 1, (unsigned char *)packed, n, P, pix_list,
                                                                                   n_active, n_chunks, n_pair_slots, lab_lut, perm);
    return cudaGetLastError();
}

// Block statistics for the pruning bound (kernels.h: launch_block_stats), read from the packed tiles so that they follow the tiles'
// compacted pixel order and slot order. One thread per (library pair slot, block) -- both images of the pair share the float4 that
// holds their L -- then one per (cell row, block). Sums run in FP32, in pixel order; launch_prune_bound allows for their rounding.
__global__ void block_stats_kernel(const unsigned char *__restrict__ lib, int64_t n_pair_slots, const unsigned char *__restrict__ cells,
                                   int n_rows, int n_chunks, float4 *__restrict__ lib_stats, float4 *__restrict__ cell_stats)
{
    constexpr int kBlocksPerChunk = MM_KP / MM_BB;
    const int n_blocks = n_chunks * kBlocksPerChunk;
    const size_t n_lib_items = (size_t)n_blocks * n_pair_slots;
    const size_t total = n_lib_items + (size_t)n_rows * n_blocks;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        if (i < n_lib_items) {
            const int b = (int)(i / n_pair_slots);
            const int64_t pr = (int64_t)(i % n_pair_slots);
            const int64_t tile = pr / (MM_TNB / 2);
            const int tp = (int)(pr % (MM_TNB / 2)), chunk = b / kBlocksPerChunk, p0 = (b % kBlocksPerChunk) * MM_BB;
            // [pair][0][p] = (L0, L1, a0, a1) (pack_library_ciede_kernel)
            const float4 *v = reinterpret_cast<const float4 *>(lib + ((size_t)tile * n_chunks + chunk) * (size_t)(MM_TNB * MM_KP * 16)) +
                              (tp * 2) * MM_KP + p0;
            float s0 = 0.0f, s1 = 0.0f, lo0 = INFINITY, lo1 = INFINITY, hi0 = -INFINITY, hi1 = -INFINITY;
#pragma unroll
            for (int p = 0; p < MM_BB; ++p) {
                const float4 q = v[p];
                s0 += q.x;
                s1 += q.y;
                lo0 = fminf(lo0, q.x);
                hi0 = fmaxf(hi0, q.x);
                lo1 = fminf(lo1, q.y);
                hi1 = fmaxf(hi1, q.y);
            }
            float4 *out = lib_stats + (size_t)b * n_pair_slots * 2 + pr * 2;
            out[0] = make_float4(s0, lo0, hi0, 0.0f);
            out[1] = make_float4(s1, lo1, hi1, 0.0f);
        } else {
            const size_t j = i - n_lib_items;
            const int row = (int)(j / n_blocks), b = (int)(j % n_blocks);
            const int chunk = b / kBlocksPerChunk, p0 = (b % kBlocksPerChunk) * MM_BB;
            const unsigned char *blk = cells + ((size_t)(row / MM_TCB) * n_chunks + chunk) * (size_t)(MM_TCB * MM_KP * 20);
            const float4 *c = reinterpret_cast<const float4 *>(blk) + (row % MM_TCB) * MM_KP + p0;
            const float *w = reinterpret_cast<const float *>(blk + (size_t)MM_TCB * MM_KP * 16) + (row % MM_TCB) * MM_KP + p0;
            const float w0 = w[0];
            float s = 0.0f, lo = INFINITY, hi = -INFINITY;
            bool uniform = true;
#pragma unroll
            for (int p = 0; p < MM_BB; ++p) {
                const float x = c[p].x;
                s += x;
                lo = fminf(lo, x);
                hi = fmaxf(hi, x);
                uniform = uniform && w[p] == w0;
            }
            cell_stats[j] = make_float4(s, lo, hi, uniform ? w0 : 0.0f);
        }
    }
}

cudaError_t launch_block_stats(const void *lib_packed, int n_lib_tiles, const void *cells_packed, int n_rows, int n_chunks,
                               float4 *lib_stats, float4 *cell_stats, cudaStream_t stream)
{
    static_assert(MM_KP % MM_BB == 0, "a block lies inside one chunk");
    const size_t total = ((size_t)n_lib_tiles * (MM_TNB / 2) + (size_t)n_rows) * n_chunks * (MM_KP / MM_BB);
    if (total == 0)
        return cudaSuccess;
    block_stats_kernel<<<grid_for(total, 256), 256, 0, stream>>>((const unsigned char *)lib_packed, (int64_t)n_lib_tiles * (MM_TNB / 2),
                                                                 (const unsigned char *)cells_packed, n_rows, n_chunks, lib_stats, cell_stats);
    return cudaGetLastError();
}

// Colour order of the library (exact pruning groups similar images into one tile): key = Morton code of each image's mean colour,
// 10 bits per channel. The means are exact integer sums over the 8-bit pixels, so every rank and every run gets the same order;
// the 5-bit Morton order is a prefix of the 10-bit one, so the key keeps locality at every scale however narrow the colour range.
__global__ void __launch_bounds__(256) library_key_kernel(const uint8_t *__restrict__ lib, size_t image_bytes, unsigned *__restrict__ key,
                                                          int *__restrict__ idx)
{
    __shared__ unsigned long long part[3][8];
    const uint8_t *img = lib + (size_t)blockIdx.x * image_bytes;
    unsigned long long sum[3] = {0, 0, 0};
    for (size_t i = threadIdx.x; i < image_bytes; i += blockDim.x)
        sum[i % 3] += img[i];
    for (int c = 0; c < 3; ++c) {
        unsigned long long v = sum[c];
        for (int o = 16; o > 0; o >>= 1)
            v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0)
            part[c][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned code = 0;
        for (int c = 0; c < 3; ++c) {
            unsigned long long t = 0;
            for (int w = 0; w < 8; ++w)
                t += part[c][w];
            const unsigned q = (unsigned)min(1023ull, t * 1024 / (image_bytes / 3 * 256));  // mean / 256, 10 bits
            for (int b = 0; b < 10; ++b)
                code |= ((q >> b) & 1u) << (3 * b + c);
        }
        key[blockIdx.x] = code;
        idx[blockIdx.x] = blockIdx.x;
    }
}

__global__ void finish_order_kernel(int *__restrict__ perm, int *__restrict__ inv, int n, int n_pad)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += gridDim.x * blockDim.x) {
        if (i >= n)
            perm[i] = i;  // padding slots keep padding columns
        inv[perm[i]] = i;
    }
}

size_t library_order_scratch_bytes(int64_t n)
{
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const unsigned *)nullptr, (unsigned *)nullptr, (const int *)nullptr, (int *)nullptr,
                                    (int)n, 0, 30);
    return (size_t)n * 12 + 256 + temp;
}

cudaError_t launch_library_order(const uint8_t *lib, int S, int64_t n, int n_pad, int *perm, int *inv_perm, void *scratch,
                                 size_t scratch_bytes, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    unsigned *key_in = (unsigned *)scratch, *key_out = key_in + n;
    int *idx = (int *)(key_out + n);
    void *temp = (unsigned char *)scratch + (((size_t)n * 12 + 255) & ~(size_t)255);
    size_t temp_bytes = scratch_bytes - (((size_t)n * 12 + 255) & ~(size_t)255);
    library_key_kernel<<<(unsigned)n, 256, 0, stream>>>(lib, (size_t)S * S * 3, key_in, idx);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_in, key_out, idx, perm, (int)n, 0, 30, stream);  // stable
    if (e != cudaSuccess)
        return e;
    finish_order_kernel<<<(unsigned)std::min<int64_t>((n_pad + 255) / 256, 1024), 256, 0, stream>>>(perm, inv_perm, (int)n, n_pad);
    return cudaGetLastError();
}

cudaError_t launch_pack_library(const float *lib, void *packed, int64_t n, int P, const int *pix_list, int n_active,
                                int n_chunks, int n_lib_tiles, PackLayout layout, cudaStream_t stream, const int *perm)
{
    if (layout == kLayoutCiede)
        return launch_pack_library_ciede(lib, false, packed, n, P, pix_list, n_active, n_chunks, n_lib_tiles, nullptr, stream, 0, 1, perm);
    cudaError_t e = cudaMemsetAsync(packed, 0, (size_t)n_lib_tiles * n_chunks * tile_geom(layout).lib_block, stream);
    if (e != cudaSuccess)
        return e;
    const size_t total = (size_t)n * n_active;
    if (total == 0)
        return cudaSuccess;
    pack_library_euclid_kernel<<<grid_for(total, 256), 256, 0, stream>>>(lib, (unsigned char *)packed, n, P, pix_list, n_active, n_chunks);
    return cudaGetLastError();
}

__global__ void extract_cells_kernel(const float *__restrict__ mains, int H, int W, const CellDesc *__restrict__ cells,
                                     int n_cells, int S, int ds, int k, AreaTab tab, const uint8_t *__restrict__ masks4,
                                     const int *__restrict__ pix_list, int n_active, int n_chunks,
                                     unsigned char *__restrict__ packed, int layout)
{
    const bool with_chroma = layout == kLayoutCiede;
    const size_t total = (size_t)n_cells * n_active;
    const size_t block_bytes = (size_t)MM_TCB * MM_KP * 20;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int q = (int)(i % n_active);
        const int c = (int)(i / n_active);
        const CellDesc cd = cells[c];
        const int p = pix_list[q];
        const int py = p / ds, px = p - py * ds;
        const float *img = mains + (size_t)cd.variant * H * W * 3;
        float v[3];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            auto tap = [&](int tp) -> float {
                // zero-filled cell buffer (PhotomosaicGeneratorBase.cpp:310-312): pixels outside the image are 0
                const int y = cd.y0 + py * k + tp / k, x = cd.x0 + px * k + tp % k;
                return (y >= 0 && y < H && x >= 0 && x < W) ? img[((size_t)y * W + x) * 3 + ch] : 0.0f;
            };
            auto tap2 = [&](int sy, int sx) -> float {
                const int y = cd.y0 + sy, x = cd.x0 + sx;
                return (y >= 0 && y < H && x >= 0 && x < W) ? img[((size_t)y * W + x) * 3 + ch] : 0.0f;
            };
            v[ch] = (k == 1) ? tap(0) : (k > 1 ? area_block_f32(k, tap) : area_general(tab, py, px, tap2));
        }
        const bool in_bound = px >= cd.bx && px < cd.bx + cd.bw && py >= cd.by && py < cd.by + cd.bh;
        const bool active = masks4[((size_t)cd.flip * ds + py) * ds + px] != 0;
        if (layout == kLayoutEuclid) {
            // pixel-major: [cell_tile][chunk][pixel][x0,x1,x2,w][64 cells] (diff_euclid.cu)
            const size_t tile = c / MM_ETC, ti = c % MM_ETC;
            const int chunk = q / MM_EKP, pi = q % MM_EKP;
            float *f = reinterpret_cast<float *>(packed + (tile * n_chunks + chunk) * (size_t)(MM_EKP * 4 * MM_ETC * 4));
            f[(pi * 4 + 0) * MM_ETC + ti] = v[0];
            f[(pi * 4 + 1) * MM_ETC + ti] = v[1];
            f[(pi * 4 + 2) * MM_ETC + ti] = v[2];
            f[(pi * 4 + 3) * MM_ETC + ti] = (in_bound && active) ? 1.0f : 0.0f;
            continue;
        }
        const size_t tile = c / MM_TCB, ti = c % MM_TCB;
        const int chunk = q / MM_KP, pi = q % MM_KP;
        unsigned char *blk = packed + (tile * n_chunks + chunk) * block_bytes;
        reinterpret_cast<float4 *>(blk)[ti * MM_KP + pi] =
            with_chroma ? half_scale_lab(v[0], v[1], v[2]) : make_float4(v[0], v[1], v[2], 0.0f);
        // the CIEDE2000 kernel returns dE/50 (stored-scale channels): the factor lives in the weight
        reinterpret_cast<float *>(blk + (size_t)MM_TCB * MM_KP * 16)[ti * MM_KP + pi] =
            (in_bound && active) ? (with_chroma ? MM_CIEDE_WEIGHT : 1.0f) : 0.0f;
    }
}

cudaError_t launch_extract_cells(const float *mains, int H, int W, const CellDesc *cells, int n_cells, int S, int ds, int k,
                                 AreaTab tab, const uint8_t *masks4, const int *pix_list, int n_active, int n_chunks,
                                 void *packed, PackLayout layout, cudaStream_t stream)
{
    const TileGeom tg = tile_geom(layout);
    const int n_tiles = (n_cells + tg.tcb - 1) / tg.tcb;
    cudaError_t e = cudaMemsetAsync(packed, 0, (size_t)n_tiles * n_chunks * tg.cell_block, stream);
    if (e != cudaSuccess)
        return e;
    const size_t total = (size_t)n_cells * n_active;
    if (total == 0)
        return cudaSuccess;
    extract_cells_kernel<<<grid_for(total, 256), 256, 0, stream>>>(mains, H, W, cells, n_cells, S, ds, k, tab, masks4, pix_list,
                                                                   n_active, n_chunks, (unsigned char *)packed, (int)layout);
    return cudaGetLastError();
}

}  // namespace mm
