// buildPhotomosaic on the GPU: composites the chosen library images into the final BGRA mosaic.
//
// Replaces PhotomosaicGeneratorBase::buildPhotomosaic (src/Photomosaic/PhotomosaicGeneratorBase.cpp:110-207):
// per size step every valid cell copies its library image through its (flipped) NORMAL-size mask into a step canvas
// in raster order (a later cell overwrites an earlier one where masks overlap), and later steps only fill pixels no
// earlier step covered. Both rules are order statistics, so the sequential blits become one scatter + one gather:
//   owner[pixel] = max over covering cells of ((n_steps - 1 - step) << 40 | raster index of the cell)   (atomicMax)
//   mosaic[pixel] = library pixel of owner[pixel]'s cell, or the background colour.
// The library stays resident from generate(); per step it is halved with OpenCV's 8U INTER_AREA like
// ImageUtility::batchResizeMat (ImageUtility.cpp:91-101) does on the BGRA copies (alpha stays 255).
// The scaled build (mosaic_build_photomosaic_scaled) is the same gather at k times the size from a render library of side k * S:
// the owner map stays at the main image's size, and output pixel (Y, X) takes the owner of base pixel (Y / k, X / k).
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "kernels.h"

namespace mm {

__global__ void build_scatter_kernel(const BuildCell *__restrict__ cells, int n_cells, int S, const uint8_t *__restrict__ masks4,
                                     int H, int W, unsigned long long step_key, unsigned long long *__restrict__ owner)
{
    // one CTA per cell, threads stride the cell's pixels
    const BuildCell c = cells[blockIdx.x];
    const uint8_t *mask = masks4 + (size_t)c.flip * S * S;
    for (int i = threadIdx.x; i < S * S; i += blockDim.x) {
        const int ly = i / S, lx = i - ly * S;
        const int y = c.y0 + ly, x = c.x0 + lx;
        if (y < 0 || y >= H || x < 0 || x >= W || mask[i] == 0)
            continue;
        atomicMax(owner + (size_t)y * W + x, step_key | (unsigned long long)c.raster);
    }
}

// Output pixel (Y, X) of the mosaic at k times the main image's size. Cell c covers it exactly when it covers base pixel
// (Y / k, X / k) in the k-scaled geometry (its rect scaled by k, its mask upsampled by nearest neighbour), so the owner map stays at
// the base size; the pixel is the cell's render tile (side k * S_s) at (Y - k * y0, X - k * x0), mirrored by the tile's orientation.
__device__ __forceinline__ unsigned gather_pixel(const unsigned long long *__restrict__ owner_row, int by, int ry, int X, int k, int n_steps,
                                                 const BuildStep *__restrict__ steps, unsigned background)
{
    const int bx = X / k;
    const unsigned long long key = owner_row[bx];
    if (key == 0ull)
        return background;
    const BuildStep st = steps[n_steps - (int)(key >> 40)];  // the high field stores n_steps - step (>= 1)
    const BuildCell c = st.cells[(key & 0xffffffffffull) - 1];
    // the base pixel lies inside the cell's rect, so by - y0 and bx - x0 are in [0, S_s) and the tile coordinates in [0, side)
    int ty = k * (by - c.y0) + ry, tx = k * (bx - c.x0) + (X - k * bx);
    if (c.orient & 2)
        ty = st.side - 1 - ty;
    if (c.orient & 1)
        tx = st.side - 1 - tx;
    const uint8_t *src = st.lib + ((size_t)c.lib_index * st.side * st.side + (size_t)ty * st.side + tx) * 3;
    return (unsigned)src[0] | (unsigned)src[1] << 8 | (unsigned)src[2] << 16 | 0xff000000u;
}

// rows [y_begin, y_end) of the (k * H) x cols BGRA mosaic into out (row y_begin first, out_stride bytes per row): every thread
// writes 4 consecutive pixels of a row, one 16-byte store where the address allows it. out and out_stride must be multiples of 4
// bytes. Column and row counters are unsigned: cols and y_end are at most INT_MAX, so X + 3 and Y + gridDim.y cannot wrap.
__global__ void build_gather_kernel(const unsigned long long *__restrict__ owner, int W, int k, int n_steps, const BuildStep *__restrict__ steps,
                                    unsigned background, int y_begin, int y_end, int cols, uint8_t *__restrict__ out, size_t out_stride)
{
    const unsigned X = (blockIdx.x * blockDim.x + threadIdx.x) * 4u, ucols = (unsigned)cols;
    if (X >= ucols)
        return;
    for (unsigned Y = (unsigned)y_begin + blockIdx.y; Y < (unsigned)y_end; Y += gridDim.y) {
        const int by = (int)Y / k, ry = (int)Y - by * k;
        const unsigned long long *orow = owner + (size_t)by * W;
        unsigned px[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            px[j] = X + j < ucols ? gather_pixel(orow, by, ry, (int)(X + j), k, n_steps, steps, background) : 0u;
        uint8_t *dst = out + (size_t)(Y - (unsigned)y_begin) * out_stride + (size_t)X * 4;
        if (X + 4 <= ucols && ((uintptr_t)dst & 15) == 0) {
            __stcs(reinterpret_cast<uint4 *>(dst), make_uint4(px[0], px[1], px[2], px[3]));  // written once, never read back here
        } else {
            for (unsigned j = 0; j < 4 && X + j < ucols; ++j)
                reinterpret_cast<unsigned *>(dst)[j] = px[j];
        }
    }
}

cudaError_t launch_build_scatter(const BuildCell *cells, int n_cells, int S, const uint8_t *masks4, int H, int W, int step, int n_steps,
                                 unsigned long long *owner, cudaStream_t stream)
{
    if (n_cells <= 0)
        return cudaSuccess;
    const unsigned long long step_key = (unsigned long long)(n_steps - step) << 40;
    build_scatter_kernel<<<n_cells, 256, 0, stream>>>(cells, n_cells, S, masks4, H, W, step_key, owner);
    return cudaGetLastError();
}

cudaError_t launch_build_gather(const unsigned long long *owner, int W, int k, int n_steps, const BuildStep *steps, const uint8_t bgra[4],
                                int y_begin, int y_end, int cols, uint8_t *out, size_t out_stride, cudaStream_t stream)
{
    if (y_end <= y_begin || cols <= 0)
        return cudaSuccess;
    const unsigned background = (unsigned)bgra[0] | (unsigned)bgra[1] << 8 | (unsigned)bgra[2] << 16 | (unsigned)bgra[3] << 24;
    const dim3 grid((unsigned)(((int64_t)cols + 1023) / 1024), (unsigned)std::min(y_end - y_begin, 65535));
    build_gather_kernel<<<grid, 256, 0, stream>>>(owner, W, k, n_steps, steps, background, y_begin, y_end, cols, out, out_stride);
    return cudaGetLastError();
}

}  // namespace mm
