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
#include <cuda_runtime.h>
#include <stdint.h>

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

__global__ void build_gather_kernel(const unsigned long long *__restrict__ owner, int H, int W, int n_steps, const BuildStep *__restrict__ steps,
                                    uchar4 background, uchar4 *__restrict__ out, size_t out_stride_px)
{
    const size_t n = (size_t)H * W;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
        const unsigned long long key = owner[i];
        uchar4 px = background;
        if (key != 0ull) {
            const BuildStep st = steps[n_steps - (int)(key >> 40)];  // the high field stores n_steps - step (>= 1)
            const BuildCell c = st.cells[(key & 0xffffffffffull) - 1];
            // tile pixel (r, c) of the cell, read at the mirrored coordinates of the tile's orientation
            const int ty = (c.orient & 2) ? st.S - 1 - (y - c.y0) : y - c.y0;
            const int tx = (c.orient & 1) ? st.S - 1 - (x - c.x0) : x - c.x0;
            const uint8_t *src = st.lib + ((size_t)c.lib_index * st.S * st.S + (size_t)ty * st.S + tx) * 3;
            px = make_uchar4(src[0], src[1], src[2], 255);
        }
        out[(size_t)y * out_stride_px + x] = px;
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

cudaError_t launch_build_gather(const unsigned long long *owner, int H, int W, int n_steps, const BuildStep *steps, const uint8_t bgra[4],
                                uint8_t *out, size_t out_stride_px, cudaStream_t stream)
{
    const size_t n = (size_t)H * W;
    if (n == 0)
        return cudaSuccess;
    size_t g = (n + 255) / 256;
    if (g > 148 * 32)
        g = 148 * 32;
    build_gather_kernel<<<(unsigned)g, 256, 0, stream>>>(owner, H, W, n_steps, steps, make_uchar4(bgra[0], bgra[1], bgra[2], bgra[3]),
                                                         reinterpret_cast<uchar4 *>(out), out_stride_px);
    return cudaGetLastError();
}

}  // namespace mm
