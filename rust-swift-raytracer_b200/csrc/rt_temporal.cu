// rt_temporal.cu — temporal accumulation: a frame's colour sums blended with the previous frame's colour history,
// reprojected through the first-hit buffers.  MUST be compiled with --fmad=false (and the nvcc defaults
// -prec-div=true -prec-sqrt=true -ftz=false): the per-pixel functions of rt_temporal.cuh then run as correctly rounded
// IEEE binary32 operations in the order written, and the result equals the CPU reference bit for bit.
//
// One launch, one thread per pixel: the pixel's sums and guides are read once, its four bilinear taps of the previous
// frame through the read-only path, and the colour, the length and optionally the RGBA8 pixel are written once.
#define RT_TU_EXACT 1
#include "rt_temporal.cuh"
#include "rt_launch.h"

#include <cuda_runtime.h>

#include <algorithm>

namespace rt {

constexpr int kTileX = 32, kTileY = 8;   // one warp per 32-pixel row segment: the current frame's reads are coalesced

// A CTA handles 32x8-pixel tiles, grid-stride over the row-major tile order.
__global__ void __launch_bounds__(kTileX * kTileY) rt_temporal_kernel(const __grid_constant__ RtTemporalParams P)
{
    const uint32_t tiles_x = (P.width + kTileX - 1) / kTileX;
    const uint64_t n_tiles = (uint64_t)tiles_x * ((P.height + kTileY - 1) / kTileY);
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t x = (uint32_t)(t % tiles_x) * kTileX + threadIdx.x;
        const uint32_t y = (uint32_t)(t / tiles_x) * kTileY + threadIdx.y;
        if (x >= P.width || y >= P.height) continue;
        const size_t p = (size_t)y * P.width + x;
        RtFloat4     c;
        float        len;
        tp_pixel(P, x, y, c, len);
        P.color[p]  = c;
        P.length[p] = len;
        if (P.pixels) P.pixels[p] = tp_rgba8(c);
    }
}

cudaError_t launch_temporal(RtTemporalParams P, const float* prev_camera12, uint32_t* grid, uint32_t* block,
                            cudaStream_t stream)
{
    if (P.mode == RT_TEMPORAL_REPROJECT) tp_setup_projection(P, prev_camera12);   // host float32, no FMA
    const dim3     blk(kTileX, kTileY);
    const uint64_t n_tiles = (uint64_t)((P.width + kTileX - 1) / kTileX) * ((P.height + kTileY - 1) / kTileY);
    const dim3     grd((unsigned)std::min<uint64_t>(n_tiles, 0x7fffffffu));
    rt_temporal_kernel<<<grd, blk, 0, stream>>>(P);
    *grid  = grd.x;
    *block = blk.x * blk.y;
    return cudaGetLastError();
}

}   // namespace rt
