// rt_svgf.cu — variance-guided filtering (SVGF, Schied et al., HPG 2017): temporal accumulation of the demodulated
// colour and its luminance moments, a per-pixel variance estimate, and the a-trous filter steered by that variance.
// MUST be compiled with --fmad=false (and the nvcc defaults -prec-div=true -prec-sqrt=true -ftz=false): the per-pixel
// functions of rt_svgf.cuh then run as correctly rounded IEEE binary32 operations in the order written, and the result
// equals the CPU reference bit for bit.
//
//   temporal:        the history lookup of §15 for colour, moments and length; writes moments and length out, the
//                    blended colour and the packed guides to scratch
//   variance:        per hit pixel, temporal or (for a young history) 7x7 spatial estimate
//   iteration i:     5x5 taps at step 2^i, colour and variance ping-pong between two scratch frames each; the first
//                    writes the next frame's colour history (illum), the last remodulates and writes the outputs
#define RT_TU_EXACT 1
#include "rt_svgf.cuh"
#include "rt_launch.h"

#include <cuda_runtime.h>

#include <algorithm>

namespace rt {

constexpr int kTileX = 32, kTileY = 8;   // one warp per 32-pixel row segment: the taps of a row are coalesced

// A CTA handles 32x8-pixel tiles, grid-stride over the row-major tile order, in each of the three kernels.
__global__ void __launch_bounds__(kTileX * kTileY) rt_svgf_temporal_kernel(const __grid_constant__ RtSvgfParams P)
{
    const uint32_t tiles_x = (P.t.width + kTileX - 1) / kTileX;
    const uint64_t n_tiles = (uint64_t)tiles_x * ((P.t.height + kTileY - 1) / kTileY);
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t x = (uint32_t)(t % tiles_x) * kTileX + threadIdx.x;
        const uint32_t y = (uint32_t)(t / tiles_x) * kTileY + threadIdx.y;
        if (x >= P.t.width || y >= P.t.height) continue;
        const size_t p = (size_t)y * P.t.width + x;
        RtFloat4 illum, gn, gx;
        RtFloat2 m;
        float    len;
        sv_temporal_pixel(P, x, y, illum, m, len, gn, gx);
        P.e[0][p]     = illum;
        P.gn[p]       = gn;
        P.gx[p]       = gx;
        P.moments[p]  = m;
        P.length[p]   = len;
    }
}

__global__ void __launch_bounds__(kTileX * kTileY) rt_svgf_variance_kernel(const __grid_constant__ RtSvgfParams P)
{
    const uint32_t tiles_x = (P.t.width + kTileX - 1) / kTileX;
    const uint64_t n_tiles = (uint64_t)tiles_x * ((P.t.height + kTileY - 1) / kTileY);
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t x = (uint32_t)(t % tiles_x) * kTileX + threadIdx.x;
        const uint32_t y = (uint32_t)(t / tiles_x) * kTileY + threadIdx.y;
        if (x >= P.t.width || y >= P.t.height) continue;
        const size_t p = (size_t)y * P.t.width + x;
        if (P.gn[p].w != 0.0f) continue;                                       // misses have no variance
        P.var[0][p] = sv_variance_pixel(P, P.moments, P.length, x, y);
    }
}

// Iteration `it` reads e[it & 1], var[it & 1] and writes e[(it + 1) & 1], var[(it + 1) & 1]; the FIRST one also writes
// illum, the LAST one the outputs instead of scratch.
template <bool FIRST, bool LAST>
__global__ void __launch_bounds__(kTileX * kTileY) rt_svgf_iter_kernel(const __grid_constant__ RtSvgfParams P,
                                                                       uint32_t it)
{
    const uint32_t  s   = 1u << it;
    const RtFloat4* ein = P.e[it & 1u];
    const float*    vin = P.var[it & 1u];
    const uint32_t tiles_x = (P.t.width + kTileX - 1) / kTileX;
    const uint64_t n_tiles = (uint64_t)tiles_x * ((P.t.height + kTileY - 1) / kTileY);
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t x = (uint32_t)(t % tiles_x) * kTileX + threadIdx.x;
        const uint32_t y = (uint32_t)(t / tiles_x) * kTileY + threadIdx.y;
        if (x >= P.t.width || y >= P.t.height) continue;
        const size_t p    = (size_t)y * P.t.width + x;
        const bool   miss = P.gn[p].w != 0.0f;
        RtFloat4     f;
        float        var = 0.0f;
        f.x = f.y = f.z = f.w = 0.0f;
        if (!miss) f = sv_filter_pixel(P, ein, vin, x, y, s, var);
        if (FIRST) P.illum[p] = miss ? dn_load(ein + p) : f;                  // a miss: stage 1 stored m
        if (!LAST) {
            if (!miss) {
                P.e[(it + 1u) & 1u][p]   = f;
                P.var[(it + 1u) & 1u][p] = var;
            }
            continue;
        }
        const float*   a = P.albedo + 3 * p;
        const RtFloat4 c = dn_finish_pixel(dn_load(P.t.accum + p), P.t.k, a[0], a[1], a[2], miss, f);
        if (P.color) P.color[p] = c;
        if (P.pixels) P.pixels[p] = dn_rgba8(c);
    }
}

template <bool FIRST, bool LAST>
static cudaError_t launch_iter(const RtSvgfParams& P, uint32_t it, dim3 grd, dim3 blk, cudaStream_t stream)
{
    rt_svgf_iter_kernel<FIRST, LAST><<<grd, blk, 0, stream>>>(P, it);
    return cudaGetLastError();
}

cudaError_t launch_svgf(RtSvgfParams P, const float* prev_camera12, uint32_t* grid, uint32_t* block,
                        cudaStream_t stream)
{
    if (P.t.mode == RT_TEMPORAL_REPROJECT) tp_setup_projection(P.t, prev_camera12);   // host float32, no FMA
    const dim3     blk(kTileX, kTileY);
    const uint64_t n_tiles = (uint64_t)((P.t.width + kTileX - 1) / kTileX) * ((P.t.height + kTileY - 1) / kTileY);
    const dim3     grd((unsigned)std::min<uint64_t>(n_tiles, 0x7fffffffu));
    rt_svgf_temporal_kernel<<<grd, blk, 0, stream>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    rt_svgf_variance_kernel<<<grd, blk, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    for (uint32_t it = 0; it < P.iterations; ++it) {
        const bool first = it == 0, last = it + 1 == P.iterations;
        e = first ? (last ? launch_iter<true, true>(P, it, grd, blk, stream) : launch_iter<true, false>(P, it, grd, blk, stream))
                  : (last ? launch_iter<false, true>(P, it, grd, blk, stream) : launch_iter<false, false>(P, it, grd, blk, stream));
        if (e != cudaSuccess) return e;
    }
    *grid  = grd.x;
    *block = blk.x * blk.y;
    return cudaSuccess;
}

}   // namespace rt
