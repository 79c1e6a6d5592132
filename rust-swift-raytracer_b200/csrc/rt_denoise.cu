// rt_denoise.cu — the denoiser: edge-avoiding a-trous wavelet filter (Dammertz et al., HPG 2010) of a frame's colour
// sums, guided by the first-hit buffers.  MUST be compiled with --fmad=false (and the nvcc defaults -prec-div=true
// -prec-sqrt=true -ftz=false): the per-pixel functions of rt_denoise.cuh then run as correctly rounded IEEE binary32
// operations in the order written, and the result equals the CPU reference bit for bit.
//
//   pack:          one pass over the inputs: e = (sum / spp) / max(albedo, 2^-10), guides packed to 32 B per pixel
//   iteration i:   5x5 taps at step 2^i, ping-pong between two scratch frames
//   last iteration: the filter, remodulation by a', the float4 colour and the RGBA8 pack fused into one kernel
#define RT_TU_EXACT 1
#include "rt_denoise.cuh"
#include "rt_launch.h"

#include <cuda_runtime.h>

#include <algorithm>

namespace rt {

constexpr int kPackBlock = 256;
constexpr int kTileX = 32, kTileY = 8;   // one warp per 32-pixel row segment: the taps of a row are coalesced

__global__ void __launch_bounds__(kPackBlock) rt_denoise_pack_kernel(const __grid_constant__ RtDenoiseParams P)
{
    const size_t n = (size_t)P.width * P.height;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const RtFloat4 sum = dn_load(P.accum + i);
        const float*   a   = P.albedo + 3 * i;
        const float*   nn  = P.normal + 3 * i;
        const float*   x   = P.position + 3 * i;
        RtFloat4 e, gn, gx;
        dn_pack_pixel(sum, P.k, a[0], a[1], a[2], nn[0], nn[1], nn[2], x[0], x[1], x[2], P.prim[i], e, gn, gx);
        P.e[0][i] = e;
        P.gn[i]   = gn;
        P.gx[i]   = gx;
    }
}

// Iteration `it` reads P.e[it & 1] and writes P.e[(it + 1) & 1]; the LAST one writes the outputs instead.  A CTA
// filters 32x8-pixel tiles, grid-stride over the row-major tile order.
template <bool LAST>
__global__ void __launch_bounds__(kTileX * kTileY) rt_denoise_iter_kernel(const __grid_constant__ RtDenoiseParams P,
                                                                          uint32_t it)
{
    const uint32_t tiles_x = (P.width + kTileX - 1) / kTileX;
    const uint64_t n_tiles = (uint64_t)tiles_x * ((P.height + kTileY - 1) / kTileY);
    const uint32_t s       = 1u << it;
    const float    sc_i    = P.sc * (float)(1u << (2u * it));          // sc * 4^i, exact
    const RtFloat4* ein    = P.e[it & 1u];
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t x = (uint32_t)(t % tiles_x) * kTileX + threadIdx.x;
        const uint32_t y = (uint32_t)(t / tiles_x) * kTileY + threadIdx.y;
        if (x >= P.width || y >= P.height) continue;
        const size_t p    = (size_t)y * P.width + x;
        const bool   miss = P.gn[p].w != 0.0f;
        RtFloat4     f;
        f.x = f.y = f.z = f.w = 0.0f;
        if (!miss) f = dn_filter_pixel(ein, P.gn, P.gx, P.width, P.height, x, y, s, sc_i, P.sn, P.sx);
        if (!LAST) {
            if (!miss) P.e[(it + 1u) & 1u][p] = f;
            continue;
        }
        const float*   a = P.albedo + 3 * p;
        const RtFloat4 c = dn_finish_pixel(dn_load(P.accum + p), P.k, a[0], a[1], a[2], miss, f);
        if (P.color) P.color[p] = c;
        if (P.pixels) P.pixels[p] = dn_rgba8(c);
    }
}

// The whole filter on `stream`: 1 + iterations launches.  *grid / *block: the geometry of the iteration kernels.
cudaError_t launch_denoise(const RtDenoiseParams& P, int num_sms, uint32_t* grid, uint32_t* block, cudaStream_t stream)
{
    const size_t n        = (size_t)P.width * P.height;
    const size_t pack_cap = (size_t)num_sms * 8;
    const int    pack     = (int)std::min<size_t>((n + kPackBlock - 1) / kPackBlock, pack_cap);
    rt_denoise_pack_kernel<<<pack, kPackBlock, 0, stream>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const dim3 blk(kTileX, kTileY);
    const uint64_t n_tiles = (uint64_t)((P.width + kTileX - 1) / kTileX) * ((P.height + kTileY - 1) / kTileY);
    const dim3     grd((unsigned)std::min<uint64_t>(n_tiles, 0x7fffffffu));
    for (uint32_t it = 0; it < P.iterations; ++it) {
        if (it + 1 == P.iterations) rt_denoise_iter_kernel<true><<<grd, blk, 0, stream>>>(P, it);
        else                        rt_denoise_iter_kernel<false><<<grd, blk, 0, stream>>>(P, it);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    *grid  = grd.x;
    *block = blk.x * blk.y;
    return cudaSuccess;
}

}   // namespace rt
