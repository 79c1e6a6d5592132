// rt_launch.h — the entry points of the kernel units (rt_kernels_exact.cu, rt_kernels_fast.cu, rt_denoise.cu,
// rt_temporal.cu, rt_svgf.cu), declared
// once for the units that define them and for rt_device.cu, which calls them.
#pragma once
#include "rt_types.h"

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace rt {

// The persistent kernels that walk the scene's hot lists.  The render kernel of the exact policy and the three
// one-ray-per-lane kernels are defined in rt_kernels_exact.cu, the render kernel of the fast policy in
// rt_kernels_fast.cu.
enum class Kernel : int { render_exact, render_fast, first_hit, ray_query, occlusion };

// The instantiation a kernel runs for one scene shape and what the occupancy API allows of it.
struct KernelGeometry {
    int    per_sm         = 0;               // resident CTAs per SM
    int    block          = 0;               // threads per CTA
    size_t hot_bytes      = 0;               // bytes of the hot lists
    bool   resident       = false;           // the hot lists are staged in shared memory
    int    walk           = RT_SPH_DIRECT;   // RT_SPH_*
    int    paths_per_lane = 1;
};

// The geometry of kernel K for the scene, with at most smem_limit bytes of dynamic shared memory per CTA.
template <Kernel K>
cudaError_t kernel_geometry(const RtSceneView& G, size_t smem_limit, bool cull, KernelGeometry* out);

// Launches kernel K with `grid` CTAs; Params is RtFrameParams for the render kernels, RtAovParams, RtRayParams and
// RtOcclusionParams for the others.
template <Kernel K, class Params>
cudaError_t launch_kernel(const Params& p, const RtSceneView& G, bool cull, int grid, size_t smem_limit,
                          cudaStream_t stream);

// The ordered sum and resolve of the sample-item mode (rt_resolve_samples_kernel), in the render's policy.
template <bool FAST>
cudaError_t launch_resolve_samples(const RtFrameParams& P, cudaStream_t stream);
cudaError_t launch_gather_rows(const uint32_t* local, uint32_t* remote, size_t n_pixels, int grid, cudaStream_t);
cudaError_t launch_selftest_division(unsigned long long n_per_thread, uint32_t seed, int grid, int block,
                                     unsigned long long* d_mismatches, cudaStream_t);
cudaError_t launch_selftest_sqrt(int grid, int block, unsigned long long* d_mismatches, cudaStream_t);
cudaError_t launch_ffma_peak(float* out, int iters, int grid, int block, cudaStream_t);
double      ffma_peak_flops_per_launch(int iters, int grid, int block);
cudaError_t launch_denoise(const RtDenoiseParams&, int num_sms, uint32_t* grid, uint32_t* block, cudaStream_t);
// rt_temporal.cu: fills P's projection constants from prev_camera12 (12 floats) when P.mode is RT_TEMPORAL_REPROJECT,
// then launches the kernel.
cudaError_t launch_temporal(RtTemporalParams P, const float* prev_camera12, uint32_t* grid, uint32_t* block, cudaStream_t);
// rt_svgf.cu: fills P.t's projection constants as launch_temporal does, then launches the 2 + P.iterations kernels.
// *grid / *block: the geometry every one of them uses.
cudaError_t launch_svgf(RtSvgfParams P, const float* prev_camera12, uint32_t* grid, uint32_t* block, cudaStream_t);

}   // namespace rt
