// rt_kernels_fast.cu — the relaxed-arithmetic render kernel (FMA contraction, approximate
// rcp/rsqrt/sqrt).  Same algorithm and RNG streams as the exact kernel; agrees with it
// statistically (RMSE), not bit for bit.  Opt-in through RtRenderOptions / Options::fast_math.
#define RT_TU_FAST 1
#include "rt_kernels.cuh"

namespace rt {

template cudaError_t kernel_geometry<Kernel::render_fast>(const RtSceneView&, size_t, bool, KernelGeometry*);
template cudaError_t launch_kernel<Kernel::render_fast>(const RtFrameParams&, const RtSceneView&, bool, int, size_t, cudaStream_t);

template cudaError_t launch_resolve_samples<true>(const RtFrameParams&, cudaStream_t);

// ---- FP32 peak microbenchmark: 16 independent FFMA chains per thread -------------------
// The roofline denominator for the render kernel (MEASURED_PEAKS.json has no FP32 figure).
#define RT_PEAK_CHAINS 16
#define RT_PEAK_UNROLL 8
__global__ void __launch_bounds__(256) rt_ffma_peak_kernel(float* out, int iters, float b, float c)
{
    float a[RT_PEAK_CHAINS];
#pragma unroll
    for (int k = 0; k < RT_PEAK_CHAINS; ++k) a[k] = (float)(threadIdx.x + k) * 1e-3f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < RT_PEAK_UNROLL; ++u)
#pragma unroll
            for (int k = 0; k < RT_PEAK_CHAINS; ++k) a[k] = fmaf(a[k], b, c);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < RT_PEAK_CHAINS; ++k) s += a[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

cudaError_t launch_ffma_peak(float* out, int iters, int grid, int block, cudaStream_t stream)
{
    rt_ffma_peak_kernel<<<grid, block, 0, stream>>>(out, iters, 0.999f, 1e-4f);
    return cudaGetLastError();
}

double ffma_peak_flops_per_launch(int iters, int grid, int block)
{
    return 2.0 * RT_PEAK_CHAINS * RT_PEAK_UNROLL * (double)iters * (double)grid * (double)block;
}

}   // namespace rt
