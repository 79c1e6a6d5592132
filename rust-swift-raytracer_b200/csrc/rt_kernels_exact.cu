// rt_kernels_exact.cu — the bit-exact render kernel.  MUST be compiled with --fmad=false
// (and the nvcc defaults -prec-div=true -prec-sqrt=true -ftz=false): every multiply, add,
// divide and square root is then a correctly rounded IEEE binary32 operation in the
// reference's association order, so the frame equals the CPU arithmetic bit for bit.
#define RT_TU_EXACT 1
#include "rt_kernels.cuh"

namespace rt {

// The exact policy's render kernel and the one-ray-per-lane kernels (exact policy only): this is the one translation
// unit that instantiates them.
template cudaError_t kernel_geometry<Kernel::render_exact>(const RtSceneView&, size_t, bool, KernelGeometry*);
template cudaError_t kernel_geometry<Kernel::first_hit>(const RtSceneView&, size_t, bool, KernelGeometry*);
template cudaError_t kernel_geometry<Kernel::ray_query>(const RtSceneView&, size_t, bool, KernelGeometry*);
template cudaError_t kernel_geometry<Kernel::occlusion>(const RtSceneView&, size_t, bool, KernelGeometry*);
template cudaError_t launch_kernel<Kernel::render_exact>(const RtFrameParams&, const RtSceneView&, bool, int, size_t, cudaStream_t);
template cudaError_t launch_kernel<Kernel::first_hit>(const RtAovParams&, const RtSceneView&, bool, int, size_t, cudaStream_t);
template cudaError_t launch_kernel<Kernel::ray_query>(const RtRayParams&, const RtSceneView&, bool, int, size_t, cudaStream_t);
template cudaError_t launch_kernel<Kernel::occlusion>(const RtOcclusionParams&, const RtSceneView&, bool, int, size_t,
                                                      cudaStream_t);

template cudaError_t launch_resolve_samples<false>(const RtFrameParams&, cudaStream_t);

// ---- self-test of the shared-reciprocal divide (rt_trace.cuh, div3 / pixel_uv) -----------
// Compares the hand-expanded sequence with the compiler's own IEEE `/` on pseudo-random
// operands whose exponents sweep the whole guarded range and beyond (so the guard and the
// fallback are exercised too).  Counts operand triples whose bits differ (NaN == NaN).
__device__ __forceinline__ bool same_bits(float a, float b)
{
    return (__float_as_uint(a) == __float_as_uint(b)) || (a != a && b != b);
}

__global__ void rt_selftest_division_kernel(unsigned long long n_per_thread, uint32_t seed,
                                            unsigned long long* mismatches)
{
    uint32_t rng = sample_seed(seed, blockIdx.x * blockDim.x + threadIdx.x, 0x5eedu);
    unsigned long long bad = 0;
    for (unsigned long long i = 0; i < n_per_thread; ++i) {
        // random mantissas; exponents: mostly moderate, sometimes extreme / zero / denormal
        uint32_t m[4], mode = xorshift32(rng);
        for (int k = 0; k < 4; ++k) m[k] = xorshift32(rng);
        float v[4];
        for (int k = 0; k < 4; ++k) {
            uint32_t bits = m[k];
            uint32_t sel  = (mode >> (8 * k)) & 0xffu;
            if (sel < 200u)      bits = (bits & 0x807fffffu) | ((117u + (bits >> 23) % 21u) << 23);   // 2^-10 .. 2^10
            else if (sel < 240u) bits = (bits & 0x807fffffu) | ((47u + (bits >> 23) % 161u) << 23);   // 2^-80 .. 2^80
            else if (sel < 250u) bits = bits;                                                          // anything (NaN, inf, denormal)
            else                 bits = bits & 0x80000000u;                                            // +-0
            v[k] = __uint_as_float(bits);
        }
        V3    a = mk(v[0], v[1], v[2]);
        float b = fabsf(v[3]);
        V3 q = div3<false>(a, b, false);
        bad += !(same_bits(q.x, a.x / b) && same_bits(q.y, a.y / b) && same_bits(q.z, a.z / b));
        // the normalisation (one range check for the root and the divides) against sqrtf and `/`
        float len = sqrtf(a.x * a.x + a.y * a.y + a.z * a.z);
        V3 nq = normalize<false>(a), np = normalize<false, true>(a);
        bad += !(same_bits(nq.x, a.x / len) && same_bits(nq.y, a.y / len) && same_bits(nq.z, a.z / len));
        bad += !(same_bits(np.x, a.x / len) && same_bits(np.y, a.y / len) && same_bits(np.z, a.z / len));
        // pixel_uv: (column + xi) / (W - 1)
        RtFrameParams P{};
        P.wm1 = (float)((m[0] % 8191u) + ((mode & 1u) ? 0u : 1u));       // includes 0 (1-pixel frame)
        P.hm1 = (float)((m[1] % 4095u) + 1u);
        float au = (float)(m[2] % 8192u) + random_f32(rng), av = (float)(m[3] % 4096u) + random_f32(rng);
        float u, w;
        pixel_uv<false>(P, au, av, u, w);
        bad += !(same_bits(u, au / P.wm1) && same_bits(w, av / P.hm1));
    }
    if (bad) atomicAdd(mismatches, bad);
}

// Every float bit pattern from +0 to +inf and a few NaNs: where sqrt_in_range() holds, the bare sequence
// sqrt_ranged() must give the bits of the compiler's IEEE sqrtf; the predicate itself must be exactly
// 2^-100 <= x <= 2^100.  Counts the patterns that violate either.
__global__ void rt_selftest_sqrt_kernel(unsigned long long* mismatches)
{
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    for (unsigned long long b = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; b <= 0x7f800010ull; b += stride) {
        const float x = __uint_as_float((uint32_t)b);
        const bool  in = sqrt_in_range(x);
        bad += in != (x >= RT_SQRT_LO && x <= RT_SQRT_HI);
        const float nx = __uint_as_float((uint32_t)b | 0x80000000u);      // negatives never pass
        if (in) {
            bad += !same_bits(sqrt_ranged(x), sqrtf(x));
            // the sphere roots' two-wide form on the negated operand: -sqrt(x) in BOTH lanes (the other lane holds a
            // second in-range value, so that the lanes cannot share a result by accident)
            const float x2 = __uint_as_float(0x0d800000u + ((uint32_t)b * 2654435761u) % 0x64000001u);
            float s0, s1;
            f2_split(neg_sqrt_pair(f2_make(nx, -x2)), s0, s1);
            bad += !same_bits(s0, -sqrtf(x));
            bad += !same_bits(s1, -sqrtf(x2));
        }
        bad += sqrt_in_range(nx);
    }
    if (bad) atomicAdd(mismatches, bad);
}

// Row gather (multi-GPU): a GPU whose frame lives in ANOTHER GPU's memory renders into a local, zeroed, full-frame
// buffer — the render kernel is exactly the single-GPU one — and this kernel then moves every pixel it finds there
// (its own tiles and whatever it stole from other shards) into the remote frame: 16-byte vector stores wherever four
// neighbouring pixels are all present (512 contiguous bytes per warp and step over NVLink instead of one 4-byte store per
// pixel), word by word at the ragged edges.  A zero word means "not rendered here": every real pixel has alpha 255.
__global__ void __launch_bounds__(256) rt_gather_rows_kernel(const uint32_t* __restrict__ local, uint32_t* __restrict__ remote,
                                                             size_t n_pixels)
{
    const size_t  n4 = n_pixels >> 2, stride = (size_t)gridDim.x * blockDim.x;
    const uint4*  src4 = reinterpret_cast<const uint4*>(local);
    uint4*        dst4 = reinterpret_cast<uint4*>(remote);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const uint4 v = src4[i];
        if (!(v.x | v.y | v.z | v.w)) continue;
        if (v.x && v.y && v.z && v.w) {
            dst4[i] = v;
        } else {
            uint32_t* d = reinterpret_cast<uint32_t*>(dst4 + i);
            if (v.x) d[0] = v.x;
            if (v.y) d[1] = v.y;
            if (v.z) d[2] = v.z;
            if (v.w) d[3] = v.w;
        }
    }
    for (size_t i = (n4 << 2) + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pixels; i += stride)
        if (local[i]) remote[i] = local[i];
}

cudaError_t launch_gather_rows(const uint32_t* local, uint32_t* remote, size_t n_pixels, int grid, cudaStream_t stream)
{
    rt_gather_rows_kernel<<<grid, 256, 0, stream>>>(local, remote, n_pixels);
    return cudaGetLastError();
}

cudaError_t launch_selftest_sqrt(int grid, int block, unsigned long long* d_mismatches, cudaStream_t stream)
{
    rt_selftest_sqrt_kernel<<<grid, block, 0, stream>>>(d_mismatches);
    return cudaGetLastError();
}

cudaError_t launch_selftest_division(unsigned long long n_per_thread, uint32_t seed, int grid, int block,
                                     unsigned long long* d_mismatches, cudaStream_t stream)
{
    rt_selftest_division_kernel<<<grid, block, 0, stream>>>(n_per_thread, seed, d_mismatches);
    return cudaGetLastError();
}

}   // namespace rt
