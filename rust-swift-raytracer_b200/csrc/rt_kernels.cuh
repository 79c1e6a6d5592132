// rt_kernels.cuh — the render kernel (sm_100a), shared by the exact and the fast
// translation units.
//
// One persistent launch per frame (or per progressive pass) replaces the reference's
// row -> column -> sample -> bounce loop nest (common.rs:320-361):
//
//   * grid = (#SMs x resident CTAs per SM) CTAs; every warp pulls work from one global
//     counter in slabs of P.reserve pixel slots (sized by the host so that a warp takes
//     dozens of slabs per frame), so the frame is balanced dynamically and there is neither a
//     CTA wave tail nor a long last-slab tail.
//   * one LANE owns one pixel at a time and adds that pixel's samples in order (float
//     addition is not associative — this is what keeps the sums bit-identical to
//     common.rs:338-340).  A lane whose path ends starts its next sample in the very next
//     iteration, and a lane whose pixel is finished takes the next pixel slot (warp-level
//     ballot/popc compaction of the slab) — no lane ever waits for its neighbours' longer
//     paths.  Each loop iteration traces exactly one ray segment per live lane, and the
//     expensive steps of that segment (normalisations, World::hit, random_unit_sphere) are
//     shared by all lanes whatever their paths are doing (rt_trace.cuh, trace_segment).
//   * the primitive list ({c, r*r} per sphere, {n, n.v0} per triangle — 16 B each) is staged
//     once per CTA into shared memory with one TMA bulk copy (cp.async.bulk + mbarrier);
//     every warp then reads it with broadcast LDS.128.  Scenes too large for shared memory
//     fall back to the same loop over global memory (L1/L2 broadcast loads).
//   * accumulate + sqrt-gamma + RGBA8 pack + vertical flip are fused at the end of each
//     pixel: one 32-bit store per pixel, no intermediate framebuffer pass.
//   * the pixel order inside a slab is 8x4 tiles, so a warp's primary rays are coherent.
#pragma once
#include "rt_launch.h"
#include "rt_trace.cuh"

#include <cuda_runtime.h>

#include <cstdlib>


namespace rt {

// bytes of the hot lists a CTA stages (block A or block B of rt_types.h)
__host__ __device__ inline uint32_t rt_hot_bytes(const RtSceneView& G, int sph_mode)
{
    if (sph_mode == RT_SPH_CULL) return (10u * G.n_groups + G.n_tri_pad) * (uint32_t)sizeof(RtFloat4);
    uint32_t b = (G.n_sph_pad + G.n_tri_pad) * (uint32_t)sizeof(RtFloat4);
    if (sph_mode == RT_SPH_FILTER) b += ((G.n_sph_pad * (uint32_t)sizeof(float)) + 15u) & ~15u;
    return b;
}

// --- TMA bulk copy (global -> shared) of the hot primitive list -------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void stage_scene_tma(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                                unsigned long long* mbar)
{
    const uint32_t bar = smem_u32(mbar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(1));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                     : "memory");
        uint32_t       dst = smem_u32(smem_dst);
        const char*    src = static_cast<const char*>(gmem_src);
        uint32_t       off = 0;
        const uint32_t CH  = 32768u;   // keep each bulk copy modest; all complete on one barrier
        while (off < bytes) {
            uint32_t n = bytes - off < CH ? bytes - off : CH;
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                ::"r"(dst + off), "l"(src + off), "r"(n), "r"(bar)
                : "memory");
            off += n;
        }
    }
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(0)
            : "memory");
    }
}

// The hot lists of a CTA — block A {sph | tri_plane}, block B {sph_filter | tri_plane | sph_r2} or block C
// {cull_bound | cull_sph | tri_plane} of rt_types.h, each one contiguous range of the scene blob — staged into the
// block's shared memory `smem` (SMEM) or addressed in global memory.  Sets the list pointers the walks read.
// The prologue of rt_render_kernel, restated for the first-hit kernel: calling this from the render kernel changes
// the SASS of one of its instantiations (DESIGN.md §11), so the render keeps its own copy.
template <bool SMEM, int SPH>
__device__ __forceinline__ void stage_hot_lists(const RtSceneView& G, unsigned char* smem, unsigned long long* mbar,
                                                const RtFloat4*& sph, const RtFloat4*& tri_plane, const float*& sph_r2,
                                                CullView& cv)
{
    if (SMEM) {
        const uint32_t hot_bytes = rt_hot_bytes(G, SPH);
        const void*    src       = SPH == RT_SPH_CULL ? (const void*)G.cull_bound
                                 : SPH == RT_SPH_FILTER ? (const void*)G.sph_filter : (const void*)G.sph;
        if (hot_bytes) stage_scene_tma(smem, src, hot_bytes, mbar);
        // The staged lists are addressed from ONE opaque copy of the block's shared-memory address.  Left to itself the
        // compiler treats `&rt_smem` as a free constant and re-derives it (S2UR SR_CgaCtaId, UMOV, UIADD3, ULEA) in
        // every iteration of the intersection loops — 6 of the 55 instructions of a FILTER group; through the opaque
        // value it stays in one uniform register and the loads become LDS [R + UR + imm].
        uint32_t hot_base = smem_u32(smem);
        asm volatile("" : "+r"(hot_base));
        const RtFloat4* const hot = reinterpret_cast<const RtFloat4*>(__cvta_shared_to_generic(hot_base));
        if (SPH == RT_SPH_CULL) {
            cv.bound  = hot;
            cv.sph9   = cv.bound + G.n_groups;
            sph       = cv.sph9;                               // not walked in list order in this mode
            tri_plane = cv.sph9 + 9u * G.n_groups;
        } else {
            sph       = hot;
            tri_plane = sph + G.n_sph_pad;
            if (SPH == RT_SPH_FILTER) sph_r2 = reinterpret_cast<const float*>(tri_plane + G.n_tri_pad);
        }
    } else {
        sph       = SPH == RT_SPH_FILTER ? G.sph_filter : G.sph;
        tri_plane = G.tri_plane;
        if (SPH == RT_SPH_FILTER) sph_r2 = G.sph_r2;
    }
}

// The float4 sums of a pixel between fused passes: ONE 16-byte access each way, at system scope
// (SASS LDG/STG.E.128.STRONG.SYS), so that the record — colour sums plus the alpha channel that
// counts the samples and thereby tags the pass — is seen whole by whichever SM or GPU traces the
// pixel's next pass, without going through a (possibly stale) L1 line.
__device__ __forceinline__ float4 accum_load(const RtFloat4* p)
{
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void accum_store(RtFloat4* p, float4 v)
{
    asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

#ifndef RT_MIN_CTAS_SMALL
#define RT_MIN_CTAS_SMALL 4   // 256-thread CTAs per SM the register allocation must allow (<= 64 registers)
#endif
#ifndef RT_MIN_CTAS_FILTER
#define RT_MIN_CTAS_FILTER 3  // FILTER kernels: 80 registers measured faster than 64 (the loop is FFMA-bound,
#endif                        // not latency-bound: C3 fast 399 -> 369 ms, exact 439 -> 431 ms)

// NP = paths per lane.  1: a lane traces one ray at a time.  2 (FILTER walk): a lane carries two independent
// paths (two pixels, or two samples in sample-item mode) and tests BOTH rays against every sphere it loads —
// half the shared-memory feed per ray-sphere test (rt_trace.cuh sphere_filter_group_n).  The doubled state
// needs ~128 registers: two 256-thread CTAs per SM, or one 512-thread CTA when the lists fill shared memory.
template <bool FAST, bool SMEM, int BLOCK, int SPH, bool TRIS, int NP>
__global__ void __launch_bounds__(BLOCK, NP == 2 ? (BLOCK == 256 ? 2 : 1)
                                         : BLOCK != 256 ? 1 : SPH != RT_SPH_DIRECT ? RT_MIN_CTAS_FILTER : RT_MIN_CTAS_SMALL)
rt_render_kernel(const __grid_constant__ RtFrameParams P, const __grid_constant__ RtSceneView G)
{
    static_assert(NP == 1 || (NP == 2 && SPH == RT_SPH_FILTER), "two paths per lane exist for the FILTER walk only");
    extern __shared__ __align__(128) unsigned char rt_smem[];
    __shared__ __align__(8) unsigned long long rt_mbar;

    // the hot lists — block A {sph | tri_plane}, block B {sph_filter | tri_plane | sph_r2} or block C
    // {cull_bound | cull_sph | tri_plane} of rt_types.h — each one contiguous range of the scene blob
    const RtFloat4* sph;
    const RtFloat4* tri_plane;
    const float*    sph_r2 = nullptr;
    CullView        cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    if (SMEM) {
        const uint32_t hot_bytes = rt_hot_bytes(G, SPH);
        const void*    src       = SPH == RT_SPH_CULL ? (const void*)G.cull_bound
                                 : SPH == RT_SPH_FILTER ? (const void*)G.sph_filter : (const void*)G.sph;
        if (hot_bytes) stage_scene_tma(rt_smem, src, hot_bytes, &rt_mbar);
        // The staged lists are addressed from ONE opaque copy of the block's shared-memory address.  Left to itself the
        // compiler treats `&rt_smem` as a free constant and re-derives it (S2UR SR_CgaCtaId, UMOV, UIADD3, ULEA) in
        // every iteration of the intersection loops — 6 of the 55 instructions of a FILTER group; through the opaque
        // value it stays in one uniform register and the loads become LDS [R + UR + imm].
        uint32_t hot_base = smem_u32(rt_smem);
        asm volatile("" : "+r"(hot_base));
        const RtFloat4* const hot = reinterpret_cast<const RtFloat4*>(__cvta_shared_to_generic(hot_base));
        if (SPH == RT_SPH_CULL) {
            cv.bound  = hot;
            cv.sph9   = cv.bound + G.n_groups;
            sph       = cv.sph9;                               // not walked in list order in this mode
            tri_plane = cv.sph9 + 9u * G.n_groups;
        } else {
            sph       = hot;
            tri_plane = sph + G.n_sph_pad;
            if (SPH == RT_SPH_FILTER) sph_r2 = reinterpret_cast<const float*>(tri_plane + G.n_tri_pad);
        }
    } else {
        sph       = SPH == RT_SPH_FILTER ? G.sph_filter : G.sph;
        tri_plane = G.tri_plane;
        if (SPH == RT_SPH_FILTER) sph_r2 = G.sph_r2;
    }

    const uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt   = (1u << lane) - 1u;

    const uint32_t subtiles_x       = (P.width + 7u) >> 3;
    const uint32_t chunks_per_strip = subtiles_x * (P.tile_rows >> 2);
    const bool     trace            = (P.spp > 0) && (P.depth > 0);
    const bool     items            = (P.flags & RT_FLAG_SAMPLE_ITEMS) != 0;      // host sets it only when trace
    const uint32_t slots_per_tile   = chunks_per_strip * 32u * (items ? (uint32_t)P.spp : 1u);
    const uint32_t passes           = P.passes > 1u ? P.passes : 1u;

    // The queue this warp draws from (P.queues[q]; q == P.n_queues: nothing left anywhere): its own shard
    // first, then — multi-GPU — the other shards.  Everything else about a queue is re-read from the
    // kernel parameters where it is needed (slab refill, slot decode), not carried in registers.
    uint32_t q = 0u;

    // warp-uniform slab of reserved pixel slots
    uint32_t pool_next = 0, pool_end = 0;

    Lane L[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
        L[p].have = false;
        L[p].fcol = L[p].frow = 0.f;
        L[p].pix_hash = L[p].out_index = 0u;
        L[p].sample = 0; L[p].seg_left = 0; L[p].rng = 1u; L[p].pend_unit = false;
        L[p].ctl = 0u;
        L[p].acc_r = L[p].acc_g = L[p].acc_b = 0.f;
        L[p].o = L[p].pend = L[p].thr = mk(0.f, 0.f, 0.f);
    }
    uint32_t segments = 0;
    for (;;) {
        // ---- 1. paths without a pixel take the next slots of the warp's slab ----
        uint32_t lacking = FULL;                  // lanes none of whose paths has a pixel
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            Lane&    Lp   = L[p];
            uint32_t need = __ballot_sync(FULL, !Lp.have);
            while (need && q < P.n_queues) {
                if (pool_next == pool_end) {
                    const uint32_t total = P.queues[q].n_tiles * slots_per_tile * passes;
                    uint32_t       base  = 0;
                    if (lane == 0)
                        base = P.n_queues > 1u ? atomicAdd_system(P.queues[q].work_counter, P.reserve)
                                               : atomicAdd(P.queues[q].work_counter, P.reserve);
                    base = __shfl_sync(FULL, base, 0);
                    if (base >= total) { ++q; continue; }      // this shard has no unassigned work left: raid the next one
                    pool_next = base;
                    pool_end  = min(base + P.reserve, total);
                    if (q && lane == 0 && P.steal_counter) atomicAdd(P.steal_counter, pool_end - pool_next);
                }
                const uint32_t avail = pool_end - pool_next;
                const uint32_t rank  = __popc(need & lt);
                if (!Lp.have && rank < avail) {
                    uint32_t  item_sample, pass;
                    const uint32_t q_tiles = P.queues[q].n_tiles;
                    PixelSlot s = decode_slot(P, pool_next + rank, subtiles_x, chunks_per_strip, P.queues[q].tile_first, q_tiles,
                                              q_tiles * slots_per_tile, item_sample, pass);
                    if (s.valid) {
                        begin_pixel(Lp, P, s.column, P.height - 1u - s.image_row, s.out_index);   // common.rs:351 (flip)
                        Lp.ctl = pass | (q << 16);
                        if (items) {                       // one sample: sums start at 0, colour goes to the sample buffer
                            Lp.sample    = (int32_t)item_sample;
                            Lp.out_index = item_sample * P.sample_stride + s.out_index;
                        } else {
                            Lp.sample = (int32_t)(pass * (uint32_t)P.spp);
                            if (pass > 0u) {
                                Lp.ctl |= RT_LANE_WAIT;     // starts from the sums of the pixel's previous pass (step 1b)
                            } else if (P.flags & RT_FLAG_ACCUM_IN) {
                                RtFloat4 a = ld4(&P.queues[0].accum[s.out_index]);
                                Lp.acc_r = a.x; Lp.acc_g = a.y; Lp.acc_b = a.z;      // a.w is re-read at the end
                            }
                        }
                    }
                }
                pool_next += min(avail, (uint32_t)__popc(need));
                need = __ballot_sync(FULL, !Lp.have);
            }
            lacking &= need;                      // `need` is the ballot of !have as it stands after the refill
        }
        if (lacking == FULL) break;               // no pixel anywhere in the warp and every queue is empty

        // ---- 1b. fused passes: a pixel's pass p continues the sums its pass p-1 stored; the alpha sum
        //          (1 + samples so far, pixel_alpha) tags the record.  Not there yet: look again next time
        //          round — the lane never blocks, so the producer (which may sit in this very warp) runs on ----
        bool ready[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            Lane& Lp = L[p];
            if (Lp.have && (Lp.ctl & RT_LANE_WAIT)) {
                const RtFloat4* ac = P.queues[(Lp.ctl >> 16) & 0xffu].accum;
                const float4    a  = accum_load(&ac[Lp.out_index]);
                if (a.w == pixel_alpha(1.0f, Lp.sample)) {
                    Lp.acc_r = a.x; Lp.acc_g = a.y; Lp.acc_b = a.z;
                    Lp.ctl &= ~RT_LANE_WAIT;
                }
            }
            ready[p] = Lp.have && !(Lp.ctl & RT_LANE_WAIT);
        }

        // ---- 2. one ray segment per live path (sample start, World::hit, scatter, accumulate) ----
        bool sample_done[NP];
        if (NP == 1) {
            sample_done[0] = false;
            if (ready[0] && trace) {
                sample_done[0] = trace_segment<FAST, SPH, TRIS>(L[0], P, G, sph, sph_r2, cv, tri_plane);
                ++segments;
            }
        } else {
            V3   o[NP], d[NP];
            Hit  h[NP];
            bool live = false;
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                sample_done[p] = false;
                o[p] = mk(0.f, 0.f, 0.f);
                d[p] = mk(NAN, NAN, NAN);                  // an idle path: never hits anything
                if (ready[p] && trace) {
                    d[p] = segment_begin<FAST>(L[p], P);
                    o[p] = L[p].o;
                    live = true;
                    ++segments;
                }
            }
            if (live) {
                closest_hit_n<FAST, TRIS, NP>(sph, sph_r2, G.n_sph, G.n_sph_pad, tri_plane, G.tri_cull, G.tri_v, G.n_tri_pad, o, d, P.one, h);
#pragma unroll
                for (int p = 0; p < NP; ++p)
                    if (ready[p] && trace) sample_done[p] = segment_end<FAST, SPH, TRIS>(L[p], G, sph, d[p], h[p]);
            }
        }

#pragma unroll
        for (int p = 0; p < NP; ++p) {
            Lane& Lp = L[p];
            // ---- 3a. sample items: hand the colour to the ordered-sum kernel ----
            if (items) {
                if (Lp.have && sample_done[p]) {
                    *reinterpret_cast<float4*>(&P.samples[Lp.out_index]) = make_float4(Lp.acc_r, Lp.acc_g, Lp.acc_b, 1.0f);
                    Lp.have = false;
                }
                continue;
            }

            // ---- 3b. the pixel's pass is complete: hand the sums on and/or resolve + pack ----
            const uint32_t pass     = Lp.ctl & 0xffffu;
            const int32_t  pass_end = (int32_t)((pass + 1u) * (uint32_t)(P.spp > 0 ? P.spp : 0));
            if (ready[p] && (!trace || Lp.sample >= pass_end)) {
                RtFloat4*  ac   = P.queues[(Lp.ctl >> 16) & 0xffu].accum;
                const bool last = pass + 1u == passes;
                // alpha: 1.0 (or the accumulator's) + one per sample; depth <= 0 still adds spp black samples
                const float a0    = (P.flags & RT_FLAG_ACCUM_IN) ? ac[Lp.out_index].w : 1.0f;
                const float acc_a = pixel_alpha(a0, pass_end);
                if (!last || (P.flags & RT_FLAG_ACCUM_OUT))
                    accum_store(&ac[Lp.out_index], make_float4(Lp.acc_r, Lp.acc_g, Lp.acc_b, acc_a));
                if (last ? !(P.flags & RT_FLAG_NO_RESOLVE) : (P.flags & RT_FLAG_RESOLVE_EACH_PASS) != 0u) {
                    P.out[Lp.out_index] = resolve_pixel<FAST>(Lp.acc_r, Lp.acc_g, Lp.acc_b, acc_a,
                                                              last ? P.resolve_spp : P.sample_begin + pass_end);
                }
                if (last && P.tile_done) {      // full-frame output: out_index = image_row * width + column
                    const uint32_t tile  = (Lp.out_index / P.width) / P.tile_rows;
                    const uint32_t rows  = min((tile + 1u) * P.tile_rows, P.height) - tile * P.tile_rows;
                    __threadfence();                   // this pixel is ordered before its count (device scope: cheap) ...
                    if (atomicAdd(&P.tile_done[tile], 1u) + 1u == rows * P.width) {
                        __threadfence_system();        // ... and the one lane that completes the tile orders all of them,
                                                       // cumulatively, before the flag the host polls
                        *reinterpret_cast<volatile unsigned int*>(&P.tile_flags[tile]) = P.tile_epoch;
                    }
                }
                Lp.have = false;
            }
        }
    }

    // ray-segment count: one atomic per warp
    unsigned long long segs = segments;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) segs += __shfl_xor_sync(FULL, segs, o);
    if (lane == 0 && P.ray_counter && segs) atomicAdd(P.ray_counter, segs);
}

// Second kernel of the RT_FLAG_SAMPLE_ITEMS mode: one thread per pixel adds the pixel's sample
// colours IN SAMPLE ORDER (common.rs:338-340; float addition is not associative, and
// 0.0f + colour == colour, so the sums are the bits the one-lane-per-pixel kernel produces),
// then resolves and packs exactly like the render kernel (common.rs:344-356).  HBM-bound:
// spp*16 B read + 4 B written per pixel, coalesced (a warp reads 512 contiguous bytes per sample).
template <bool FAST>
__global__ void __launch_bounds__(256) rt_resolve_samples_kernel(const __grid_constant__ RtFrameParams P)
{
    const uint32_t rows_out = P.n_tiles * P.tile_rows;
    const uint32_t local    = blockIdx.x * blockDim.x + threadIdx.x;          // index among this shard's pixel rows
    if (local >= rows_out * P.width) return;
    const uint32_t r = local / P.width, x = local - r * P.width;
    const uint32_t strip = r / P.tile_rows, yin = r - strip * P.tile_rows;
    const uint32_t image_row = rt_shard_tile(P.tile_first, P.tile_stride, strip) * P.tile_rows + yin;
    if (image_row >= P.height) return;
    const uint32_t out_row = (P.flags & RT_FLAG_COMPACT_OUT) ? r : image_row;
    const uint32_t idx     = out_row * P.width + x;
    float acc_r = 0.f, acc_g = 0.f, acc_b = 0.f, a0 = 1.0f;                 // Color::new(0,0,0), common.rs:333
    if (P.flags & RT_FLAG_ACCUM_IN) {
        RtFloat4 a = ld4(&P.accum[idx]);
        acc_r = a.x; acc_g = a.y; acc_b = a.z; a0 = a.w;
    }
    for (int32_t s = 0; s < P.spp; ++s) {
        const float4 c = *reinterpret_cast<const float4*>(&P.samples[(size_t)s * P.sample_stride + idx]);
        acc_r += c.x; acc_g += c.y; acc_b += c.z;
    }
    const float acc_a = pixel_alpha(a0, P.spp);
    if (P.flags & RT_FLAG_ACCUM_OUT) *reinterpret_cast<float4*>(&P.accum[idx]) = make_float4(acc_r, acc_g, acc_b, acc_a);
    if (!(P.flags & RT_FLAG_NO_RESOLVE)) P.out[idx] = resolve_pixel<FAST>(acc_r, acc_g, acc_b, acc_a, P.resolve_spp);
}

template <bool FAST>
cudaError_t launch_resolve_samples(const RtFrameParams& P, cudaStream_t stream)
{
    const uint64_t n = (uint64_t)P.n_tiles * P.tile_rows * P.width;
    if (n == 0) return cudaSuccess;
    rt_resolve_samples_kernel<FAST><<<(unsigned)((n + 255u) / 256u), 256, 0, stream>>>(P);
    return cudaGetLastError();
}

// Launch geometry.  Small primitive lists leave room for several 256-thread CTAs per SM;
// a list that fills most of shared memory (thousands of primitives) allows only one CTA
// per SM, which then has to be 1024 threads wide to keep the SM's schedulers fed.
constexpr int      kBlockSmall    = 256;
#ifndef RT_BLOCK_LARGE
#define RT_BLOCK_LARGE 1024
#endif
constexpr int      kBlockLarge    = RT_BLOCK_LARGE;
constexpr int      kBlockLarge2   = RT_BLOCK_LARGE / 2;   // two paths per lane: half the threads, twice the registers
constexpr size_t   kLargeSmemFrom = 56 * 1024;   // above this, < 4 CTAs of 256 threads would fit
constexpr uint32_t kFilterFrom    = RT_FILTER_FROM;   // spheres from which the kernels filter first

struct RenderVariant { bool smem; int block; int sph; bool tris; size_t hot_bytes; int np; };

// Paths per lane of the FILTER kernels.  Measured with the FFMA2 filter (profiles/r02_bench.md): one path per lane
// is as fast as two on C3 exact (302 vs 304 ms), 3 % slower on C3 fast-math (290 vs 281 ms) and 17 % FASTER on C5
// (194 vs 233 ms: sixteen warps per SM do not hide the latencies of its long, divergent paths), so one is the
// default; RT_PATHS_PER_LANE=2 selects the two-path kernels.
inline int filter_paths_per_lane()
{
    static const int np = [] { const char* e = getenv("RT_PATHS_PER_LANE"); return (e && *e == '2') ? 2 : 1; }();
    return np;
}

inline RenderVariant choose_variant(const RtSceneView& G, size_t smem_limit, bool cull)
{
    RenderVariant v;
    // the sphere count, not the padded list: 57-63 spheres pad to 64 but stay below RT_FILTER_FROM (no block C either)
    v.sph       = (cull && G.n_groups > 0) ? RT_SPH_CULL : G.n_sph >= kFilterFrom ? RT_SPH_FILTER : RT_SPH_DIRECT;
    v.tris      = G.n_tri_pad > 0;
    v.hot_bytes = rt_hot_bytes(G, v.sph);
    v.smem      = v.hot_bytes <= smem_limit;
    v.np        = v.sph == RT_SPH_FILTER ? filter_paths_per_lane() : 1;
    v.block     = (v.smem && v.hot_bytes > kLargeSmemFrom) ? (v.np == 2 ? kBlockLarge2 : kBlockLarge) : kBlockSmall;
    return v;
}

// The geometry of the one-ray-per-lane kernels (first hit, ray and occlusion queries): the walk, staging and CTA width
// choose_variant picks for the render of the same world, with one path per lane.
inline RenderVariant choose_aov_variant(const RtSceneView& G, size_t smem_limit, bool cull)
{
    RenderVariant v = choose_variant(G, smem_limit, cull);
    if (v.np == 2) {
        v.np = 1;
        if (v.block == kBlockLarge2) v.block = kBlockLarge;
    }
    return v;
}

// ---- first-hit buffers ---------------------------------------------------------------------------------------------
// One World::hit per pixel: the camera ray of sample A.sample_begin (rt_trace.cuh first_hit), its HitRecord written to
// the buffers A names.  Persistent grid; every CTA stages the hot lists once (stage_hot_lists), then each warp takes
// 8x4-pixel sub-tiles in a grid-stride loop, so that its primary rays are as coherent as the render's.  The lanes of a
// warp store 4 rows of 8 neighbouring pixels: every store instruction covers whole 32-byte sectors (depth, prim) or
// 96 contiguous bytes per row (the float3 buffers), each buffer written once.  Exact policy only.
template <bool SMEM, int BLOCK, int SPH, bool TRIS>
__global__ void __launch_bounds__(BLOCK, BLOCK != 256 ? 1 : SPH != RT_SPH_DIRECT ? RT_MIN_CTAS_FILTER : RT_MIN_CTAS_SMALL)
rt_aov_kernel(const __grid_constant__ RtAovParams A, const __grid_constant__ RtSceneView G)
{
    extern __shared__ __align__(128) unsigned char rt_smem[];
    __shared__ __align__(8) unsigned long long rt_mbar;
    const RtFloat4* sph;
    const RtFloat4* tri_plane;
    const float*    sph_r2 = nullptr;
    CullView        cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    stage_hot_lists<SMEM, SPH>(G, rt_smem, &rt_mbar, sph, tri_plane, sph_r2, cv);

    const uint32_t lane       = threadIdx.x & 31u;
    const uint32_t subtiles_x = (A.width + 7u) >> 3;
    const uint32_t n_sub      = subtiles_x * ((A.height + 3u) >> 2);      // < 2^31 (host check)
    const uint32_t warps      = gridDim.x * (uint32_t)(BLOCK / 32);
    for (uint32_t s = blockIdx.x * (uint32_t)(BLOCK / 32) + (threadIdx.x >> 5); s < n_sub; s += warps) {
        const uint32_t sy = s / subtiles_x, sx = s - sy * subtiles_x;
        const uint32_t x = sx * 8u + (lane & 7u), row = sy * 4u + (lane >> 3);
        if (x >= A.width || row >= A.height) continue;
        const AovRecord r = first_hit<false, SPH, TRIS>(A, G, sph, sph_r2, cv, tri_plane, x, row);
        const size_t    i = (size_t)row * A.width + x;
        if (A.depth) A.depth[i] = r.t;
        if (A.position) { A.position[3 * i] = r.pos.x; A.position[3 * i + 1] = r.pos.y; A.position[3 * i + 2] = r.pos.z; }
        if (A.normal) { A.normal[3 * i] = r.n.x; A.normal[3 * i + 1] = r.n.y; A.normal[3 * i + 2] = r.n.z; }
        if (A.albedo) { A.albedo[3 * i] = r.albedo.x; A.albedo[3 * i + 1] = r.albedo.y; A.albedo[3 * i + 2] = r.albedo.z; }
        if (A.prim) A.prim[i] = r.prim;
    }
}

// ---- ray queries ---------------------------------------------------------------------------------------------------
// World::hit of n caller-supplied rays with a per-ray t_max (rt_trace.cuh ray_hit), the record of ray i written to
// element i of the buffers R names.  The skeleton of rt_aov_kernel: persistent grid, hot lists staged once per CTA,
// then each warp takes 32 consecutive rays in a grid-stride loop — two 16-byte read-only loads per ray, each buffer
// written once, the lanes' stores contiguous.  No scratch, no atomics.  Exact policy only.
template <bool SMEM, int BLOCK, int SPH, bool TRIS>
__global__ void __launch_bounds__(BLOCK, BLOCK != 256 ? 1 : SPH != RT_SPH_DIRECT ? RT_MIN_CTAS_FILTER : RT_MIN_CTAS_SMALL)
rt_ray_kernel(const __grid_constant__ RtRayParams R, const __grid_constant__ RtSceneView G)
{
    extern __shared__ __align__(128) unsigned char rt_smem[];
    __shared__ __align__(8) unsigned long long rt_mbar;
    const RtFloat4* sph;
    const RtFloat4* tri_plane;
    const float*    sph_r2 = nullptr;
    CullView        cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    stage_hot_lists<SMEM, SPH>(G, rt_smem, &rt_mbar, sph, tri_plane, sph_r2, cv);

    // one induction variable: ray i = 32 * (warp's chunk) + lane, stepping 32 * (warps in the grid)
    const uint32_t end    = ((R.n + 31u) >> 5) << 5;                     // R.n < 2^31 (host check)
    const uint32_t stride = gridDim.x * (uint32_t)BLOCK;
    const float4*  rays   = reinterpret_cast<const float4*>(R.rays);
    for (uint32_t i = (blockIdx.x * (uint32_t)(BLOCK / 32) + (threadIdx.x >> 5)) * 32u + (threadIdx.x & 31u); i < end; i += stride) {
        if (i >= R.n) continue;
        const float4 a = __ldg(&rays[2u * (size_t)i]), b = __ldg(&rays[2u * (size_t)i + 1u]);
        RtFloat4 r0, r1;
        r0.x = a.x; r0.y = a.y; r0.z = a.z; r0.w = a.w;
        r1.x = b.x; r1.y = b.y; r1.z = b.z; r1.w = b.w;
        const AovRecord r = ray_hit<SPH, TRIS>(G, sph, sph_r2, cv, tri_plane, r0, r1, R.one);
        const size_t    k = i;                                           // the record of ray i
        if (R.depth) R.depth[k] = r.t;
        if (R.position) { R.position[3 * k] = r.pos.x; R.position[3 * k + 1] = r.pos.y; R.position[3 * k + 2] = r.pos.z; }
        if (R.normal) { R.normal[3 * k] = r.n.x; R.normal[3 * k + 1] = r.n.y; R.normal[3 * k + 2] = r.n.z; }
        if (R.albedo) { R.albedo[3 * k] = r.albedo.x; R.albedo[3 * k + 1] = r.albedo.y; R.albedo[3 * k + 2] = r.albedo.z; }
        if (R.prim) R.prim[k] = r.prim;
    }
}

// ---- occlusion queries ---------------------------------------------------------------------------------------------
// Does World::hit return a hit for each of n caller-supplied rays (rt_trace.cuh ray_occluded)?  The skeleton of
// rt_ray_kernel — persistent grid, hot lists staged once per CTA, 32 consecutive rays per warp, two 16-byte read-only
// loads per ray — and one byte stored per ray.  A lane whose ray is answered early leaves the walk and waits for the
// warp's other lanes.  No scratch, no atomics.  Exact policy only.
template <bool SMEM, int BLOCK, int SPH, bool TRIS>
__global__ void __launch_bounds__(BLOCK, BLOCK != 256 ? 1 : SPH != RT_SPH_DIRECT ? RT_MIN_CTAS_FILTER : RT_MIN_CTAS_SMALL)
rt_occlusion_kernel(const __grid_constant__ RtOcclusionParams Q, const __grid_constant__ RtSceneView G)
{
    extern __shared__ __align__(128) unsigned char rt_smem[];
    __shared__ __align__(8) unsigned long long rt_mbar;
    const RtFloat4* sph;
    const RtFloat4* tri_plane;
    const float*    sph_r2 = nullptr;
    CullView        cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    stage_hot_lists<SMEM, SPH>(G, rt_smem, &rt_mbar, sph, tri_plane, sph_r2, cv);

    const uint32_t end    = ((Q.n + 31u) >> 5) << 5;                     // Q.n < 2^31 (host check)
    const uint32_t stride = gridDim.x * (uint32_t)BLOCK;
    const float4*  rays   = reinterpret_cast<const float4*>(Q.rays);
    for (uint32_t i = (blockIdx.x * (uint32_t)(BLOCK / 32) + (threadIdx.x >> 5)) * 32u + (threadIdx.x & 31u); i < end; i += stride) {
        if (i >= Q.n) continue;
        const float4 a = __ldg(&rays[2u * (size_t)i]), b = __ldg(&rays[2u * (size_t)i + 1u]);
        RtFloat4 r0, r1;
        r0.x = a.x; r0.y = a.y; r0.z = a.z; r0.w = a.w;
        r1.x = b.x; r1.y = b.y; r1.z = b.z; r1.w = b.w;
        Q.occluded[i] = (uint8_t)ray_occluded<SPH, TRIS>(G, sph, sph_r2, cv, tri_plane, r0, r1, Q.one);
    }
}

// ---- host-side dispatch -------------------------------------------------------------------------------------------
// KernelOf<K> names the template of kernel K (rt_launch.h): get<SMEM, BLOCK, SPH, TRIS, NP>() is an instantiation,
// choose() its geometry, and two_paths whether it has the two-paths-per-lane instantiations (the render only).
template <bool FAST>
struct RenderKernelOf {
    static constexpr bool two_paths = true;
    template <bool SMEM, int BLOCK, int SPH, bool TRIS, int NP>
    static constexpr auto get() { return rt_render_kernel<FAST, SMEM, BLOCK, SPH, TRIS, NP>; }
    static RenderVariant choose(const RtSceneView& G, size_t smem_limit, bool cull) { return choose_variant(G, smem_limit, cull); }
};
struct LaneKernelOf {
    static constexpr bool two_paths = false;
    static RenderVariant choose(const RtSceneView& G, size_t smem_limit, bool cull) { return choose_aov_variant(G, smem_limit, cull); }
};
template <Kernel K> struct KernelOf;
template <> struct KernelOf<Kernel::render_exact> : RenderKernelOf<false> {};
template <> struct KernelOf<Kernel::render_fast> : RenderKernelOf<true> {};
template <> struct KernelOf<Kernel::first_hit> : LaneKernelOf {
    template <bool SMEM, int BLOCK, int SPH, bool TRIS, int NP>
    static constexpr auto get() { static_assert(NP == 1); return rt_aov_kernel<SMEM, BLOCK, SPH, TRIS>; }
};
template <> struct KernelOf<Kernel::ray_query> : LaneKernelOf {
    template <bool SMEM, int BLOCK, int SPH, bool TRIS, int NP>
    static constexpr auto get() { static_assert(NP == 1); return rt_ray_kernel<SMEM, BLOCK, SPH, TRIS>; }
};
template <> struct KernelOf<Kernel::occlusion> : LaneKernelOf {
    template <bool SMEM, int BLOCK, int SPH, bool TRIS, int NP>
    static constexpr auto get() { static_assert(NP == 1); return rt_occlusion_kernel<SMEM, BLOCK, SPH, TRIS>; }
};

// f(kernel pointer, block) for the variant's instantiation of kernel K.  Large sphere lists get the FILTER (or, on
// request, CULL) kernels; worlds without triangles get kernels without the triangle code.
template <class KO, bool SMEM, int BLOCK, int SPH, int NP, class F>
cudaError_t with_tris(const RenderVariant& v, F&& f)
{
    return v.tris ? f(KO::template get<SMEM, BLOCK, SPH, true, NP>(), BLOCK)
                  : f(KO::template get<SMEM, BLOCK, SPH, false, NP>(), BLOCK);
}
template <class KO, int SPH, int NP, class F>
cudaError_t with_staging(const RenderVariant& v, F&& f)
{
    constexpr int large = NP == 2 ? kBlockLarge2 : kBlockLarge;
    if (!v.smem) return with_tris<KO, false, kBlockSmall, SPH, NP>(v, f);
    if (v.block == large) return with_tris<KO, true, large, SPH, NP>(v, f);
    return with_tris<KO, true, kBlockSmall, SPH, NP>(v, f);
}
template <Kernel K, class F>
cudaError_t with_kernel(const RenderVariant& v, F&& f)
{
    using KO = KernelOf<K>;
    if constexpr (KO::two_paths)
        if (v.np == 2) return with_staging<KO, RT_SPH_FILTER, 2>(v, f);      // FILTER walk only
    if (v.sph == RT_SPH_CULL) return with_staging<KO, RT_SPH_CULL, 1>(v, f);
    if (v.sph == RT_SPH_FILTER) return with_staging<KO, RT_SPH_FILTER, 1>(v, f);
    return with_staging<KO, RT_SPH_DIRECT, 1>(v, f);
}

// A kernel that stages its hot lists may use up to smem_limit bytes of dynamic shared memory.
template <class Fn>
cudaError_t allow_staging(Fn* k, const RenderVariant& v, size_t smem_limit)
{
    return v.smem ? cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_limit) : cudaSuccess;
}

template <Kernel K, class Params>
cudaError_t launch_kernel(const Params& p, const RtSceneView& G, bool cull, int grid, size_t smem_limit,
                          cudaStream_t stream)
{
    const RenderVariant v = KernelOf<K>::choose(G, smem_limit, cull);
    return with_kernel<K>(v, [&](auto k, int block) -> cudaError_t {
        const cudaError_t e = allow_staging(k, v, smem_limit);
        if (e != cudaSuccess) return e;
        k<<<grid, block, v.smem ? v.hot_bytes : 0, stream>>>(p, G);
        return cudaGetLastError();
    });
}

template <Kernel K>
cudaError_t kernel_geometry(const RtSceneView& G, size_t smem_limit, bool cull, KernelGeometry* out)
{
    const RenderVariant v = KernelOf<K>::choose(G, smem_limit, cull);
    out->block = v.block; out->hot_bytes = v.hot_bytes; out->resident = v.smem; out->walk = v.sph; out->paths_per_lane = v.np;
    return with_kernel<K>(v, [&](auto k, int block) -> cudaError_t {
        const cudaError_t e = allow_staging(k, v, smem_limit);
        if (e != cudaSuccess) return e;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&out->per_sm, k, block, v.smem ? v.hot_bytes : 0);
    });
}

}   // namespace rt
