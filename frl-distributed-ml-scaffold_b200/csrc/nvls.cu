// K7 — fused gradient all-reduce + optimizer update + weight broadcast over NVSwitch multicast
// (NVLS), one kernel per gradient bucket (sm_100a, world_size > 1).
//
// The reference step is "DDP all-reduces every bucket, then torch.optim updates every replica"
// (reference solver.py:287-289 + solver_worker.py:586-592): every GPU receives the full reduced
// gradient and every GPU streams the full 20-28 B/param optimizer update.  Here each rank owns
// 1/world of every bucket:
//
//   barrier      every rank has finished writing this bucket's gradients
//   reduce       g = multimem.ld_reduce(add) on the bucket's MULTICAST address: the NVSwitch
//                sums the world_size copies in flight; only this rank's shard crosses its link
//   update       torch-exact SGD/Adam/RMSprop on the shard (fp32 master + state, local HBM)
//   broadcast    multimem.st of the new bf16 shadow weights (BF16 mode) or fp32 weights (FP32
//                mode) to the multicast address: the switch replicates them into every replica
//   barrier      all replicas have every shard
//
// Per GPU and step this moves S(1 + 1/world) bytes per direction over NVLink (S = gradient
// bytes) — what an NVLS all-reduce alone moves — and divides the optimizer's HBM traffic and
// state updates by world_size.  No NCCL call, no separate update launch.
//
// Cross-GPU synchronisation uses the symmetric-memory signal pads: block 0 of rank r raises flag r
// in every peer's pad and consumes flag `peer` in its own (CAS 0->1 / 1->0, system scope), then
// releases / collects the other blocks through local flags, so the grid can span every SM.
// Data movement is 16 bytes per multimem instruction.
#include <stdlib.h>

#include "frl_common.cuh"
#include "optim_rules.cuh"

namespace frl {

constexpr int kNThreads = 512;

__device__ __forceinline__ void mm_ld_reduce_bf16x8(const void* mc, uint32_t (&r)[4]) {
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(mc) : "memory");
}
__device__ __forceinline__ void mm_ld_reduce_f32x4(const void* mc, float (&r)[4]) {
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]) : "l"(mc) : "memory");
}
__device__ __forceinline__ void mm_st_b128(void* mc, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(mc), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Cross-GPU rendezvous, done by block 0 only: thread t < world raises flag `rank` in peer t's pad
// and consumes flag `t` in its own (CAS 0->1 / 1->0, system scope).
__device__ __forceinline__ void meet_peers_block0(uint32_t* const* pads, int rank, int world, int base) {
    if (threadIdx.x < world) {
        const int peer = threadIdx.x;
        uint32_t* put = pads[peer] + base + rank;
        uint32_t* wait = pads[rank] + base + peer;
        __threadfence_system();                                   // release everything before
        while (atomicCAS_system(put, 0u, 1u) != 0u) { __nanosleep(100); }
        while (atomicCAS_system(wait, 1u, 0u) != 1u) { __nanosleep(100); }
        __threadfence_system();                                   // acquire everything after
    }
    __syncthreads();
}

// local scratch (uint32, zero-initialised once): [0] = finished-block counter, [8 + b] = go flag of block b
__device__ __forceinline__ void kernel_entry_barrier(uint32_t* const* pads, int rank, int world, int base,
                                                     uint32_t* local) {
    if (blockIdx.x == 0) {
        meet_peers_block0(pads, rank, world, base);               // every rank's gradients are written
        for (int b = threadIdx.x + 1; b < static_cast<int>(gridDim.x); b += blockDim.x)
            atomicExch(local + 8 + b, 1u);                        // release the other blocks
    } else {
        if (threadIdx.x == 0) {
            while (atomicCAS(local + 8 + blockIdx.x, 1u, 0u) != 1u) { __nanosleep(200); }
            __threadfence();
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void kernel_exit_barrier(uint32_t* const* pads, int rank, int world, int base,
                                                    uint32_t* local) {
    __syncthreads();
    if (blockIdx.x != 0) {
        if (threadIdx.x == 0) {
            __threadfence_system();                               // my multimem stores before the count
            atomicAdd(local, 1u);
        }
        return;
    }
    if (threadIdx.x == 0) {
        while (atomicAdd(local, 0u) != gridDim.x - 1) { __nanosleep(100); }
        atomicExch(local, 0u);
        __threadfence_system();
    }
    __syncthreads();
    meet_peers_block0(pads, rank, world, base + 32);              // every replica has every shard
}

struct NvlsCommon {
    uint32_t* const* pads;
    uint32_t* local;
    int rank, world, pad_base;
    int sync_inside;      // 0: the caller brackets the launch with frl_nvls_barrier
    int64_t n;            // bucket elements
    float gscale;
    const float* dyn;
};

// BF16 mode: bf16 gradients in, fp32 master/state local, bf16 shadow multicast out. 8 elems / item.
// The switch round trip of multimem.ld_reduce is the long latency here (microseconds), so every
// thread first issues kNRemote of them back to back and only then walks the items, loading the
// (short-latency) local master/state slices item by item.
// How many remote loads a thread keeps in flight is a template parameter (FRL_B200_NVLS_INFLIGHT,
// default 4).  Deeper pipelines (8, 16) were tried to let a small grid cover NVLink's
// bandwidth-latency product; measured at world 2 (the case with the largest shard per rank) they
// do not pay: 74 CTAs x depth 4 = 1.170 ms/step, 32 x 8 = 1.190, 74 x 16 = 1.198, 16 x 16 = 1.648.
template <typename Rule, int NS, int kNRemote>
__global__ void __launch_bounds__(kNThreads)
nvls_update_bf16(float* __restrict__ p_, float* __restrict__ s0_, float* __restrict__ s1_,
                 float* __restrict__ s2_, const __nv_bfloat16* mc_g, __nv_bfloat16* mc_lp,
                 Rule rule, NvlsCommon c) {
    if (c.dyn) rule.patch(c.dyn);
    if (c.sync_inside) kernel_entry_barrier(c.pads, c.rank, c.world, c.pad_base, c.local);
    const int64_t per = ((c.n + c.world - 1) / c.world + 7) / 8 * 8;
    const int64_t lo = static_cast<int64_t>(c.rank) * per;
    int64_t hi = lo + per;
    if (hi > c.n) hi = c.n;
    const int64_t items = hi > lo ? (hi - lo + 7) / 8 : 0;        // arena buckets are multiples of 8
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kNThreads;
    const f32x4 zero{0.f, 0.f, 0.f, 0.f};
    const float gs = c.gscale;
    for (int64_t it0 = static_cast<int64_t>(blockIdx.x) * kNThreads + threadIdx.x; it0 < items;
         it0 += stride * kNRemote) {
        uint32_t g[kNRemote][4];
#pragma unroll
        for (int u = 0; u < kNRemote; ++u) {
            const int64_t it = it0 + u * stride;
            if (it < items) mm_ld_reduce_bf16x8(mc_g + lo + it * 8, g[u]);
        }
#pragma unroll
        for (int u = 0; u < kNRemote; ++u) {
            const int64_t it = it0 + u * stride;
            if (it >= items) break;
            const int64_t e = lo + it * 8;
            f32x4 vp[2], a0[2], a1[2], a2[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                vp[h] = ld_stream(reinterpret_cast<const f32x4*>(p_ + e) + h);
                a0[h] = NS > 0 ? ld_stream(reinterpret_cast<const f32x4*>(s0_ + e) + h) : zero;
                a1[h] = NS > 1 ? ld_stream(reinterpret_cast<const f32x4*>(s1_ + e) + h) : zero;
                a2[h] = NS > 2 ? ld_stream(reinterpret_cast<const f32x4*>(s2_ + e) + h) : zero;
            }
            rule(vp[0].x, bf16lo(g[u][0]) * gs, a0[0].x, a1[0].x, a2[0].x);
            rule(vp[0].y, bf16hi(g[u][0]) * gs, a0[0].y, a1[0].y, a2[0].y);
            rule(vp[0].z, bf16lo(g[u][1]) * gs, a0[0].z, a1[0].z, a2[0].z);
            rule(vp[0].w, bf16hi(g[u][1]) * gs, a0[0].w, a1[0].w, a2[0].w);
            rule(vp[1].x, bf16lo(g[u][2]) * gs, a0[1].x, a1[1].x, a2[1].x);
            rule(vp[1].y, bf16hi(g[u][2]) * gs, a0[1].y, a1[1].y, a2[1].y);
            rule(vp[1].z, bf16lo(g[u][3]) * gs, a0[1].z, a1[1].z, a2[1].z);
            rule(vp[1].w, bf16hi(g[u][3]) * gs, a0[1].w, a1[1].w, a2[1].w);
            mm_st_b128(mc_lp + e, pack_bf16(vp[0].x, vp[0].y), pack_bf16(vp[0].z, vp[0].w),
                       pack_bf16(vp[1].x, vp[1].y), pack_bf16(vp[1].z, vp[1].w));
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                st_stream(reinterpret_cast<f32x4*>(p_ + e) + h, vp[h]);
                if (NS > 0) st_stream(reinterpret_cast<f32x4*>(s0_ + e) + h, a0[h]);
                if (NS > 1) st_stream(reinterpret_cast<f32x4*>(s1_ + e) + h, a1[h]);
                if (NS > 2) st_stream(reinterpret_cast<f32x4*>(s2_ + e) + h, a2[h]);
            }
        }
    }
    if (c.sync_inside) kernel_exit_barrier(c.pads, c.rank, c.world, c.pad_base, c.local);
    else __threadfence_system();                                  // my multimem stores before the grid ends
}

// FP32 mode: fp32 gradients in, parameters ARE the master: multicast the new fp32 weights.
template <typename Rule, int NS, int kNRemote>
__global__ void __launch_bounds__(kNThreads)
nvls_update_f32(const float* __restrict__ p_, float* __restrict__ s0_, float* __restrict__ s1_,
                float* __restrict__ s2_, const float* mc_g, float* mc_p, Rule rule, NvlsCommon c) {
    if (c.dyn) rule.patch(c.dyn);
    if (c.sync_inside) kernel_entry_barrier(c.pads, c.rank, c.world, c.pad_base, c.local);
    const int64_t per = ((c.n + c.world - 1) / c.world + 7) / 8 * 8;
    const int64_t lo = static_cast<int64_t>(c.rank) * per;
    int64_t hi = lo + per;
    if (hi > c.n) hi = c.n;
    const int64_t items = hi > lo ? (hi - lo + 3) / 4 : 0;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kNThreads;
    const f32x4 zero{0.f, 0.f, 0.f, 0.f};
    const float gs = c.gscale;
    for (int64_t it0 = static_cast<int64_t>(blockIdx.x) * kNThreads + threadIdx.x; it0 < items;
         it0 += stride * kNRemote) {
        float g[kNRemote][4];
#pragma unroll
        for (int u = 0; u < kNRemote; ++u) {
            const int64_t it = it0 + u * stride;
            if (it < items) mm_ld_reduce_f32x4(mc_g + lo + it * 4, g[u]);
        }
#pragma unroll
        for (int u = 0; u < kNRemote; ++u) {
            const int64_t it = it0 + u * stride;
            if (it >= items) break;
            const int64_t e = lo + it * 4;
            f32x4 vp = ld_stream(reinterpret_cast<const f32x4*>(p_ + e));
            f32x4 a0 = NS > 0 ? ld_stream(reinterpret_cast<const f32x4*>(s0_ + e)) : zero;
            f32x4 a1 = NS > 1 ? ld_stream(reinterpret_cast<const f32x4*>(s1_ + e)) : zero;
            f32x4 a2 = NS > 2 ? ld_stream(reinterpret_cast<const f32x4*>(s2_ + e)) : zero;
            rule(vp.x, g[u][0] * gs, a0.x, a1.x, a2.x);
            rule(vp.y, g[u][1] * gs, a0.y, a1.y, a2.y);
            rule(vp.z, g[u][2] * gs, a0.z, a1.z, a2.z);
            rule(vp.w, g[u][3] * gs, a0.w, a1.w, a2.w);
            mm_st_b128(mc_p + e, __float_as_uint(vp.x), __float_as_uint(vp.y), __float_as_uint(vp.z),
                       __float_as_uint(vp.w));
            if (NS > 0) st_stream(reinterpret_cast<f32x4*>(s0_ + e), a0);
            if (NS > 1) st_stream(reinterpret_cast<f32x4*>(s1_ + e), a1);
            if (NS > 2) st_stream(reinterpret_cast<f32x4*>(s2_ + e), a2);
        }
    }
    if (c.sync_inside) kernel_exit_barrier(c.pads, c.rank, c.world, c.pad_base, c.local);
    else __threadfence_system();                                  // my multimem stores before the grid ends
}

template <typename Rule, int NS>
static int launch_nvls(const Rule& rule, float* p, float* s0, float* s1, float* s2, const void* mc_g,
                       void* mc_out, int64_t n, int rank, int world, void* const* pads, int pad_base,
                       void* local_scratch, int max_blocks, double gscale, const float* dyn, int g_dtype,
                       int flags, void* stream, const char* name) {
    FRL_REQUIRE(p && mc_g && mc_out && pads, FRL_E_ARG, "%s: null pointer", name);
    FRL_REQUIRE(world >= 2 && world <= 32 && rank >= 0 && rank < world, FRL_E_ARG, "%s: rank/world", name);
    FRL_REQUIRE(n >= 0 && n % 8 == 0, FRL_E_ARG, "%s: bucket size must be a multiple of 8 elements", name);
    FRL_REQUIRE(g_dtype == FRL_F32 || g_dtype == FRL_BF16, FRL_E_DTYPE, "%s: g_dtype", name);
    FRL_REQUIRE(aligned16(p) && aligned16(s0) && aligned16(s1) && aligned16(s2) && aligned16(mc_g) &&
                aligned16(mc_out), FRL_E_ALIGN, "%s: 16-byte alignment", name);
    FRL_REQUIRE(max_blocks >= 1 && max_blocks <= 1024 && local_scratch, FRL_E_ARG,
                "%s: max_blocks in 1..1024 and a local scratch are required", name);
    NvlsCommon c{reinterpret_cast<uint32_t* const*>(pads), static_cast<uint32_t*>(local_scratch), rank,
                 world, pad_base, (flags & FRL_NVLS_EXTERNAL_SYNC) ? 0 : 1, n,
                 static_cast<float>(gscale), dyn};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // remote loads in flight per thread: FRL_B200_NVLS_INFLIGHT (4 | 8 | 16), default by world size
    static const int env_depth = [] {
        const char* e = getenv("FRL_B200_NVLS_INFLIGHT");
        return e ? atoi(e) : 0;
    }();
    const int depth = env_depth > 0 ? env_depth : 4;   // measured at world 2: 4 -> 1.170, 8 -> 1.190, 16 -> 1.198 ms/step
    // the grid must be identical on every rank: it depends on arguments only
#define FRL_NV(NR)                                                                                    \
    do {                                                                                              \
        if (g_dtype == FRL_BF16)                                                                      \
            nvls_update_bf16<Rule, NS, NR><<<max_blocks, kNThreads, 0, st>>>(                         \
                p, s0, s1, s2, static_cast<const __nv_bfloat16*>(mc_g), static_cast<__nv_bfloat16*>(mc_out), rule, c); \
        else                                                                                          \
            nvls_update_f32<Rule, NS, NR><<<max_blocks, kNThreads, 0, st>>>(                          \
                p, s0, s1, s2, static_cast<const float*>(mc_g), static_cast<float*>(mc_out), rule, c); \
    } while (0)
    if (depth >= 16) FRL_NV(16);
    else if (depth >= 8) FRL_NV(8);
    else FRL_NV(4);
#undef FRL_NV
    return after_launch(name);
}

}  // namespace frl

using namespace frl;

extern "C" int frl_nvls_sgd(float* p, float* buf, const void* mc_g, void* mc_out, int64_t n, int rank,
                            int world, void* const* signal_pads_dev, int pad_base, void* local_scratch,
                            int max_blocks, double lr, double mu, double dampening, double wd, double grad_scale,
                            const float* dyn, int first_step, int g_dtype, int flags, void* stream) {
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_nvls_sgd: momentum needs buf");
    const SgdRule r = make_sgd_rule(lr, mu, dampening, wd, first_step);
    if (mu != 0.0)
        return launch_nvls<SgdRule, 1>(r, p, buf, nullptr, nullptr, mc_g, mc_out, n, rank, world,
                                       signal_pads_dev, pad_base, local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_sgd");
    return launch_nvls<SgdRule, 0>(r, p, nullptr, nullptr, nullptr, mc_g, mc_out, n, rank, world,
                                   signal_pads_dev, pad_base, local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream,
                                   "frl_nvls_sgd");
}

extern "C" int frl_nvls_adam(float* p, float* m, float* v, float* vmax, const void* mc_g, void* mc_out,
                             int64_t n, int rank, int world, void* const* signal_pads_dev, int pad_base,
                             void* local_scratch, int max_blocks, double lr, double beta1, double beta2, double eps, double wd,
                             int64_t step, double grad_scale, const float* dyn, int g_dtype, int flags, void* stream) {
    FRL_REQUIRE(m && v && step >= 1, FRL_E_ARG, "frl_nvls_adam: state/step");
    if (vmax)
        return launch_nvls<AdamRule<true>, 3>(make_adam_rule<true>(lr, beta1, beta2, eps, wd, step), p, m, v,
                                              vmax, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                              local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_adam");
    return launch_nvls<AdamRule<false>, 2>(make_adam_rule<false>(lr, beta1, beta2, eps, wd, step), p, m, v,
                                           nullptr, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                           local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_adam");
}

extern "C" int frl_nvls_adamw(float* p, float* m, float* v, float* vmax, const void* mc_g, void* mc_out,
                              int64_t n, int rank, int world, void* const* signal_pads_dev, int pad_base,
                              void* local_scratch, int max_blocks, double lr, double beta1, double beta2, double eps, double wd,
                              int64_t step, double grad_scale, const float* dyn, int g_dtype, int flags, void* stream) {
    FRL_REQUIRE(m && v && step >= 1, FRL_E_ARG, "frl_nvls_adamw: state/step");
    if (vmax)
        return launch_nvls<AdamRule<true, true>, 3>(make_adam_rule<true, true>(lr, beta1, beta2, eps, wd, step), p, m, v,
                                                    vmax, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                                    local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_adamw");
    return launch_nvls<AdamRule<false, true>, 2>(make_adam_rule<false, true>(lr, beta1, beta2, eps, wd, step), p, m, v,
                                                 nullptr, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                                 local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_adamw");
}

extern "C" int frl_nvls_rmsprop(float* p, float* sq, float* buf, const void* mc_g, void* mc_out, int64_t n,
                                int rank, int world, void* const* signal_pads_dev, int pad_base,
                                void* local_scratch, int max_blocks, double lr, double alpha, double eps, double wd, double mu,
                                double grad_scale, const float* dyn, int g_dtype, int flags, void* stream) {
    FRL_REQUIRE(sq, FRL_E_ARG, "frl_nvls_rmsprop: null sq");
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_nvls_rmsprop: momentum needs buf");
    if (mu != 0.0)
        return launch_nvls<RmspropRule<true>, 2>(make_rmsprop_rule<true>(lr, alpha, eps, wd, mu), p, sq, buf,
                                                 nullptr, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                                 local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_rmsprop");
    return launch_nvls<RmspropRule<false>, 1>(make_rmsprop_rule<false>(lr, alpha, eps, wd, mu), p, sq, nullptr,
                                              nullptr, mc_g, mc_out, n, rank, world, signal_pads_dev, pad_base,
                                              local_scratch, max_blocks, grad_scale, dyn, g_dtype, flags, stream, "frl_nvls_rmsprop");
}


// Cross-GPU rendezvous as its own 1-CTA launch.  With FRL_NVLS_EXTERNAL_SYNC the bucket sequence on
// the side stream is  barrier(slot 0) -> frl_nvls_* -> barrier(slot 1): while a rank waits for
// slower peers only one warp is resident, instead of a whole grid of spinning CTAs that keeps the
// backward GEMMs of this rank off the SMs; the update kernel itself then never waits.
namespace frl {
__global__ void __launch_bounds__(32)
nvls_barrier_kernel(uint32_t* const* pads, int rank, int world, int base) {
    meet_peers_block0(pads, rank, world, base);
}
}  // namespace frl

extern "C" int frl_nvls_barrier(void* const* signal_pads_dev, int rank, int world, int pad_slot,
                                void* stream) {
    FRL_REQUIRE(signal_pads_dev, FRL_E_ARG, "frl_nvls_barrier: null pads");
    FRL_REQUIRE(world >= 2 && world <= 32 && rank >= 0 && rank < world, FRL_E_ARG, "frl_nvls_barrier: rank/world");
    FRL_REQUIRE(pad_slot >= 0 && pad_slot < 8, FRL_E_ARG, "frl_nvls_barrier: pad_slot in 0..7");
    frl::nvls_barrier_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<uint32_t* const*>(signal_pads_dev), rank, world, pad_slot * 32);
    return frl::after_launch("frl_nvls_barrier");
}
