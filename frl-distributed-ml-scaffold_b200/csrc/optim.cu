// K2 — fused optimizer update over a flat bucket of the parameter arena (sm_100a).
//
// One streaming pass: read the (already all-reduced) gradient bucket, the fp32 master weights
// and the optimizer state; apply torch 2.11's update rule in fp32; write master, state and —
// in bf16 mode — the bf16 shadow weights the next forward reads.  Gradient scaling (1/world,
// clip coefficient) is folded into the gradient read, so the flatten / pre-divide / copy-out
// passes of the stock DDP reducer do not exist here.
//
// HBM-bound: 20 B/param (SGD-momentum), 28 B/param (Adam, RMSprop+momentum), 36 B/param
// (Adam+amsgrad); +2 B with a bf16 shadow, -2 B with a bf16 gradient.
//
// Layout: every thread owns 4 consecutive elements per item, so fp32 arrays move as fully
// coalesced 16-byte accesses (bf16 as 8-byte).  Each thread issues the loads of UNROLL items
// before the first use (UNROLL * (2 + NSTATE) independent 128-bit loads in flight), which is
// what keeps ~100 KB per SM outstanding — the amount Little's law asks for at ~6.5 TB/s.
#include "frl_common.cuh"
#include "optim_rules.cuh"

namespace frl {

constexpr int kThreads = 256;
constexpr int kUnroll = 4;
constexpr int kTileVec = kThreads * kUnroll;   // vec4 items per tile

// ---- gradient vector load (scaled, as fp32) ---------------------------------------------------
__device__ __forceinline__ f32x4 load_grad4(const f32x4* g, int64_t i) { return ld_stream_ro(g + i); }
__device__ __forceinline__ f32x4 load_grad4(const bf16x4* g, int64_t i) {
    const bf16x4 r = ld_stream_ro(g + i);
    return f32x4{bf16lo(r.a), bf16hi(r.a), bf16lo(r.b), bf16hi(r.b)};
}
__device__ __forceinline__ float load_grad1(const f32x4* g, int64_t e) {
    return reinterpret_cast<const float*>(g)[e];
}
__device__ __forceinline__ float load_grad1(const bf16x4* g, int64_t e) {
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g)[e]);
}

template <typename Rule>
__device__ __forceinline__ void apply4(const Rule& r, f32x4& p, const f32x4& g, float gs,
                                       f32x4& s0, f32x4& s1, f32x4& s2) {
    r(p.x, g.x * gs, s0.x, s1.x, s2.x);
    r(p.y, g.y * gs, s0.y, s1.y, s2.y);
    r(p.z, g.z * gs, s0.z, s1.z, s2.z);
    r(p.w, g.w * gs, s0.w, s1.w, s2.w);
}

// NS = number of state arrays actually touched (0..3).
template <typename Rule, typename GVec, int NS, bool HAS_LP>
__global__ void __launch_bounds__(kThreads)
update_kernel(float* __restrict__ p_, const GVec* __restrict__ g, float* __restrict__ s0_,
              float* __restrict__ s1_, float* __restrict__ s2_, bf16x4* __restrict__ lp,
              int64_t n, Rule rule, float gscale, const float* __restrict__ gscale_dev,
              const float* __restrict__ dyn) {
    if (dyn) rule.patch(dyn);      // per-step scalars from device memory (CUDA-graph replays)
    f32x4* p = reinterpret_cast<f32x4*>(p_);
    f32x4* s0 = reinterpret_cast<f32x4*>(s0_);
    f32x4* s1 = reinterpret_cast<f32x4*>(s1_);
    f32x4* s2 = reinterpret_cast<f32x4*>(s2_);
    const float gs = gscale_dev ? gscale * __ldg(gscale_dev) : gscale;
    const int64_t n_vec = n >> 2;
    const int64_t n_tiles = (n_vec + kTileVec - 1) / kTileVec;
    const f32x4 zero{0.f, 0.f, 0.f, 0.f};

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t base = tile * kTileVec + threadIdx.x;
        f32x4 vp[kUnroll], vg[kUnroll], a0[kUnroll], a1[kUnroll], a2[kUnroll];
        if (base + (kUnroll - 1) * kThreads < n_vec) {      // whole tile in range for this thread
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                const int64_t i = base + j * kThreads;
                vg[j] = load_grad4(g, i);
                vp[j] = ld_stream(p + i);
                a0[j] = NS > 0 ? ld_stream(s0 + i) : zero;
                a1[j] = NS > 1 ? ld_stream(s1 + i) : zero;
                a2[j] = NS > 2 ? ld_stream(s2 + i) : zero;
            }
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                const int64_t i = base + j * kThreads;
                apply4(rule, vp[j], vg[j], gs, a0[j], a1[j], a2[j]);
                st_stream(p + i, vp[j]);
                if (NS > 0) st_stream(s0 + i, a0[j]);
                if (NS > 1) st_stream(s1 + i, a1[j]);
                if (NS > 2) st_stream(s2 + i, a2[j]);
                if (HAS_LP) st_stream(lp + i, bf16x4{pack_bf16(vp[j].x, vp[j].y), pack_bf16(vp[j].z, vp[j].w)});
            }
        } else {
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                const int64_t i = base + j * kThreads;
                if (i >= n_vec) break;
                f32x4 qg = load_grad4(g, i), qp = ld_stream(p + i);
                f32x4 q0 = NS > 0 ? ld_stream(s0 + i) : zero;
                f32x4 q1 = NS > 1 ? ld_stream(s1 + i) : zero;
                f32x4 q2 = NS > 2 ? ld_stream(s2 + i) : zero;
                apply4(rule, qp, qg, gs, q0, q1, q2);
                st_stream(p + i, qp);
                if (NS > 0) st_stream(s0 + i, q0);
                if (NS > 1) st_stream(s1 + i, q1);
                if (NS > 2) st_stream(s2 + i, q2);
                if (HAS_LP) st_stream(lp + i, bf16x4{pack_bf16(qp.x, qp.y), pack_bf16(qp.z, qp.w)});
            }
        }
    }
    // scalar tail: n % 4 trailing elements
    const int64_t tail0 = n_vec << 2;
    if (blockIdx.x == 0 && tail0 + threadIdx.x < n) {
        const int64_t e = tail0 + threadIdx.x;
        float pe = p_[e], d0 = 0.f, d1 = 0.f, d2 = 0.f;
        if (NS > 0) d0 = s0_[e];
        if (NS > 1) d1 = s1_[e];
        if (NS > 2) d2 = s2_[e];
        rule(pe, load_grad1(g, e) * gs, d0, d1, d2);
        p_[e] = pe;
        if (NS > 0) s0_[e] = d0;
        if (NS > 1) s1_[e] = d1;
        if (NS > 2) s2_[e] = d2;
        if (HAS_LP) reinterpret_cast<__nv_bfloat16*>(lp)[e] = __float2bfloat16_rn(pe);
    }
}

// grid: one resident wave — (CTAs that fit per SM for this instantiation) x SM count, capped by
// the number of tiles; the grid-stride loop walks the rest, so there is no partial last wave.
template <typename K>
static int grid_for(K kernel, int64_t n) {
    static int occ = 0;            // per template instantiation
    if (occ == 0) {
        int o = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kernel, kThreads, 0) != cudaSuccess || o < 1) o = 2;
        occ = o;
    }
    const int64_t tiles = (n / 4 + kTileVec - 1) / kTileVec;
    const int64_t cap = static_cast<int64_t>(sm_count()) * occ;
    int64_t g = tiles < cap ? tiles : cap;
    return g < 1 ? 1 : static_cast<int>(g);
}

template <typename Rule, int NS>
static int launch_update(const Rule& rule, float* p, const void* g, float* s0, float* s1, float* s2,
                         void* p_lp, int64_t n, float gscale, const float* gscale_dev,
                         const float* dyn, int g_dtype, cudaStream_t st, const char* name) {
    FRL_REQUIRE(n >= 0, FRL_E_ARG, "%s: n < 0", name);
    if (n == 0) return 0;
    FRL_REQUIRE(p && g, FRL_E_ARG, "%s: null p/g", name);
    FRL_REQUIRE(g_dtype == FRL_F32 || g_dtype == FRL_BF16, FRL_E_DTYPE, "%s: g_dtype %d", name, g_dtype);
    FRL_REQUIRE(aligned16(p) && aligned16(g) && aligned16(s0) && aligned16(s1) && aligned16(s2) &&
                aligned16(p_lp), FRL_E_ALIGN, "%s: arrays must be 16-byte aligned", name);
    bf16x4* lp = static_cast<bf16x4*>(p_lp);
#define FRL_LAUNCH(GV, LP)                                                                      \
    update_kernel<Rule, GV, NS, LP><<<grid_for(update_kernel<Rule, GV, NS, LP>, n), kThreads, 0, st>>>( \
        p, static_cast<const GV*>(g), s0, s1, s2, lp, n, rule, gscale, gscale_dev, dyn)
    if (g_dtype == FRL_F32) { if (lp) FRL_LAUNCH(f32x4, true); else FRL_LAUNCH(f32x4, false); }
    else                    { if (lp) FRL_LAUNCH(bf16x4, true); else FRL_LAUNCH(bf16x4, false); }
#undef FRL_LAUNCH
    return after_launch(name);
}


// =============================================================================================
// K2-mt / K1 — multi-tensor forms: gradients read in place from wherever autograd produced them
// =============================================================================================
// Convolution and normalisation layers hand their parameter gradients to autograd as freshly
// allocated tensors (cuDNN writes them; there is no `out=`).  The stock pipeline then copies every
// one of them into a DDP bucket and back (reference solver.py:287-289 -> torch Reducer: +16 B per
// parameter and a copy launch per tensor).  Here a SEGMENT TABLE in device memory
// (frl_grad_seg: gradient pointer + dtype + arena offset + length per parameter tensor) lets
//   * frl_*_mt        : the fused update read each gradient where it lies (1 GPU: the flatten
//                       pass does not exist at all, the arena's `grad` vector is not touched);
//   * frl_flatten_grads: ONE launch per bucket gather the bucket's gradients into the arena slice
//                       NCCL / the NVLS kernel reduce (world > 1: copy-in only, cast and pre-scale
//                       folded in, no copy-out, no per-tensor launches).
// Work is cut into tiles of kTileElems arena elements that never straddle a segment;
// tile_prefix[s] = first tile of segment s (n_segs + 1 entries), tile_seg[t] = segment of tile t
// (both built once on the host: sizes never change).  Interior tiles run the flat kernel's body;
// only the last tile of a tensor is bounds-checked.
constexpr int kTileElems = kTileVec * 4;

struct SegView {
    const void* g;
    int64_t arena_off, numel;
    int g_dtype;
    int64_t t_in;      // tile index inside the segment
};

// tile -> segment through a per-tile int32 map built once on the host (sizes never change): one
// L2-resident 4-byte read per 16 KB+ of streamed data
__device__ __forceinline__ SegView find_segment(const frl_grad_seg* __restrict__ segs,
                                                const int64_t* __restrict__ tile_prefix,
                                                const int32_t* __restrict__ tile_seg, int64_t tile) {
    const int si = __ldg(tile_seg + tile);
    SegView v;
    v.g = segs[si].g;
    v.arena_off = segs[si].arena_off;
    v.numel = segs[si].numel;
    v.g_dtype = segs[si].g_dtype;
    v.t_in = tile - __ldg(tile_prefix + si);
    return v;
}

// 4 consecutive gradient elements starting at element e of a segment, zero-filled past its end
__device__ __forceinline__ f32x4 seg_load4(const SegView& sv, int64_t e) {
    if (e + 4 <= sv.numel) {
        if (sv.g_dtype == FRL_F32) return ld_stream_ro(reinterpret_cast<const f32x4*>(static_cast<const float*>(sv.g) + e));
        const bf16x4 r = ld_stream_ro(reinterpret_cast<const bf16x4*>(static_cast<const __nv_bfloat16*>(sv.g) + e));
        return f32x4{bf16lo(r.a), bf16hi(r.a), bf16lo(r.b), bf16hi(r.b)};
    }
    float t[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (e + k < sv.numel)
            t[k] = sv.g_dtype == FRL_F32 ? static_cast<const float*>(sv.g)[e + k]
                                         : __bfloat162float(static_cast<const __nv_bfloat16*>(sv.g)[e + k]);
    return f32x4{t[0], t[1], t[2], t[3]};
}

// interior tile (every vector of the tile lies inside the gradient tensor): the flat kernel's body
template <typename Rule, typename GVec, int NS, bool HAS_LP>
__device__ __forceinline__ void mt_full_tile(const Rule& rule, float gs, f32x4* p, f32x4* s0, f32x4* s1,
                                             f32x4* s2, bf16x4* lp, const GVec* g, int64_t a0, int64_t v0) {
    const f32x4 zero{0.f, 0.f, 0.f, 0.f};
    f32x4 vp[kUnroll], vg[kUnroll], a_0[kUnroll], a_1[kUnroll], a_2[kUnroll];
#pragma unroll
    for (int j = 0; j < kUnroll; ++j) {
        const int64_t v = v0 + j * kThreads, i = a0 + v;
        vg[j] = load_grad4(g, v);
        vp[j] = ld_stream(p + i);
        a_0[j] = NS > 0 ? ld_stream(s0 + i) : zero;
        a_1[j] = NS > 1 ? ld_stream(s1 + i) : zero;
        a_2[j] = NS > 2 ? ld_stream(s2 + i) : zero;
    }
#pragma unroll
    for (int j = 0; j < kUnroll; ++j) {
        const int64_t i = a0 + v0 + j * kThreads;
        apply4(rule, vp[j], vg[j], gs, a_0[j], a_1[j], a_2[j]);
        st_stream(p + i, vp[j]);
        if (NS > 0) st_stream(s0 + i, a_0[j]);
        if (NS > 1) st_stream(s1 + i, a_1[j]);
        if (NS > 2) st_stream(s2 + i, a_2[j]);
        if (HAS_LP) st_stream(lp + i, bf16x4{pack_bf16(vp[j].x, vp[j].y), pack_bf16(vp[j].z, vp[j].w)});
    }
}

template <typename Rule, int NS, bool HAS_LP>
__global__ void __launch_bounds__(kThreads)
update_mt_kernel(float* __restrict__ p_, float* __restrict__ s0_, float* __restrict__ s1_,
                 float* __restrict__ s2_, bf16x4* __restrict__ lp,
                 const frl_grad_seg* __restrict__ segs, const int64_t* __restrict__ tile_prefix,
                 const int32_t* __restrict__ tile_seg, int64_t n_tiles, Rule rule, float gscale,
                 const float* __restrict__ gscale_dev, const float* __restrict__ dyn) {
    if (dyn) rule.patch(dyn);
    f32x4* p = reinterpret_cast<f32x4*>(p_);
    f32x4* s0 = reinterpret_cast<f32x4*>(s0_);
    f32x4* s1 = reinterpret_cast<f32x4*>(s1_);
    f32x4* s2 = reinterpret_cast<f32x4*>(s2_);
    const float gs = gscale_dev ? gscale * __ldg(gscale_dev) : gscale;
    const f32x4 zero{0.f, 0.f, 0.f, 0.f};
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const SegView sv = find_segment(segs, tile_prefix, tile_seg, tile);
        const int64_t v0 = sv.t_in * kTileVec + threadIdx.x;      // vec4 index inside the segment
        const int64_t a0 = sv.arena_off >> 2;                     // vec4 index of the segment in the arena
        if ((sv.t_in + 1) * kTileVec <= (sv.numel >> 2)) {        // CTA-uniform: interior tile
            if (sv.g_dtype == FRL_F32)
                mt_full_tile<Rule, f32x4, NS, HAS_LP>(rule, gs, p, s0, s1, s2, lp,
                                                      static_cast<const f32x4*>(sv.g), a0, v0);
            else
                mt_full_tile<Rule, bf16x4, NS, HAS_LP>(rule, gs, p, s0, s1, s2, lp,
                                                       static_cast<const bf16x4*>(sv.g), a0, v0);
            continue;
        }
        // last tile of a segment (or a small tensor): bounds-checked, element-wise at the very end
        const int64_t seg_vec = (sv.numel + 3) >> 2;              // arena slices are padded to 8
#pragma unroll 1
        for (int j = 0; j < kUnroll; ++j) {
            const int64_t v = v0 + j * kThreads;
            if (v >= seg_vec) break;
            const int64_t i = a0 + v;
            f32x4 qg = seg_load4(sv, v << 2), qp = ld_stream(p + i);
            f32x4 q0 = NS > 0 ? ld_stream(s0 + i) : zero;
            f32x4 q1 = NS > 1 ? ld_stream(s1 + i) : zero;
            f32x4 q2 = NS > 2 ? ld_stream(s2 + i) : zero;
            apply4(rule, qp, qg, gs, q0, q1, q2);
            st_stream(p + i, qp);
            if (NS > 0) st_stream(s0 + i, q0);
            if (NS > 1) st_stream(s1 + i, q1);
            if (NS > 2) st_stream(s2 + i, q2);
            if (HAS_LP) st_stream(lp + i, bf16x4{pack_bf16(qp.x, qp.y), pack_bf16(qp.z, qp.w)});
        }
    }
}

template <typename DVec>
__device__ __forceinline__ void store_flat4(DVec* dst, int64_t i, const f32x4& v);
template <> __device__ __forceinline__ void store_flat4<f32x4>(f32x4* dst, int64_t i, const f32x4& v) {
    st_stream(dst + i, v);
}
template <> __device__ __forceinline__ void store_flat4<bf16x4>(bf16x4* dst, int64_t i, const f32x4& v) {
    st_stream(dst + i, bf16x4{pack_bf16(v.x, v.y), pack_bf16(v.z, v.w)});
}

template <typename DVec>
__global__ void __launch_bounds__(kThreads)
flatten_kernel(DVec* __restrict__ dst, const frl_grad_seg* __restrict__ segs,
               const int64_t* __restrict__ tile_prefix, const int32_t* __restrict__ tile_seg,
               int64_t n_tiles, float scale) {
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const SegView sv = find_segment(segs, tile_prefix, tile_seg, tile);
        const int64_t seg_vec = (sv.numel + 3) >> 2;
        const int64_t v0 = sv.t_in * kTileVec + threadIdx.x;
        const int64_t a0 = sv.arena_off >> 2;
        f32x4 vg[kUnroll];
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const int64_t v = v0 + j * kThreads;
            if (v < seg_vec) vg[j] = seg_load4(sv, v << 2);
        }
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const int64_t v = v0 + j * kThreads;
            if (v >= seg_vec) break;
            f32x4 q = vg[j];
            if (scale != 1.f) { q.x *= scale; q.y *= scale; q.z *= scale; q.w *= scale; }
            store_flat4<DVec>(dst, a0 + v, q);
        }
    }
}

template <typename K>
static int grid_for_tiles(K kernel, int64_t n_tiles) {
    static int occ = 0;
    if (occ == 0) {
        int o = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kernel, kThreads, 0) != cudaSuccess || o < 1) o = 2;
        occ = o;
    }
    const int64_t cap = static_cast<int64_t>(sm_count()) * occ;
    const int64_t g = n_tiles < cap ? n_tiles : cap;
    return g < 1 ? 1 : static_cast<int>(g);
}

template <typename Rule, int NS>
static int launch_update_mt(const Rule& rule, float* p, float* s0, float* s1, float* s2, void* p_lp,
                            const frl_grad_seg* segs, const int64_t* tile_prefix, const int32_t* tile_seg,
                            int64_t n_tiles, float gscale, const float* gscale_dev, const float* dyn,
                            cudaStream_t st, const char* name) {
    FRL_REQUIRE(n_tiles >= 0, FRL_E_ARG, "%s: negative tile count", name);
    if (n_tiles == 0) return 0;
    FRL_REQUIRE(p && segs && tile_prefix && tile_seg, FRL_E_ARG, "%s: null p/segs/tile_prefix/tile_seg", name);
    FRL_REQUIRE(aligned16(p) && aligned16(s0) && aligned16(s1) && aligned16(s2) && aligned16(p_lp),
                FRL_E_ALIGN, "%s: arrays must be 16-byte aligned", name);
    bf16x4* lp = static_cast<bf16x4*>(p_lp);
    if (lp)
        update_mt_kernel<Rule, NS, true><<<grid_for_tiles(update_mt_kernel<Rule, NS, true>, n_tiles), kThreads, 0, st>>>(
            p, s0, s1, s2, lp, segs, tile_prefix, tile_seg, n_tiles, rule, gscale, gscale_dev, dyn);
    else
        update_mt_kernel<Rule, NS, false><<<grid_for_tiles(update_mt_kernel<Rule, NS, false>, n_tiles), kThreads, 0, st>>>(
            p, s0, s1, s2, lp, segs, tile_prefix, tile_seg, n_tiles, rule, gscale, gscale_dev, dyn);
    return after_launch(name);
}

}  // namespace frl

using namespace frl;

extern "C" int frl_sgd_momentum(float* p, const void* g, float* buf, void* p_lp, int64_t n,
                                double lr, double mu, double dampening, double wd,
                                double grad_scale, const float* grad_scale_dev,
                                const float* dyn, int first_step, int g_dtype, void* stream) {
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_sgd_momentum: momentum needs buf");
    SgdRule r{static_cast<float>(-lr), static_cast<float>(mu), static_cast<float>(1.0 - dampening),
              static_cast<float>(wd), first_step ? 1 : 0, (mu != 0.0) ? 1 : 0};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float gs = static_cast<float>(grad_scale);
    if (mu != 0.0)
        return launch_update<SgdRule, 1>(r, p, g, buf, nullptr, nullptr, p_lp, n, gs,
                                         grad_scale_dev, dyn, g_dtype, st, "frl_sgd_momentum");
    return launch_update<SgdRule, 0>(r, p, g, nullptr, nullptr, nullptr, p_lp, n, gs,
                                     grad_scale_dev, dyn, g_dtype, st, "frl_sgd_momentum");
}

extern "C" int frl_adam(float* p, const void* g, float* m, float* v, float* vmax, void* p_lp,
                        int64_t n, double lr, double beta1, double beta2, double eps, double wd,
                        int64_t step, double grad_scale, const float* grad_scale_dev,
                        const float* dyn, int g_dtype, void* stream) {
    FRL_REQUIRE(m && v, FRL_E_ARG, "frl_adam: null state");
    FRL_REQUIRE(step >= 1, FRL_E_ARG, "frl_adam: step must be >= 1");
    // bias corrections in double, as torch computes them from Python floats
    const double bc1 = 1.0 - pow(beta1, static_cast<double>(step));
    const double bc2 = 1.0 - pow(beta2, static_cast<double>(step));
    const float neg_step = static_cast<float>(-(lr / bc1));
    const float bc2s = static_cast<float>(sqrt(bc2));
    const float w1 = static_cast<float>(1.0 - beta1);
    const float w2 = static_cast<float>(1.0 - beta2);
    const float b2 = static_cast<float>(beta2), epsf = static_cast<float>(eps), wdf = static_cast<float>(wd);
    const float gs = static_cast<float>(grad_scale);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (vmax) {
        AdamRule<true> r{w1, b2, w2, epsf, wdf, neg_step, bc2s};
        return launch_update<AdamRule<true>, 3>(r, p, g, m, v, vmax, p_lp, n, gs,
                                                grad_scale_dev, dyn, g_dtype, st, "frl_adam");
    }
    AdamRule<false> r{w1, b2, w2, epsf, wdf, neg_step, bc2s};
    return launch_update<AdamRule<false>, 2>(r, p, g, m, v, nullptr, p_lp, n, gs,
                                             grad_scale_dev, dyn, g_dtype, st, "frl_adam");
}

// AdamW: the same kernel as frl_adam with the decoupled rule (p *= 1 - lr*wd, g not decayed)
extern "C" int frl_adamw(float* p, const void* g, float* m, float* v, float* vmax, void* p_lp,
                         int64_t n, double lr, double beta1, double beta2, double eps, double wd,
                         int64_t step, double grad_scale, const float* grad_scale_dev,
                         const float* dyn, int g_dtype, void* stream) {
    FRL_REQUIRE(m && v, FRL_E_ARG, "frl_adamw: null state");
    FRL_REQUIRE(step >= 1, FRL_E_ARG, "frl_adamw: step must be >= 1");
    const float gs = static_cast<float>(grad_scale);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (vmax)
        return launch_update<AdamRule<true, true>, 3>(make_adam_rule<true, true>(lr, beta1, beta2, eps, wd, step),
                                                      p, g, m, v, vmax, p_lp, n, gs, grad_scale_dev, dyn,
                                                      g_dtype, st, "frl_adamw");
    return launch_update<AdamRule<false, true>, 2>(make_adam_rule<false, true>(lr, beta1, beta2, eps, wd, step),
                                                   p, g, m, v, nullptr, p_lp, n, gs, grad_scale_dev, dyn,
                                                   g_dtype, st, "frl_adamw");
}

extern "C" int frl_rmsprop(float* p, const void* g, float* sq, float* buf, void* p_lp, int64_t n,
                           double lr, double alpha, double eps, double wd, double mu,
                           double grad_scale, const float* grad_scale_dev, const float* dyn,
                           int g_dtype, void* stream) {
    FRL_REQUIRE(sq, FRL_E_ARG, "frl_rmsprop: null sq");
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_rmsprop: momentum needs buf");
    const float af = static_cast<float>(alpha), oma = static_cast<float>(1.0 - alpha);
    const float epsf = static_cast<float>(eps), wdf = static_cast<float>(wd);
    const float muf = static_cast<float>(mu), nlr = static_cast<float>(-lr);
    const float gs = static_cast<float>(grad_scale);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (mu != 0.0) {
        RmspropRule<true> r{af, oma, epsf, wdf, muf, nlr};
        return launch_update<RmspropRule<true>, 2>(r, p, g, sq, buf, nullptr, p_lp, n, gs,
                                                   grad_scale_dev, dyn, g_dtype, st, "frl_rmsprop");
    }
    RmspropRule<false> r{af, oma, epsf, wdf, muf, nlr};
    return launch_update<RmspropRule<false>, 1>(r, p, g, sq, nullptr, nullptr, p_lp, n, gs,
                                                grad_scale_dev, dyn, g_dtype, st, "frl_rmsprop");
}

// ---- multi-tensor entry points -------------------------------------------------------------------

extern "C" int64_t frl_mt_tile_elems(void) { return kTileElems; }

extern "C" int frl_flatten_grads(const frl_grad_seg* segs_dev, const int64_t* tile_prefix_dev,
                                 const int32_t* tile_seg_dev, int64_t n_tiles, void* arena_grad, int dst_dtype,
                                 double scale, void* stream) {
    FRL_REQUIRE(n_tiles >= 0, FRL_E_ARG, "frl_flatten_grads: negative tile count");
    if (n_tiles == 0) return 0;
    FRL_REQUIRE(segs_dev && tile_prefix_dev && tile_seg_dev && arena_grad, FRL_E_ARG, "frl_flatten_grads: null pointer");
    FRL_REQUIRE(dst_dtype == FRL_F32 || dst_dtype == FRL_BF16, FRL_E_DTYPE, "frl_flatten_grads: dst dtype %d", dst_dtype);
    FRL_REQUIRE(aligned16(arena_grad), FRL_E_ALIGN, "frl_flatten_grads: arena must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float sc = static_cast<float>(scale);
    if (dst_dtype == FRL_F32)
        flatten_kernel<f32x4><<<grid_for_tiles(flatten_kernel<f32x4>, n_tiles), kThreads, 0, st>>>(
            static_cast<f32x4*>(arena_grad), segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, sc);
    else
        flatten_kernel<bf16x4><<<grid_for_tiles(flatten_kernel<bf16x4>, n_tiles), kThreads, 0, st>>>(
            static_cast<bf16x4*>(arena_grad), segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, sc);
    return after_launch("frl_flatten_grads");
}

extern "C" int frl_sgd_momentum_mt(float* p, float* buf, void* p_lp, const frl_grad_seg* segs_dev,
                                   const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles,
                                   double lr, double mu, double dampening, double wd, double grad_scale,
                                   const float* grad_scale_dev, const float* dyn, int first_step, void* stream) {
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_sgd_momentum_mt: momentum needs buf");
    const SgdRule r = make_sgd_rule(lr, mu, dampening, wd, first_step);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float gs = static_cast<float>(grad_scale);
    if (mu != 0.0)
        return launch_update_mt<SgdRule, 1>(r, p, buf, nullptr, nullptr, p_lp, segs_dev, tile_prefix_dev, tile_seg_dev,
                                            n_tiles, gs, grad_scale_dev, dyn, st, "frl_sgd_momentum_mt");
    return launch_update_mt<SgdRule, 0>(r, p, nullptr, nullptr, nullptr, p_lp, segs_dev, tile_prefix_dev, tile_seg_dev,
                                        n_tiles, gs, grad_scale_dev, dyn, st, "frl_sgd_momentum_mt");
}

extern "C" int frl_adam_mt(float* p, float* m, float* v, float* vmax, void* p_lp, const frl_grad_seg* segs_dev,
                           const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double beta1,
                           double beta2, double eps, double wd, int64_t step, double grad_scale,
                           const float* grad_scale_dev, const float* dyn, void* stream) {
    FRL_REQUIRE(m && v, FRL_E_ARG, "frl_adam_mt: null state");
    FRL_REQUIRE(step >= 1, FRL_E_ARG, "frl_adam_mt: step must be >= 1");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float gs = static_cast<float>(grad_scale);
    if (vmax)
        return launch_update_mt<AdamRule<true>, 3>(make_adam_rule<true>(lr, beta1, beta2, eps, wd, step), p, m, v, vmax,
                                                   p_lp, segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, gs,
                                                   grad_scale_dev, dyn, st, "frl_adam_mt");
    return launch_update_mt<AdamRule<false>, 2>(make_adam_rule<false>(lr, beta1, beta2, eps, wd, step), p, m, v, nullptr,
                                                p_lp, segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, gs,
                                                grad_scale_dev, dyn, st, "frl_adam_mt");
}

extern "C" int frl_adamw_mt(float* p, float* m, float* v, float* vmax, void* p_lp, const frl_grad_seg* segs_dev,
                            const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double beta1,
                            double beta2, double eps, double wd, int64_t step, double grad_scale,
                            const float* grad_scale_dev, const float* dyn, void* stream) {
    FRL_REQUIRE(m && v, FRL_E_ARG, "frl_adamw_mt: null state");
    FRL_REQUIRE(step >= 1, FRL_E_ARG, "frl_adamw_mt: step must be >= 1");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float gs = static_cast<float>(grad_scale);
    if (vmax)
        return launch_update_mt<AdamRule<true, true>, 3>(make_adam_rule<true, true>(lr, beta1, beta2, eps, wd, step),
                                                         p, m, v, vmax, p_lp, segs_dev, tile_prefix_dev, tile_seg_dev,
                                                         n_tiles, gs, grad_scale_dev, dyn, st, "frl_adamw_mt");
    return launch_update_mt<AdamRule<false, true>, 2>(make_adam_rule<false, true>(lr, beta1, beta2, eps, wd, step),
                                                      p, m, v, nullptr, p_lp, segs_dev, tile_prefix_dev, tile_seg_dev,
                                                      n_tiles, gs, grad_scale_dev, dyn, st, "frl_adamw_mt");
}

extern "C" int frl_rmsprop_mt(float* p, float* sq, float* buf, void* p_lp, const frl_grad_seg* segs_dev,
                              const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double alpha,
                              double eps, double wd, double mu, double grad_scale, const float* grad_scale_dev,
                              const float* dyn, void* stream) {
    FRL_REQUIRE(sq, FRL_E_ARG, "frl_rmsprop_mt: null sq");
    FRL_REQUIRE(mu == 0.0 || buf != nullptr, FRL_E_ARG, "frl_rmsprop_mt: momentum needs buf");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float gs = static_cast<float>(grad_scale);
    if (mu != 0.0)
        return launch_update_mt<RmspropRule<true>, 2>(make_rmsprop_rule<true>(lr, alpha, eps, wd, mu), p, sq, buf, nullptr,
                                                      p_lp, segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, gs,
                                                      grad_scale_dev, dyn, st, "frl_rmsprop_mt");
    return launch_update_mt<RmspropRule<false>, 1>(make_rmsprop_rule<false>(lr, alpha, eps, wd, mu), p, sq, nullptr, nullptr,
                                                   p_lp, segs_dev, tile_prefix_dev, tile_seg_dev, n_tiles, gs,
                                                   grad_scale_dev, dyn, st, "frl_rmsprop_mt");
}
