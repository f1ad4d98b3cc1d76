// Update rules shared by the single-GPU update kernel (optim.cu) and the fused NVLS
// reduce + update + broadcast kernel (nvls.cu).  Scalar, fp32, torch 2.11 operation order.
#pragma once
#include "frl_common.cuh"

namespace frl {

// ---- update rules (scalar, fp32) ------------------------------------------------------------
struct SgdRule {
    float neg_lr, mu, one_minus_damp, wd;
    int first_step, has_buf;
    static constexpr int kStates = 1;
    __device__ __forceinline__ void patch(const float* dyn) { neg_lr = -__ldg(dyn); }
    __device__ __forceinline__ void operator()(float& p, float g, float& buf, float&, float&) const {
        g = fmaf(wd, p, g);
        if (has_buf) {
            buf = first_step ? g : fmaf(mu, buf, one_minus_damp * g);
            g = buf;
        }
        p = fmaf(neg_lr, g, p);
    }
};

// Adam's moment update and step, shared by the coupled and the decoupled rule:
// m.lerp_(g, 1-beta1) ; v.mul_(beta2).addcmul_(g, g, 1-beta2) ; p.addcdiv_(m, sqrt(v)/bc2_sqrt + eps, -step_size)
template <bool AMSGRAD>
__device__ __forceinline__ void adam_moments_step(float& p, float g, float& m, float& v, float& vmax, float w1,
                                                  float beta2, float w2, float eps, float neg_step_size,
                                                  float bc2_sqrt) {
    m = fmaf(w1, g - m, m);                       // exp_avg.lerp_(g, 1-beta1), weight < 0.5 branch
    v = fmaf(w2 * g, g, v * beta2);               // mul_(beta2).addcmul_(g, g, 1-beta2)
    float vv = v;
    if (AMSGRAD) { vmax = fmaxf(vmax, v); vv = vmax; }
    const float denom = sqrtf(vv) / bc2_sqrt + eps;
    p = fmaf(neg_step_size, m / denom, p);        // addcdiv_(m, denom, -step_size)
}

// torch.optim.Adam: L2 weight decay added to the gradient (DECOUPLED = false).
template <bool AMSGRAD, bool DECOUPLED = false>
struct AdamRule {
    float w1;               // 1 - beta1   (lerp weight)
    float beta2, w2;        // beta2, 1 - beta2
    float eps, wd;
    float neg_step_size;    // -lr / (1 - beta1^t)
    float bc2_sqrt;         // sqrt(1 - beta2^t)
    static constexpr int kStates = AMSGRAD ? 3 : 2;
    __device__ __forceinline__ void patch(const float* dyn) {
        neg_step_size = __ldg(dyn);
        bc2_sqrt = __ldg(dyn + 1);
    }
    __device__ __forceinline__ void operator()(float& p, float g, float& m, float& v, float& vmax) const {
        g = fmaf(wd, p, g);                       // grad.add(param, alpha=weight_decay)
        adam_moments_step<AMSGRAD>(p, g, m, v, vmax, w1, beta2, w2, eps, neg_step_size, bc2_sqrt);
    }
};

// torch.optim.AdamW = Adam(decoupled_weight_decay=True): the weight is scaled by
// keep = 1 - lr*wd first and the gradient is not decayed.  Same state, same bytes moved; `keep`
// sits where the coupled rule keeps `wd`, and changes with lr, so it is dyn[2] under graph replay.
template <bool AMSGRAD>
struct AdamRule<AMSGRAD, true> {
    float w1;
    float beta2, w2;
    float eps, keep;        // keep = fp32(1 - lr * weight_decay), formed in double
    float neg_step_size;
    float bc2_sqrt;
    static constexpr int kStates = AMSGRAD ? 3 : 2;
    __device__ __forceinline__ void patch(const float* dyn) {
        neg_step_size = __ldg(dyn);
        bc2_sqrt = __ldg(dyn + 1);
        keep = __ldg(dyn + 2);
    }
    __device__ __forceinline__ void operator()(float& p, float g, float& m, float& v, float& vmax) const {
        p *= keep;                                // param.mul_(1 - lr * weight_decay)
        adam_moments_step<AMSGRAD>(p, g, m, v, vmax, w1, beta2, w2, eps, neg_step_size, bc2_sqrt);
    }
};

template <bool MOMENTUM>
struct RmspropRule {
    float alpha, one_minus_alpha, eps, wd, mu, neg_lr;
    static constexpr int kStates = MOMENTUM ? 2 : 1;
    __device__ __forceinline__ void patch(const float* dyn) { neg_lr = -__ldg(dyn); }
    __device__ __forceinline__ void operator()(float& p, float g, float& sq, float& buf, float&) const {
        g = fmaf(wd, p, g);
        sq = fmaf(one_minus_alpha * g, g, sq * alpha);
        const float avg = sqrtf(sq) + eps;
        float upd = g / avg;
        if (MOMENTUM) { buf = fmaf(mu, buf, upd); upd = buf; }
        p = fmaf(neg_lr, upd, p);
    }
};


// ---- host-side construction from the double-precision hyper-parameters -----------------------
static inline SgdRule make_sgd_rule(double lr, double mu, double dampening, double wd, int first_step) {
    return SgdRule{static_cast<float>(-lr), static_cast<float>(mu), static_cast<float>(1.0 - dampening),
                   static_cast<float>(wd), first_step ? 1 : 0, (mu != 0.0) ? 1 : 0};
}
template <bool AMS, bool DECOUPLED = false>
static inline AdamRule<AMS, DECOUPLED> make_adam_rule(double lr, double beta1, double beta2, double eps,
                                                      double wd, int64_t step) {
    // bias corrections in double, as torch computes them from Python floats
    const double bc1 = 1.0 - pow(beta1, static_cast<double>(step));
    const double bc2 = 1.0 - pow(beta2, static_cast<double>(step));
    // coupled: wd itself; decoupled: 1 - lr*wd, as torch forms it from Python floats
    const double wd_slot = DECOUPLED ? 1.0 - lr * wd : wd;
    return AdamRule<AMS, DECOUPLED>{static_cast<float>(1.0 - beta1), static_cast<float>(beta2),
                                    static_cast<float>(1.0 - beta2), static_cast<float>(eps),
                                    static_cast<float>(wd_slot), static_cast<float>(-(lr / bc1)),
                                    static_cast<float>(sqrt(bc2))};
}
template <bool MOM>
static inline RmspropRule<MOM> make_rmsprop_rule(double lr, double alpha, double eps, double wd, double mu) {
    return RmspropRule<MOM>{static_cast<float>(alpha), static_cast<float>(1.0 - alpha), static_cast<float>(eps),
                            static_cast<float>(wd), static_cast<float>(mu), static_cast<float>(-lr)};
}

}  // namespace frl
