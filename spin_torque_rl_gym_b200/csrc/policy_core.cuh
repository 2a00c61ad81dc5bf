// policy_core.cuh — per-env arithmetic of K9, the ActorCriticPolicy forward pass (include/stg.h, stg_policy_act_f32 /
// stg_policy_value_f32), shared by policy_kernels.cu and the host build in tests/test_actor_critic_policy.py.
//
// Specification: Stable-Baselines3's ActorCriticPolicy.forward for PPO's MlpPolicy (net_arch pi=[64, 64], vf=[64, 64], tanh)
// with a DiagGaussianDistribution, in float32. Sampling and log-probability follow torch's expression order
// (Normal.rsample: loc + eps * scale; Normal.log_prob: -((value - loc) ** 2) / (2 * var) - log_scale - log(sqrt(2 pi))), every
// product, sum and quotient rounded on its own (Pk<float>, no contraction), so the device and the host give the same bits for
// the same means. The layer products are fma chains in ascending k; their order is the contract, not their rounding.
#pragma once

#include <stdint.h>
#include <math.h>

#include "llgs_core.cuh"
#include "vecnorm_core.cuh"
#include "../../include/stg.h"

namespace stg {

constexpr int kPolObs = STG_POLICY_OBS;
constexpr int kPolHidden = STG_POLICY_HIDDEN;
constexpr float kLogSqrt2Pi = 0.91893853320467274f;   // math.log(math.sqrt(2 * math.pi)), rounded to float32 as torch does

STG_HD float pol_div(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(a, b);
#else
    volatile float r = a / b; return r;
#endif
}

// one output of a dense layer: b, then fma(x[k], W[k * n_out + o], .) for k = 0 .. K-1
STG_HD float pol_dot(const float* x, int K, const float* W, int n_out, int o, float b) {
    float acc = b;
    for (int k = 0; k < K; ++k) acc = fmaf(x[k], W[k * n_out + o], acc);
    return acc;
}

// the two standard normals of env `gid` at noise draw `draw`
STG_HD void pol_eps(uint32_t k0, uint32_t k1, uint64_t gid, uint64_t draw, float& e0, float& e1) {
    uint32_t o[4];
    Philox{k0, k1}((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)draw, (uint32_t)(draw >> 32), o);
    box_muller(o[0], o[1], e0, e1);
}

// Normal.rsample: loc + eps * scale
STG_HD float pol_sample(float mean, float eps, float std) {
    using K = Pk<float>;
    return K::add(mean, K::mul(eps, std));
}

// one dimension of Normal.log_prob(a)
STG_HD float pol_log_prob_term(float a, float mean, float std, float log_scale) {
    using K = Pk<float>;
    const float d = K::add(a, -mean);
    const float var = K::mul(std, std);
    const float q = pol_div(-K::mul(d, d), K::mul(2.0f, var));
    return K::add(K::add(q, -log_scale), -kLogSqrt2Pi);
}

// np.clip to the [-1, 1] Box, then gymnasium's RescaleAction to [lo, hi]
STG_HD float pol_rescale(float a, float lo, float hi) {
    using K = Pk<float>;
    const float c = fminf(fmaxf(a, -1.0f), 1.0f);
    return K::add(lo, K::mul(K::add(hi, -lo), K::mul(K::add(c, 1.0f), 0.5f)));
}

// The whole forward pass of one env on the host (the kernel computes the same chains, tiled): means, value and, when
// `sample`, the action and its log-probability.
STG_HD void pol_forward_row(const float* w, const float* obs, uint32_t k0, uint32_t k1, uint64_t gid, uint64_t draw,
                            bool sample, float mean[2], float action[2], float& value, float& log_prob) {
    float h1[kPolHidden], h2[kPolHidden];
    for (int o = 0; o < kPolHidden; ++o) h1[o] = tanhf(pol_dot(obs, kPolObs, w + STG_POLICY_VF_W1, 64, o, w[STG_POLICY_VF_B1 + o]));
    for (int o = 0; o < kPolHidden; ++o) h2[o] = tanhf(pol_dot(h1, 64, w + STG_POLICY_VF_W2, 64, o, w[STG_POLICY_VF_B2 + o]));
    value = pol_dot(h2, 64, w + STG_POLICY_VAL_W, 1, 0, w[STG_POLICY_VAL_B]);
    for (int o = 0; o < kPolHidden; ++o) h1[o] = tanhf(pol_dot(obs, kPolObs, w + STG_POLICY_PI_W1, 64, o, w[STG_POLICY_PI_B1 + o]));
    for (int o = 0; o < kPolHidden; ++o) h2[o] = tanhf(pol_dot(h1, 64, w + STG_POLICY_PI_W2, 64, o, w[STG_POLICY_PI_B2 + o]));
    for (int d = 0; d < 2; ++d) mean[d] = pol_dot(h2, 64, w + STG_POLICY_ACT_W, 2, d, w[STG_POLICY_ACT_B + d]);
    float e[2] = {0.0f, 0.0f};
    if (sample) pol_eps(k0, k1, gid, draw, e[0], e[1]);
    log_prob = 0.0f;
    for (int d = 0; d < 2; ++d) {
        action[d] = sample ? pol_sample(mean[d], e[d], w[STG_POLICY_STD + d]) : mean[d];
        const float t = pol_log_prob_term(action[d], mean[d], w[STG_POLICY_STD + d], w[STG_POLICY_LOG_SCALE + d]);
        log_prob = d == 0 ? t : Pk<float>::add(log_prob, t);
    }
}

// ---- K10: the per-row arithmetic of SB3's PPO loss and its gradient (include/stg.h, stg_policy_ppo_grad_f32) ------------
// Gradients here are unscaled: the critic's are d/d(.) of sum((return - vpred)^2) / 2, the actor's of -sum(pmin); the fold
// multiplies them by 2 vf_coef / B and 1 / B.

struct PolPpoCoef {
    float clip_range, ratio_lo, ratio_hi, clip_range_vf;
    bool clip_value;
};

// loss sums of a row, in the order of STG_PPO_PART_LOSS
enum { kPpoPmin = 0, kPpoSq = 1, kPpoKl = 2, kPpoClipped = 3 };

constexpr float kEntropyConst = 1.4189385332046727f;  // 0.5 + 0.5 * math.log(2 * math.pi), rounded to float32 as torch does

// torch's (adv - adv.mean()) / (adv.std() + 1e-8) for one row; stats = {mean, std} or NULL
STG_HD float pol_ppo_advantage(float adv, const float* stats) {
    using K = Pk<float>;
    return stats ? pol_div(K::add(adv, -stats[0]), K::add(stats[1], 1e-8f)) : adv;
}

// d tanh: g * (1 - h^2) with h = tanh(.)
STG_HD float pol_dtanh(float g, float h) {
    using K = Pk<float>;
    return K::mul(g, K::add(1.0f, -K::mul(h, h)));
}

// The value part of a row: adds (return - vpred)^2 to sums[kPpoSq] and returns d/d value of half of it
STG_HD float pol_ppo_value_row(float v, float old_v, float ret, const PolPpoCoef& c, double* sums) {
    using K = Pk<float>;
    float vpred = v;
    bool pass = true;
    if (c.clip_value) {
        const float dv = K::add(v, -old_v);
        vpred = K::add(old_v, fminf(fmaxf(dv, -c.clip_range_vf), c.clip_range_vf));
        pass = dv >= -c.clip_range_vf && dv <= c.clip_range_vf;        // clamp passes the gradient on the closed interval
    }
    const float e = K::add(ret, -vpred);
    sums[kPpoSq] += (double)K::mul(e, e);
    return pass ? -e : 0.0f;
}

// The policy part of a row with (normalised) advantage `adv`: adds its pmin, kl and clipped flag to `sums` and returns
// d(-pmin)/d logp
STG_HD float pol_ppo_policy_row(float logp, float old_logp, float adv, const PolPpoCoef& c, double* sums) {
    using K = Pk<float>;
    const float lr = K::add(logp, -old_logp);
    const float r = expf(lr);
    const float cr = fminf(fmaxf(r, c.ratio_lo), c.ratio_hi);
    const float p1 = K::mul(adv, r), p2 = K::mul(adv, cr);
    // torch.min: the whole gradient to the smaller side, half to each at a tie; clamp: on [lo, hi] only
    const float w1 = p1 < p2 ? 1.0f : (p1 == p2 ? 0.5f : 0.0f);
    const float w2 = p2 < p1 ? 1.0f : (p1 == p2 ? 0.5f : 0.0f);
    const bool inside = r >= c.ratio_lo && r <= c.ratio_hi;
    const float dmin = K::add(w1 * adv, inside ? w2 * adv : 0.0f);
    const float rm1 = K::add(r, -1.0f);
    sums[kPpoPmin] += (double)fminf(p1, p2);
    sums[kPpoKl] += (double)K::add(rm1, -lr);
    sums[kPpoClipped] += fabsf(rm1) > c.clip_range ? 1.0 : 0.0;
    return K::mul(-dmin, r);                                              // exp's backward: times its result
}

// The policy part of an A2C row (SB3's A2C.train(): policy_loss = -(A * logp).mean()): adds A * logp to sums[kPpoPmin], so
// that the fold's -sum / B is A2C's policy loss, and returns d(-A logp)/d logp. The kl and clipped sums stay 0.
STG_HD float pol_a2c_policy_row(float logp, float adv, double* sums) {
    sums[kPpoPmin] += (double)Pk<float>::mul(adv, logp);
    return -adv;
}

// the loss a K10 instance computes: SB3's PPO (clipped surrogate, optional value clip) or A2C (plain policy gradient,
// unclipped value MSE; old values and old log-probabilities are not read)
enum PolLoss { kLossPpo = 0, kLossA2c = 1 };

// the policy part of a row under loss L: d(policy loss term)/d logp
template <PolLoss L>
STG_HD float pol_policy_row(float logp, float old_logp, float adv, const PolPpoCoef& c, double* sums) {
    return L == kLossA2c ? pol_a2c_policy_row(logp, adv, sums) : pol_ppo_policy_row(logp, old_logp, adv, c, sums);
}

// Normal.log_prob's backward for a row with d(.)/d logp = gl and scale = STD: d/d mean_d and d/d log_std_d
STG_HD void pol_ppo_gauss_row(float gl, const float act[2], const float mean[2], const float* w, float gm[2], float gs[2]) {
    using K = Pk<float>;
    for (int d = 0; d < 2; ++d) {
        const float std = w[STG_POLICY_STD + d];
        const float dd = K::add(act[d], -mean[d]);
        const float q = pol_div(dd, K::mul(std, std));
        gm[d] = K::mul(gl, q);
        gs[d] = K::mul(gl, K::add(K::mul(q, dd), -1.0f));
    }
}

STG_HD bool pol_ppo_is_critic(int p) {
    return (p >= STG_POLICY_VF_W1 && p < STG_POLICY_ACT_W) || (p >= STG_POLICY_VAL_W && p < STG_POLICY_LOG_STD);
}

// parameter p of the gradient from its unscaled sum over the B rows
STG_HD float pol_ppo_grad_value(int p, double sum, int64_t batch, float ent_coef, float vf_coef) {
    double g = pol_ppo_is_critic(p) ? sum * (2.0 * (double)vf_coef / (double)batch) : sum / (double)batch;
    if (p >= STG_POLICY_LOG_STD && p < STG_POLICY_LOG_STD + 2) g -= (double)ent_coef;   // the entropy term
    return (float)g;
}

// the six losses of include/stg.h from the four loss sums
STG_HD void pol_ppo_losses(const double* sums, const float* w, int64_t batch, float ent_coef, float vf_coef, float* out) {
    const double n = (double)batch;
    double h = 0.0;
    for (int d = 0; d < 2; ++d) h += (double)Pk<float>::add(kEntropyConst, w[STG_POLICY_LOG_SCALE + d]);
    const double pl = -sums[kPpoPmin] / n, vl = sums[kPpoSq] / n, el = -h;
    out[0] = (float)(pl + (double)ent_coef * el + (double)vf_coef * vl);
    out[1] = (float)pl;
    out[2] = (float)vl;
    out[3] = (float)el;
    out[4] = (float)(sums[kPpoKl] / n);
    out[5] = (float)(sums[kPpoClipped] / n);
}

// ---- K12: advantage statistics across ranks (include/stg.h, stg_ppo_adv_moments_f64 / stg_ppo_adv_merge_f32) -------------
// Moment vectors (n, mean, M2) of the raw advantages, merged with K8's Chan update (vecnorm_core.cuh).

// the moments of adv[begin], adv[begin + stride], ... below n: sums shifted by the first of those rows, as K8's threads do
STG_HD void pol_adv_moments(const float* adv, int64_t begin, int64_t n, int64_t stride, double out[3]) {
    double cnt = 0.0, s1 = 0.0, s2 = 0.0;
    const double x0 = begin < n ? (double)adv[begin] : 0.0;
    for (int64_t i = begin; i < n; i += stride) {
        const double d = (double)adv[i] - x0;
        s1 += d;
        s2 += d * d;
        cnt += 1.0;
    }
    out[0] = cnt;
    vn_shifted_to_moments(cnt, x0, s1, s2, out[1], out[2]);
}

// a <- a (+) b, a the left operand
STG_HD void pol_adv_merge(double a[3], const double b[3]) {
    double w, c;
    vn_chan_weights(a[0], b[0], w, c);
    vn_chan_feature(a[1], a[2], b[1], b[2], w, c);
    a[0] = a[0] + b[0];
}

// the fold of stg_ppo_adv_merge_f32: `ranks` moment vectors in rank order, then torch's mean and std (correction 1)
STG_HD void pol_adv_stats(const double* moments, int ranks, float out[2]) {
    double acc[3] = {0.0, 0.0, 0.0};
    for (int r = 0; r < ranks; ++r) pol_adv_merge(acc, moments + 3 * (int64_t)r);
    const double n = acc[0];
    out[0] = n > 0.0 ? (float)acc[1] : NAN;
    out[1] = n > 0.0 ? (float)dsqrt(ddiv(acc[2], dadd(n, -1.0))) : NAN;   // n = 1: 0 / 0
}

// One row's forward pass (K9's chains) and backward pass on the host: adds its unscaled gradient to grad (the d_grad layout)
// and its loss sums to sums. `adv` is already normalised. The kernel computes the same per-row quantities, tiled; its
// weight-gradient sums run over the rows of a tile in FP32 instead of one product per row. With L = kLossA2c, old_value and
// old_logp are not read and c.clip_value must be false.
template <PolLoss L = kLossPpo>
STG_HD void pol_backward_row(const float* w, const float* obs, const float act[2], float old_value, float old_logp, float adv,
                             float ret, const PolPpoCoef& c, double* grad, double* sums) {
    float h1[kPolHidden], h2[kPolHidden], d2[kPolHidden];
    for (int net = 0; net < 2; ++net) {                                   // the critic, then the actor
        const int w1 = net ? STG_POLICY_PI_W1 : STG_POLICY_VF_W1, b1 = net ? STG_POLICY_PI_B1 : STG_POLICY_VF_B1;
        const int w2 = net ? STG_POLICY_PI_W2 : STG_POLICY_VF_W2, b2 = net ? STG_POLICY_PI_B2 : STG_POLICY_VF_B2;
        for (int o = 0; o < kPolHidden; ++o) h1[o] = tanhf(pol_dot(obs, kPolObs, w + w1, 64, o, w[b1 + o]));
        for (int o = 0; o < kPolHidden; ++o) h2[o] = tanhf(pol_dot(h1, 64, w + w2, 64, o, w[b2 + o]));
        if (net == 0) {
            const float v = pol_dot(h2, 64, w + STG_POLICY_VAL_W, 1, 0, w[STG_POLICY_VAL_B]);
            const float gv = pol_ppo_value_row(v, old_value, ret, c, sums);
            for (int k = 0; k < kPolHidden; ++k) {
                grad[STG_POLICY_VAL_W + k] += (double)h2[k] * gv;
                d2[k] = pol_dtanh(Pk<float>::mul(w[STG_POLICY_VAL_W + k], gv), h2[k]);
            }
            grad[STG_POLICY_VAL_B] += gv;
        } else {
            float mean[2], gm[2], gs[2], logp = 0.0f;
            for (int d = 0; d < 2; ++d) {
                mean[d] = pol_dot(h2, 64, w + STG_POLICY_ACT_W, 2, d, w[STG_POLICY_ACT_B + d]);
                const float t = pol_log_prob_term(act[d], mean[d], w[STG_POLICY_STD + d], w[STG_POLICY_LOG_SCALE + d]);
                logp = d == 0 ? t : Pk<float>::add(logp, t);
            }
            const float gl = pol_policy_row<L>(logp, old_logp, adv, c, sums);
            pol_ppo_gauss_row(gl, act, mean, w, gm, gs);
            for (int k = 0; k < kPolHidden; ++k) {
                grad[STG_POLICY_ACT_W + k] += (double)h2[k] * gm[0];
                grad[STG_POLICY_ACT_W + 64 + k] += (double)h2[k] * gm[1];
                const float s = Pk<float>::add(Pk<float>::mul(w[STG_POLICY_ACT_W + 2 * k], gm[0]),
                                               Pk<float>::mul(w[STG_POLICY_ACT_W + 2 * k + 1], gm[1]));
                d2[k] = pol_dtanh(s, h2[k]);
            }
            for (int d = 0; d < 2; ++d) {
                grad[STG_POLICY_ACT_B + d] += gm[d];
                grad[STG_POLICY_LOG_STD + d] += gs[d];
            }
        }
        for (int o = 0; o < kPolHidden; ++o) {
            grad[b2 + o] += d2[o];
            for (int k = 0; k < kPolHidden; ++k) grad[w2 + o * 64 + k] += (double)h1[k] * d2[o];
        }
        for (int k = 0; k < kPolHidden; ++k) {                             // d1[k] = (W2 d2)[k] * (1 - h1[k]^2), ascending o
            float acc = 0.0f;
            for (int o = 0; o < kPolHidden; ++o) acc = fmaf(w[w2 + k * 64 + o], d2[o], acc);
            const float d1 = pol_dtanh(acc, h1[k]);
            grad[b1 + k] += d1;
            for (int i = 0; i < kPolObs; ++i) grad[w1 + k * kPolObs + i] += (double)obs[i] * d1;
        }
    }
}

}  // namespace stg
