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

}  // namespace stg
