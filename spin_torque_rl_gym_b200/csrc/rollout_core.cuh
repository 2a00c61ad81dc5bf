// rollout_core.cuh — one step of the generalised-advantage-estimation recurrence (K6) and the keyed permutation of the PPO
// minibatch gather (K7), shared by rollout_kernels.cu and the host builds in tests/test_rollout_gae.py and
// tests/test_rollout_minibatch.py.
//
// Specification: Stable-Baselines3's RolloutBuffer.compute_returns_and_advantage in float32, together with the bootstrap of
// truncated episodes in OnPolicyAlgorithm.collect_rollouts (`rewards[idx] += gamma * terminal_value`), in SB3's expression
// order. Every product and sum is rounded on its own (Pk<float>::mul / add: __fmul_rn / __fadd_rn on the device, volatile
// stores on the host), so no compiler may contract any of them into an FMA and the result is the same bits everywhere.
#pragma once

#include <stdint.h>

#include "llgs_core.cuh"

namespace stg {

// Step t of the backward walk, given adv_{t+1} (0 after the last step) and v_next = value_{t+1} (last_value at t = T-1):
//   r_t      = reward_t + gamma * final_value_t            where trunc_t && !term_t, else reward_t
//   nnt_t    = 1 - (term_t | trunc_t)
//   delta_t  = (r_t + (gamma * v_next) * nnt_t) - value_t
//   adv_t    = delta_t + (gamma_lambda * nnt_t) * adv_{t+1}
//   return_t = adv_t + value_t
// final_value_t is selected, never multiplied by zero: for envs whose episode did not end it is a stale row (NaN allowed).
STG_HD float gae_step(float reward, float value, float v_next, bool term, bool trunc, float final_value, float gamma,
                      float gamma_lambda, float adv_next, float& ret) {
    using K = Pk<float>;
    const float r = (trunc && !term) ? K::add(reward, K::mul(gamma, final_value)) : reward;
    const float nnt = (term || trunc) ? 0.0f : 1.0f;
    const float delta = K::add(K::add(r, K::mul(K::mul(gamma, v_next), nnt)), K::neg(value));
    const float adv = K::add(delta, K::mul(K::mul(gamma_lambda, nnt), adv_next));
    ret = K::add(adv, value);
    return adv;
}

// ---- K7: the keyed permutation behind RolloutCollector.get() ----------------------------------------------------------------

// murmur3's 32-bit finaliser: the round function of the Feistel network below.
STG_HD uint32_t fmix32(uint32_t h) {
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

// Half width of the network for a domain of M >= 1 elements: 2 * half is the smallest even number >= 2 with 2^(2 half) >= M,
// so 2^(2 half) < 4 M and, for M <= 2^62, half <= 31 (all round arithmetic is 32-bit).
STG_HD int rollout_permute_half_bits(int64_t M) {
    const uint64_t m = (uint64_t)(M - 1);
#if defined(__CUDA_ARCH__)
    const int bits = m ? 64 - __clzll((long long)m) : 0;
#else
    const int bits = m ? 64 - __builtin_clzll(m) : 0;
#endif
    return bits < 2 ? 1 : (bits + 1) / 2;
}

// One pass of the balanced 8-round Feistel network over [0, 2^(2 half)): a bijection for any keys.
STG_HD uint64_t rollout_feistel(const uint32_t round_keys[8], int half, uint64_t x) {
    const uint32_t mask = (1u << half) - 1u;
    uint32_t l = (uint32_t)(x >> half), r = (uint32_t)x & mask;
    for (int k = 0; k < 8; ++k) {
        const uint32_t n = l ^ (fmix32(r ^ round_keys[k]) & mask);
        l = r;
        r = n;
    }
    return ((uint64_t)l << half) | r;
}

// Position p in [0, M) of the keyed permutation of [0, M), 1 <= M <= 2^62: the network applied to p, then re-applied (cycle
// walking) while the result lies outside [0, M). Walking follows p's cycle of the network's permutation of [0, 2^(2 half)) to the
// next element inside [0, M), which makes the restriction a bijection of [0, M); since 2^(2 half) < 4 M, fewer than 4 passes
// are expected. The result is a flat index t * n_envs + i into the collector's time-major [n_steps][n_envs] planes.
STG_HD int64_t rollout_permute(const uint32_t round_keys[8], int64_t M, int64_t p) {
    const int half = rollout_permute_half_bits(M);
    uint64_t x = (uint64_t)p;
    do {
        x = rollout_feistel(round_keys, half, x);
    } while (x >= (uint64_t)M);
    return (int64_t)x;
}

}  // namespace stg
