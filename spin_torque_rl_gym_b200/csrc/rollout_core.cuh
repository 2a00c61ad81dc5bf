// rollout_core.cuh — one step of the generalised-advantage-estimation recurrence (K6), shared by rollout_kernels.cu and the
// host build in tests/test_rollout_gae.py.
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

}  // namespace stg
