// rollout_kernels.cu — K6: generalised advantage estimation over a stored rollout (include/stg.h, stg_rollout_gae_f32), and
// K7: shuffled PPO minibatches gathered from it (stg_rollout_minibatch_f32, below K6).
// Replaces Stable-Baselines3's RolloutBuffer.compute_returns_and_advantage (a Python loop over time with NumPy over envs)
// plus the TimeLimit.truncated bootstrap of OnPolicyAlgorithm.collect_rollouts; the arithmetic is rollout_core.cuh.
//
// Layout: every plane is [T][N] (time-major, the collector's layout). One env per thread walks t = T-1 .. 0, so each load and
// store of a warp is one contiguous 128-B (f32) / 32-B (u8) segment. HBM-bound: 10 B read and 8 B written per (step, env),
// plus 4 B read where a truncated episode is bootstrapped. The recurrence is serial in t, so a thread must keep several steps
// of loads in flight to cover HBM latency (at N = 131,072 there are only ~28 warps per SM): the walk goes in chunks of
// kGaeDepth steps whose reward / value / final-value loads are all issued before the chunk's dependent chain runs, and the
// flags of the NEXT chunk are loaded alongside, so the final-value loads (only where trunc && !term) never wait for a flag
// load of their own. Offsets are int64: 2048 steps x 1,048,576 envs is exactly 2^31 elements.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stg.h"
#include "rollout_core.cuh"

namespace stg {

constexpr int kGaeThreads = 128;
constexpr int kGaeDepth = 8;      // steps per chunk: 72 registers, seven CTAs per SM (16 steps: 128 registers)

__global__ void __launch_bounds__(kGaeThreads) rollout_gae_kernel(const StgGaeArgs a) {
    constexpr int D = kGaeDepth;
    const int64_t N = a.n_envs;
    const int64_t i = (int64_t)blockIdx.x * kGaeThreads + threadIdx.x;
    if (i >= N) return;
    const float gamma = a.gamma, gamma_lambda = a.gamma_lambda;
    float v_next = __ldcs(a.d_last_value + i);
    float adv = 0.0f;
    int64_t t = a.n_steps - 1;
    // the n_steps % D latest steps one at a time, so that every chunk below is complete
#pragma unroll 1
    for (int64_t k = a.n_steps % D; k > 0; --k, --t) {
        const int64_t o = t * N + i;
        const bool te = __ldcs(a.d_terminated + o), tr = __ldcs(a.d_truncated + o);
        const float v = __ldcs(a.d_value + o);
        const float fv = (tr && !te) ? __ldcs(a.d_final_value + o) : 0.0f;
        float ret;
        adv = gae_step(__ldcs(a.d_reward + o), v, v_next, te, tr, fv, gamma, gamma_lambda, adv, ret);
        v_next = v;
        __stcs(a.d_advantage + o, adv);
        if (a.d_return) __stcs(a.d_return + o, ret);
    }
    if (t < 0) return;
    // chunks of D steps t, t-1, ..., t-D+1 (bit j of the flag masks = step t - j). The chunk's flags were loaded during the
    // previous chunk, so its reward / value / final-value loads all issue at once; the next chunk's flags load alongside.
    uint8_t te[D], tr[D];
    uint32_t mterm = 0, mtrunc = 0;
    {
        const int64_t o = t * N + i;
#pragma unroll
        for (int j = 0; j < D; ++j) {
            mterm |= (__ldcs(a.d_terminated + o - j * N) != 0 ? 1u : 0u) << j;
            mtrunc |= (__ldcs(a.d_truncated + o - j * N) != 0 ? 1u : 0u) << j;
        }
    }
#pragma unroll 1
    for (; t >= 0; t -= D) {
        // opaque to the optimiser: otherwise every address below becomes an induction variable of its own, two registers each
        int64_t o = t * N + i;
        asm volatile("" : "+l"(o));
        const uint32_t mboot = mtrunc & ~mterm;
        float r[D], v[D], fv[D];
        {
            const float *pr = a.d_reward + o, *pv = a.d_value + o, *pf = a.d_final_value + o;
#pragma unroll
            for (int j = 0; j < D; ++j, pr -= N, pv -= N, pf -= N) {
                r[j] = __ldcs(pr);
                v[j] = __ldcs(pv);
                fv[j] = (mboot >> j & 1u) ? __ldcs(pf) : 0.0f;
            }
        }
        if (t >= D) {
            const uint8_t *pe = a.d_terminated + o - D * N, *pt = a.d_truncated + o - D * N;
#pragma unroll
            for (int j = 0; j < D; ++j, pe -= N, pt -= N) {
                te[j] = __ldcs(pe);
                tr[j] = __ldcs(pt);
            }
        }
        {
            float *pa = a.d_advantage + o, *pq = a.d_return ? a.d_return + o : nullptr;
#pragma unroll
            for (int j = 0; j < D; ++j, pa -= N) {
                float ret;
                adv = gae_step(r[j], v[j], v_next, mterm >> j & 1u, mtrunc >> j & 1u, fv[j], gamma, gamma_lambda, adv, ret);
                v_next = v[j];
                __stcs(pa, adv);
                if (pq) {
                    __stcs(pq, ret);
                    pq -= N;
                }
            }
        }
        if (t >= D) {
            mterm = mtrunc = 0;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                mterm |= (te[j] != 0 ? 1u : 0u) << j;
                mtrunc |= (tr[j] != 0 ? 1u : 0u) << j;
            }
        }
    }
}

// K7: one PPO minibatch (stg_rollout_minibatch_f32). One output row per thread: the row's sample index comes from the keyed
// permutation (rollout_core.cuh, pure integer arithmetic, no memory), then every requested plane is gathered. The planes are
// dense [T][N] (x 12 / x 2), so the flat time-major index f addresses a row directly: no division into (t, i) is needed.
// All loads of a row are issued before its first store. The reads are random, so a sample costs whole 32-B sectors: 2 for the
// 48-B observation row (48 f is a multiple of 16, so the row never touches a third sector), 1 for the action, 1 per scalar.
// The outputs are written with ordinary stores: the training step reads the minibatch right after, so it may stay in L2.
constexpr int kMinibatchThreads = 256;

__global__ void __launch_bounds__(kMinibatchThreads) rollout_minibatch_kernel(const StgMinibatchArgs a) {
    const int64_t k = (int64_t)blockIdx.x * kMinibatchThreads + threadIdx.x;
    if (k >= a.batch) return;
    const int64_t f = rollout_permute(a.round_keys, a.n_steps * a.n_envs, a.start + k);
    float4 o0, o1, o2;
    float2 act;
    float v, lp, adv, ret;
    if (a.d_obs) {
        const float4* src = reinterpret_cast<const float4*>(a.d_obs + f * 12);
        o0 = __ldg(src);
        o1 = __ldg(src + 1);
        o2 = __ldg(src + 2);
    }
    if (a.d_action) act = __ldg(reinterpret_cast<const float2*>(a.d_action) + f);
    if (a.d_value) v = __ldg(a.d_value + f);
    if (a.d_log_prob) lp = __ldg(a.d_log_prob + f);
    if (a.d_advantage) adv = __ldg(a.d_advantage + f);
    if (a.d_return) ret = __ldg(a.d_return + f);
    if (a.d_obs) {
        float4* dst = reinterpret_cast<float4*>(a.d_obs_out + k * 12);
        dst[0] = o0;
        dst[1] = o1;
        dst[2] = o2;
    }
    if (a.d_action) reinterpret_cast<float2*>(a.d_action_out)[k] = act;
    if (a.d_value) a.d_value_out[k] = v;
    if (a.d_log_prob) a.d_log_prob_out[k] = lp;
    if (a.d_advantage) a.d_advantage_out[k] = adv;
    if (a.d_return) a.d_return_out[k] = ret;
}

}  // namespace stg

extern "C" int stg_rollout_minibatch_f32(const StgMinibatchArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgMinibatchArgs& a = *args;
    if (a.n_steps < 0 || a.n_envs < 0 || a.start < 0 || a.batch < 0) return STG_E_SIZE;
    if (a.n_envs > 0 && a.n_steps > INT64_MAX / a.n_envs) return STG_E_SIZE;
    const int64_t M = a.n_steps * a.n_envs;
    if (M > ((int64_t)1 << 62)) return STG_E_SIZE;
    if (a.batch == 0 || M == 0) return STG_OK;
    if (a.start > M - a.batch) return STG_E_SIZE;
    const void* pairs[6][2] = {{a.d_obs, a.d_obs_out},         {a.d_action, a.d_action_out},
                               {a.d_value, a.d_value_out},     {a.d_log_prob, a.d_log_prob_out},
                               {a.d_advantage, a.d_advantage_out}, {a.d_return, a.d_return_out}};
    bool any = false;
    for (const auto& p : pairs) {
        if (!p[0] != !p[1]) return STG_E_NULL;
        any = any || p[0];
    }
    if (!any) return STG_E_NULL;
    if (((uintptr_t)a.d_obs | (uintptr_t)a.d_obs_out) & 15u) return STG_E_ALIGN;
    if (((uintptr_t)a.d_action | (uintptr_t)a.d_action_out) & 7u) return STG_E_ALIGN;
    const int64_t grid = (a.batch + stg::kMinibatchThreads - 1) / stg::kMinibatchThreads;
    if (grid > 0x7fffffff) return STG_E_SIZE;
    stg::rollout_minibatch_kernel<<<(unsigned)grid, stg::kMinibatchThreads, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

extern "C" int stg_rollout_gae_f32(const StgGaeArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgGaeArgs& a = *args;
    if (a.n_steps < 0 || a.n_envs < 0) return STG_E_SIZE;
    if (a.n_steps == 0 || a.n_envs == 0) return STG_OK;
    if (a.n_steps > INT64_MAX / a.n_envs) return STG_E_SIZE;
    if (!a.d_reward || !a.d_value || !a.d_terminated || !a.d_truncated || !a.d_final_value || !a.d_last_value || !a.d_advantage)
        return STG_E_NULL;
    const int64_t grid = (a.n_envs + stg::kGaeThreads - 1) / stg::kGaeThreads;
    if (grid > 0x7fffffff) return STG_E_SIZE;
    stg::rollout_gae_kernel<<<(unsigned)grid, stg::kGaeThreads, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}
