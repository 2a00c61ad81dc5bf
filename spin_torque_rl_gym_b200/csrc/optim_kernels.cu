// optim_kernels.cu — K11: the clipped Adam step of the ActorCriticPolicy (include/stg.h, stg_policy_adam_f32). The arithmetic
// is optim_core.cuh; this file runs it in one CTA.
//
// The 10,181 parameters are too few to spread over the GPU: one CTA of STG_ADAM_THREADS threads reads the gradient twice (the
// norm, then the update) and each moment and parameter once, and the launch replaces the dozen small launches and the host work
// of clip_grad_norm_ + Adam.step(). Thread 0 evaluates the gate and writes the log; the decision reaches the other threads through
// shared memory, so nothing is read back to the host and a closed gate costs one launch that returns.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stg.h"
#include "optim_core.cuh"

namespace stg {

__global__ void __launch_bounds__(kAdamThreads) policy_adam_kernel(const StgAdamArgs a) {
    __shared__ double part[kAdamThreads];
    __shared__ int open;
    __shared__ float step;
    const int t = threadIdx.x;
    if (t == 0) {
        int go = a.d_gate == nullptr || *a.d_gate != 0;
        if (go && a.d_losses != nullptr) {
            const float* l = a.d_losses;
            if (a.d_log != nullptr) {
                double* log = a.d_log;
                log[STG_ADAM_LOG_PG] += (double)l[1];
                log[STG_ADAM_LOG_VALUE] += (double)l[2];
                log[STG_ADAM_LOG_ENTROPY] += (double)l[3];
                log[STG_ADAM_LOG_CLIP] += (double)l[5];
                log[STG_ADAM_LOG_COUNT] += 1.0;
                log[STG_ADAM_LOG_EPOCH_KL] += (double)l[4];
                log[STG_ADAM_LOG_EPOCH_COUNT] += 1.0;
                log[STG_ADAM_LOG_LAST_LOSS] = (double)l[0];
            }
            if ((a.flags & STG_ADAM_TARGET_KL) && (double)l[4] > 1.5 * a.target_kl) {
                *a.d_gate = 0;
                go = 0;
            }
        }
        if (go) {
            step = Pk<float>::add(*a.d_step, 1.0f);
            *a.d_step = step;
        }
        open = go;
    }
    __syncthreads();
    if (!open) return;

    float coef = 1.0f;
    if (a.flags & STG_ADAM_CLIP) {
        part[t] = adam_norm_chain(a.d_grad, STG_POLICY_PARAMS, t);
        __syncthreads();
        for (int h = kAdamThreads / 2; h >= 1; h /= 2) {
            if (t < h) part[t] = adam_dadd(part[t], part[t + h]);
            __syncthreads();
        }
        coef = adam_clip_coef(part[0], a.max_grad_norm);
    }
    const AdamCoef c = adam_coef(step, a.lr, a.beta1, a.beta2, a.eps);
    const bool clip = (a.flags & STG_ADAM_CLIP) != 0;
#pragma unroll 1
    for (int s = 0; s < STG_ADAM_TENSORS; ++s) {
        const int off = adam_offset(s), len = adam_offset(s + 1) - off;
        float* p = a.d_param[s];
        for (int j = t; j < len; j += kAdamThreads) {
            const int i = off + j;
            float g = a.d_grad[i];
            if (clip) {
                g = Pk<float>::mul(g, coef);
                a.d_grad[i] = g;
            }
            float m = a.d_exp_avg[i], v = a.d_exp_avg_sq[i];
            p[j] = adam_element(p[j], g, m, v, c);
            a.d_exp_avg[i] = m;
            a.d_exp_avg_sq[i] = v;
        }
    }
}

}  // namespace stg

extern "C" int stg_policy_adam_f32(const StgAdamArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgAdamArgs& a = *args;
    uintptr_t any = 0;
    for (int s = 0; s < STG_ADAM_TENSORS; ++s) {
        if (!a.d_param[s]) return STG_E_NULL;
        any |= (uintptr_t)a.d_param[s];
    }
    if (!a.d_grad || !a.d_exp_avg || !a.d_exp_avg_sq || !a.d_step) return STG_E_NULL;
    any |= (uintptr_t)a.d_grad | (uintptr_t)a.d_exp_avg | (uintptr_t)a.d_exp_avg_sq | (uintptr_t)a.d_step |
           (uintptr_t)a.d_losses | (uintptr_t)a.d_gate;
    if ((any & 3u) || ((uintptr_t)a.d_log & 7u)) return STG_E_ALIGN;
    if (a.flags & ~(STG_ADAM_CLIP | STG_ADAM_TARGET_KL)) return STG_E_ENUM;
    if ((a.flags & STG_ADAM_TARGET_KL) && (!a.d_losses || !a.d_gate)) return STG_E_NULL;
    stg::policy_adam_kernel<<<1, stg::kAdamThreads, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}
