// optim_core.cuh — arithmetic of K11, the clipped Adam step (include/stg.h, stg_policy_adam_f32), shared by optim_kernels.cu and
// the host build in tests/test_ppo_train.py.
//
// Specification: torch.nn.utils.clip_grad_norm_ followed by torch.optim.Adam's single-tensor update (foreach=False,
// capturable=False, no weight decay, no amsgrad), in torch's order of operations. Every float32 product, sum, quotient and
// square root is rounded on its own (no contraction) and the FP64 norm is summed in the fixed order of adam_norm_chain and
// adam_norm_tree, so for the same scalars the device and the host give the same bits. The one exception is adam_coef's double
// pow: CUDA's is accurate to 2 ulp where glibc's is correctly rounded in practice, so in rare steps step_size or bc2_sqrt can
// differ in their last float32 bit between the two builds. (The bias corrections cannot come from the host: the step count
// lives on the device, and reading it would synchronise every step.)
#pragma once

#include <stdint.h>
#include <math.h>

#include "llgs_core.cuh"
#include "../../include/stg.h"

namespace stg {

constexpr int kAdamThreads = STG_ADAM_THREADS;

// offset of parameter segment s in the K10 gradient layout; s = STG_ADAM_TENSORS gives the end of the last one
STG_HD int adam_offset(int s) {
    const int o[STG_ADAM_TENSORS + 1] = {
        STG_PPO_GRAD_PI_W1, STG_PPO_GRAD_PI_B1, STG_PPO_GRAD_PI_W2, STG_PPO_GRAD_PI_B2, STG_PPO_GRAD_VF_W1, STG_PPO_GRAD_VF_B1,
        STG_PPO_GRAD_VF_W2, STG_PPO_GRAD_VF_B2, STG_PPO_GRAD_ACT_W, STG_PPO_GRAD_ACT_B, STG_PPO_GRAD_VAL_W,
        STG_PPO_GRAD_VAL_B, STG_PPO_GRAD_LOG_STD, STG_POLICY_PARAMS};
    return o[s];
}

STG_HD float adam_div(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(a, b);
#else
    volatile float r = a / b; return r;
#endif
}

STG_HD float adam_sub(float a, float b) { return Pk<float>::add(a, -b); }

STG_HD float adam_sqrt(float a) {
#if defined(__CUDA_ARCH__)
    return __fsqrt_rn(a);
#else
    volatile float r = sqrtf(a); return r;
#endif
}

STG_HD double adam_dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}

STG_HD double adam_dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}

// thread t's partial sum of squares: elements t, t + kAdamThreads, ... in ascending order
STG_HD double adam_norm_chain(const float* g, int n, int t) {
    double s = 0.0;
    for (int i = t; i < n; i += kAdamThreads) s = adam_dadd(s, adam_dmul((double)g[i], (double)g[i]));
    return s;
}

// the tree over the kAdamThreads partials, in place (the host form of the kernel's shared-memory tree); returns the sum
STG_HD double adam_norm_tree(double* part) {
    for (int h = kAdamThreads / 2; h >= 1; h /= 2)
        for (int t = 0; t < h; ++t) part[t] = adam_dadd(part[t], part[t + h]);
    return part[0];
}

// clip_grad_norm_'s coefficient for the FP64 sum of squares, clamped to 1 (NaN stays NaN)
STG_HD float adam_clip_coef(double sumsq, double max_norm) {
    const float total = (float)sqrt(sumsq);
    const float c = Pk<float>::mul(adam_div(1.0f, Pk<float>::add(total, 1e-6f)), (float)max_norm);
    return c > 1.0f ? 1.0f : c;
}

// the float32 scalars of one Adam step at the incremented step count
struct AdamCoef {
    float w1, b2, w2, eps, step_size, bc2_sqrt;
};

STG_HD AdamCoef adam_coef(float step, double lr, double beta1, double beta2, double eps) {
    const double s = (double)step;
    const double bc1 = 1.0 - pow(beta1, s), bc2 = 1.0 - pow(beta2, s);
    AdamCoef c;
    c.w1 = (float)(1.0 - beta1);
    c.b2 = (float)beta2;
    c.w2 = (float)(1.0 - beta2);
    c.eps = (float)eps;
    c.step_size = (float)(lr / bc1);
    c.bc2_sqrt = (float)sqrt(bc2);
    return c;
}

// one element: the moments m, v are updated in place and the new parameter is returned
STG_HD float adam_element(float p, float g, float& m, float& v, const AdamCoef& c) {
    const float d = adam_sub(g, m);
    m = c.w1 < 0.5f ? Pk<float>::add(m, Pk<float>::mul(c.w1, d))
                    : adam_sub(g, Pk<float>::mul(d, adam_sub(1.0f, c.w1)));
    v = Pk<float>::add(Pk<float>::mul(v, c.b2), Pk<float>::mul(Pk<float>::mul(c.w2, g), g));
    const float denom = Pk<float>::add(adam_div(adam_sqrt(v), c.bc2_sqrt), c.eps);
    return adam_sub(p, adam_div(Pk<float>::mul(c.step_size, m), denom));
}

}  // namespace stg
