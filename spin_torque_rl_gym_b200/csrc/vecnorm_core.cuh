// vecnorm_core.cuh — the arithmetic of K8, VecNormalize on the GPU (vecnorm_kernels.cu), shared with the host builds in
// tests/test_vec_normalize.py.
//
// Specification: Stable-Baselines3's VecNormalize (step_wait, reset, _update_reward, normalize_obs, normalize_reward) and
// RunningMeanStd.update_from_moments, in SB3's expression order on float64 data. Every operation of that specification is
// rounded on its own (dmul / dadd / ddiv / dsqrt: __dmul_rn, __dadd_rn, __ddiv_rn, __dsqrt_rn on the device, volatile or
// correctly rounded operations on the host), so no compiler may contract them and the results are NumPy's bits everywhere.
// The batch moments themselves are a parallel reduction (Chan et al.'s pairwise update in a fixed tree): they equal NumPy's
// np.mean / np.var up to FP64 summation order, and contraction is allowed there.
#pragma once

#include <math.h>
#include <stdint.h>

#include "llgs_core.cuh"

namespace stg {

constexpr int kVnObs = 12;                 // STT observation width
constexpr int kVnFeat = kVnObs + 1;        // the 12 observation columns and the discounted return
constexpr int kVnMoments = 1 + 2 * kVnFeat;    // (n, mean[13], M2[13])

STG_HD double dsqrt(double x) {
#if defined(__CUDA_ARCH__)
    return __dsqrt_rn(x);
#else
    return sqrt(x);
#endif
}

// np.clip(x, -c, c) for c >= 0: NaN stays NaN
STG_HD double vn_clip(double x, double c) { return x < -c ? -c : (x > c ? c : x); }

// np.sqrt(rms.var + epsilon): the denominator of both normalisations
STG_HD double vn_scale(double var, double epsilon) { return dsqrt(dadd(var, epsilon)); }

// _normalize_obs: np.clip((obs - mean) / scale, -clip_obs, clip_obs) in float64, then .astype(np.float32)
STG_HD float vn_norm_obs(float x, double mean, double scale, double clip_obs) {
    return (float)vn_clip(ddiv(dadd((double)x, -mean), scale), clip_obs);
}

// normalize_reward: np.clip(reward / scale, -clip_reward, clip_reward) in float64
STG_HD double vn_norm_reward(double r, double scale, double clip_reward) { return vn_clip(ddiv(r, scale), clip_reward); }

// _update_reward: returns * gamma + reward, two roundings
STG_HD double vn_return(double ret, double gamma, double reward) { return dadd(dmul(ret, gamma), reward); }

// RunningMeanStd.update_from_moments for one feature, SB3's expression order:
//   delta = batch_mean - mean;  tot_count = count + batch_count
//   new_mean = mean + delta * batch_count / tot_count
//   m_2 = var * count + batch_var * batch_count + np.square(delta) * count * batch_count / (count + batch_count)
//   new_var = m_2 / (count + batch_count)
// The new count, batch_count + count, is the caller's (it is shared by the features).
STG_HD void vn_update_from_moments(double& mean, double& var, double count, double batch_mean, double batch_var,
                                   double batch_count) {
    const double delta = dadd(batch_mean, -mean);
    const double tot_count = dadd(count, batch_count);
    const double new_mean = dadd(mean, ddiv(dmul(delta, batch_count), tot_count));
    const double m_a = dmul(var, count);
    const double m_b = dmul(batch_var, batch_count);
    const double m_2 = dadd(dadd(m_a, m_b), ddiv(dmul(dmul(dmul(delta, delta), count), batch_count), dadd(count, batch_count)));
    mean = new_mean;
    var = ddiv(m_2, dadd(count, batch_count));
}

// ---- batch moments -----------------------------------------------------------------------------------------------------------
// A thread accumulates its rows shifted by its first row x0: s1 = sum(x - x0), s2 = sum((x - x0)^2) (no division per element;
// a constant column gives exactly zero). Then (n, mean, M2) = (n, x0 + s1/n, s2 - s1^2/n).
STG_HD void vn_shifted_to_moments(double n, double x0, double s1, double s2, double& mean, double& m2) {
    if (n == 0.0) {
        mean = 0.0;
        m2 = 0.0;
        return;
    }
    const double q = s1 / n;
    mean = x0 + q;
    const double r = s2 - s1 * q;
    m2 = r > 0.0 ? r : 0.0;
}

// Chan's pairwise update: (n_a, mean_a, M2_a) <- (n_a, mean_a, M2_a) (+) (n_b, mean_b, M2_b), a the left operand. The weights are
// shared by the features: w = n_b / n, c = n_a n_b / n. An empty operand has n = mean = M2 = 0 (vn_shifted_to_moments), and
// merging it changes no bit: w = 0 (n_b = 0), or w = 1 and c = 0 (n_a = 0); two empty operands give w = 0.
STG_HD void vn_chan_weights(double na, double nb, double& w, double& c) {
    const double n = na + nb;
    w = n > 0.0 ? nb / n : 0.0;
    c = na * w;
}
STG_HD void vn_chan_feature(double& mean_a, double& m2_a, double mean_b, double m2_b, double w, double c) {
    const double d = mean_b - mean_a;
    mean_a = mean_a + d * w;
    m2_a = m2_a + m2_b + d * d * c;
}

// Moment vector v = (n, mean[13], M2[13]): a <- a (+) b
STG_HD void vn_chan_merge(double* a, const double* b) {
    double w, c;
    vn_chan_weights(a[0], b[0], w, c);
    for (int f = 0; f < kVnFeat; ++f) vn_chan_feature(a[1 + f], a[1 + kVnFeat + f], b[1 + f], b[1 + kVnFeat + f], w, c);
    a[0] = a[0] + b[0];
}

// The fold of the merge launch: g moment vectors [g][27] in rank order, left to right, into out[27].
STG_HD void vn_fold(const double* vecs, int g, double* out) {
    for (int k = 0; k < kVnMoments; ++k) out[k] = 0.0;
    for (int r = 0; r < g; ++r) vn_chan_merge(out, vecs + (int64_t)r * kVnMoments);
}

}  // namespace stg
