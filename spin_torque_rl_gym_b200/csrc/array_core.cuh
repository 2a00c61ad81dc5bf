// array_core.cuh — K3: one SpinTorqueArray-v0 step of one crossbar array (envs/array_env.py:358-551 of the reference).
//
// The affected devices are updated SEQUENTIALLY and in place, each seeing the already-updated neighbours through the
// coupling sum (Gauss-Seidel order is part of the reference's semantics), with a derivative frozen at the pre-pulse state
// and ten renormalised Euler substeps. All arithmetic FP64; products and sums are kept unfused (dmul/dadd) where the
// reference's NumPy code rounds twice, so the result agrees with the oracle to the last bits.
#pragma once

#include "../../include/stg.h"
#include "llgs_core.cuh"

namespace stg {

STG_HD void cross_u(const double* a, const double* b, double* c) {   // np.cross: unfused multiply / subtract
    c[0] = dadd(dmul(a[1], b[2]), -dmul(a[2], b[1]));
    c[1] = dadd(dmul(a[2], b[0]), -dmul(a[0], b[2]));
    c[2] = dadd(dmul(a[0], b[1]), -dmul(a[1], b[0]));
}
STG_HD double dot_u(const double* a, const double* b) {
    return dadd(dadd(dmul(a[0], b[0]), dmul(a[1], b[1])), dmul(a[2], b[2]));
}
STG_HD double norm_u(const double* a) { return sqrt(dot_u(a, a)); }

// np.add.reduce over n doubles (pairwise summation, numpy/_core/src/umath/loops_utils.h.src): bit-compatible for n <= 128,
// recursive halves above that.
STG_HD double numpy_sum(const double* v, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r = dadd(r, v[i]);
        return r;
    }
    if (n <= 128) {
        double r[8];
        for (int k = 0; k < 8; ++k) r[k] = v[k];
        int i;
        for (i = 8; i < n - (n % 8); i += 8)
            for (int k = 0; k < 8; ++k) r[k] = dadd(r[k], v[i + k]);
        double res = dadd(dadd(dadd(r[0], r[1]), dadd(r[2], r[3])), dadd(dadd(r[4], r[5]), dadd(r[6], r[7])));
        for (; i < n; ++i) res = dadd(res, v[i]);
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return dadd(numpy_sum(v, n2), numpy_sum(v + n2, n - n2));
}

// intrinsic field of one device (device.compute_effective_field(m, 0): devices/stt_mram.py:56-76 / sot / vcma forms)
STG_HD void array_intrinsic_field(const StgArrayParams& p, const double* m, double* h) {
    double mm[3] = {m[0], m[1], m[2]};
    if (p.device_kind == STG_DEV_STT) {
        const double n = norm_u(m);
        mm[0] = m[0] / n; mm[1] = m[1] / n; mm[2] = m[2] / n;
    }
    const double s = dmul(p.hk, dot_u(mm, p.easy_axis));
    for (int k = 0; k < 3; ++k) h[k] = dmul(s, p.easy_axis[k]);
    if (p.device_kind != STG_DEV_STT)
        for (int k = 0; k < 3; ++k) h[k] = dadd(h[k], dmul(dmul(-p.saturation_magnetization, p.demag_n[k]), mm[k]));
}

// _simulate_device_dynamics (envs/array_env.py:497-531): frozen derivative, 10 renormalised Euler substeps
STG_HD void array_device_dynamics(const double* m0, double cur, double dur, const double* h, double* out) {
    if (!(fabs(cur) > 1e-12)) { out[0] = m0[0]; out[1] = m0[1]; out[2] = m0[2]; return; }
    const double z[3] = {0.0, 0.0, 1.0};
    double mp[3], mmp[3], tau[3], dm[3], mdm[3];
    cross_u(m0, z, mp);
    cross_u(m0, mp, mmp);
    const double pre = dmul(0.1, cur);
    for (int k = 0; k < 3; ++k) tau[k] = dmul(pre, mmp[k]);
    cross_u(m0, h, dm);
    for (int k = 0; k < 3; ++k) dm[k] = dmul(-2.21e5, dm[k]);
    cross_u(m0, dm, mdm);
    for (int k = 0; k < 3; ++k) dm[k] = dadd(dadd(dm[k], dmul(0.01, mdm[k])), tau[k]);
    const double dt = ddiv(dur, 10.0);
    double m[3] = {m0[0], m0[1], m0[2]};
    for (int s = 0; s < 10; ++s) {
        for (int k = 0; k < 3; ++k) m[k] = dadd(m[k], dmul(dm[k], dt));
        const double n = norm_u(m);
        for (int k = 0; k < 3; ++k) m[k] = ddiv(m[k], n);
    }
    out[0] = m[0]; out[1] = m[1]; out[2] = m[2];
}

STG_HD double array_resistance(const StgArrayParams& p, const double* m) {
    double f[FI_COUNT];
    f[FI_KIND] = (double)p.device_kind;
    f[FI_RP] = p.resistance_parallel; f[FI_RAP] = p.resistance_antiparallel;
    f[FI_TMR] = (p.resistance_antiparallel - p.resistance_parallel) / p.resistance_parallel;
    f[FI_REFX] = p.reference_magnetization[0]; f[FI_REFY] = p.reference_magnetization[1];
    f[FI_REFZ] = p.reference_magnetization[2];
    f[FI_RSERIES] = p.series_resistance;
    return resistance(f, m[0], m[1], m[2]);
}

// action -> (first affected device, count, stride, J, T) (envs/array_env.py:413-442)
struct ArrayAction {
    int first, count, stride;
    double cur, dur;
};
STG_HD ArrayAction array_parse_action(const StgArrayParams& p, const float* act) {
    ArrayAction a;
    const int nd = p.n_rows * p.n_cols;
    double cur, dur;
    if (p.action_mode == STG_ARRAY_GLOBAL) {      // [J, T] is read as [idx, J]; the duration defaults to 1 ns (:415-416)
        cur = (double)act[1];
        dur = 1e-9;
    } else {
        cur = (double)act[1];
        dur = (double)act[2];
    }
    // np.clip keeps NaN (both comparisons are false); fmin/fmax would drop it. A NaN current then drives nothing and costs no
    // energy (|NaN| > 1e-12 is false), and a NaN duration propagates through the dynamics and the energy, as in the reference.
    auto clip = [](double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); };
    a.cur = clip(cur, -p.max_current, p.max_current);
    a.dur = clip(dur, 1e-12, p.max_duration);
    const float a0 = act[0];
    // int(np.clip(action[0], 0, hi)) on a float32 scalar. The reference raises on a NaN index; a kernel cannot, so it takes 0.
    auto clip_idx = [](float v, int hi) {
        float c = fminf(fmaxf(v, 0.0f), (float)hi);
        if (!(c == c)) c = 0.0f;
        return (int)c;
    };
    if (p.action_mode == STG_ARRAY_INDIVIDUAL) { a.first = clip_idx(a0, nd - 1); a.count = 1; a.stride = 1; }
    else if (p.action_mode == STG_ARRAY_ROW) { a.first = clip_idx(a0, p.n_rows - 1) * p.n_cols; a.count = p.n_cols; a.stride = 1; }
    else if (p.action_mode == STG_ARRAY_COLUMN) { a.first = clip_idx(a0, p.n_cols - 1); a.count = p.n_rows; a.stride = p.n_cols; }
    else { a.first = 0; a.count = nd; a.stride = 1; }
    return a;
}

// sequential in-place update of the affected devices; pattern [nd][3] (shared memory on the device). Returns step energy.
STG_HD double array_apply_action(const StgArrayParams& p, const double* coupling, double* pattern, const ArrayAction& a) {
    const int nd = p.n_rows * p.n_cols;
    double energy = 0.0;
    for (int q = 0; q < a.count; ++q) {
        const int i = a.first + q * a.stride;
        double* m = pattern + 3 * i;
        double h[3], hc[3] = {0.0, 0.0, 0.0};
        array_intrinsic_field(p, m, h);
        if (coupling) {
            const double* row = coupling + (int64_t)i * nd;
            for (int j = 0; j < nd; ++j) {
                if (j == i) continue;
                const double c = row[j];
                hc[0] = dadd(hc[0], dmul(c, pattern[3 * j]));
                hc[1] = dadd(hc[1], dmul(c, pattern[3 * j + 1]));
                hc[2] = dadd(hc[2], dmul(c, pattern[3 * j + 2]));
            }
        }
        for (int k = 0; k < 3; ++k) h[k] = dadd(h[k], hc[k]);
        double fin[3];
        array_device_dynamics(m, a.cur, a.dur, h, fin);
        m[0] = fin[0]; m[1] = fin[1]; m[2] = fin[2];
        if (fabs(a.cur) > 1e-12) {                 // resistance of the UPDATED magnetisation (NumPy view aliasing, :447-461)
            const double r = array_resistance(p, m);
            const double v = dmul(dmul(a.cur, r), p.area);
            energy = dadd(energy, dmul(ddiv(dmul(v, v), r), a.dur));
        }
    }
    return energy;
}

// reward (envs/array_env.py:182-221) from similarity / energy / improvement / per-device magnitudes
STG_HD double array_reward(const StgArrayParams& p, bool success, double sim, double energy, double improvement,
                           double uniformity_std) {
    double total = 0.0;
    total = dadd(total, dmul(10.0, success ? 10.0 : dmul(sim, 5.0)));
    total = dadd(total, dmul(-p.energy_penalty_weight, ddiv(-energy, 1e-12)));
    total = dadd(total, dmul(1.0, improvement));
    const double u = dadd(1.0, -uniformity_std);
    total = dadd(total, dmul(2.0, u > 0.0 ? u : 0.0));
    return total;
}

// std of the magnitudes exactly like np.std: sqrt(mean(|x - mean(x)|^2)) with NumPy's pairwise sums. scratch: nd doubles.
STG_HD double array_magnitude_std(const double* pattern, int nd, double* scratch) {
    for (int i = 0; i < nd; ++i) scratch[i] = norm_u(pattern + 3 * i);
    const double mean = ddiv(numpy_sum(scratch, nd), (double)nd);
    for (int i = 0; i < nd; ++i) { const double d = dadd(scratch[i], -mean); scratch[i] = dmul(d, d); }
    return sqrt(ddiv(numpy_sum(scratch, nd), (double)nd));
}
STG_HD double array_similarity(const double* pattern, const double* target, int nd, double* scratch) {
    for (int i = 0; i < nd; ++i) scratch[i] = dot_u(pattern + 3 * i, target + 3 * i);
    return ddiv(numpy_sum(scratch, nd), (double)nd);
}

}  // namespace stg
