// array_kernels.cu — K3 launch + C-ABI. The pattern and the target live in shared memory for the whole step (coalesced FP64
// loads, coalesced f32 observation stores); the Gauss-Seidel device update is sequential in device order (part of the
// reference's semantics) and the reductions are NumPy-ordered sums. Default kernel for 8..128 devices: four arrays per
// warp, eight lanes per array (array_step_kernel8); other sizes / STG_F_ARRAY_ONE_WARP: one warp per array.
// HBM-bound: ~ (24+24) B read + (24+24) B written per device and step.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stg.h"
#include "array_core.cuh"

namespace stg {

constexpr int kArrayBlock = 32;     // one warp per crossbar array; 24 CTAs (= arrays) resident per SM hide the FP64 latency
constexpr int kArrayMinBlocks = 24;

__device__ __forceinline__ void array_draw_pattern(const StgArrayStepArgs& a, int64_t arr, uint32_t episode, int nd,
                                                   double* pattern) {
    Philox ph{(uint32_t)a.seed, (uint32_t)(a.seed >> 32)};
    const uint64_t gid = a.array_offset + (uint64_t)arr;
    for (int i = threadIdx.x; i < nd; i += blockDim.x) {
        uint32_t o[4];
        float z0, z1, z2, z3;
        uint32_t attempt = 0;
        do {
            ph((uint32_t)gid, (uint32_t)(gid >> 32), episode, ((uint32_t)i << 4) + attempt, o);
            box_muller(o[0], o[1], z0, z1);
            box_muller(o[2], o[3], z2, z3);
            ++attempt;
        } while (z0 * z0 + z1 * z1 + z2 * z2 < 1e-12f && attempt < 8);
        const double n = sqrt((double)z0 * z0 + (double)z1 * z1 + (double)z2 * z2);
        pattern[3 * i] = z0 / n; pattern[3 * i + 1] = z1 / n; pattern[3 * i + 2] = z2 / n;
    }
}

__device__ __forceinline__ void array_store_obs(float* obs, const double* pattern, const double* target, int nd) {
    // [D][6] f32: consecutive threads write consecutive floats
    for (int q = threadIdx.x; q < nd * 6; q += blockDim.x) {
        const int d = q / 6, c = q % 6;
        obs[q] = (float)(c < 3 ? pattern[3 * d + c] : target[3 * d + c - 3]);
    }
}

__global__ void __launch_bounds__(kArrayBlock, kArrayMinBlocks) array_step_kernel(const __grid_constant__ StgArrayStepArgs a) {
    extern __shared__ double smem[];
    const int nd = a.params.n_rows * a.params.n_cols;
    double* pattern = smem;                 // [nd][3]
    double* target = smem + 3 * nd;         // [nd][3]
    double* scratch = smem + 6 * nd;        // [nd]
    __shared__ double s_out[6];
    __shared__ int s_flags[3];
    const int64_t arr = blockIdx.x;
    double* gp = a.d_pattern + arr * nd * 3;
    const double* gt = a.d_target + arr * nd * 3;
    for (int q = threadIdx.x; q < nd * 3; q += blockDim.x) { pattern[q] = gp[q]; target[q] = gt[q]; }
    __syncthreads();
    const StgArrayParams& p = a.params;
    __shared__ double s_prev, s_energy, s_sim, s_mean;
    __shared__ ArrayAction s_act;
    // per-device dot products / norms in parallel, NumPy-ordered sums by lane 0 (bit-identical to the sequential form)
    for (int i = threadIdx.x; i < nd; i += blockDim.x) scratch[i] = dot_u(pattern + 3 * i, target + 3 * i);
    __syncthreads();
    if (threadIdx.x == 0) {
        s_prev = ddiv(numpy_sum(scratch, nd), (double)nd);
        s_act = array_parse_action(p, a.d_action + arr * a.action_stride);
        s_energy = array_apply_action(p, a.d_coupling, pattern, s_act);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nd; i += blockDim.x) scratch[i] = dot_u(pattern + 3 * i, target + 3 * i);
    __syncthreads();
    if (threadIdx.x == 0) s_sim = ddiv(numpy_sum(scratch, nd), (double)nd);
    __syncthreads();
    for (int i = threadIdx.x; i < nd; i += blockDim.x) scratch[i] = norm_u(pattern + 3 * i);
    __syncthreads();
    if (threadIdx.x == 0) s_mean = ddiv(numpy_sum(scratch, nd), (double)nd);
    __syncthreads();
    for (int i = threadIdx.x; i < nd; i += blockDim.x) { const double d = dadd(scratch[i], -s_mean); scratch[i] = dmul(d, d); }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double prev = s_prev, energy = s_energy, sim = s_sim;
        const ArrayAction act = s_act;
        const bool success = sim >= p.success_threshold;
        const double sd = sqrt(ddiv(numpy_sum(scratch, nd), (double)nd));
        const double reward = array_reward(p, success, sim, energy, dadd(sim, -prev), sd);
        const int step = a.d_step_count[arr] + 1;
        const double tot = dadd(a.d_total_energy[arr], energy);
        const bool trunc = step >= p.max_steps;
        a.d_reward[arr] = reward;
        a.d_terminated[arr] = success ? 1 : 0;
        a.d_truncated[arr] = trunc ? 1 : 0;
        if (a.d_step_energy) a.d_step_energy[arr] = energy;
        if (a.d_similarity) a.d_similarity[arr] = sim;
        const bool reset = (a.flags & STG_F_AUTORESET) && (success || trunc);
        a.d_step_count[arr] = reset ? 0 : step;
        a.d_total_energy[arr] = reset ? 0.0 : tot;
        s_flags[0] = reset ? 1 : 0;
        if (a.d_stats) {
            double* st = a.d_stats + (blockIdx.x % STG_STAT_REPLICAS) * STG_NSTATS;
            atomicAdd(st + STG_STAT_STEPS, 1.0);
            atomicAdd(st + STG_STAT_SUBSTEPS, 10.0 * act.count);
            if (success) atomicAdd(st + STG_STAT_TERMINATED, 1.0);
            else if (trunc) atomicAdd(st + STG_STAT_TRUNCATED, 1.0);
            atomicAdd(st + STG_STAT_ENERGY, energy);
            atomicAdd(st + STG_STAT_REWARD, reward);
            if (success || trunc) atomicAdd(st + STG_STAT_EPLEN, (double)step);
        }
    }
    __syncthreads();
    const bool reset = s_flags[0] != 0;
    if (reset) {
        if (a.d_final_obs) array_store_obs(a.d_final_obs + arr * nd * 6, pattern, target, nd);
        __syncthreads();
        const uint32_t ep = (uint32_t)a.d_episode[arr] + 1u;
        __syncthreads();
        if (threadIdx.x == 0) a.d_episode[arr] = (int32_t)ep;
        array_draw_pattern(a, arr, ep, nd, pattern);
        __syncthreads();
    }       // final_obs of a running array is not written (include/stg.h: valid where terminated | truncated)
    for (int q = threadIdx.x; q < nd * 3; q += blockDim.x) gp[q] = pattern[q];
    array_store_obs(a.d_obs + arr * nd * 6, pattern, target, nd);
}

// ---- four arrays per warp, eight lanes per array ----------------------------------------------------------------------------
// The one-warp kernel above executes ~4,800 warp-instructions per 8x8 array with 6 of 32 lanes active on average (ncu,
// profiles/): every NumPy-ordered sum and the device update run on lane 0. Here a group of 8 lanes owns one array:
//   * lane k IS accumulator r[k] of NumPy's pairwise sum (same additions in the same order); the final
//     ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) is an xor-shuffle tree (IEEE addition commutes, so every lane holds the same bits);
//   * lanes 0..2 carry the x, y, z components through the sequential coupling sum and the ten renormalised Euler substeps
//     (one software sqrt and one division per substep instead of one sqrt and three divisions in a single lane);
//   * loads and stores use the whole warp over the four arrays, which are contiguous in HBM.
// All results are bit-identical to the one-warp kernel and to the host sequence in array_core.cuh.
constexpr int kGroupLanes = 8;
constexpr int kGroupsPerWarp = 4;
// Shared-memory stride of one array in doubles: pattern 3nd, target 3nd, scratch / coupling row nd, rounded so that the stride
// is 8 (mod 16) doubles = 64 (mod 128) bytes. With a stride that is a multiple of 128 bytes (8x8: 3,584 B) the four groups of
// a warp map to the same 16 banks and every group-parallel 64-bit access is a 4-way conflict (ncu: 2.9e6 conflicts per
// launch, short-scoreboard + MIO-throttle stalls 7 per issue); alternating the groups between the two halves of the banks
// leaves the two wavefronts a 32-lane 64-bit access needs anyway.
__host__ __device__ inline int array8_stride(int nd) {
    const int per = 7 * nd + (nd & 1);
    return per + ((8 - per % 16) + 16) % 16;
}
constexpr int kArray8MinBlocks = 14;     // 14.2 KB of shared memory per CTA at 8x8: ncu reports 14 resident CTAs per SM
                                         // (shared-memory limit), so 4,096 CTAs are 1.98 waves

template <int ND_T, typename F>
__device__ __forceinline__ double group_numpy_sum(unsigned gmask, int l8, int n_rt, F v) {      // 8 <= n <= 128
    const int n = ND_T ? ND_T : n_rt;
    const int nfull = n - (n % 8);
    double r = v(l8);
#pragma unroll
    for (int i = 8; i < nfull; i += 8) r = dadd(r, v(i + l8));
    r = dadd(r, __shfl_xor_sync(gmask, r, 1));
    r = dadd(r, __shfl_xor_sync(gmask, r, 2));
    r = dadd(r, __shfl_xor_sync(gmask, r, 4));
    for (int i = nfull; i < n; ++i) r = dadd(r, v(i));
    return r;
}

// Sequential in-place update of the affected devices by one 8-lane group (array_apply_action in array_core.cuh is the
// one-thread form). The coupling row of device q+1 is fetched into registers while device q is integrated, so the
// L2 latency of the row never sits on the dependent chain; rowbuf is the group's scratch region (free until the norms).
template <int ND_T>
__device__ __forceinline__ double group_apply_action(const StgArrayParams& p, const double* coupling, double* pattern,
                                                     double* rowbuf, const ArrayAction& a, unsigned gmask, int l8) {
    constexpr int RN = ND_T ? ND_T / kGroupLanes : 16;          // row values per lane (nd <= 128)
    const int nd = ND_T ? ND_T : p.n_rows * p.n_cols;
    const int c = l8 < 3 ? l8 : 0;                 // lanes 3..7 shadow component 0 so the group never diverges
    const bool drive = fabs(a.cur) > 1e-12;
    double energy = 0.0;
    double rn[RN];
    auto fetch_row = [&](int i) {
        const double* row = coupling + (int64_t)i * nd;
#pragma unroll
        for (int k = 0; k < RN; ++k) {
            const int j = l8 + kGroupLanes * k;
            rn[k] = (ND_T || j < nd) ? row[j] : 0.0;
        }
    };
    if (coupling && a.count > 0) fetch_row(a.first);
    for (int q = 0; q < a.count; ++q) {
        const int i = a.first + q * a.stride;
        double* m = pattern + 3 * i;
        double h[3];
        array_intrinsic_field(p, m, h);
        if (coupling) {
#pragma unroll
            for (int k = 0; k < RN; ++k) {
                const int j = l8 + kGroupLanes * k;
                if (ND_T || j < nd) rowbuf[j] = rn[k];
            }
            __syncwarp(gmask);
            if (q + 1 < a.count) fetch_row(i + a.stride);       // in flight during this device's update
            double hcv = 0.0;
#pragma unroll 16
            for (int j = 0; j < nd; ++j) {
                const double t = dmul(rowbuf[j], pattern[3 * j + c]);
                hcv = (j == i) ? hcv : dadd(hcv, t);
            }
            h[0] = dadd(h[0], __shfl_sync(gmask, hcv, 0, kGroupLanes));
            h[1] = dadd(h[1], __shfl_sync(gmask, hcv, 1, kGroupLanes));
            h[2] = dadd(h[2], __shfl_sync(gmask, hcv, 2, kGroupLanes));
        } else {
            for (int k = 0; k < 3; ++k) h[k] = dadd(h[k], 0.0);
        }
        if (drive) {      // _simulate_device_dynamics (envs/array_env.py:497-531), see array_device_dynamics
            const double m0[3] = {m[0], m[1], m[2]};
            const double z[3] = {0.0, 0.0, 1.0};
            double mp[3], mmp[3], dm[3], mdm[3];
            cross_u(m0, z, mp);
            cross_u(m0, mp, mmp);
            const double pre = dmul(0.1, a.cur);
            cross_u(m0, h, dm);
            for (int k = 0; k < 3; ++k) dm[k] = dmul(-2.21e5, dm[k]);
            cross_u(m0, dm, mdm);
            // component of this lane by selects (a runtime index would push the vectors to local memory)
            auto pick = [c](const double* v) { return c == 0 ? v[0] : (c == 1 ? v[1] : v[2]); };
            const double dc = dadd(dadd(pick(dm), dmul(0.01, pick(mdm))), dmul(pre, pick(mmp)));
            const double dt = ddiv(a.dur, 10.0);
            double mc = pick(m0);
            for (int s = 0; s < 10; ++s) {
                mc = dadd(mc, dmul(dc, dt));
                const double sq = dmul(mc, mc);
                const double n = sqrt(dadd(dadd(__shfl_sync(gmask, sq, 0, kGroupLanes), __shfl_sync(gmask, sq, 1, kGroupLanes)),
                                           __shfl_sync(gmask, sq, 2, kGroupLanes)));
                mc = ddiv(mc, n);
            }
            __syncwarp(gmask);
            if (l8 < 3) m[l8] = mc;
            __syncwarp(gmask);
            const double r = array_resistance(p, m);          // resistance of the UPDATED magnetisation (:447-461)
            const double v = dmul(dmul(a.cur, r), p.area);
            energy = dadd(energy, dmul(ddiv(dmul(v, v), r), a.dur));
        }
        __syncwarp(gmask);
    }
    return energy;
}

__device__ __forceinline__ void group_draw_pattern(const StgArrayStepArgs& a, int64_t arr, uint32_t episode, int nd,
                                                   double* pattern, int l8) {
    Philox ph{(uint32_t)a.seed, (uint32_t)(a.seed >> 32)};
    const uint64_t gid = a.array_offset + (uint64_t)arr;
    for (int i = l8; i < nd; i += kGroupLanes) {
        uint32_t o[4];
        float z0, z1, z2, z3;
        uint32_t attempt = 0;
        do {
            ph((uint32_t)gid, (uint32_t)(gid >> 32), episode, ((uint32_t)i << 4) + attempt, o);
            box_muller(o[0], o[1], z0, z1);
            box_muller(o[2], o[3], z2, z3);
            ++attempt;
        } while (z0 * z0 + z1 * z1 + z2 * z2 < 1e-12f && attempt < 8);
        const double n = sqrt((double)z0 * z0 + (double)z1 * z1 + (double)z2 * z2);
        pattern[3 * i] = z0 / n; pattern[3 * i + 1] = z1 / n; pattern[3 * i + 2] = z2 / n;
    }
}

// two f32 packed into the bit pattern of one f64 slot: observations are built IN PLACE over the target rows (a device's six
// f32 outputs overlay exactly its own three f64 target values), written through the same double-typed array
__device__ __forceinline__ double pack2f(float lo, float hi) { return __hiloint2double(__float_as_int(hi), __float_as_int(lo)); }

// ND_T: devices per array at compile time (0 = runtime), lets the copy loops unroll so every load is in flight before the
// first use. VEC: 16-byte global/shared accesses (even device count, 16-byte aligned buffers; checked at launch).
template <int ND_T, bool VEC>
__global__ void __launch_bounds__(32, kArray8MinBlocks) array_step_kernel8(const __grid_constant__ StgArrayStepArgs a) {
    extern __shared__ __align__(16) double smem[];
    const StgArrayParams& p = a.params;
    const int nd = ND_T ? ND_T : p.n_rows * p.n_cols;
    const int per = array8_stride(nd);
    const int lane = threadIdx.x, g = lane >> 3, l8 = lane & 7;
    const unsigned gmask = 0xFFu << (8 * g);
    const int64_t arr0 = (int64_t)blockIdx.x * kGroupsPerWarp;
    const int64_t left = a.n_arrays - arr0;
    const int narr = left < kGroupsPerWarp ? (int)left : kGroupsPerWarp;
    const bool valid = g < narr;
    const int64_t arr = arr0 + g;
    // per-array scalars first: their latency hides behind the bulk load
    float act_raw[3] = {0.0f, 0.0f, 0.0f};
    int step_prev = 0;
    double tot_prev = 0.0;
    if (valid) {
        const float* ga = a.d_action + arr * a.action_stride;
        act_raw[0] = ga[0]; act_raw[1] = ga[1];
        if (p.action_mode != STG_ARRAY_GLOBAL) act_raw[2] = ga[2];
        step_prev = a.d_step_count[arr];
        tot_prev = a.d_total_energy[arr];
    }
    double* gp0 = a.d_pattern + arr0 * nd * 3;
    const double* gt0 = a.d_target + arr0 * nd * 3;
    if (VEC) {
#ifndef STG_ARRAY_NO_BULK
        // bulk asynchronous copies global -> shared (cp.async.bulk = UBLKCP, completion on an mbarrier): the 2 x narr tensors of
        // 3 nd doubles never pass through registers, so the load costs the warp ten instructions instead of 48 LDG.128 + 48
        // STS.128 and their MIO-queue / long-scoreboard stalls (16 % of the stall samples of the LDG / STS form, profiles/)
        __shared__ __align__(8) uint64_t s_bar;
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
        if (lane == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            const uint32_t bytes = (uint32_t)(3 * nd * sizeof(double));
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2u * (uint32_t)narr * bytes) : "memory");
#pragma unroll
            for (int ar = 0; ar < kGroupsPerWarp; ++ar) {
                if (ar < narr) {
                    const uint32_t dp = (uint32_t)__cvta_generic_to_shared(smem + ar * per);
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(dp), "l"(gp0 + ar * 3 * nd), "r"(bytes), "r"(bar) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(dp + bytes), "l"(gt0 + ar * 3 * nd), "r"(bytes), "r"(bar) : "memory");
                }
            }
        }
        __syncwarp();
        uint32_t done = 0;
        while (!done) {
            asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                         : "=r"(done) : "r"(bar), "r"(0u) : "memory");
        }
#else
        const int n2 = 3 * nd / 2;                   // 16-byte words per array and tensor
        const double2* gp2 = reinterpret_cast<const double2*>(gp0);
        const double2* gt2 = reinterpret_cast<const double2*>(gt0);
#pragma unroll
        for (int ar = 0; ar < kGroupsPerWarp; ++ar) {
            if (ar < narr) {
                double2* sp = reinterpret_cast<double2*>(smem + ar * per);
                double2* st = reinterpret_cast<double2*>(smem + ar * per + 3 * nd);
#pragma unroll
                for (int q = lane; q < n2; q += 32) { sp[q] = gp2[ar * n2 + q]; st[q] = gt2[ar * n2 + q]; }
            }
        }
#endif
    } else {
        for (int ar = 0; ar < narr; ++ar)
            for (int q = lane; q < 3 * nd; q += 32) {
                smem[ar * per + q] = gp0[ar * 3 * nd + q];
                smem[ar * per + 3 * nd + q] = gt0[ar * 3 * nd + q];
            }
    }
    __syncwarp();
    double* pattern = smem + g * per;
    double* target = pattern + 3 * nd;
    double* scratch = target + 3 * nd;              // coupling row during the device update, per-device norms afterwards
    bool reset = false;
    int aff_first = 0, aff_count = 0, aff_stride = 1;     // devices this step updated (pattern write-back)
    double st_v[STG_NSTATS];
#pragma unroll
    for (int q = 0; q < STG_NSTATS; ++q) st_v[q] = 0.0;
    if (valid) {
        const double fnd = (double)nd;
        // x / nd. For a power-of-two device count known at compile time the quotient equals x * 2^-k bit for bit (an exact
        // scaling; no result here is anywhere near the subnormal range), which takes four software FP64 divisions off the chain.
        constexpr bool kPow2 = ND_T > 0 && (ND_T & (ND_T - 1)) == 0;
        auto over_nd = [&](double x) { return kPow2 ? dmul(x, 1.0 / (double)(ND_T > 0 ? ND_T : 1)) : ddiv(x, fnd); };
        auto dots = [&](int i) { return dot_u(pattern + 3 * i, target + 3 * i); };
        const double prev = over_nd(group_numpy_sum<ND_T>(gmask, l8, nd, dots));
        const ArrayAction act = array_parse_action(p, act_raw);
        aff_first = act.first; aff_count = act.count; aff_stride = act.stride;
        const double energy = group_apply_action<ND_T>(p, a.d_coupling, pattern, scratch, act, gmask, l8);
        const double sim = over_nd(group_numpy_sum<ND_T>(gmask, l8, nd, dots));
#pragma unroll
        for (int i = l8; i < nd; i += kGroupLanes) scratch[i] = norm_u(pattern + 3 * i);
        __syncwarp(gmask);
        const double mean = over_nd(group_numpy_sum<ND_T>(gmask, l8, nd, [&](int i) { return scratch[i]; }));
        const double var = group_numpy_sum<ND_T>(gmask, l8, nd, [&](int i) { const double d = dadd(scratch[i], -mean); return dmul(d, d); });
        const double sd = sqrt(over_nd(var));
        const bool success = sim >= p.success_threshold;
        const double reward = array_reward(p, success, sim, energy, dadd(sim, -prev), sd);
        const int step = step_prev + 1;
        const bool trunc = step >= p.max_steps;
        reset = (a.flags & STG_F_AUTORESET) && (success || trunc);
        if (l8 == 0) {
            a.d_reward[arr] = reward;
            a.d_terminated[arr] = success ? 1 : 0;
            a.d_truncated[arr] = trunc ? 1 : 0;
            if (a.d_step_energy) a.d_step_energy[arr] = energy;
            if (a.d_similarity) a.d_similarity[arr] = sim;
            a.d_step_count[arr] = reset ? 0 : step;
            a.d_total_energy[arr] = reset ? 0.0 : dadd(tot_prev, energy);
            st_v[STG_STAT_STEPS] = 1.0;
            st_v[STG_STAT_SUBSTEPS] = 10.0 * act.count;
            st_v[STG_STAT_TERMINATED] = success ? 1.0 : 0.0;
            st_v[STG_STAT_TRUNCATED] = (!success && trunc) ? 1.0 : 0.0;
            st_v[STG_STAT_ENERGY] = energy;
            st_v[STG_STAT_REWARD] = reward;
            st_v[STG_STAT_EPLEN] = (success || trunc) ? (double)step : 0.0;
        }
        // observation rows [p_x p_y p_z t_x t_y t_z] as f32, in place over the target rows
#pragma unroll
        for (int d = l8; d < nd; d += kGroupLanes) {
            const double t0 = target[3 * d], t1 = target[3 * d + 1], t2 = target[3 * d + 2];
            target[3 * d] = pack2f((float)pattern[3 * d], (float)pattern[3 * d + 1]);
            target[3 * d + 1] = pack2f((float)pattern[3 * d + 2], (float)t0);
            target[3 * d + 2] = pack2f((float)t1, (float)t2);
        }
        __syncwarp(gmask);
        if (reset) {
            if (a.d_final_obs) {       // pre-reset observation
                double* fo = reinterpret_cast<double*>(a.d_final_obs + arr * nd * 6);
                for (int q = l8; q < 3 * nd; q += kGroupLanes) fo[q] = target[q];
            }
            const uint32_t ep = (uint32_t)a.d_episode[arr] + 1u;
            __syncwarp(gmask);
            if (l8 == 0) a.d_episode[arr] = (int32_t)ep;
            group_draw_pattern(a, arr, ep, nd, pattern, l8);
            for (int d = l8; d < nd; d += kGroupLanes) {      // refresh the pattern half of the rows, keep the f32 target half
                const float t0 = __int_as_float(__double2hiint(target[3 * d + 1]));
                target[3 * d] = pack2f((float)pattern[3 * d], (float)pattern[3 * d + 1]);
                target[3 * d + 1] = pack2f((float)pattern[3 * d + 2], t0);
            }
        }
    }
    // statistics (K5 input): fire-and-forget atomics from the four group leaders into this CTA's copy of the vector
    // (include/stg.h, STG_STAT_REPLICAS). A shuffle reduction across the groups put 32 SHFL on the dependent chain of this
    // latency-bound kernel (11 % of the stall samples); un-replicated, the 114,688 atomics of a 16,384-array launch land on one
    // L2 line and the step takes 91 us instead of 43 us.
    if (a.d_stats && valid && l8 == 0) {
        double* st = a.d_stats + (blockIdx.x % STG_STAT_REPLICAS) * STG_NSTATS;
#pragma unroll
        for (int q = 0; q < STG_NSTATS; ++q)
            if (st_v[q] != 0.0) atomicAdd(st + q, st_v[q]);
    }
    __syncwarp();
    // Pattern write-back: only the rows this step changed - the affected devices (1 of 64 in individual mode) - unless the array
    // was reset (new random pattern) or every device was driven; the final-observation rows of running arrays are not written
    // (include/stg.h: valid where terminated | truncated). The observations of the four arrays are contiguous in HBM:
    // whole-warp coalesced stores.
    const bool bulk_pattern = reset || 2 * aff_count > nd;
    if (valid && !bulk_pattern) {
        double* gp = gp0 + (int64_t)g * nd * 3;
        for (int q = l8; q < 3 * aff_count; q += kGroupLanes) {
            const int d = aff_first + (q / 3) * aff_stride, c = q - 3 * (q / 3);
            gp[3 * d + c] = pattern[3 * d + c];
        }
    }
    const unsigned bulk_bits = __ballot_sync(0xffffffffu, valid && bulk_pattern && l8 == 0);   // bit 8*ar: whole pattern of array ar
    if (VEC) {
        // (a bulk asynchronous copy shared -> global of these rows was measured: no gain, 25.4 us either way)
        const int n2 = 3 * nd / 2;
        double2* gp2 = reinterpret_cast<double2*>(gp0);
        double2* go2 = reinterpret_cast<double2*>(a.d_obs + arr0 * nd * 6);
#pragma unroll
        for (int ar = 0; ar < kGroupsPerWarp; ++ar) {
            if (ar < narr) {
                const double2* sp = reinterpret_cast<const double2*>(smem + ar * per);
                const double2* so = reinterpret_cast<const double2*>(smem + ar * per + 3 * nd);
                const bool bp = (bulk_bits >> (8 * ar)) & 1u;
#pragma unroll
                for (int q = lane; q < n2; q += 32) {
                    if (bp) gp2[ar * n2 + q] = sp[q];
                    go2[ar * n2 + q] = so[q];
                }
            }
        }
    } else {
        for (int ar = 0; ar < narr; ++ar) {
            const double* pat = smem + ar * per;
            const double* so = pat + 3 * nd;
            double* go = reinterpret_cast<double*>(a.d_obs + (arr0 + ar) * nd * 6);      // 6 f32 = 3 f64 slots per device
            const bool bp = (bulk_bits >> (8 * ar)) & 1u;
            for (int q = lane; q < 3 * nd; q += 32) {
                if (bp) gp0[ar * 3 * nd + q] = pat[q];
                go[q] = so[q];
            }
        }
    }
}

__global__ void __launch_bounds__(kArrayBlock) array_reset_kernel(const __grid_constant__ StgArrayStepArgs a,
                                                                   const uint8_t* mask, const double* pattern0) {
    extern __shared__ double smem[];
    const int nd = a.params.n_rows * a.params.n_cols;
    double* pattern = smem;
    double* target = smem + 3 * nd;
    const int64_t arr = blockIdx.x;
    if (mask && !mask[arr]) return;
    double* gp = a.d_pattern + arr * nd * 3;
    const double* gt = a.d_target + arr * nd * 3;
    const uint32_t ep = (uint32_t)a.d_episode[arr] + 1u;
    if (pattern0) {
        for (int q = threadIdx.x; q < nd * 3; q += blockDim.x) pattern[q] = pattern0[arr * nd * 3 + q];
    } else {
        array_draw_pattern(a, arr, ep, nd, pattern);
    }
    for (int q = threadIdx.x; q < nd * 3; q += blockDim.x) target[q] = gt[q];
    __syncthreads();
    for (int q = threadIdx.x; q < nd * 3; q += blockDim.x) gp[q] = pattern[q];
    if (a.d_obs) array_store_obs(a.d_obs + arr * nd * 6, pattern, target, nd);
    if (threadIdx.x == 0) {
        a.d_episode[arr] = (int32_t)ep;
        a.d_step_count[arr] = 0;
        a.d_total_energy[arr] = 0.0;
    }
}

}  // namespace stg

static int check_array_args(const StgArrayStepArgs& a) {
    const int nd = a.params.n_rows * a.params.n_cols;
    if (a.n_arrays < 0 || a.params.n_rows <= 0 || a.params.n_cols <= 0 || nd > STG_ARRAY_MAX_DEVICES) return STG_E_SIZE;
    if (a.params.action_mode < STG_ARRAY_INDIVIDUAL || a.params.action_mode > STG_ARRAY_GLOBAL) return STG_E_ENUM;
    if (a.params.device_kind < STG_DEV_STT || a.params.device_kind > STG_DEV_VCMA) return STG_E_ENUM;
    if (!a.d_pattern || !a.d_target || !a.d_total_energy || !a.d_step_count || !a.d_episode) return STG_E_NULL;
    return STG_OK;
}

// A launch may use 48 KB of static plus dynamic shared memory without the opt-in, so the kernel's static part counts too
// (the one-warp step kernel's 80 B push 1x877 = 49,112 B of dynamic shared memory over the line). The static size is a
// property of the compiled kernel: it is queried once per kernel and kept in *static_bytes (-1 = not yet known).
static int opt_in_shared_memory(const void* kernel, size_t dynamic_bytes, int* static_bytes) {
    if (*static_bytes < 0) {
        cudaFuncAttributes fa;
        const cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
        if (e != cudaSuccess) return (int)e;
        *static_bytes = (int)fa.sharedSizeBytes;
    }
    if (dynamic_bytes + (size_t)*static_bytes <= 48 * 1024) return STG_OK;
    return (int)cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dynamic_bytes);
}

extern "C" int stg_array_step_f64(const StgArrayStepArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgArrayStepArgs& a = *args;
    int rc = check_array_args(a);
    if (rc != STG_OK) return rc;
    if (!a.d_action || !a.d_obs || !a.d_reward || !a.d_terminated || !a.d_truncated) return STG_E_NULL;
    if (a.action_stride < (a.params.action_mode == STG_ARRAY_GLOBAL ? 2 : 3)) return STG_E_SIZE;
    if (a.n_arrays == 0) return STG_OK;
    const int nd = a.params.n_rows * a.params.n_cols;
    // four arrays per warp, eight lanes each. The observation rows are written as 8-byte words (6 f32 per device = 3 words),
    // so d_obs / d_final_obs must be 8-byte aligned for this kernel; anything else takes the one-warp kernel.
    const auto aligned = [](const void* q, uintptr_t n) { return (reinterpret_cast<uintptr_t>(q) & (n - 1)) == 0; };
    if (nd >= 8 && nd <= 128 && !(a.flags & STG_F_ARRAY_ONE_WARP) && aligned(a.d_obs, 8) &&
        (!a.d_final_obs || aligned(a.d_final_obs, 8))) {
        // <= 28.2 KB; the last group needs no trailing pad (8x8: 14,528 B + 1 KB reserved per CTA; 14 CTAs fit the 233,472 B of an
        // SM). The pad is 0..15 doubles depending on nd (0 at 10x12), so it is computed, not assumed.
        const int tail_pad = stg::array8_stride(nd) - (7 * nd + (nd & 1));
        const size_t smem8 = sizeof(double) * ((size_t)stg::array8_stride(nd) * stg::kGroupsPerWarp - (size_t)tail_pad);
        const unsigned grid = (unsigned)((a.n_arrays + stg::kGroupsPerWarp - 1) / stg::kGroupsPerWarp);
        const bool vec = nd % 2 == 0 && aligned(a.d_pattern, 16) && aligned(a.d_target, 16) && aligned(a.d_obs, 16) &&
                         (!a.d_final_obs || aligned(a.d_final_obs, 16));
        static bool carveout_set = false;
        if (!carveout_set) {       // shared-memory-heavy split so >= 12 CTAs x 16 KB are resident per SM
            cudaFuncSetAttribute(stg::array_step_kernel8<64, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            cudaFuncSetAttribute(stg::array_step_kernel8<0, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            cudaFuncSetAttribute(stg::array_step_kernel8<0, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            carveout_set = true;
        }
        if (vec && nd == 64) stg::array_step_kernel8<64, true><<<grid, 32, smem8, (cudaStream_t)stream>>>(a);
        else if (vec) stg::array_step_kernel8<0, true><<<grid, 32, smem8, (cudaStream_t)stream>>>(a);
        else stg::array_step_kernel8<0, false><<<grid, 32, smem8, (cudaStream_t)stream>>>(a);
        return (int)cudaGetLastError();
    }
    const size_t smem = sizeof(double) * 7 * (size_t)nd;
    static int static_smem = -1;
    rc = opt_in_shared_memory((const void*)stg::array_step_kernel, smem, &static_smem);
    if (rc != STG_OK) return rc;
    stg::array_step_kernel<<<(unsigned)a.n_arrays, stg::kArrayBlock, smem, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

extern "C" int stg_array_reset(const StgArrayStepArgs* args, const uint8_t* d_mask, const double* d_pattern0, void* stream) {
    if (!args) return STG_E_NULL;
    const StgArrayStepArgs& a = *args;
    int rc = check_array_args(a);
    if (rc != STG_OK) return rc;
    if (a.n_arrays == 0) return STG_OK;
    const int nd = a.params.n_rows * a.params.n_cols;
    const size_t smem = sizeof(double) * 6 * (size_t)nd;
    static int static_smem = -1;
    rc = opt_in_shared_memory((const void*)stg::array_reset_kernel, smem, &static_smem);
    if (rc != STG_OK) return rc;
    stg::array_reset_kernel<<<(unsigned)a.n_arrays, stg::kArrayBlock, smem, (cudaStream_t)stream>>>(a, d_mask, d_pattern0);
    return (int)cudaGetLastError();
}
