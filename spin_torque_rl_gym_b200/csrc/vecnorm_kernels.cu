// vecnorm_kernels.cu — K8: VecNormalize on the GPU (include/stg.h, stg_vecnorm_moments_f32 / stg_vecnorm_merge_f64 /
// stg_vecnorm_apply_f32). Replaces Stable-Baselines3's VecNormalize with RunningMeanStd; the arithmetic is vecnorm_core.cuh.
//
// A wrapped env step is three launches after K1, with no host round trip:
//   moments  grid of STG_VECNORM_GRID(n) CTAs (a function of n alone). Each thread reads rows i, i + stride, ... as three 16-B
//            loads plus the reward and the return, writes the updated return, and accumulates 13 columns shifted by its first
//            row. Threads convert to (n, mean, M2) and merge by Chan's update through a fixed tree (warp shuffles, then the
//            CTA's eight warps); each CTA writes its partial to the work buffer, and the last CTA to finish (a counter in the work
//            buffer) folds the partials in a fixed tree over CTA indices. Which CTA is last does not change a bit. 72 B per env.
//   merge    one CTA: thread 0 folds the rank vectors in rank order, threads 0..12 apply update_from_moments to one feature
//            each, and the counts are written after a barrier. A separate launch, so no CTA of the moments grid reads
//            statistics this one writes.
//   apply    one env per thread: the CTA first computes sqrt(var + eps) for the 13 features into shared memory, then each
//            thread normalises its row (IEEE division, no contraction), its final row if the episode ended, and its reward, and
//            zeroes its return if the episode ended. 114 B per env plus 104 B per ended env.
// Observations are loaded through the read-only path with default caching: apply reads them again right after, and at
// 1,048,576 envs the 50 MB of observations K1 just wrote fit in the 126 MB L2.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stg.h"
#include "vecnorm_core.cuh"

namespace stg {

constexpr int kVnThreads = STG_VECNORM_THREADS;
constexpr int kVnWarps = kVnThreads / 32;
static_assert(kVnMoments == STG_VECNORM_MOMENTS && kVnFeat == STG_VECNORM_FEATURES, "stg.h and vecnorm_core.cuh disagree");

// Chan merge of this lane's vector with the one `off` lanes up (shuffle-down tree: lane 0 ends with the warp's vector), the
// arithmetic of vn_chan_merge one feature at a time, so that only two shuffled values are live
__device__ __forceinline__ void vn_warp_merge(double v[kVnMoments]) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double nb = __shfl_down_sync(0xffffffffu, v[0], off);
        double w, c;
        vn_chan_weights(v[0], nb, w, c);
#pragma unroll
        for (int f = 0; f < kVnFeat; ++f) {
            const double mb = __shfl_down_sync(0xffffffffu, v[1 + f], off);
            const double m2b = __shfl_down_sync(0xffffffffu, v[1 + kVnFeat + f], off);
            vn_chan_feature(v[1 + f], v[1 + kVnFeat + f], mb, m2b, w, c);
        }
        v[0] = v[0] + nb;
    }
}

// the CTA's vector on thread 0 (fixed tree: warps, then the eight warp vectors by warp 0)
__device__ __forceinline__ void vn_block_merge(double v[kVnMoments], double (*sm)[kVnMoments]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    vn_warp_merge(v);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kVnMoments; ++k) sm[warp][k] = v[k];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < kVnMoments; ++k) v[k] = lane < kVnWarps ? sm[lane][k] : 0.0;
        vn_warp_merge(v);
    }
}

struct VnRow {
    float4 o[3];
    double reward, ret;
};

__device__ __forceinline__ void vn_load(const StgVecNormArgs& a, int64_t i, bool with_ret, VnRow& r) {
    const float4* p = reinterpret_cast<const float4*>(a.d_obs) + i * 3;
    r.o[0] = __ldg(p);
    r.o[1] = __ldg(p + 1);
    r.o[2] = __ldg(p + 2);
    if (with_ret) {
        r.reward = __ldg(a.d_reward + i);
        r.ret = a.d_returns[i];
    }
}

__global__ void __launch_bounds__(kVnThreads, 2) vecnorm_moments_kernel(const StgVecNormArgs a) {
    __shared__ double sm[kVnWarps][kVnMoments];
    __shared__ bool is_last;
    const int64_t N = a.n_envs;
    const int64_t stride = (int64_t)gridDim.x * kVnThreads;
    const bool with_ret = a.d_reward != nullptr;
    const double gamma = a.gamma;
    // the thread's first row is the shift of its sums (observation columns kept as the f32 values they are)
    float x0[kVnObs];
    double r0 = 0.0, s1[kVnFeat], s2[kVnFeat];
    double n = 0.0;
#pragma unroll
    for (int f = 0; f < kVnFeat; ++f) s1[f] = s2[f] = 0.0;
    int64_t i = (int64_t)blockIdx.x * kVnThreads + threadIdx.x;
    VnRow cur;
    cur.reward = cur.ret = 0.0;
    if (i < N) {
        vn_load(a, i, with_ret, cur);
        const float* c = reinterpret_cast<const float*>(cur.o);
#pragma unroll
        for (int f = 0; f < kVnObs; ++f) x0[f] = c[f];
        if (with_ret) r0 = vn_return(cur.ret, gamma, cur.reward);
    }
    // software pipeline: the loads of row i + stride are issued before row i is accumulated
    for (; i < N; i += stride) {
        VnRow nxt;
        nxt.reward = nxt.ret = 0.0;
        if (i + stride < N) vn_load(a, i + stride, with_ret, nxt);
        const float* c = reinterpret_cast<const float*>(cur.o);
#pragma unroll
        for (int f = 0; f < kVnObs; ++f) {
            const double d = (double)c[f] - (double)x0[f];
            s1[f] += d;
            s2[f] += d * d;
        }
        if (with_ret) {
            const double r = vn_return(cur.ret, gamma, cur.reward);
            a.d_returns[i] = r;
            const double d = r - r0;
            s1[kVnObs] += d;
            s2[kVnObs] += d * d;
        }
        n += 1.0;
        cur = nxt;
    }
    double v[kVnMoments];
    v[0] = n;
#pragma unroll
    for (int f = 0; f < kVnObs; ++f) vn_shifted_to_moments(n, x0[f], s1[f], s2[f], v[1 + f], v[1 + kVnFeat + f]);
    vn_shifted_to_moments(n, r0, s1[kVnObs], s2[kVnObs], v[1 + kVnObs], v[1 + kVnFeat + kVnObs]);
    vn_block_merge(v, sm);
    if (gridDim.x == 1) {
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < kVnMoments; ++k) a.d_moments[k] = v[k];
        }
        return;
    }
    unsigned int* counter = reinterpret_cast<unsigned int*>(a.d_work + STG_VECNORM_MAX_CTAS * kVnMoments);
    if (threadIdx.x == 0) {
        double* part = a.d_work + (int64_t)blockIdx.x * kVnMoments;
#pragma unroll
        for (int k = 0; k < kVnMoments; ++k) part[k] = v[k];
        __threadfence();
        is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // the last CTA: thread t folds partials t, t + 256 (grid <= 296) in order, then the same fixed tree as above
    const unsigned G = gridDim.x;
#pragma unroll
    for (int k = 0; k < kVnMoments; ++k) v[k] = 0.0;
    for (unsigned b = threadIdx.x; b < G; b += kVnThreads) {
        const double* p = a.d_work + (int64_t)b * kVnMoments;       // vn_chan_merge(v, p), loaded through L2
        const double nb = __ldcg(p);
        double w, c;
        vn_chan_weights(v[0], nb, w, c);
#pragma unroll
        for (int f = 0; f < kVnFeat; ++f)
            vn_chan_feature(v[1 + f], v[1 + kVnFeat + f], __ldcg(p + 1 + f), __ldcg(p + 1 + kVnFeat + f), w, c);
        v[0] = v[0] + nb;
    }
    __syncthreads();                  // sm is reused
    vn_block_merge(v, sm);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kVnMoments; ++k) a.d_moments[k] = v[k];
        *counter = 0u;
    }
}

__global__ void __launch_bounds__(32) vecnorm_merge_kernel(const StgVecNormArgs a) {
    __shared__ double batch[kVnMoments];
    const int f = threadIdx.x;
    if (f == 0) vn_fold(a.d_moments, a.n_ranks, batch);
    __syncthreads();
    const double bn = batch[0];
    const bool train = (a.flags & STG_VECNORM_TRAINING) != 0u;
    const bool upd_obs = train && (a.flags & STG_VECNORM_NORM_OBS) != 0u && bn > 0.0;
    const bool upd_ret = train && a.d_reward != nullptr && bn > 0.0;
    double* s = a.d_stats;
    const double obs_count = s[STG_VECNORM_OBS_COUNT], ret_count = s[STG_VECNORM_RET_COUNT];
    if (f < kVnObs && upd_obs) {
        double mean = s[STG_VECNORM_OBS_MEAN + f], var = s[STG_VECNORM_OBS_VAR + f];
        vn_update_from_moments(mean, var, obs_count, batch[1 + f], ddiv(batch[1 + kVnFeat + f], bn), bn);
        s[STG_VECNORM_OBS_MEAN + f] = mean;
        s[STG_VECNORM_OBS_VAR + f] = var;
    }
    if (f == kVnObs && upd_ret) {
        double mean = s[STG_VECNORM_RET_MEAN], var = s[STG_VECNORM_RET_VAR];
        vn_update_from_moments(mean, var, ret_count, batch[1 + kVnObs], ddiv(batch[1 + kVnFeat + kVnObs], bn), bn);
        s[STG_VECNORM_RET_MEAN] = mean;
        s[STG_VECNORM_RET_VAR] = var;
    }
    __syncthreads();                  // every thread has read the old counts
    if (f == 0 && upd_obs) s[STG_VECNORM_OBS_COUNT] = dadd(bn, obs_count);
    if (f == 1 && upd_ret) s[STG_VECNORM_RET_COUNT] = dadd(bn, ret_count);
}

__device__ __forceinline__ void vn_norm_row(const float* src, float* dst, int64_t i, const double* mean, const double* scale,
                                            double clip, bool norm) {
    const float4* p = reinterpret_cast<const float4*>(src) + i * 3;
    float4* q = reinterpret_cast<float4*>(dst) + i * 3;
    float4 v[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
    if (norm) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            v[j].x = vn_norm_obs(v[j].x, mean[4 * j], scale[4 * j], clip);
            v[j].y = vn_norm_obs(v[j].y, mean[4 * j + 1], scale[4 * j + 1], clip);
            v[j].z = vn_norm_obs(v[j].z, mean[4 * j + 2], scale[4 * j + 2], clip);
            v[j].w = vn_norm_obs(v[j].w, mean[4 * j + 3], scale[4 * j + 3], clip);
        }
    }
    q[0] = v[0];
    q[1] = v[1];
    q[2] = v[2];
}

__global__ void __launch_bounds__(kVnThreads) vecnorm_apply_kernel(const StgVecNormArgs a) {
    __shared__ double mean[kVnObs], scale[kVnFeat];
    const int t = threadIdx.x;
    if (t < kVnObs) {
        mean[t] = a.d_stats[STG_VECNORM_OBS_MEAN + t];
        scale[t] = vn_scale(a.d_stats[STG_VECNORM_OBS_VAR + t], a.epsilon);
    } else if (t == kVnObs) {
        scale[t] = vn_scale(a.d_stats[STG_VECNORM_RET_VAR], a.epsilon);
    }
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * kVnThreads + t;
    if (i >= a.n_envs) return;
    const bool norm_obs = (a.flags & STG_VECNORM_NORM_OBS) != 0u;
    bool ended = false;
    if (a.d_terminated) ended = (__ldg(a.d_terminated + i) | __ldg(a.d_truncated + i)) != 0;
    if (a.d_obs) vn_norm_row(a.d_obs, a.d_obs_out, i, mean, scale, a.clip_obs, norm_obs);
    if (a.d_final_obs && ended) vn_norm_row(a.d_final_obs, a.d_final_obs_out, i, mean, scale, a.clip_obs, norm_obs);
    if (a.d_reward) {
        const double r = __ldg(a.d_reward + i);
        a.d_reward_out[i] = (a.flags & STG_VECNORM_NORM_REWARD) ? vn_norm_reward(r, scale[kVnObs], a.clip_reward) : r;
    }
    if (a.d_returns && ended) a.d_returns[i] = 0.0;
}

}  // namespace stg

extern "C" int stg_vecnorm_moments_f32(const StgVecNormArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgVecNormArgs& a = *args;
    if (a.n_envs < 0) return STG_E_SIZE;
    if (a.n_envs == 0) return STG_OK;
    if (!a.d_obs || !a.d_moments || !a.d_work || (a.d_reward && !a.d_returns)) return STG_E_NULL;
    if ((uintptr_t)a.d_obs & 15u) return STG_E_ALIGN;
    const int64_t grid = STG_VECNORM_GRID(a.n_envs);
    stg::vecnorm_moments_kernel<<<(unsigned)grid, stg::kVnThreads, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

extern "C" int stg_vecnorm_merge_f64(const StgVecNormArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgVecNormArgs& a = *args;
    if (a.n_ranks < 1) return STG_E_SIZE;
    if (!a.d_moments || !a.d_stats) return STG_E_NULL;
    stg::vecnorm_merge_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

extern "C" int stg_vecnorm_apply_f32(const StgVecNormArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgVecNormArgs& a = *args;
    if (a.n_envs < 0) return STG_E_SIZE;
    if (a.n_envs == 0) return STG_OK;
    if (!a.d_stats) return STG_E_NULL;
    const bool obs = a.d_obs || a.d_obs_out, fin = a.d_final_obs || a.d_final_obs_out, rew = a.d_reward || a.d_reward_out;
    if ((obs && !(a.d_obs && a.d_obs_out)) || (fin && !(a.d_final_obs && a.d_final_obs_out)) ||
        (rew && !(a.d_reward && a.d_reward_out)))
        return STG_E_NULL;
    if (!obs && !fin && !rew) return STG_E_NULL;
    if (!a.d_terminated != !a.d_truncated) return STG_E_NULL;
    if (fin && !a.d_terminated) return STG_E_NULL;
    if (((uintptr_t)a.d_obs | (uintptr_t)a.d_obs_out | (uintptr_t)a.d_final_obs | (uintptr_t)a.d_final_obs_out) & 15u)
        return STG_E_ALIGN;
    const int64_t grid = (a.n_envs + stg::kVnThreads - 1) / stg::kVnThreads;
    if (grid > 0x7fffffff) return STG_E_SIZE;
    stg::vecnorm_apply_kernel<<<(unsigned)grid, stg::kVnThreads, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}
