// policy_kernels.cu — K9: ActorCriticPolicy rollout inference (include/stg.h, stg_policy_act_f32 / stg_policy_value_f32). The
// per-env arithmetic is policy_core.cuh; this file tiles it.
//
// Both kernels are persistent: each CTA copies the 40.75 KB weight buffer into shared memory once and then walks tiles of
// kPolTile envs. A tile's observations are stored transposed (x[k][env]) and each layer is a [tile x K] . [K x 64] product,
// register-tiled like an SGEMM microkernel: thread (ty, tx) owns envs ty*4 .. ty*4+3 and outputs tx*4 .. tx*4+3 and
// 32+tx*4 .. 32+tx*4+3, so per k it issues three 128-bit shared loads (4 activations, 8 weights, conflict-free) for 32 FFMAs.
// The tanh of each layer is written back transposed (h[o][env]) for the next layer; the plane's row stride kPolTile + 4 spreads
// those 128-bit stores over the banks. Every output is one fma chain in ascending k started from the bias, the same in every
// thread and every tile, so the bits of an env do not depend on where it lands. The critic runs first (its head kept in a
// register), then the actor; the heads (64 -> 1, 64 -> 2) are one env per thread.
//
// The value kernel compacts: each CTA scans its contiguous range of 256-row windows, appends the rows whose mask is set to a
// queue in shared memory (warp ballots, in row order) and computes the critic whenever kPolTile rows are queued, so a step
// where 1 % of the envs ended costs the mask scan plus 1 % of the dense work.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stg.h"
#include "policy_core.cuh"

namespace stg {

constexpr int kPolThreads = 256;
constexpr int kPolEnvsPerThread = 4;
constexpr int kPolTile = 32 * kPolEnvsPerThread;       // 32 env groups x 8 output groups = 256 threads
constexpr int kPolStride = kPolTile + 4;               // row stride of the transposed activation planes
constexpr int kPolWindow = kPolThreads;                // rows scanned per step of the value kernel
static_assert(STG_POLICY_FLOATS % 4 == 0 && STG_POLICY_HIDDEN == 64 && STG_POLICY_OBS == 12, "layout of stg.h");

struct PolShared {
    float w[STG_POLICY_FLOATS];
    float x[kPolObs * kPolStride];
    float h[kPolHidden * kPolStride];
    int64_t rows[kPolTile + kPolWindow];              // value kernel: queue of selected rows
    int warp_count[kPolThreads / 32];
};

__device__ __forceinline__ void pol_load_weights(PolShared& s, const float* __restrict__ w) {
    const float4* src = reinterpret_cast<const float4*>(w);
    float4* dst = reinterpret_cast<float4*>(s.w);
    for (int i = threadIdx.x; i < STG_POLICY_FLOATS / 4; i += kPolThreads) dst[i] = __ldg(src + i);
}

// observations of tile rows r < count into s.x (transposed, zero rows past count); row r is env row_of(r)
template <typename RowOf>
__device__ __forceinline__ void pol_load_tile(PolShared& s, const float* __restrict__ obs, float* obs_copy, int count,
                                              RowOf row_of) {
    for (int q = threadIdx.x; q < 3 * kPolTile; q += kPolThreads) {
        const int r = q / 3, part = q - 3 * r;
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (r < count) {
            const int64_t g = row_of(r);
            v = __ldg(reinterpret_cast<const float4*>(obs) + g * 3 + part);
            if (obs_copy) reinterpret_cast<float4*>(obs_copy)[g * 3 + part] = v;
        }
        float* col = s.x + (part * 4) * kPolStride + r;
        col[0] = v.x;
        col[kPolStride] = v.y;
        col[2 * kPolStride] = v.z;
        col[3 * kPolStride] = v.w;
    }
}

// s.h[o][env] = tanh(b[o] + sum_k in[k][env] W[k][o]) for the whole tile. `in` may be s.h: every thread has finished reading
// it at the first barrier. Ends with a barrier.
template <int K>
__device__ __forceinline__ void pol_layer(PolShared& s, const float* in, int w_off, int b_off) {
    const int tx = threadIdx.x & 7, ty = threadIdx.x >> 3;
    const float* W = s.w + w_off;
    float acc[kPolEnvsPerThread][8];
    {
        const float4 b0 = *reinterpret_cast<const float4*>(s.w + b_off + tx * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(s.w + b_off + 32 + tx * 4);
#pragma unroll
        for (int i = 0; i < kPolEnvsPerThread; ++i) {
            acc[i][0] = b0.x; acc[i][1] = b0.y; acc[i][2] = b0.z; acc[i][3] = b0.w;
            acc[i][4] = b1.x; acc[i][5] = b1.y; acc[i][6] = b1.z; acc[i][7] = b1.w;
        }
    }
#pragma unroll 16
    for (int k = 0; k < K; ++k) {
        const float4 xv = *reinterpret_cast<const float4*>(in + k * kPolStride + ty * kPolEnvsPerThread);
        const float4 w0 = *reinterpret_cast<const float4*>(W + k * 64 + tx * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(W + k * 64 + 32 + tx * 4);
        const float xa[4] = {xv.x, xv.y, xv.z, xv.w};
        const float wa[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < kPolEnvsPerThread; ++i) {
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(xa[i], wa[j], acc[i][j]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int o = (j < 4 ? 0 : 32) + tx * 4 + (j & 3);
        *reinterpret_cast<float4*>(s.h + o * kPolStride + ty * kPolEnvsPerThread) =
            make_float4(tanhf(acc[0][j]), tanhf(acc[1][j]), tanhf(acc[2][j]), tanhf(acc[3][j]));
    }
    __syncthreads();
}

// head output `o` of a 64 -> n_out layer for tile env `e` (one thread per env)
__device__ __forceinline__ float pol_head(const PolShared& s, int e, int w_off, int n_out, int o, float b) {
    float acc = b;
#pragma unroll 16
    for (int k = 0; k < kPolHidden; ++k) acc = fmaf(s.h[k * kPolStride + e], s.w[w_off + k * n_out + o], acc);
    return acc;
}

// the critic of the tile in s.x: V of tile env threadIdx.x (threads < kPolTile)
__device__ __forceinline__ float pol_critic(PolShared& s) {
    pol_layer<kPolObs>(s, s.x, STG_POLICY_VF_W1, STG_POLICY_VF_B1);
    pol_layer<kPolHidden>(s, s.h, STG_POLICY_VF_W2, STG_POLICY_VF_B2);
    float v = 0.0f;
    if (threadIdx.x < kPolTile) v = pol_head(s, threadIdx.x, STG_POLICY_VAL_W, 1, 0, s.w[STG_POLICY_VAL_B]);
    return v;
}

__global__ void __launch_bounds__(kPolThreads, 2) policy_act_kernel(const StgPolicyArgs a) {
    extern __shared__ __align__(16) unsigned char pol_smem[];
    PolShared& s = *reinterpret_cast<PolShared*>(pol_smem);
    pol_load_weights(s, a.d_weights);
    const int64_t n = a.n_envs, tiles = (n + kPolTile - 1) / kPolTile;
    const bool sample = (a.flags & STG_POLICY_DETERMINISTIC) == 0u;
    const int e = threadIdx.x;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * kPolTile;
        const int count = n - base < kPolTile ? (int)(n - base) : kPolTile;
        pol_load_tile(s, a.d_obs, a.d_obs_copy, count, [base](int r) { return base + r; });
        __syncthreads();
        const float v = pol_critic(s);
        // the actor's first layer writes s.h only after its first barrier: the critic head above has read it by then
        pol_layer<kPolObs>(s, s.x, STG_POLICY_PI_W1, STG_POLICY_PI_B1);
        pol_layer<kPolHidden>(s, s.h, STG_POLICY_PI_W2, STG_POLICY_PI_B2);
        if (e < count) {
            const int64_t i = base + e;
            float mean[2], act[2], eps[2] = {0.0f, 0.0f};
            mean[0] = pol_head(s, e, STG_POLICY_ACT_W, 2, 0, s.w[STG_POLICY_ACT_B]);
            mean[1] = pol_head(s, e, STG_POLICY_ACT_W, 2, 1, s.w[STG_POLICY_ACT_B + 1]);
            if (sample) pol_eps(a.key[0], a.key[1], a.env_offset + (uint64_t)i, a.draw, eps[0], eps[1]);
            float lp = 0.0f;
#pragma unroll
            for (int d = 0; d < 2; ++d) {
                act[d] = sample ? pol_sample(mean[d], eps[d], s.w[STG_POLICY_STD + d]) : mean[d];
                const float t = pol_log_prob_term(act[d], mean[d], s.w[STG_POLICY_STD + d], s.w[STG_POLICY_LOG_SCALE + d]);
                lp = d == 0 ? t : Pk<float>::add(lp, t);
            }
            if (a.d_action) reinterpret_cast<float2*>(a.d_action)[i] = make_float2(act[0], act[1]);
            if (a.d_env_action)
                reinterpret_cast<float2*>(a.d_env_action)[i] =
                    make_float2(pol_rescale(act[0], a.action_low[0], a.action_high[0]),
                                pol_rescale(act[1], a.action_low[1], a.action_high[1]));
            if (a.d_value) a.d_value[i] = v;
            if (a.d_log_prob) a.d_log_prob[i] = lp;
        }
        // the next tile's loads write s.x (last read before the actor's barriers) and its first layer writes s.h after a
        // barrier, so the actor heads above need no barrier of their own
    }
}

__device__ __forceinline__ void pol_value_tile(PolShared& s, const StgPolicyArgs& a, int count) {
    pol_load_tile(s, a.d_obs, nullptr, count, [&s](int r) { return s.rows[r]; });
    __syncthreads();
    const float v = pol_critic(s);
    if ((int)threadIdx.x < count) a.d_value[s.rows[threadIdx.x]] = v;
    __syncthreads();                  // s.rows is rewritten next
}

__global__ void __launch_bounds__(kPolThreads, 2) policy_value_kernel(const StgPolicyArgs a) {
    extern __shared__ __align__(16) unsigned char pol_smem[];
    PolShared& s = *reinterpret_cast<PolShared*>(pol_smem);
    pol_load_weights(s, a.d_weights);
    const int64_t n = a.n_envs, windows = (n + kPolWindow - 1) / kPolWindow;
    const int64_t per_cta = (windows + gridDim.x - 1) / gridDim.x;
    const int64_t w0 = blockIdx.x * per_cta, w1 = w0 + per_cta < windows ? w0 + per_cta : windows;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    int queued = 0;                   // the same in every thread
    for (int64_t w = w0; w < w1; ++w) {
        const int64_t g = w * kPolWindow + t;
        const bool sel = g < n && (a.d_mask == nullptr || __ldg(a.d_mask + g) != 0);
        const unsigned ballot = __ballot_sync(0xffffffffu, sel);
        if (lane == 0) s.warp_count[warp] = __popc(ballot);
        __syncthreads();
        int before = queued, total = queued;
#pragma unroll
        for (int q = 0; q < kPolThreads / 32; ++q) {
            const int c = s.warp_count[q];
            before += q < warp ? c : 0;
            total += c;
        }
        if (sel) s.rows[before + __popc(ballot & ((1u << lane) - 1u))] = g;
        __syncthreads();
        queued = total;
        while (queued >= kPolTile) {
            pol_value_tile(s, a, kPolTile);
            const int rest = queued - kPolTile;
            const int64_t moved = t < rest ? s.rows[kPolTile + t] : 0;
            __syncthreads();
            if (t < rest) s.rows[t] = moved;
            __syncthreads();
            queued = rest;
        }
    }
    if (queued > 0) pol_value_tile(s, a, queued);
}

struct PolLaunch {
    int sms = 0, per_sm = 0;
};

// per device: SM count and resident CTAs per SM of the two kernels (their shared-memory footprint bounds it at 2)
static int pol_configure(PolLaunch& out) {
    static PolLaunch cache[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev >= 0 && dev < 64 && cache[dev].sms > 0) {
        out = cache[dev];
        return 0;
    }
    const int smem = (int)sizeof(PolShared);
    PolLaunch l;
    if ((e = cudaFuncSetAttribute(policy_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(policy_value_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess ||
        (e = cudaDeviceGetAttribute(&l.sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&l.per_sm, policy_act_kernel, kPolThreads, smem)) != cudaSuccess)
        return (int)e;
    if (l.per_sm < 1) l.per_sm = 1;
    if (dev >= 0 && dev < 64) cache[dev] = l;
    out = l;
    return 0;
}

static int pol_check(const StgPolicyArgs& a) {
    if (((uintptr_t)a.d_obs | (uintptr_t)a.d_weights | (uintptr_t)a.d_obs_copy) & 15u) return STG_E_ALIGN;
    if (((uintptr_t)a.d_action | (uintptr_t)a.d_env_action) & 7u) return STG_E_ALIGN;
    if (a.flags & ~STG_POLICY_DETERMINISTIC) return STG_E_ENUM;
    return STG_OK;
}

}  // namespace stg

extern "C" int stg_policy_act_f32(const StgPolicyArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgPolicyArgs& a = *args;
    if (a.n_envs < 0) return STG_E_SIZE;
    if (a.n_envs == 0) return STG_OK;
    if (!a.d_obs || !a.d_weights) return STG_E_NULL;
    if (!a.d_obs_copy && !a.d_action && !a.d_env_action && !a.d_value && !a.d_log_prob) return STG_E_NULL;
    if (int rc = stg::pol_check(a)) return rc;
    stg::PolLaunch l;
    if (int rc = stg::pol_configure(l)) return rc;
    const int64_t tiles = (a.n_envs + stg::kPolTile - 1) / stg::kPolTile;
    const int64_t grid = tiles < (int64_t)l.sms * l.per_sm ? tiles : (int64_t)l.sms * l.per_sm;
    stg::policy_act_kernel<<<(unsigned)grid, stg::kPolThreads, sizeof(stg::PolShared), (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

extern "C" int stg_policy_value_f32(const StgPolicyArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgPolicyArgs& a = *args;
    if (a.n_envs < 0) return STG_E_SIZE;
    if (a.n_envs == 0) return STG_OK;
    if (!a.d_obs || !a.d_weights || !a.d_value) return STG_E_NULL;
    if (int rc = stg::pol_check(a)) return rc;
    stg::PolLaunch l;
    if (int rc = stg::pol_configure(l)) return rc;
    const int64_t windows = (a.n_envs + stg::kPolWindow - 1) / stg::kPolWindow;
    const int64_t grid = windows < (int64_t)l.sms * l.per_sm ? windows : (int64_t)l.sms * l.per_sm;
    stg::policy_value_kernel<<<(unsigned)grid, stg::kPolThreads, sizeof(stg::PolShared), (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}
