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

__device__ __forceinline__ void pol_load_weights(float* sw, const float* __restrict__ w) {
    const float4* src = reinterpret_cast<const float4*>(w);
    float4* dst = reinterpret_cast<float4*>(sw);
    for (int i = threadIdx.x; i < STG_POLICY_FLOATS / 4; i += kPolThreads) dst[i] = __ldg(src + i);
}

// observations of tile rows r < count into the plane sx (transposed, zero rows past count); row r is env row_of(r)
template <typename RowOf>
__device__ __forceinline__ void pol_load_tile(float* sx, const float* __restrict__ obs, float* obs_copy, int count,
                                              RowOf row_of) {
    for (int q = threadIdx.x; q < 3 * kPolTile; q += kPolThreads) {
        const int r = q / 3, part = q - 3 * r;
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (r < count) {
            const int64_t g = row_of(r);
            v = __ldg(reinterpret_cast<const float4*>(obs) + g * 3 + part);
            if (obs_copy) reinterpret_cast<float4*>(obs_copy)[g * 3 + part] = v;
        }
        float* col = sx + (part * 4) * kPolStride + r;
        col[0] = v.x;
        col[kPolStride] = v.y;
        col[2 * kPolStride] = v.z;
        col[3 * kPolStride] = v.w;
    }
}

// out[o][env] = tanh(b[o] + sum_k in[k][env] W[k][o]) for the whole tile (sw: the weights in shared memory). `in` may be
// `out`: every thread has finished reading it at the first barrier. Ends with a barrier.
template <int K>
__device__ __forceinline__ void pol_layer(const float* sw, const float* in, float* out, int w_off, int b_off) {
    const int tx = threadIdx.x & 7, ty = threadIdx.x >> 3;
    const float* W = sw + w_off;
    float acc[kPolEnvsPerThread][8];
    {
        const float4 b0 = *reinterpret_cast<const float4*>(sw + b_off + tx * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(sw + b_off + 32 + tx * 4);
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
        *reinterpret_cast<float4*>(out + o * kPolStride + ty * kPolEnvsPerThread) =
            make_float4(tanhf(acc[0][j]), tanhf(acc[1][j]), tanhf(acc[2][j]), tanhf(acc[3][j]));
    }
    __syncthreads();
}

// head output `o` of a 64 -> n_out layer on the plane h for tile env `e` (one thread per env)
__device__ __forceinline__ float pol_head(const float* sw, const float* h, int e, int w_off, int n_out, int o, float b) {
    float acc = b;
#pragma unroll 16
    for (int k = 0; k < kPolHidden; ++k) acc = fmaf(h[k * kPolStride + e], sw[w_off + k * n_out + o], acc);
    return acc;
}

// the critic of the tile in s.x: V of tile env threadIdx.x (threads < kPolTile)
__device__ __forceinline__ float pol_critic(PolShared& s) {
    pol_layer<kPolObs>(s.w, s.x, s.h, STG_POLICY_VF_W1, STG_POLICY_VF_B1);
    pol_layer<kPolHidden>(s.w, s.h, s.h, STG_POLICY_VF_W2, STG_POLICY_VF_B2);
    float v = 0.0f;
    if (threadIdx.x < kPolTile) v = pol_head(s.w, s.h, threadIdx.x, STG_POLICY_VAL_W, 1, 0, s.w[STG_POLICY_VAL_B]);
    return v;
}

__global__ void __launch_bounds__(kPolThreads, 2) policy_act_kernel(const StgPolicyArgs a) {
    extern __shared__ __align__(16) unsigned char pol_smem[];
    PolShared& s = *reinterpret_cast<PolShared*>(pol_smem);
    pol_load_weights(s.w, a.d_weights);
    const int64_t n = a.n_envs, tiles = (n + kPolTile - 1) / kPolTile;
    const bool sample = (a.flags & STG_POLICY_DETERMINISTIC) == 0u;
    const int e = threadIdx.x;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * kPolTile;
        const int count = n - base < kPolTile ? (int)(n - base) : kPolTile;
        pol_load_tile(s.x, a.d_obs, a.d_obs_copy, count, [base](int r) { return base + r; });
        __syncthreads();
        const float v = pol_critic(s);
        // the actor's first layer writes s.h only after its first barrier: the critic head above has read it by then
        pol_layer<kPolObs>(s.w, s.x, s.h, STG_POLICY_PI_W1, STG_POLICY_PI_B1);
        pol_layer<kPolHidden>(s.w, s.h, s.h, STG_POLICY_PI_W2, STG_POLICY_PI_B2);
        if (e < count) {
            const int64_t i = base + e;
            float mean[2], act[2], eps[2] = {0.0f, 0.0f};
            mean[0] = pol_head(s.w, s.h, e, STG_POLICY_ACT_W, 2, 0, s.w[STG_POLICY_ACT_B]);
            mean[1] = pol_head(s.w, s.h, e, STG_POLICY_ACT_W, 2, 1, s.w[STG_POLICY_ACT_B + 1]);
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
    pol_load_tile(s.x, a.d_obs, nullptr, count, [&s](int r) { return s.rows[r]; });
    __syncthreads();
    const float v = pol_critic(s);
    if ((int)threadIdx.x < count) a.d_value[s.rows[threadIdx.x]] = v;
    __syncthreads();                  // s.rows is rewritten next
}

__global__ void __launch_bounds__(kPolThreads, 2) policy_value_kernel(const StgPolicyArgs a) {
    extern __shared__ __align__(16) unsigned char pol_smem[];
    PolShared& s = *reinterpret_cast<PolShared*>(pol_smem);
    pol_load_weights(s.w, a.d_weights);
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

// ---- K10: PPO and A2C loss and gradient (stg_policy_ppo_grad_f32, stg_policy_a2c_grad_f32) -------------------------------
// A grid of STG_PPO_GRID(B) persistent CTAs walks tiles of kPolTile rows (CTA b: tiles b, b + grid, ...). Per tile and network
// (the critic, then the actor, so that only one network's activations are held):
//   forward   pol_layer twice: h1 into plane a, h2 into plane h (K9's chains and bits);
//   head      one row per thread: the value or the means and log-probability (pol_head), the loss terms and the head
//             gradient into s.g (pol_ppo_value_row / pol_ppo_policy_row / pol_ppo_gauss_row);
//   delta2    warp w takes outputs o = w + 8j, lane l rows 4l .. 4l+3: d2 = (W_head g) * (1 - h2^2) written over h2, with
//             the head-weight and bias-2 tile sums reduced over the warp by xor shuffles (the same bits in every lane);
//   dW2       thread (kg = t & 15, og = t >> 4) sums h1[kg + 16i][e] d2[4og + j][e] over the tile's rows: a 4 x 4 register
//             tile, per 4 rows 8 conflict-free 128-bit loads (a quarter warp reads 8 k rows 132 floats apart) for 64 FFMA;
//   delta1    d1[k][e] = (sum_o W2[k][o] d2[o][e]) (1 - h1^2), written over h1: thread (eg, kg) owns rows 4eg .. 4eg+3 and
//             k = 8kg .. 8kg+7, a quarter warp shares kg (its W2 loads broadcast) and reads 8 consecutive row groups of d2;
//             per 4 o 12 loads for 128 FFMA, one fma chain in ascending o per output;
//   dW1, b1   thread (o = t >> 2, kq = t & 3) sums x[kq + 4i][e] d1[o][e] and d1[o][e] over the rows.
// Every weight-gradient tile sum is one FP32 fma chain over the tile's rows in ascending order; each thread adds its tile sums
// in FP64 to its CTA's partial in d_work (always the same thread for the same element, so no atomics). The per-row sums (loss
// terms, log_std) are FP64 in the row's thread and reduced in thread order at the end. ppo_fold_kernel then sums the partials
// in CTA order. Shared memory: 40.75 KB of weights, x, two 64-row planes and two 128-row gradient channels, 113.0 KB, so two
// CTAs fit on an SM. The loss is a template parameter: the A2C instance takes pol_a2c_policy_row as its policy head, has no
// value clip and reads neither old plane; the tiling, the backward pass and the fold are the same code.
constexpr int kPpoSums = 6;                             // per-row FP64 sums: the four loss sums and d/d log_std
static_assert(STG_PPO_TILE == kPolTile && kPolThreads == 256, "stg.h and the K10 tiling disagree");

struct PpoShared {
    float w[STG_POLICY_FLOATS];
    float x[kPolObs * kPolStride];
    float a[kPolHidden * kPolStride];                 // h1, then d1
    float h[kPolHidden * kPolStride];                 // h2, then d2
    float g[2][kPolTile];                              // head gradient of each row: d/d value, or d/d mean_0, mean_1
};

__device__ __forceinline__ void ppo_add(double* part, int idx, float v, bool first) {
    part[idx] = first ? (double)v : part[idx] + (double)v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// d2 over h2 in place and the tile sums of the head weights, the head bias and bias 2 (n_out = 1: critic, 2: actor)
template <int NOUT>
__device__ __forceinline__ void ppo_delta2(PpoShared& s, int w_head, int g_head, int b_head, int b2, double* part, bool first) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 g[NOUT];
#pragma unroll
    for (int d = 0; d < NOUT; ++d) g[d] = *reinterpret_cast<const float4*>(&s.g[d][lane * 4]);
    if (warp == 0) {
#pragma unroll
        for (int d = 0; d < NOUT; ++d) {
            const float t = warp_sum(((g[d].x + g[d].y) + g[d].z) + g[d].w);
            if (lane == 0) ppo_add(part, b_head + d, t, first);
        }
    }
#pragma unroll 2
    for (int j = 0; j < kPolHidden / 8; ++j) {
        const int o = warp + 8 * j;
        float4* hp = reinterpret_cast<float4*>(s.h + o * kPolStride + lane * 4);
        const float4 h = *hp;
        float wh[NOUT];
#pragma unroll
        for (int d = 0; d < NOUT; ++d) wh[d] = s.w[w_head + o * NOUT + d];
        const float hv[4] = {h.x, h.y, h.z, h.w};
        float dv[4], hw[NOUT], db = 0.0f;
#pragma unroll
        for (int d = 0; d < NOUT; ++d) hw[d] = 0.0f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float gi[2] = {(&g[0].x)[i], NOUT > 1 ? (&g[NOUT - 1].x)[i] : 0.0f};
            float sum = Pk<float>::mul(wh[0], gi[0]);
#pragma unroll
            for (int d = 1; d < NOUT; ++d) sum = Pk<float>::add(sum, Pk<float>::mul(wh[d], gi[d]));
            dv[i] = pol_dtanh(sum, hv[i]);
#pragma unroll
            for (int d = 0; d < NOUT; ++d) hw[d] = fmaf(hv[i], gi[d], hw[d]);
            db += dv[i];
        }
        *hp = make_float4(dv[0], dv[1], dv[2], dv[3]);
#pragma unroll
        for (int d = 0; d < NOUT; ++d) hw[d] = warp_sum(hw[d]);
        db = warp_sum(db);
        if (lane == 0) {
#pragma unroll
            for (int d = 0; d < NOUT; ++d) ppo_add(part, g_head + d * kPolHidden + o, hw[d], first);
            ppo_add(part, b2 + o, db, first);
        }
    }
    __syncthreads();
}

// dW2[o][k] += sum over the tile's rows of h1[k][e] d2[o][e]
__device__ __forceinline__ void ppo_dw2(const PpoShared& s, int gw2, double* part, bool first) {
    const int kg = threadIdx.x & 15, og = threadIdx.x >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
#pragma unroll 4
    for (int e = 0; e < kPolTile; e += 4) {
        float4 hv[4], dv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) hv[i] = *reinterpret_cast<const float4*>(s.a + (kg + 16 * i) * kPolStride + e);
#pragma unroll
        for (int j = 0; j < 4; ++j) dv[j] = *reinterpret_cast<const float4*>(s.h + (og * 4 + j) * kPolStride + e);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[i][j] = fmaf(hv[i].x, dv[j].x, acc[i][j]);
                acc[i][j] = fmaf(hv[i].y, dv[j].y, acc[i][j]);
                acc[i][j] = fmaf(hv[i].z, dv[j].z, acc[i][j]);
                acc[i][j] = fmaf(hv[i].w, dv[j].w, acc[i][j]);
            }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) ppo_add(part, gw2 + (og * 4 + j) * kPolHidden + kg + 16 * i, acc[i][j], first);
    __syncthreads();                  // plane a is overwritten next
}

// d1 = (W2 d2) (1 - h1^2) over h1 in plane a
__device__ __forceinline__ void ppo_delta1(PpoShared& s, int w2) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int eg = (lane & 7) + 8 * (warp & 3), kg = (lane >> 3) + 4 * (warp >> 2);
    const float* W = s.w + w2 + kg * 8 * kPolHidden;
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int m = 0; m < 8; ++m) acc[i][m] = 0.0f;
#pragma unroll 2
    for (int o = 0; o < kPolHidden; o += 4) {
        float4 dv[4], wv[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) dv[q] = *reinterpret_cast<const float4*>(s.h + (o + q) * kPolStride + eg * 4);
#pragma unroll
        for (int m = 0; m < 8; ++m) wv[m] = *reinterpret_cast<const float4*>(W + m * kPolHidden + o);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float d[4] = {(&dv[q].x)[0], (&dv[q].x)[1], (&dv[q].x)[2], (&dv[q].x)[3]};
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                const float wq = (&wv[m].x)[q];
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i][m] = fmaf(wq, d[i], acc[i][m]);
            }
        }
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        float4* hp = reinterpret_cast<float4*>(s.a + (kg * 8 + m) * kPolStride + eg * 4);
        const float4 h = *hp;
        *hp = make_float4(pol_dtanh(acc[0][m], h.x), pol_dtanh(acc[1][m], h.y), pol_dtanh(acc[2][m], h.z),
                          pol_dtanh(acc[3][m], h.w));
    }
    __syncthreads();
}

// dW1[o][k] += sum of x[k][e] d1[o][e], db1[o] += sum of d1[o][e], over the tile's rows
__device__ __forceinline__ void ppo_dw1(const PpoShared& s, int gw1, int gb1, double* part, bool first) {
    const int o = threadIdx.x >> 2, kq = threadIdx.x & 3;
    float acc[3] = {0.0f, 0.0f, 0.0f}, db = 0.0f;
#pragma unroll 4
    for (int e = 0; e < kPolTile; e += 4) {
        const float4 dv = *reinterpret_cast<const float4*>(s.a + o * kPolStride + e);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float4 xv = *reinterpret_cast<const float4*>(s.x + (kq + 4 * i) * kPolStride + e);
            acc[i] = fmaf(xv.x, dv.x, acc[i]);
            acc[i] = fmaf(xv.y, dv.y, acc[i]);
            acc[i] = fmaf(xv.z, dv.z, acc[i]);
            acc[i] = fmaf(xv.w, dv.w, acc[i]);
        }
        db = (((db + dv.x) + dv.y) + dv.z) + dv.w;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) ppo_add(part, gw1 + o * kPolObs + kq + 4 * i, acc[i], first);
    if (kq == 0) ppo_add(part, gb1 + o, db, first);
}

template <PolLoss kLoss>
__global__ void __launch_bounds__(kPolThreads, 2) policy_ppo_grad_kernel(const StgPpoArgs a) {
    extern __shared__ __align__(16) unsigned char pol_smem[];
    PpoShared& s = *reinterpret_cast<PpoShared*>(pol_smem);
    pol_load_weights(s.w, a.d_weights);
    const int64_t n = a.batch, tiles = (n + kPolTile - 1) / kPolTile;
    const int e = threadIdx.x;
    const PolPpoCoef c{a.clip_range, a.ratio_lo, a.ratio_hi, a.clip_range_vf,
                       kLoss == kLossPpo && (a.flags & STG_PPO_CLIP_VF) != 0u};
    float stats[2] = {0.0f, 0.0f};
    if (a.d_adv_stats) stats[0] = __ldg(a.d_adv_stats), stats[1] = __ldg(a.d_adv_stats + 1);
    double* part = a.d_work + (int64_t)blockIdx.x * STG_PPO_PART;
    double sums[kPpoSums];
#pragma unroll
    for (int k = 0; k < kPpoSums; ++k) sums[k] = 0.0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * kPolTile;
        const int count = n - base < kPolTile ? (int)(n - base) : kPolTile;
        const bool first = tile == blockIdx.x;
        pol_load_tile(s.x, a.d_obs, nullptr, count, [base](int r) { return base + r; });
        __syncthreads();
        // ---- critic
        pol_layer<kPolObs>(s.w, s.x, s.a, STG_POLICY_VF_W1, STG_POLICY_VF_B1);
        pol_layer<kPolHidden>(s.w, s.a, s.h, STG_POLICY_VF_W2, STG_POLICY_VF_B2);
        if (e < kPolTile) {
            const float v = pol_head(s.w, s.h, e, STG_POLICY_VAL_W, 1, 0, s.w[STG_POLICY_VAL_B]);
            float gv = 0.0f;
            if (e < count) {
                const float old_v = kLoss == kLossPpo ? __ldg(a.d_old_value + base + e) : 0.0f;
                gv = pol_ppo_value_row(v, old_v, __ldg(a.d_return + base + e), c, sums);
            }
            s.g[0][e] = gv;
        }
        __syncthreads();
        ppo_delta2<1>(s, STG_POLICY_VAL_W, STG_POLICY_VAL_W, STG_POLICY_VAL_B, STG_POLICY_VF_B2, part, first);
        ppo_dw2(s, STG_POLICY_VF_W2, part, first);
        ppo_delta1(s, STG_POLICY_VF_W2);
        ppo_dw1(s, STG_POLICY_VF_W1, STG_POLICY_VF_B1, part, first);
        // ---- actor (its first layer writes plane a only after its first barrier, when dW1 above has read it)
        pol_layer<kPolObs>(s.w, s.x, s.a, STG_POLICY_PI_W1, STG_POLICY_PI_B1);
        pol_layer<kPolHidden>(s.w, s.a, s.h, STG_POLICY_PI_W2, STG_POLICY_PI_B2);
        if (e < kPolTile) {
            float mean[2], gm[2] = {0.0f, 0.0f}, gs[2];
            mean[0] = pol_head(s.w, s.h, e, STG_POLICY_ACT_W, 2, 0, s.w[STG_POLICY_ACT_B]);
            mean[1] = pol_head(s.w, s.h, e, STG_POLICY_ACT_W, 2, 1, s.w[STG_POLICY_ACT_B + 1]);
            if (e < count) {
                const int64_t i = base + e;
                const float2 av = __ldg(reinterpret_cast<const float2*>(a.d_action) + i);
                const float act[2] = {av.x, av.y};
                float lp = 0.0f;
#pragma unroll
                for (int d = 0; d < 2; ++d) {
                    const float t = pol_log_prob_term(act[d], mean[d], s.w[STG_POLICY_STD + d], s.w[STG_POLICY_LOG_SCALE + d]);
                    lp = d == 0 ? t : Pk<float>::add(lp, t);
                }
                const float adv = pol_ppo_advantage(__ldg(a.d_advantage + i), a.d_adv_stats ? stats : nullptr);
                const float old_lp = kLoss == kLossPpo ? __ldg(a.d_old_log_prob + i) : 0.0f;
                const float gl = pol_policy_row<kLoss>(lp, old_lp, adv, c, sums);
                pol_ppo_gauss_row(gl, act, mean, s.w, gm, gs);
                sums[4] += (double)gs[0];
                sums[5] += (double)gs[1];
            }
            s.g[0][e] = gm[0];
            s.g[1][e] = gm[1];
        }
        __syncthreads();
        ppo_delta2<2>(s, STG_POLICY_ACT_W, STG_POLICY_ACT_W, STG_POLICY_ACT_B, STG_POLICY_PI_B2, part, first);
        ppo_dw2(s, STG_POLICY_PI_W2, part, first);
        ppo_delta1(s, STG_POLICY_PI_W2);
        ppo_dw1(s, STG_POLICY_PI_W1, STG_POLICY_PI_B1, part, first);
        __syncthreads();              // the next tile's observations overwrite s.x
    }
    // the per-row sums of the CTA, in thread order
    double* red = reinterpret_cast<double*>(s.a);
    if (e < kPolTile) {
#pragma unroll
        for (int k = 0; k < kPpoSums; ++k) red[k * kPolTile + e] = sums[k];
    }
    __syncthreads();
    if (e < kPpoSums) {
        double t = 0.0;
        for (int r = 0; r < kPolTile; ++r) t += red[e * kPolTile + r];
        part[e < 4 ? STG_PPO_PART_LOSS + e : STG_POLICY_LOG_STD + e - 4] = t;
    }
}

// slot p of `parts` vectors of STG_PPO_PART doubles, summed in vector order from 0.0
__device__ __forceinline__ double ppo_fold_slot(const double* vecs, int parts, int p) {
    double t = 0.0;
#pragma unroll 8
    for (int b = 0; b < parts; ++b) t += __ldcg(vecs + (int64_t)b * STG_PPO_PART + p);
    return t;
}

enum PpoFold { kFoldScale, kFoldRaw, kFoldRanks };

// The fold of K10 and K12 over `parts` vectors of STG_PPO_PART doubles (K10's CTA partials, or K12's per-rank sums):
//   kFoldScale  sums in vector order, scales them (pol_ppo_grad_value, pol_ppo_losses) with B = a.batch into d_grad and
//               d_losses: stg_policy_ppo_grad_f32;
//   kFoldRaw    writes the same sums unscaled, with the row count a.batch, into `raw`: stg_policy_ppo_sums_f32;
//   kFoldRanks  as kFoldScale with B = the folded count slot: stg_policy_ppo_finish_f32.
template <PpoFold kMode>
__global__ void __launch_bounds__(kPolThreads) policy_ppo_fold_kernel(const StgPpoArgs a, const double* vecs, int parts,
                                                                     double* raw) {
    const int p = blockIdx.x * kPolThreads + threadIdx.x;
    if (p > STG_POLICY_PARAMS) return;
    const int64_t batch = kMode == kFoldRanks ? (int64_t)ppo_fold_slot(vecs, parts, STG_PPO_PART_COUNT) : a.batch;
    if (p < STG_POLICY_PARAMS) {
        const double t = ppo_fold_slot(vecs, parts, p);
        if (kMode == kFoldRaw) raw[p] = t;
        else a.d_grad[p] = pol_ppo_grad_value(p, t, batch, a.ent_coef, a.vf_coef);
        return;
    }
    double t[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = ppo_fold_slot(vecs, parts, STG_PPO_PART_LOSS + k);
    if (kMode == kFoldRaw) {
#pragma unroll
        for (int k = 0; k < 4; ++k) raw[STG_PPO_PART_LOSS + k] = t[k];
        raw[STG_PPO_PART_COUNT] = (double)a.batch;
        for (int k = STG_PPO_PART_COUNT + 1; k < STG_PPO_PART; ++k) raw[k] = 0.0;
    } else {
        pol_ppo_losses(t, a.d_weights, batch, a.ent_coef, a.vf_coef, a.d_losses);
    }
}

// K12: the advantage moments of one local minibatch, one CTA (include/stg.h). Chan merge of this lane's vector with the one
// `off` lanes up, a shuffle-down tree: lane 0 ends with the warp's vector.
constexpr int kAdvThreads = STG_PPO_ADV_THREADS;
static_assert(STG_PPO_ADV_MOMENTS == 3 && kAdvThreads == 32 * 32, "stg.h and the K12 moments tree disagree");

__device__ __forceinline__ void ppo_adv_warp_merge(double v[3]) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double b[3] = {__shfl_down_sync(0xffffffffu, v[0], off), __shfl_down_sync(0xffffffffu, v[1], off),
                             __shfl_down_sync(0xffffffffu, v[2], off)};
        pol_adv_merge(v, b);
    }
}

__global__ void __launch_bounds__(kAdvThreads) ppo_adv_moments_kernel(const float* __restrict__ adv, int64_t n,
                                                                      double* out) {
    __shared__ double sm[32][3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double v[3];
    pol_adv_moments(adv, threadIdx.x, n, kAdvThreads, v);
    ppo_adv_warp_merge(v);
    if (lane == 0) sm[warp][0] = v[0], sm[warp][1] = v[1], sm[warp][2] = v[2];
    __syncthreads();
    if (warp == 0) {
        v[0] = sm[lane][0], v[1] = sm[lane][1], v[2] = sm[lane][2];
        ppo_adv_warp_merge(v);
        if (lane == 0) out[0] = v[0], out[1] = v[1], out[2] = v[2];
    }
}

__global__ void __launch_bounds__(32) ppo_adv_merge_kernel(const double* moments, int ranks, float* stats) {
    if (threadIdx.x == 0) pol_adv_stats(moments, ranks, stats);
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
        (e = cudaFuncSetAttribute(policy_ppo_grad_kernel<kLossPpo>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(PpoShared))) != cudaSuccess ||
        (e = cudaFuncSetAttribute(policy_ppo_grad_kernel<kLossA2c>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(PpoShared))) != cudaSuccess ||
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

namespace stg {

// K10's argument checks, with the gradient and loss outputs required or not (K12's sums); the A2C instance reads neither old
// plane, so under kLossA2c they may be NULL and are not checked
template <PolLoss kLoss>
static int ppo_check(const StgPpoArgs& a, bool outputs) {
    const bool old = kLoss == kLossPpo;
    if (a.batch < 1) return STG_E_SIZE;
    if (!a.d_weights || !a.d_obs || !a.d_action || (old && (!a.d_old_value || !a.d_old_log_prob)) || !a.d_advantage ||
        !a.d_return || (outputs && (!a.d_grad || !a.d_losses)) || !a.d_work)
        return STG_E_NULL;
    if (((uintptr_t)a.d_weights | (uintptr_t)a.d_obs) & 15u) return STG_E_ALIGN;
    if (((uintptr_t)a.d_action | (uintptr_t)a.d_work) & 7u) return STG_E_ALIGN;
    const uintptr_t old_planes = old ? ((uintptr_t)a.d_old_value | (uintptr_t)a.d_old_log_prob) : 0u;
    if ((old_planes | (uintptr_t)a.d_advantage | (uintptr_t)a.d_return | (uintptr_t)a.d_adv_stats | (uintptr_t)a.d_grad |
         (uintptr_t)a.d_losses) & 3u)
        return STG_E_ALIGN;
    return STG_OK;
}

// flags K10 accepts under kLoss: STG_PPO_CLIP_VF for PPO, none for A2C (it has no value clip)
template <PolLoss kLoss>
static int ppo_check_flags(const StgPpoArgs& a) {
    return a.flags & ~(kLoss == kLossPpo ? STG_PPO_CLIP_VF : 0u) ? STG_E_ENUM : STG_OK;
}

// the gradient kernel of K10 under kLoss into d_work, then the fold of its grid partials in `kMode`
template <PolLoss kLoss, PpoFold kMode>
static int ppo_launch(const StgPpoArgs& a, double* raw, cudaStream_t s) {
    PolLaunch l;
    if (int rc = pol_configure(l)) return rc;
    const int grid = (int)STG_PPO_GRID(a.batch);
    policy_ppo_grad_kernel<kLoss><<<grid, kPolThreads, sizeof(PpoShared), s>>>(a);
    if (cudaError_t e = cudaGetLastError()) return (int)e;
    policy_ppo_fold_kernel<kMode><<<STG_POLICY_PARAMS / kPolThreads + 1, kPolThreads, 0, s>>>(a, a.d_work, grid, raw);
    return (int)cudaGetLastError();
}

}  // namespace stg

namespace stg {

// stg_policy_{ppo,a2c}_grad_f32
template <PolLoss kLoss>
static int ppo_grad_entry(const StgPpoArgs* args, void* stream) {
    if (!args) return STG_E_NULL;
    const StgPpoArgs& a = *args;
    if (int rc = ppo_check<kLoss>(a, true)) return rc;
    if (int rc = ppo_check_flags<kLoss>(a)) return rc;
    return ppo_launch<kLoss, kFoldScale>(a, nullptr, (cudaStream_t)stream);
}

// stg_policy_{ppo,a2c}_sums_f32
template <PolLoss kLoss>
static int ppo_sums_entry(const StgPpoArgs* args, double* d_sums, void* stream) {
    if (!args) return STG_E_NULL;
    const StgPpoArgs& a = *args;
    if (a.batch < 1) return STG_E_SIZE;
    if (!d_sums) return STG_E_NULL;
    if (int rc = ppo_check<kLoss>(a, false)) return rc;
    if ((uintptr_t)d_sums & 7u) return STG_E_ALIGN;
    if (int rc = ppo_check_flags<kLoss>(a)) return rc;
    return ppo_launch<kLoss, kFoldRaw>(a, d_sums, (cudaStream_t)stream);
}

}  // namespace stg

extern "C" int stg_policy_ppo_grad_f32(const StgPpoArgs* args, void* stream) {
    return stg::ppo_grad_entry<stg::kLossPpo>(args, stream);
}

extern "C" int stg_policy_ppo_sums_f32(const StgPpoArgs* args, double* d_sums, void* stream) {
    return stg::ppo_sums_entry<stg::kLossPpo>(args, d_sums, stream);
}

extern "C" int stg_policy_a2c_grad_f32(const StgPpoArgs* args, void* stream) {
    return stg::ppo_grad_entry<stg::kLossA2c>(args, stream);
}

extern "C" int stg_policy_a2c_sums_f32(const StgPpoArgs* args, double* d_sums, void* stream) {
    return stg::ppo_sums_entry<stg::kLossA2c>(args, d_sums, stream);
}

extern "C" int stg_policy_ppo_finish_f32(const StgPpoArgs* args, const double* d_sums, int32_t ranks, void* stream) {
    if (!args) return STG_E_NULL;
    const StgPpoArgs& a = *args;
    if (ranks < 1) return STG_E_SIZE;
    if (!a.d_weights || !a.d_grad || !a.d_losses || !d_sums) return STG_E_NULL;
    if ((uintptr_t)a.d_weights & 15u || (uintptr_t)d_sums & 7u || ((uintptr_t)a.d_grad | (uintptr_t)a.d_losses) & 3u)
        return STG_E_ALIGN;
    stg::policy_ppo_fold_kernel<stg::kFoldRanks><<<STG_POLICY_PARAMS / stg::kPolThreads + 1, stg::kPolThreads, 0,
                                                   (cudaStream_t)stream>>>(a, d_sums, ranks, nullptr);
    return (int)cudaGetLastError();
}

extern "C" int stg_ppo_adv_moments_f64(const float* d_adv, int64_t n, double* d_out, void* stream) {
    if (n < 0) return STG_E_SIZE;
    if (!d_out || (n > 0 && !d_adv)) return STG_E_NULL;
    if ((uintptr_t)d_adv & 3u || (uintptr_t)d_out & 7u) return STG_E_ALIGN;
    stg::ppo_adv_moments_kernel<<<1, stg::kAdvThreads, 0, (cudaStream_t)stream>>>(d_adv, n, d_out);
    return (int)cudaGetLastError();
}

extern "C" int stg_ppo_adv_merge_f32(const double* d_moments, int32_t ranks, float* d_stats, void* stream) {
    if (ranks < 1) return STG_E_SIZE;
    if (!d_moments || !d_stats) return STG_E_NULL;
    if ((uintptr_t)d_moments & 7u || (uintptr_t)d_stats & 3u) return STG_E_ALIGN;
    stg::ppo_adv_merge_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_moments, ranks, d_stats);
    return (int)cudaGetLastError();
}
