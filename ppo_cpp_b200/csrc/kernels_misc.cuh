// HBM-bound kernels of the path: synthetic env, VecNormalize, GAE, advantage statistics,
// gradient reduction, global-norm clip + Adam, layout conversion.
#pragma once
#include <cooperative_groups.h>

#include "device_common.cuh"
#include "sync_prims.cuh"

namespace ppo {

// ------------------------------------------------------------------------------------------------
// Synthetic GPU-resident env (SURVEY §8d): s' = 0.9 s + 0.1 clamp(a,-1,1) + 0.01 xi, reward = s'[0]-s[0],
// 334-step episodes with per-env phase offset, reset to 0.1*U(-1,1).  One thread per env.
struct SynthEnv {
    float* state;      // [n][D]
    uint32_t* t_env;   // [n]
    uint32_t* resets;  // [n]
    uint64_t seed;
    uint32_t env_id0;
    int n, D;
};

__device__ __forceinline__ void synth_reset_state(const SynthEnv& e, int i, float* s /*[D] out*/) {
    const uint2 key = make_uint2((uint32_t)e.seed, (uint32_t)(e.seed >> 32));
    const uint32_t gid = e.env_id0 + (uint32_t)i, rc = e.resets[i];
    for (int blk = 0; blk * 4 < e.D; ++blk) {
        const uint4 w = philox4x32_10(make_uint4(gid, rc, (uint32_t)blk, PPO_TAG_ENVRESET), key);
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (blk * 4 + k < e.D) s[blk * 4 + k] = __fmul_rn(0.1f, __fsub_rn(__fmul_rn(2.0f, u32_to_unit(wv[k])), 1.0f));
    }
    e.resets[i] = rc + 1;
}

__global__ void synth_env_reset_kernel(SynthEnv e, float* __restrict__ obs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e.n) return;
    e.resets[i] = 0;
    e.t_env[i] = (e.env_id0 + (uint32_t)i) % 334u;
    float s[32];
    synth_reset_state(e, i, s);
    for (int k = 0; k < e.D; ++k) {
        e.state[(size_t)i * e.D + k] = s[k];
        obs[(size_t)i * e.D + k] = s[k];
    }
}

__global__ void synth_env_step_kernel(SynthEnv e, const float* __restrict__ actions, float* __restrict__ obs,
                                      float* __restrict__ rew, float* __restrict__ done) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e.n) return;
    float s[32];
    const uint32_t t = e.t_env[i];
    float s0 = 0.f;
    for (int blk = 0; blk * 4 < e.D; ++blk) {
        float xi[4];
        normal4(e.seed, e.env_id0 + (uint32_t)i, t, (uint32_t)blk, PPO_TAG_ENVNOISE, xi);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int k = blk * 4 + q;
            if (k < e.D) {
                const float sk = e.state[(size_t)i * e.D + k];
                if (k == 0) s0 = sk;
                float a = actions[(size_t)i * e.D + k];
                a = a < -1.f ? -1.f : (a > 1.f ? 1.f : a);
                s[k] = __fadd_rn(__fadd_rn(__fmul_rn(0.9f, sk), __fmul_rn(0.1f, a)), __fmul_rn(0.01f, xi[q]));
            }
        }
    }
    rew[i] = __fsub_rn(s[0], s0);
    e.t_env[i] = t + 1;
    if ((t + 1) % 334u == 0u) {
        done[i] = 1.f;
        synth_reset_state(e, i, s);
    } else {
        done[i] = 0.f;
    }
    for (int k = 0; k < e.D; ++k) {
        e.state[(size_t)i * e.D + k] = s[k];
        obs[(size_t)i * e.D + k] = s[k];
    }
}

// ------------------------------------------------------------------------------------------------
// VecNormalize (env/env_normalize.hpp:64-116, common/running_statistics.hpp:26-104).
// Running statistics live on the device: mean/var fp32 [D], count double — as in the reference.
struct NormStats {
    float* obs_mean;   // [D]
    float* obs_var;    // [D]
    double* obs_count; // [1]
    float* ret_mean;   // [1]
    float* ret_var;    // [1]
    double* ret_count; // [1]
};

// Chan merge exactly as RunningStatistics::update_from_moments (running_statistics.hpp:88-104): doubles are
// converted to the fp32 matrix scalar one at a time, left to right.
__device__ __forceinline__ void chan_merge(float& mean, float& var, double count, float bmean, float bvar, double bcount) {
    const double total = count + bcount;
    const float delta = __fsub_rn(bmean, mean);
    const float new_mean = __fadd_rn(mean, __fdiv_rn(__fmul_rn(delta, (float)bcount), (float)total));
    const float m_a = __fmul_rn(var, (float)count);
    const float m_b = __fmul_rn(bvar, (float)bcount);
    const float cross = __fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(delta, delta), (float)count), (float)bcount), (float)total);
    const float m_2 = __fadd_rn(__fadd_rn(m_a, m_b), cross);
    mean = new_mean;
    var = __fdiv_rn(m_2, (float)total);
}

// Pass A: ret = ret*gamma + rew; per-column (sum, sum of squares) in double for the D obs columns and the
// return column.  Thread i walks elements i, i+S, ... with S a multiple of D so its column never changes
// (coalesced, all lanes busy).  Per-CTA partials -> moments_partial[cta][2*(D+1)]; the last CTA to finish sums
// them in fixed order into moments[2*(D+1)+1] (last entry = row count) and, when fuse_merge, performs the
// Chan merge into the running statistics (single GPU).  Multi-GPU: allreduce `moments`, then norm_merge_kernel.
struct MomentsArgs {
    const float* raw_obs;  // [n][D]
    const float* raw_rew;  // [n] or NULL (reset: observations only)
    float* ret;            // [n] in/out
    int n, D;
    float gamma;
    double* partial;       // [grid][2*(D+1)]
    double* moments;       // [2*(D+1)+1]
    unsigned int* ticket;
    NormStats st;
    int fuse_merge, update_obs, update_ret;
};

__device__ __forceinline__ void norm_merge(const MomentsArgs& a, const double* mom, int tid, int nthreads) {
    const int D = a.D;
    const double rows = mom[2 * (D + 1)];
    for (int c = tid; c <= D; c += nthreads) {
        const bool is_ret = (c == D);
        if (is_ret ? !a.update_ret : !a.update_obs) continue;
        // colwise().mean() and sum((x-mean)^2)/rows of the reference, evaluated in double from sums taken
        // around a pivot (the running mean before this update; identical on every rank) and rounded once
        const double pivot = is_ret ? 0.0 : (double)a.st.obs_mean[c];
        const double m1 = mom[c] / rows;
        const double mean_d = pivot + m1;
        double var_d = mom[D + 1 + c] / rows - m1 * m1;
        if (var_d < 0.0) var_d = 0.0;
        const float bmean = (float)mean_d, bvar = (float)var_d;
        if (is_ret) {
            float m = *a.st.ret_mean, v = *a.st.ret_var;
            chan_merge(m, v, *a.st.ret_count, bmean, bvar, rows);
            *a.st.ret_mean = m; *a.st.ret_var = v;
        } else {
            float m = a.st.obs_mean[c], v = a.st.obs_var[c];
            chan_merge(m, v, *a.st.obs_count, bmean, bvar, rows);
            a.st.obs_mean[c] = m; a.st.obs_var[c] = v;
        }
    }
    __syncthreads();
    if (tid == 0) {
        if (a.update_obs) *a.st.obs_count = rows + *a.st.obs_count;
        if (a.update_ret) *a.st.ret_count = rows + *a.st.ret_count;
    }
}

__global__ void norm_moments_kernel(const MomentsArgs a) {
    extern __shared__ double sm[];  // [blockDim][2] then [2*(D+1)]
    const int D = a.D, tid = threadIdx.x, nth = blockDim.x;
    const size_t S = (size_t)gridDim.x * nth;  // multiple of D by construction
    const size_t total = (size_t)a.n * D;
    double s = 0.0, q = 0.0;
    // sums are taken around a per-column pivot (the current running mean) to keep the sum of squares well
    // conditioned; norm_merge adds the pivot back
    const int col = (int)(((size_t)blockIdx.x * nth + tid) % D);
    const float pivot = a.st.obs_mean[col];
    for (size_t e = (size_t)blockIdx.x * nth + tid; e < total; e += S) {
        const double x = (double)a.raw_obs[e] - (double)pivot;
        s += x;
        q += x * x;
    }
    sm[tid * 2] = s;
    sm[tid * 2 + 1] = q;
    // return column
    double rs = 0.0, rq = 0.0;
    if (a.raw_rew) {
        for (size_t i = (size_t)blockIdx.x * nth + tid; i < (size_t)a.n; i += S) {
            const float r = __fadd_rn(__fmul_rn(a.ret[i], a.gamma), a.raw_rew[i]);  // env_normalize.hpp:71
            a.ret[i] = r;
            rs += (double)r;
            rq += (double)r * (double)r;
        }
    }
    rs = warp_sum(rs);
    rq = warp_sum(rq);
    double* colsum = sm + 2 * nth;            // [2*(D+1)]
    double* wred = colsum + 2 * (D + 1);      // [2*32]
    if ((tid & 31) == 0) { wred[(tid >> 5) * 2] = rs; wred[(tid >> 5) * 2 + 1] = rq; }
    __syncthreads();
    if (tid < D) {  // threads with the same (tid % D) hold the same column
        double cs = 0.0, cq = 0.0;
        for (int j = tid; j < nth; j += D) { cs += sm[j * 2]; cq += sm[j * 2 + 1]; }
        colsum[tid] = cs;
        colsum[D + 1 + tid] = cq;
    } else if (tid == D) {
        double cs = 0.0, cq = 0.0;
        for (int w = 0; w < (nth + 31) / 32; ++w) { cs += wred[w * 2]; cq += wred[w * 2 + 1]; }
        colsum[D] = cs;
        colsum[2 * D + 1] = cq;
    }
    __syncthreads();
    double* mine = a.partial + (size_t)blockIdx.x * 2 * (D + 1);
    for (int c = tid; c < 2 * (D + 1); c += nth) mine[c] = colsum[c];
    __threadfence();
    __shared__ bool last;
    __syncthreads();
    if (tid == 0) last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last block adds the per-block partials in a fixed order: G threads per column take interleaved blocks (loads batched eight
    // deep), then the G sums are added in order.  (One thread per column walking all blocks was a chain of 296 dependent L2 round
    // trips: 59 k of the kernel's 66 k cycles at 65 536 envs — profiles/r2_small_kernels_ncu.txt.)
    {
        const int W2 = 2 * (D + 1);
        const int G = max(1, min(nth / W2, 8));
        double* gp = sm;  // [G][W2] <= [nth][2]
        if (tid < G * W2) {
            const int g = tid / W2, c = tid - g * W2;
            double t = 0.0;
            unsigned b = (unsigned)g;
            for (; b + 7u * G < gridDim.x; b += 8u * G) {
                double v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = __ldcg(a.partial + (size_t)(b + i * G) * W2 + c);
#pragma unroll
                for (int i = 0; i < 8; ++i) t += v[i];
            }
            for (; b < gridDim.x; b += G) t += __ldcg(a.partial + (size_t)b * W2 + c);
            gp[tid] = t;
        }
        __syncthreads();
        for (int c = tid; c < W2; c += nth) {
            double t = 0.0;
            for (int g = 0; g < G; ++g) t += gp[g * W2 + c];
            colsum[c] = t;
        }
    }
    __syncthreads();
    for (int c = tid; c < D; c += nth) {
        a.moments[c] = colsum[c];
        a.moments[D + 1 + c] = colsum[D + 1 + c];
    }
    if (tid == 0) {
        a.moments[D] = colsum[D];
        a.moments[2 * D + 1] = colsum[2 * D + 1];
        a.moments[2 * (D + 1)] = (double)a.n;
        *a.ticket = 0u;
    }
    __syncthreads();
    __threadfence();
    if (a.fuse_merge) norm_merge(a, a.moments, tid, nth);
}

__global__ void norm_merge_kernel(const MomentsArgs a) { norm_merge(a, a.moments, threadIdx.x, blockDim.x); }

// Pass B: normalise + clip observations and rewards, reset ret on done, publish current obs/dones and store
// this step's rewards (env_normalize.hpp:74-91, matrix_clamp.hpp:32-35, runner.hpp:116-129).
struct ApplyArgs {
    const float* raw_obs;  // [n][D]
    const float* raw_rew;  // [n] or NULL (reset)
    const float* done;     // [n] or NULL
    float* ret;            // [n]
    int n, D;
    NormStats st;
    int norm_obs, norm_reward;
    float clip_obs, clip_rew, eps;
    float* obs_out;      // [n][D] normalised observation (Runner::obs)
    float* rew_out;      // [n] normalised reward or NULL
    float* dones_out;    // [n] or NULL (Runner::dones)
    float* rew_store;    // rollout true_rewards[t] or NULL
    float* urew_store;   // rollout unnormalized_rewards[t] or NULL
    uint32_t* step_ctr;  // incremented once per env step (Philox step counter) or NULL
};

__global__ void norm_apply_kernel(const ApplyArgs a) {
    const size_t total = (size_t)a.n * a.D;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int c = (int)(e % a.D);
        float x = a.raw_obs[e];
        if (a.norm_obs) {
            const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(a.st.obs_var[c], a.eps)));
            x = __fmul_rn(__fsub_rn(x, a.st.obs_mean[c]), inv);
            x = fminf(fmaxf(x, -a.clip_obs), a.clip_obs);  // cwiseMax(lo).cwiseMin(hi)
        }
        a.obs_out[e] = x;
    }
    if (a.raw_rew) {
        const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(*a.st.ret_var, a.eps)));
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)a.n; i += stride) {
            const float raw = a.raw_rew[i];
            float r = raw;
            if (a.norm_reward) {
                r = __fmul_rn(raw, inv);  // no mean subtraction (env_normalize.hpp:80)
                r = fminf(fmaxf(r, -a.clip_rew), a.clip_rew);
            }
            const float dn = a.done[i];
            a.ret[i] = __fmul_rn(a.ret[i], __fsub_rn(1.0f, dn));  // env_normalize.hpp:88
            if (a.rew_out) a.rew_out[i] = r;
            if (a.dones_out) a.dones_out[i] = dn;
            if (a.rew_store) a.rew_store[i] = r;
            if (a.urew_store) a.urew_store[i] = raw;
        }
    }
    if (a.step_ctr && blockIdx.x == 0 && threadIdx.x == 0) *a.step_ctr += 1u;
}

// ------------------------------------------------------------------------------------------------
// VecNormalize over a recorded trajectory [T][n][D] (ppo_vecnorm_replay): the result of T consecutive
// EnvNormalize::step calls (env_normalize.hpp:64-92) computed in three HBM-bound passes instead of T latency-bound
// launch pairs.  The running statistics at step t depend on all rows of steps <= t, but only through per-step batch
// moments, so: (1) per-env discounted return scan along t (sequential per env, coalesced across envs) -> rt[t][n];
// (2) per-step column sums of obs and rt around a fixed pivot, all steps in parallel; (3) one warp replays the T Chan
// merges in order and records the statistics in force at every step; (4) normalise + clip, all steps in parallel.
struct ReplayArgs {
    const float *raw_obs, *raw_rew, *done;  // [T][n][D], [T][n], [T][n]
    float* ret;                             // [n] in/out: discounted return carried across calls
    float* rt;                              // [T][n] scratch: ret after the step's reward, before the done reset
    double* partial;                        // [T][NB][2*(D+1)]
    float* bmom;                            // [T][2*(D+1)]: batch mean[D+1], batch variance[D+1] of every step
    float* stats;                           // [T][2*D+1]: mean[D], inv_std[D], inv_ret_std
    int T, n, D, NB;
    NormStats st;
    int update_obs, update_ret, norm_obs, norm_reward;
    float gamma, clip_obs, clip_rew, eps;
    float *obs_out, *rew_out;
};

__global__ void replay_ret_kernel(const ReplayArgs a) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n) return;
    float r = a.ret[e];
    constexpr int RB = 8;
    for (int t0 = 0; t0 < a.T; t0 += RB) {
        float rw[RB], dn[RB];
#pragma unroll
        for (int i = 0; i < RB; ++i) {
            const bool in = t0 + i < a.T;
            rw[i] = in ? __ldg(a.raw_rew + (size_t)(t0 + i) * a.n + e) : 0.f;
            dn[i] = in ? __ldg(a.done + (size_t)(t0 + i) * a.n + e) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < RB; ++i) {
            if (t0 + i < a.T) {
                r = __fadd_rn(__fmul_rn(r, a.gamma), rw[i]);  // env_normalize.hpp:71
                a.rt[(size_t)(t0 + i) * a.n + e] = r;
                r = __fmul_rn(r, __fsub_rn(1.0f, dn[i]));      // env_normalize.hpp:88
            }
        }
    }
    a.ret[e] = r;
}

// grid (NB, T); blockDim = D * k.  Thread stride is a multiple of D, so a thread's column (pair) never changes.
__global__ void replay_moments_kernel(const ReplayArgs a) {
    extern __shared__ double sm[];  // [blockDim][4], then [2*32] warp partials of the return column
    const int D = a.D, tid = threadIdx.x, nth = blockDim.x, t = blockIdx.y;
    const size_t S = (size_t)gridDim.x * nth, total = (size_t)a.n * D;
    const float* x0 = a.raw_obs + (size_t)t * total;
    const bool vec2 = (D & 1) == 0 && nth % (D / 2) == 0 && (total & 1) == 0;  // 8-byte loads: D even keeps rows 8-byte aligned
    // pivot = the running mean when the replay starts (fixed for all steps)
    if (vec2) {
        const int cp = tid % (D / 2);
        const double p0 = (double)a.st.obs_mean[2 * cp], p1 = (double)a.st.obs_mean[2 * cp + 1];
        const float2* x2 = reinterpret_cast<const float2*>(x0);
        double s0 = 0.0, q0 = 0.0, s1 = 0.0, q1 = 0.0;
        // two-level sums: runs of 4 elements in fp32 (around the pivot, so the terms are O(std)), runs added in double -
        // the fp64 pipe (conversions included) was the bound of the all-double loop
        const float f0 = (float)p0, f1 = (float)p1;
        size_t e = (size_t)blockIdx.x * nth + tid;
        for (; e + 3 * S < total / 2; e += 4 * S) {
            const float2 v0 = __ldg(x2 + e), v1 = __ldg(x2 + e + S), v2 = __ldg(x2 + e + 2 * S), v3 = __ldg(x2 + e + 3 * S);
            const float a0 = v0.x - f0, a1 = v1.x - f0, a2 = v2.x - f0, a3 = v3.x - f0;
            const float b0 = v0.y - f1, b1 = v1.y - f1, b2 = v2.y - f1, b3 = v3.y - f1;
            s0 += (double)((a0 + a1) + (a2 + a3));
            q0 += (double)(fmaf(a0, a0, a1 * a1) + fmaf(a2, a2, a3 * a3));
            s1 += (double)((b0 + b1) + (b2 + b3));
            q1 += (double)(fmaf(b0, b0, b1 * b1) + fmaf(b2, b2, b3 * b3));
        }
        for (; e < total / 2; e += S) {
            const float2 v = __ldg(x2 + e);
            const float a0 = v.x - f0, b0 = v.y - f1;
            s0 += (double)a0; q0 += (double)(a0 * a0);
            s1 += (double)b0; q1 += (double)(b0 * b0);
        }
        sm[tid * 4] = s0; sm[tid * 4 + 1] = q0; sm[tid * 4 + 2] = s1; sm[tid * 4 + 3] = q1;
    } else {
        const int col = (int)(((size_t)blockIdx.x * nth + tid) % D);
        const double pivot = (double)a.st.obs_mean[col];
        double s = 0.0, q = 0.0;
        for (size_t e = (size_t)blockIdx.x * nth + tid; e < total; e += S) {
            const double x = (double)__ldg(x0 + e) - pivot;
            s += x;
            q += x * x;
        }
        sm[tid * 4] = s; sm[tid * 4 + 1] = q;
    }
    double rs = 0.0, rq = 0.0;
    for (size_t i = (size_t)blockIdx.x * nth + tid; i < (size_t)a.n; i += S) {
        const double r = (double)__ldg(a.rt + (size_t)t * a.n + i);
        rs += r;
        rq += r * r;
    }
    rs = warp_sum(rs);
    rq = warp_sum(rq);
    double* wred = sm + 4 * nth;
    if ((tid & 31) == 0) { wred[(tid >> 5) * 2] = rs; wred[(tid >> 5) * 2 + 1] = rq; }
    __syncthreads();
    double* mine = a.partial + ((size_t)t * gridDim.x + blockIdx.x) * 2 * (D + 1);
    if (tid < D) {
        double cs = 0.0, cq = 0.0;
        if (vec2) {
            const int k = 2 * (tid & 1);
            for (int j = tid >> 1; j < nth; j += D / 2) { cs += sm[j * 4 + k]; cq += sm[j * 4 + k + 1]; }
        } else {
            for (int j = tid; j < nth; j += D) { cs += sm[j * 4]; cq += sm[j * 4 + 1]; }
        }
        mine[tid] = cs;
        mine[D + 1 + tid] = cq;
    } else if (tid == D) {
        double cs = 0.0, cq = 0.0;
        for (int w = 0; w < (nth + 31) / 32; ++w) { cs += wred[w * 2]; cq += wred[w * 2 + 1]; }
        mine[D] = cs;
        mine[2 * D + 1] = cq;
    }
}

// grid T, 64 threads: per-step column sums over the NB block partials (fixed order) -> batch mean / variance of step t
// (colwise().mean() and sum((x-mean)^2)/rows of the reference, evaluated in double and rounded once)
__global__ void replay_reduce_kernel(const ReplayArgs a) {
    const int D = a.D, W2 = 2 * (D + 1), c = threadIdx.x, t = blockIdx.x;
    if (c > D) return;
    const double* p = a.partial + (size_t)t * a.NB * W2;
    double s0 = 0.0, s1 = 0.0, q0 = 0.0, q1 = 0.0;
    int b = 0;
    for (; b + 2 <= a.NB; b += 2) {
        s0 += p[(size_t)b * W2 + c]; q0 += p[(size_t)b * W2 + D + 1 + c];
        s1 += p[(size_t)(b + 1) * W2 + c]; q1 += p[(size_t)(b + 1) * W2 + D + 1 + c];
    }
    for (; b < a.NB; ++b) { s0 += p[(size_t)b * W2 + c]; q0 += p[(size_t)b * W2 + D + 1 + c]; }
    const double rows = (double)a.n;
    const double pivot = c == D ? 0.0 : (double)a.st.obs_mean[c];  // unchanged until replay_merge_kernel runs
    const double m1 = (s0 + s1) / rows;
    double var_d = (q0 + q1) / rows - m1 * m1;
    if (var_d < 0.0) var_d = 0.0;
    a.bmom[(size_t)t * W2 + c] = (float)(pivot + m1);
    a.bmom[(size_t)t * W2 + D + 1 + c] = (float)var_d;
}

// one CTA: the per-step batch moments are staged through shared memory in chunks (all threads), warp 0 replays the
// Chan merges in order (lane c < D: obs column c, lane D: the return column), all threads turn the recorded variances
// into 1/sqrt(var + eps) and write the statistics of every step
constexpr int REPLAY_CH = 128;
__global__ void __launch_bounds__(256) replay_merge_kernel(const ReplayArgs a) {
    extern __shared__ float smf[];  // [REPLAY_CH][2*(D+1)] batch moments, then [REPLAY_CH][2*(D+1)] running (mean, var)
    const int D = a.D, W2 = 2 * (D + 1), SW = 2 * D + 1, c = threadIdx.x;
    float* run = smf + (size_t)REPLAY_CH * W2;
    const bool lane_on = c <= D;
    const bool is_ret = c == D;
    const bool upd = lane_on && (is_ret ? a.update_ret : a.update_obs);
    float mean = 0.f, var = 1.f;
    double count = 0.0;
    if (lane_on) {
        mean = is_ret ? *a.st.ret_mean : a.st.obs_mean[c];
        var = is_ret ? *a.st.ret_var : a.st.obs_var[c];
        count = is_ret ? *a.st.ret_count : *a.st.obs_count;
    }
    const double rows = (double)a.n;
    for (int t0 = 0; t0 < a.T; t0 += REPLAY_CH) {
        const int nt = min(REPLAY_CH, a.T - t0);
        if (a.update_obs || a.update_ret)
            for (int i = threadIdx.x; i < nt * W2; i += blockDim.x) smf[i] = a.bmom[(size_t)t0 * W2 + i];
        __syncthreads();
        if (lane_on) {
            for (int t = 0; t < nt; ++t) {
                if (upd) {
                    chan_merge(mean, var, count, smf[t * W2 + c], smf[t * W2 + D + 1 + c], rows);
                    count = rows + count;
                }
                run[t * W2 + c] = mean;
                run[t * W2 + D + 1 + c] = var;
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < nt * SW; i += blockDim.x) {
            const int t = i / SW, k = i % SW;
            float v;
            if (k < D) v = run[t * W2 + k];
            else {
                const int col = k - D;  // D + col < 2D: obs column col; k == 2D: the return column
                v = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(run[t * W2 + D + 1 + col], a.eps)));
            }
            a.stats[(size_t)t0 * SW + i] = v;
        }
        __syncthreads();
    }
    if (upd) {
        if (is_ret) { *a.st.ret_mean = mean; *a.st.ret_var = var; *a.st.ret_count = count; }
        else {
            a.st.obs_mean[c] = mean; a.st.obs_var[c] = var;
            if (c == 0) *a.st.obs_count = count;
        }
    }
}

// grid (blocks, T): normalise + clip step t with the statistics in force after its update (env_normalize.hpp:74-86)
__global__ void replay_apply_kernel(const ReplayArgs a) {
    extern __shared__ float ss[];  // [2*D+1]
    const int D = a.D, t = blockIdx.y;
    for (int i = threadIdx.x; i < 2 * D + 1; i += blockDim.x) ss[i] = a.stats[(size_t)t * (2 * D + 1) + i];
    __syncthreads();
    const size_t total = (size_t)a.n * D, stride = (size_t)gridDim.x * blockDim.x;
    const float2* x2 = reinterpret_cast<const float2*>(a.raw_obs + (size_t)t * total);  // D even: rows are 8-byte aligned
    float2* o2 = reinterpret_cast<float2*>(a.obs_out + (size_t)t * total);
    if ((total & 3) == 0) {  // 16-byte accesses over the flat step block
        const float4* x4 = reinterpret_cast<const float4*>(a.raw_obs + (size_t)t * total);
        float4* o4 = reinterpret_cast<float4*>(a.obs_out + (size_t)t * total);
#pragma unroll 4
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total / 4; e += stride) {
            float4 x = __ldcs(x4 + e);  // streamed once: evict first
            if (a.norm_obs) {
                int c = (int)((4 * e) % D);
                x.x = fminf(fmaxf(__fmul_rn(__fsub_rn(x.x, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
                c = c + 1 == D ? 0 : c + 1;
                x.y = fminf(fmaxf(__fmul_rn(__fsub_rn(x.y, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
                c = c + 1 == D ? 0 : c + 1;
                x.z = fminf(fmaxf(__fmul_rn(__fsub_rn(x.z, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
                c = c + 1 == D ? 0 : c + 1;
                x.w = fminf(fmaxf(__fmul_rn(__fsub_rn(x.w, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
            }
            __stcs(o4 + e, x);
        }
    } else if ((D & 1) == 0) {
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total / 2; e += stride) {
            const int c = (int)((2 * e) % D);
            float2 x = __ldg(x2 + e);
            if (a.norm_obs) {
                x.x = fminf(fmaxf(__fmul_rn(__fsub_rn(x.x, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
                x.y = fminf(fmaxf(__fmul_rn(__fsub_rn(x.y, ss[c + 1]), ss[D + c + 1]), -a.clip_obs), a.clip_obs);
            }
            o2[e] = x;
        }
    } else {
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
            const int c = (int)(e % D);
            float x = __ldg(a.raw_obs + (size_t)t * total + e);
            if (a.norm_obs) x = fminf(fmaxf(__fmul_rn(__fsub_rn(x, ss[c]), ss[D + c]), -a.clip_obs), a.clip_obs);
            a.obs_out[(size_t)t * total + e] = x;
        }
    }
    if (a.rew_out) {
        const float inv = ss[2 * D];
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)a.n; i += stride) {
            float r = __ldg(a.raw_rew + (size_t)t * a.n + i);
            if (a.norm_reward) r = fminf(fmaxf(__fmul_rn(r, inv), -a.clip_rew), a.clip_rew);  // no mean subtraction (env_normalize.hpp:80)
            a.rew_out[(size_t)t * a.n + i] = r;
        }
    }
}

__global__ void clamp_kernel(const float* __restrict__ x, size_t n, float lo, float hi, float* __restrict__ out) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = fminf(fmaxf(x[i], lo), hi);
}

__global__ void bump_counter_kernel(uint32_t* c) { *c += 1u; }

// ------------------------------------------------------------------------------------------------
// GAE(lambda) reverse scan (Runner::set_returns, runner.hpp:159-191) over time-major [T][N] buffers.
// One thread per (env, chunk of `chunk` steps).  A chunk that does not end at T-1 first runs `warm` extra
// steps ahead of it starting from lastgaelam = 0: the recurrence contracts by gamma*lam per step (and is reset exactly
// by every done flag), so after `warm` steps the carried value equals the sequential one to below fp32 resolution
// while every arithmetic operation stays the reference's (bit-identical results in practice).  The launcher derives
// `warm` from gamma*lam ((gamma*lam)^warm <= 2^-46; 0.9405 -> 520) and switches to the affine-carry kernels below when
// gamma*lam is too close to 1 for any warm-up to contract.
__global__ void gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const float* __restrict__ dones,
                           const float* __restrict__ last_val, const float* __restrict__ last_done, int T, int N,
                           float gamma, float lam, int chunk, int warm, float* __restrict__ adv_out,
                           float* __restrict__ ret_out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (e >= N) return;
    const int t_lo = c * chunk;
    const int t_hi = min(T, t_lo + chunk) - 1;  // inclusive
    const int t_start = min(T - 1, t_hi + warm);
    const float gl = __fmul_rn(gamma, lam);
    float last = 0.f;
    float nextv = (t_start == T - 1) ? last_val[e] : val[(size_t)(t_start + 1) * N + e];
    float nextnt = 1.0f - ((t_start == T - 1) ? last_done[e] : dones[(size_t)(t_start + 1) * N + e]);
    // batches of GAE_B steps: all 3*GAE_B loads of a batch are issued before the (sequential) recurrence consumes them,
    // so that enough bytes are in flight per thread to cover the HBM latency (16 M transitions: 45 % -> see profiles/)
    constexpr int GAE_B = 8;
    int t = t_start;
    for (; t - (GAE_B - 1) >= t_lo; t -= GAE_B) {
        float vv[GAE_B], rr[GAE_B], dd[GAE_B];
#pragma unroll
        for (int u = 0; u < GAE_B; ++u) {
            const size_t idx = (size_t)(t - u) * N + e;
            vv[u] = __ldg(val + idx);
            rr[u] = __ldg(rew + idx);
            dd[u] = __ldg(dones + idx);
        }
#pragma unroll
        for (int u = 0; u < GAE_B; ++u) {
            const size_t idx = (size_t)(t - u) * N + e;
            const float delta = __fsub_rn(__fadd_rn(rr[u], __fmul_rn(gamma, __fmul_rn(nextv, nextnt))), vv[u]);
            last = __fadd_rn(delta, __fmul_rn(gl, __fmul_rn(nextnt, last)));
            if (t - u <= t_hi) {
                if (adv_out) adv_out[idx] = last;
                ret_out[idx] = __fadd_rn(last, vv[u]);
            }
            nextv = vv[u];
            nextnt = 1.0f - dd[u];
        }
    }
    for (; t >= t_lo; --t) {
        const size_t idx = (size_t)t * N + e;
        const float v = val[idx];
        const float delta = __fsub_rn(__fadd_rn(rew[idx], __fmul_rn(gamma, __fmul_rn(nextv, nextnt))), v);
        last = __fadd_rn(delta, __fmul_rn(gl, __fmul_rn(nextnt, last)));
        if (t <= t_hi) {
            if (adv_out) adv_out[idx] = last;
            ret_out[idx] = __fadd_rn(last, v);
        }
        nextv = v;
        nextnt = 1.0f - dones[idx];
    }
}

// Exact chunking for ANY gamma, lam (gamma*lam close to or equal to 1, where no warm-up length contracts): pass 1 reduces
// every (env, chunk) to the affine map  last_out = A * last_in + B  of its steps (fp64), pass 2 (gae_kernel_carry)
// composes the maps of the chunks above it into the chunk's incoming `lastgaelam` and then runs the chunk with the
// reference's fp32 operation order.  The carried value is the exact recurrence rounded once instead of the sequential
// fp32 one: the two differ by the rounding the sequential fp32 scan itself accumulates (a few ulp).
__global__ void gae_affine_kernel(const float* __restrict__ rew, const float* __restrict__ val, const float* __restrict__ dones,
                                  const float* __restrict__ last_val, const float* __restrict__ last_done, int T, int N,
                                  float gamma, float lam, int chunk, double2* __restrict__ ab) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (e >= N) return;
    const int t_lo = c * chunk;
    const int t_hi = min(T, t_lo + chunk) - 1;
    const double g = (double)gamma, gl = (double)__fmul_rn(gamma, lam);
    double A = 1.0, B = 0.0;
    double nextv = (t_hi == T - 1) ? (double)last_val[e] : (double)val[(size_t)(t_hi + 1) * N + e];
    double nextnt = 1.0 - ((t_hi == T - 1) ? (double)last_done[e] : (double)dones[(size_t)(t_hi + 1) * N + e]);
    for (int t = t_hi; t >= t_lo; --t) {
        const size_t idx = (size_t)t * N + e;
        const double v = (double)__ldg(val + idx);
        const double delta = (double)__ldg(rew + idx) + g * nextv * nextnt - v;
        const double ct = gl * nextnt;
        B = delta + ct * B;
        A = ct * A;
        nextv = v;
        nextnt = 1.0 - (double)__ldg(dones + idx);
    }
    ab[(size_t)c * N + e] = make_double2(A, B);
}

__global__ void gae_kernel_carry(const float* __restrict__ rew, const float* __restrict__ val, const float* __restrict__ dones,
                                 const float* __restrict__ last_val, const float* __restrict__ last_done, int T, int N,
                                 float gamma, float lam, int chunk, int nchunks, const double2* __restrict__ ab,
                                 float* __restrict__ adv_out, float* __restrict__ ret_out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (e >= N) return;
    double carry = 0.0;
    for (int cc = nchunks - 1; cc > c; --cc) {
        const double2 m = ab[(size_t)cc * N + e];
        carry = m.x * carry + m.y;
    }
    const int t_lo = c * chunk;
    const int t_hi = min(T, t_lo + chunk) - 1;
    const float gl = __fmul_rn(gamma, lam);
    float last = (float)carry;
    float nextv = (t_hi == T - 1) ? last_val[e] : val[(size_t)(t_hi + 1) * N + e];
    float nextnt = 1.0f - ((t_hi == T - 1) ? last_done[e] : dones[(size_t)(t_hi + 1) * N + e]);
    for (int t = t_hi; t >= t_lo; --t) {
        const size_t idx = (size_t)t * N + e;
        const float v = __ldg(val + idx);
        const float delta = __fsub_rn(__fadd_rn(__ldg(rew + idx), __fmul_rn(gamma, __fmul_rn(nextv, nextnt))), v);
        last = __fadd_rn(delta, __fmul_rn(gl, __fmul_rn(nextnt, last)));
        if (adv_out) adv_out[idx] = last;
        ret_out[idx] = __fadd_rn(last, v);
        nextv = v;
        nextnt = 1.0f - __ldg(dones + idx);
    }
}

// ------------------------------------------------------------------------------------------------
// Update-phase helpers.
// perm (semantic flat rows, row = env*T + t of the GLOBAL batch) -> gather list of physical rows:
// Eigen `perm * buf` writes out[perm[i]] = in[i] (ppo2.hpp:291-296), so minibatch slot s reads row i with perm[i]==s.
// physical row of semantic row i: env_g = i / T, t = i % T, rank r = env_g / Nl, el = env_g % Nl -> r*T*Nl + t*Nl + el
__global__ void build_gather_kernel(const int* __restrict__ perm, int n_batch, int T, int Nl, int* __restrict__ gather) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_batch) return;
    const int env_g = i / T, t = i - env_g * T;
    const int r = env_g / Nl, el = env_g - r * Nl;
    gather[perm[i]] = r * T * Nl + t * Nl + el;
}

// per-minibatch advantage statistics (ppo2.hpp:401-405): one CTA per minibatch.
// mean = sum(ret-val)/B ; var = sum((adv-mean)^2)/B ; denom = float(sqrt(var) + 1e-8)
// blockIdx.y = epoch when the gather lists / statistics of several epochs are laid out with the given strides
__global__ void advnorm_stats_kernel(const float* __restrict__ ret, const float* __restrict__ val,
                                     const int* __restrict__ gather, int B, float2* __restrict__ stats,
                                     size_t gather_stride = 0, int stats_stride = 0) {
    __shared__ double red[32];
    __shared__ float s_mean;
    const int k = blockIdx.x, tid = threadIdx.x;
    if (gather) gather += (size_t)blockIdx.y * gather_stride;
    stats += (size_t)blockIdx.y * stats_stride;
    const int* g = gather ? gather + (size_t)k * B : nullptr;
    // the gathered rows are random 4-byte reads: 8 independent (index -> row) chains in flight per thread
    constexpr int U = 8;
    double s = 0.0;
    {
        int i = tid;
        for (; i + (U - 1) * (int)blockDim.x < B; i += U * blockDim.x) {
            int row[U];
            float d[U];
#pragma unroll
            for (int u = 0; u < U; ++u) row[u] = g ? __ldg(g + i + u * blockDim.x) : (k * B + i + u * (int)blockDim.x);
#pragma unroll
            for (int u = 0; u < U; ++u) d[u] = __fsub_rn(__ldg(ret + row[u]), __ldg(val + row[u]));
#pragma unroll
            for (int u = 0; u < U; ++u) s += (double)d[u];
        }
        for (; i < B; i += blockDim.x) {
            const int row = g ? g[i] : (k * B + i);
            s += (double)__fsub_rn(ret[row], val[row]);
        }
    }
    s = warp_sum(s);
    if ((tid & 31) == 0) red[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) t += red[w];
        s_mean = (float)(t / (double)B);
    }
    __syncthreads();
    const float mean = s_mean;
    double q = 0.0;
    {
        int i = tid;
        for (; i + (U - 1) * (int)blockDim.x < B; i += U * blockDim.x) {
            int row[U];
            float d[U];
#pragma unroll
            for (int u = 0; u < U; ++u) row[u] = g ? __ldg(g + i + u * blockDim.x) : (k * B + i + u * (int)blockDim.x);
#pragma unroll
            for (int u = 0; u < U; ++u) d[u] = __fsub_rn(__fsub_rn(__ldg(ret + row[u]), __ldg(val + row[u])), mean);
#pragma unroll
            for (int u = 0; u < U; ++u) q += (double)__fmul_rn(d[u], d[u]);
        }
        for (; i < B; i += blockDim.x) {
            const int row = g ? g[i] : (k * B + i);
            const float d = __fsub_rn(__fsub_rn(ret[row], val[row]), mean);
            q += (double)__fmul_rn(d, d);
        }
    }
    q = warp_sum(q);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = q;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) t += red[w];
        const float var = (float)(t / (double)B);
        const float denom = (float)((double)__fsqrt_rn(var) + 1e-8);
        stats[k] = make_float2(mean, denom);
    }
}

__global__ void advnorm_apply_kernel(const float* __restrict__ ret, const float* __restrict__ val, int n,
                                     const float2* __restrict__ stats, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 st = *stats;
    out[i] = __fdiv_rn(__fsub_rn(__fsub_rn(ret[i], val[i]), st.x), st.y);
}

// sum the per-CTA partial slabs column-wise (fixed order, double accumulation) -> grad[PS];
// also per-block sum of squares of the first P columns (for the global norm when no allreduce follows).
__global__ void grad_reduce_kernel(const float* __restrict__ partial, int G, int PS, int P, float* __restrict__ grad,
                                   double* __restrict__ sq_partial) {
    __shared__ double red[32];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    double t = 0.0;
    if (c < PS) {
        for (int g = 0; g < G; ++g) t += (double)partial[(size_t)g * PS + c];
        grad[c] = (float)t;
    }
    const float gf = (c < P) ? (float)t : 0.f;
    double q = warp_sum((double)gf * (double)gf);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)blockDim.x / 32; ++w) s += red[w];
        sq_partial[blockIdx.x] = s;
    }
}

__global__ void sqnorm_kernel(const float* __restrict__ grad, int P, double* __restrict__ sq_partial) {
    __shared__ double red[32];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const float gf = (c < P) ? grad[c] : 0.f;
    double q = warp_sum((double)gf * (double)gf);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)blockDim.x / 32; ++w) s += red[w];
        sq_partial[blockIdx.x] = s;
    }
}

// clip_by_global_norm (GRAPH:24102-25392) + ApplyAdam for all 13 tensors flat + beta-power update
// (GRAPH:25426-31383; TF 1.14 ApplyAdam: epsilon outside the sqrt, not bias-corrected).
struct AdamArgs {
    float* params;
    float* m;
    float* v;
    const float* grad;         // [PS] summed over CTAs (and ranks); columns P.. hold the loss sums
    const double* sq_partial;  // [nblk]
    int nblk, P;
    const UpdateScalars* sc;  // lr of this update (device)
    float beta1, beta2, eps, clip_norm;
    const float* bpow_in;  // [2] beta1_power, beta2_power
    float* bpow_out;       // [2]
    float invB, inv_world;
    float* loss_row;       // [5] this step's pg, vf, entropy, approxkl, clipfrac
    float* gnorm_out;      // [1]
};

__global__ void adam_kernel(const AdamArgs a) {
    __shared__ float s_scale;
    __shared__ double s_ss[256];
    const float lr = a.sc->lr;
    {  // sum of the per-block partials in a fixed order: strided per thread, then a tree (every block does the same)
        double t = 0.0;
        for (int b = threadIdx.x; b < a.nblk; b += blockDim.x) t += a.sq_partial[b];
        s_ss[threadIdx.x] = t;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o && threadIdx.x + o < blockDim.x) s_ss[threadIdx.x] += s_ss[threadIdx.x + o];
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) {
        const double ss = s_ss[0];
        const float gnorm = (float)sqrt(ss);  // sqrt(2 * sum L2Loss(g_i))
        const float inv = __fdiv_rn(1.0f, gnorm), invc = __fdiv_rn(1.0f, a.clip_norm);
        float scale = __fmul_rn(a.clip_norm, fminf(inv, invc));
        if (!isfinite(gnorm)) scale = __int_as_float(0x7fc00000);  // GRAPH:24493-24543
        s_scale = scale;
        if (blockIdx.x == 0) {
            *a.gnorm_out = gnorm;
            const float* L = a.grad + a.P;
            a.loss_row[0] = L[L_PG] * a.invB;
            a.loss_row[1] = 0.5f * (L[L_VF] * a.invB);
            a.loss_row[2] = L[L_ENT] * a.inv_world;
            a.loss_row[3] = 0.5f * (L[L_KL] * a.invB);
            a.loss_row[4] = L[L_CLIP] * a.invB;
            a.bpow_out[0] = __fmul_rn(a.bpow_in[0], a.beta1);
            a.bpow_out[1] = __fmul_rn(a.bpow_in[1], a.beta2);
        }
    }
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.P) return;
    const float b1p = a.bpow_in[0], b2p = a.bpow_in[1];
    const float alpha = __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.0f, b2p))), __fsub_rn(1.0f, b1p));
    const float g = __fmul_rn(a.grad[i], s_scale);
    float m = a.m[i], v = a.v[i];
    m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), __fsub_rn(1.0f, a.beta1)));
    v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), __fsub_rn(1.0f, a.beta2)));
    a.m[i] = m;
    a.v[i] = v;
    a.params[i] = __fsub_rn(a.params[i], __fdiv_rn(__fmul_rn(m, alpha), __fadd_rn(__fsqrt_rn(v), a.eps)));
}

// Fused gradient step: column-reduce the CTA slabs -> (multi-GPU: allreduce through the peer mailboxes) -> global norm
// -> clip -> Adam, in ONE cooperative launch (replaces grad_reduce_kernel + ncclAllReduce + sqnorm_kernel + adam_kernel).
// A block owns 64-column chunks (chunk = blockIdx.x + j * gridDim.x, j < RA_MAXJ), 4 row groups of threads per chunk.
//   phase 1  sum the G slabs per column (fixed order: 4 interleaved row groups in fp32, combined in double)
//   phase 1b multi-GPU: store the block's columns into slot [seq & 1][rank] of EVERY rank's mailbox (NVLink P2P stores),
//            signal channel = blockIdx.x, wait for the same block of every peer, add the `world` slots in rank order
//            (every rank adds the same numbers in the same order -> replicas stay bit-identical)
//   phase 2  per-block sum of squares -> grid barrier -> global norm, clip scale, TF ApplyAdam on the block's columns
//            straight from registers, loss row, beta powers.
constexpr int RA_MAXJ = 4;
struct ReduceAdamArgs {
    const float* partial;
    int G, PS;
    float* grad;  // [PS] written for inspection / loss sums
    double* sq_partial;
    AdamArgs adam;
    unsigned* bar_ctr;  // grid barrier counter (monotonic) and generations completed (device-resident so that the
    unsigned* bar_gen;  // launch can be replayed from a CUDA graph)
    PeerMailbox mbox;   // world == 1: unused
    unsigned* mbox_seq; // device-resident sequence number of the gradient exchange
    // Sum-of-squares partials as LL words instead of a grid barrier (or NULL): every block stores its partial (a double and the
    // sequence number of the step in one 16-byte word) into the row of EVERY block, [parity][destination][source], and polls its
    // own row — one polling thread per word, no barrier between the column sums and Adam.  sq_seq: device-resident sequence number.
    uint4* sq_ll;
    unsigned* sq_seq;
};

// Body shared by the stand-alone cooperative kernel and the persistent epoch kernel (kernels_umma.cuh): `blk` of `nblk`
// blocks of 256 threads.  b1p / b2p are the beta powers BEFORE this step.  Contains one grid barrier.
// EXT: the 8 KB combine buffer is the caller's (16-byte aligned shared memory, `ext_part`) instead of a static array — the
// persistent epoch kernel lends an operand block that is idle during the gradient step.
template <bool EXT = false>
__device__ __forceinline__ void reduce_adam_device(const ReduceAdamArgs& r, int blk, int nblk, GridBarrier& bar, unsigned seq,
                                                   float b1p, float b2p, float* loss_row, long long* prof = nullptr, unsigned sqseq = 0u,
                                                   float* ext_part = nullptr) {
    __shared__ __align__(16) float part_static[EXT ? 1 : RA_MAXJ][8][64];
    float (*part)[8][64] = EXT ? reinterpret_cast<float (*)[8][64]>(ext_part) : part_static;
    __shared__ double red[8];
    __shared__ double s_parts[256];
    __shared__ float s_scale;
    const AdamArgs& a = r.adam;
    const int lane_c = threadIdx.x & 63, rg = threadIdx.x >> 6;
    const int nchunks = (r.PS + 63) >> 6;
    const int world = r.mbox.world;
    int pi = 0;
#define RA_PROF()                                                   \
    do {                                                            \
        if (prof && threadIdx.x == 0 && pi < 8) prof[pi++] = clock64(); \
    } while (0)
    RA_PROF();
    float gsum[1];
    double q = 0.0;
    static_assert(RA_MAXJ == 4, "one 64-thread group per chunk of a block");
    // phase 1: thread (column quad cq of the chunk, slab group sg) loads slabs sg, sg + 16, ... as float4 (rows are 16-byte
    // aligned: PS % 4 == 0); every load of this thread (all its chunks, 4 slabs at a time) is independent of the others
    const int cq = threadIdx.x & 15, sg = threadIdx.x >> 4;
    float4 acc4[RA_MAXJ];
#pragma unroll
    for (int j = 0; j < RA_MAXJ; ++j) acc4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
    for (int g0 = sg; g0 < r.G; g0 += 64) {  // one L2 round trip for G <= 64
        float4 v[RA_MAXJ][4];
#pragma unroll
        for (int j = 0; j < RA_MAXJ; ++j) {
            const int c = (blk + j * nblk) * 64 + 4 * cq;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int g = g0 + 16 * u;
                v[j][u] = (c < r.PS && g < r.G) ? __ldcg(reinterpret_cast<const float4*>(r.partial + (size_t)g * r.PS + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int j = 0; j < RA_MAXJ; ++j)
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                acc4[j].x += v[j][u].x; acc4[j].y += v[j][u].y; acc4[j].z += v[j][u].z; acc4[j].w += v[j][u].w;
            }
    }
    RA_PROF();
    // the two slab groups of a warp by a shuffle, the eight warps through shared memory (fixed order, combined in double)
#pragma unroll
    for (int j = 0; j < RA_MAXJ; ++j) {
        acc4[j].x += __shfl_xor_sync(0xffffffffu, acc4[j].x, 16);
        acc4[j].y += __shfl_xor_sync(0xffffffffu, acc4[j].y, 16);
        acc4[j].z += __shfl_xor_sync(0xffffffffu, acc4[j].z, 16);
        acc4[j].w += __shfl_xor_sync(0xffffffffu, acc4[j].w, 16);
    }
    __syncthreads();
    if ((threadIdx.x & 31) < 16) {
#pragma unroll
        for (int j = 0; j < RA_MAXJ; ++j) *reinterpret_cast<float4*>(&part[j][threadIdx.x >> 5][4 * cq]) = acc4[j];
    }
    __syncthreads();
    // From here on thread group rg (64 threads, one per column) owns chunk blk + rg * nblk (RA_MAXJ groups = RA_MAXJ chunks): the
    // groups combine, exchange and update their chunks side by side instead of group 0 walking through all of them.
    const int mychunk = blk + rg * nblk;
    const int c = mychunk * 64 + lane_c;
    const bool have = mychunk < nchunks;  // uniform per group
    float gs = 0.f;
    {
        float t4[8];
#pragma unroll
        for (int w = 0; w < 8; ++w) t4[w] = part[rg][w][lane_c];
        const double t = (((double)t4[0] + (double)t4[1]) + ((double)t4[2] + (double)t4[3])) + (((double)t4[4] + (double)t4[5]) + ((double)t4[6] + (double)t4[7]));
        if (have) gs = (float)t;
    }
    if (world > 1 && have && c < r.PS) {
        // LL store of (value, seq) into every rank's slot of this rank, then the `world` values of the column added in rank order
        // (the same order on every rank; four ranks' values in flight together)
        for (int dst = 0; dst < world; ++dst) ll_store(r.mbox.ll_slot(dst, seq, r.mbox.rank) + c, __float_as_uint(gs), seq);
        float t = 0.f;
        for (int s0 = 0; s0 < world; s0 += 4) {
            unsigned w[4];
            r.mbox.ll_wait4(seq, (size_t)c, s0, w);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (s0 + k < world) t += __uint_as_float(w[k]);
        }
        gs = t;
    }
    if (have) {
        if (c < r.PS) r.grad[c] = gs;
        if (c < a.P) q += (double)gs * (double)gs;
    }
    gsum[0] = gs;
    q = warp_sum(q);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
    __syncthreads();
    const double q_blk = ((red[0] + red[1]) + (red[2] + red[3])) + ((red[4] + red[5]) + (red[6] + red[7]));
    if (threadIdx.x == 0) r.sq_partial[blk] = q_blk;
    // Adam state of this thread's column: only this thread ever touches it, so it can be fetched ahead of the exchange
    const bool mine = have && c < a.P;
    float am = mine ? __ldcg(a.m + c) : 0.f;
    float av = mine ? __ldcg(a.v + c) : 0.f;
    const float ap = mine ? __ldcg(a.params + c) : 0.f;
    const float lr = a.sc->lr;  // (ahead of the exchange as well: after it, its latency would add to every minibatch)
    RA_PROF();
    const bool ll = r.sq_ll != nullptr;  // (nblk <= 256)
    if (ll) {
        const unsigned long long qb = (unsigned long long)__double_as_longlong(q_blk);
        uint4* const base = r.sq_ll + (size_t)(sqseq & 1u) * nblk * nblk;
        for (int dst = threadIdx.x; dst < nblk; dst += blockDim.x) {
            uint4* p = base + (size_t)dst * nblk + blk;
            asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"((unsigned)qb), "r"(sqseq), "r"((unsigned)(qb >> 32)), "r"(sqseq) : "memory");
        }
        if ((int)threadIdx.x < nblk) {
            const uint4* p = base + (size_t)blk * nblk + threadIdx.x;
            uint4 v;
            unsigned long long t0 = 0;
            unsigned spins = 0;
            while (true) {
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
                if (v.y == sqseq && v.w == sqseq) break;
                if (((++spins) & 0x3ffu) == 0u) {  // bounded like the mailbox waits (a block of this grid never arrived)
                    if (t0 == 0) t0 = globaltimer_ns();
                    if (globaltimer_ns() - t0 > 4000000000ull) {
                        *r.mbox.err = 1u;
                        break;
                    }
                }
            }
            s_parts[threadIdx.x] = __longlong_as_double((long long)(((unsigned long long)v.z << 32) | (unsigned long long)v.x));
        }
        __syncthreads();
    } else {
        bar.sync();
    }
    RA_PROF();
    if (threadIdx.x < 32) {
        double ss = 0.0;
        for (int b = threadIdx.x; b < nblk; b += 32) ss += ll ? s_parts[b] : __ldcg(r.sq_partial + b);
        // fixed-order combine: lane partials summed by a butterfly (same order in every block and on every rank)
        ss = warp_sum(ss);
        if (threadIdx.x == 0) {
            const float gnorm = (float)sqrt(ss);
            const float inv = __fdiv_rn(1.0f, gnorm), invc = __fdiv_rn(1.0f, a.clip_norm);
            float scale = __fmul_rn(a.clip_norm, fminf(inv, invc));
            if (!isfinite(gnorm)) scale = __int_as_float(0x7fc00000);
            s_scale = scale;
            if (blk == 0) *a.gnorm_out = gnorm;
        }
    }
    __syncthreads();
    RA_PROF();
    const int loss_chunk = (a.P >> 6);  // the chunk that holds column P (the loss sums start there)
    if (blk == loss_chunk % nblk && threadIdx.x == 0) {
        // columns P.. may straddle into another block's chunk: read through L2 (the LL variant is only used when they do not:
        // this block wrote them itself, before the __syncthreads above)
        const float* Ls = r.grad + a.P;
        float L[5];
        for (int k = 0; k < 5; ++k) L[k] = __ldcg(Ls + k);
        loss_row[0] = L[L_PG] * a.invB;
        loss_row[1] = 0.5f * (L[L_VF] * a.invB);
        loss_row[2] = L[L_ENT] * a.inv_world;
        loss_row[3] = 0.5f * (L[L_KL] * a.invB);
        loss_row[4] = L[L_CLIP] * a.invB;
    }
    if (mine) {
        const float alpha = __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.0f, b2p))), __fsub_rn(1.0f, b1p));
        const float g = __fmul_rn(gsum[0], s_scale);
        am = __fadd_rn(am, __fmul_rn(__fsub_rn(g, am), __fsub_rn(1.0f, a.beta1)));
        av = __fadd_rn(av, __fmul_rn(__fsub_rn(__fmul_rn(g, g), av), __fsub_rn(1.0f, a.beta2)));
        a.m[c] = am;
        a.v[c] = av;
        a.params[c] = __fsub_rn(ap, __fdiv_rn(__fmul_rn(am, alpha), __fadd_rn(__fsqrt_rn(av), a.eps)));
    }
    RA_PROF();
#undef RA_PROF
}

__global__ void __launch_bounds__(256) grad_reduce_adam_coop_kernel(const ReduceAdamArgs r) {
    GridBarrier bar{r.bar_ctr, gridDim.x, *r.bar_gen};
    const unsigned seq = r.mbox.world > 1 ? (*r.mbox_seq + 1u) : 0u;
    const unsigned sqseq = r.sq_ll ? (*r.sq_seq + 1u) : 0u;
    const float b1p = r.adam.bpow_in[0], b2p = r.adam.bpow_in[1];
    reduce_adam_device(r, (int)blockIdx.x, (int)gridDim.x, bar, seq, b1p, b2p, r.adam.loss_row, nullptr, sqseq);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        r.adam.bpow_out[0] = __fmul_rn(b1p, r.adam.beta1);
        r.adam.bpow_out[1] = __fmul_rn(b2p, r.adam.beta2);
        *r.bar_gen = bar.gen;
        if (r.mbox.world > 1) *r.mbox_seq = seq;
        // (every block has read sq_seq by now: block 0 got here only after polling a partial of each of them)
        if (r.sq_ll) *r.sq_seq = sqseq;
    }
}

// The same gradient step for parameter vectors too long for RA_MAXJ chunks per block (the W family: [256,256] has 2 285
// chunks): a block walks its chunks blk, blk + nblk, ... in passes — (A) column sums of every owned chunk, stored to r.grad
// and, multi-GPU, into every rank's mailbox slot; (B) multi-GPU: all peers' values of every owned chunk (the NVLink flights of
// all chunks overlap), summed in rank order; sum of squares; grid barrier; (C) clip + Adam per chunk, the gradient re-read
// from r.grad (this block wrote it).  Same arithmetic and summation order as reduce_adam_device.
__global__ void __launch_bounds__(256) grad_reduce_adam_big_kernel(const ReduceAdamArgs r) {
    __shared__ float part[4][64];
    __shared__ double red[8];
    __shared__ float s_scale;
    GridBarrier bar{r.bar_ctr, gridDim.x, *r.bar_gen};
    const AdamArgs& a = r.adam;
    const int blk = blockIdx.x, nblk = gridDim.x;
    const int lane_c = threadIdx.x & 63, rg = threadIdx.x >> 6;
    const int nchunks = (r.PS + 63) >> 6;
    const int world = r.mbox.world;
    const unsigned seq = world > 1 ? (*r.mbox_seq + 1u) : 0u;
    const float b1p = a.bpow_in[0], b2p = a.bpow_in[1];
    const float lr = a.sc->lr;
    double q = 0.0;
    for (int chunk0 = blk; chunk0 < nchunks; chunk0 += 4 * nblk) {  // pass A, four chunks per trip: their loads are in flight together
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
        for (int g0 = rg; g0 < r.G; g0 += 64) {
            float v[4][16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = (chunk0 + j * nblk) * 64 + lane_c;
#pragma unroll
                for (int u = 0; u < 16; ++u) {
                    const int g = g0 + 4 * u;
                    v[j][u] = (c < r.PS && g < r.G) ? __ldcg(r.partial + (size_t)g * r.PS + c) : 0.f;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int u = 0; u < 16; ++u) acc[j] += v[j][u];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int chunk = chunk0 + j * nblk;
            if (chunk >= nchunks) break;  // block-uniform
            const int c = chunk * 64 + lane_c;
            __syncthreads();
            part[rg][lane_c] = acc[j];
            __syncthreads();
            if (rg == 0 && c < r.PS) {
                const double t = ((double)part[0][lane_c] + (double)part[1][lane_c]) + ((double)part[2][lane_c] + (double)part[3][lane_c]);
                const float gs = (float)t;
                if (world > 1) {
                    for (int dst = 0; dst < world; ++dst) ll_store(r.mbox.ll_slot(dst, seq, r.mbox.rank) + c, __float_as_uint(gs), seq);
                } else {
                    r.grad[c] = gs;
                    if (c < a.P) q += (double)gs * (double)gs;
                }
            }
        }
    }
    if (world > 1 && rg == 0) {  // pass B
        for (int chunk = blk; chunk < nchunks; chunk += nblk) {
            const int c = chunk * 64 + lane_c;
            if (c < r.PS) {
                float t = 0.f;
                for (int s0 = 0; s0 < world; s0 += 4) {
                    unsigned w[4];
                    r.mbox.ll_wait4(seq, (size_t)c, s0, w);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (s0 + k < world) t += __uint_as_float(w[k]);
                }
                r.grad[c] = t;
                if (c < a.P) q += (double)t * (double)t;
            }
        }
    }
    q = warp_sum(q);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
    __syncthreads();
    if (threadIdx.x == 0) r.sq_partial[blk] = red[0] + red[1];
    bar.sync();
    if (threadIdx.x < 32) {
        double ss = 0.0;
        for (int b = threadIdx.x; b < nblk; b += 32) ss += __ldcg(r.sq_partial + b);
        ss = warp_sum(ss);
        if (threadIdx.x == 0) {
            const float gnorm = (float)sqrt(ss);
            const float inv = __fdiv_rn(1.0f, gnorm), invc = __fdiv_rn(1.0f, a.clip_norm);
            float scale = __fmul_rn(a.clip_norm, fminf(inv, invc));
            if (!isfinite(gnorm)) scale = __int_as_float(0x7fc00000);
            s_scale = scale;
            if (blk == 0) *a.gnorm_out = gnorm;
        }
    }
    __syncthreads();
    if (blk == 0 && threadIdx.x == 0) {  // the loss sums may sit in another block's chunk: every chunk passed the barrier
        const float* Ls = r.grad + a.P;
        float L[5];
        for (int k = 0; k < 5; ++k) L[k] = __ldcg(Ls + k);
        a.loss_row[0] = L[L_PG] * a.invB;
        a.loss_row[1] = 0.5f * (L[L_VF] * a.invB);
        a.loss_row[2] = L[L_ENT] * a.inv_world;
        a.loss_row[3] = 0.5f * (L[L_KL] * a.invB);
        a.loss_row[4] = L[L_CLIP] * a.invB;
    }
    if (rg == 0) {  // pass C, four chunks per trip: the sixteen loads of a trip are in flight together
        const float alpha = __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.0f, b2p))), __fsub_rn(1.0f, b1p));
        for (int chunk0 = blk; chunk0 < nchunks; chunk0 += 4 * nblk) {
            float gg[4], mm[4], vv[4], pp[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = (chunk0 + j * nblk) * 64 + lane_c;
                const bool ok = c < a.P;
                gg[j] = ok ? __ldcg(r.grad + c) : 0.f;
                mm[j] = ok ? __ldcg(a.m + c) : 0.f;
                vv[j] = ok ? __ldcg(a.v + c) : 0.f;
                pp[j] = ok ? __ldcg(a.params + c) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = (chunk0 + j * nblk) * 64 + lane_c;
                if (c < a.P) {
                    const float g = __fmul_rn(gg[j], s_scale);
                    float m = mm[j], v = vv[j];
                    m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), __fsub_rn(1.0f, a.beta1)));
                    v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), __fsub_rn(1.0f, a.beta2)));
                    a.m[c] = m;
                    a.v[c] = v;
                    a.params[c] = __fsub_rn(pp[j], __fdiv_rn(__fmul_rn(m, alpha), __fadd_rn(__fsqrt_rn(v), a.eps)));
                }
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.bpow_out[0] = __fmul_rn(b1p, a.beta1);
        a.bpow_out[1] = __fmul_rn(b2p, a.beta2);
        *r.bar_gen = bar.gen;
        if (world > 1) *r.mbox_seq = seq;
    }
}

// mean over the rows of the per-step loss table (colwise().mean(), ppo2.hpp:335)
__global__ void loss_mean_kernel(const float* __restrict__ rows, int nrows, float* __restrict__ out) {
    const int c = threadIdx.x;
    if (c >= 5) return;
    float s = 0.f;
    for (int r = 0; r < nrows; ++r) s += rows[r * 5 + c];
    out[c] = s / (float)nrows;
}

// physical (slab, time-major) <-> reference flat layout (row = env*T + t) conversion for export/import
__global__ void export_flat_kernel(const float* __restrict__ phys, int T, int N, int W, float* __restrict__ flat) {
    const size_t total = (size_t)T * N * W;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int w = (int)(e % W);
        const size_t row = e / W;  // flat row = env*T + t
        const int env = (int)(row / T), t = (int)(row % T);
        flat[e] = phys[((size_t)t * N + env) * W + w];
    }
}
__global__ void import_flat_kernel(const float* __restrict__ flat, int T, int N, int W, float* __restrict__ phys) {
    const size_t total = (size_t)T * N * W;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int w = (int)(e % W);
        const size_t row = e / W;
        const int env = (int)(row / T), t = (int)(row % T);
        phys[((size_t)t * N + env) * W + w] = flat[e];
    }
}

}  // namespace ppo
