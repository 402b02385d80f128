// Generic tile-based MLP kernels ("T family"): any hidden sizes, fp32 FFMA on CUDA cores.
//
// One CTA owns a tile of TM samples.  Activations of the tile live in shared memory feature-major
// ([feature][sample], leading dimension TM) so that a thread's 4x4 register tile reads 4 samples with one
// LDS.128; weights ([in,out] row-major as in the TF graph) are read through the read-only path and stay in
// L1/L2 — they are tiny (334 floats for the reference's [4,5] net, 48 KB for [64,64]).
//   policy_tile_kernel : pi/V forward + Gaussian sample (Philox) + neglogp      (MlpPolicy::step/value, policies.hpp:33-77)
//   train_tile_kernel  : loss forward + hand-derived backward -> per-CTA partial gradients (GRAPH:9210-23699)
#pragma once
#include "device_common.cuh"

namespace ppo {

constexpr int NT = 256;  // threads per CTA for the tile kernels

// Cs[n][m] = act( sum_k As[k][m] * W[k][n] + b[n] )      As: [K][TM] smem, W: [K][N] global, Cs: [N][TM] smem; act = FA (ACT_NONE: linear)
template <int TM, int FA>
__device__ __forceinline__ void tile_fwd(const float* __restrict__ As, int K, const float* __restrict__ W,
                                         const float* __restrict__ b, int N, float* __restrict__ Cs) {
    constexpr int MG = TM / 4, NGS = NT / MG;
    const int mg = threadIdx.x % MG, ng0 = threadIdx.x / MG;
    const int ngroups = (N + 3) >> 2;
    const bool vec = (N & 3) == 0;
    for (int ng = ng0; ng < ngroups; ng += NGS) {
        const int n = ng << 2;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (vec) {
#pragma unroll 4
            for (int k = 0; k < K; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(As + k * TM + mg * 4);
                const float4 w = __ldg(reinterpret_cast<const float4*>(W + (size_t)k * N + n));
                const float av[4] = {a.x, a.y, a.z, a.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(wv[i], av[j], acc[i][j]);
            }
        } else {
#pragma unroll 2
            for (int k = 0; k < K; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(As + k * TM + mg * 4);
                const float av[4] = {a.x, a.y, a.z, a.w};
                float wv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) wv[i] = (n + i < N) ? __ldg(W + (size_t)k * N + n + i) : 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(wv[i], av[j], acc[i][j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (n + i < N) {
                const float bb = __ldg(b + n + i);
                float4 o;
                o.x = acc[i][0] + bb; o.y = acc[i][1] + bb; o.z = acc[i][2] + bb; o.w = acc[i][3] + bb;
                if (FA != ACT_NONE) { o.x = act_fwd<FA>(o.x); o.y = act_fwd<FA>(o.y); o.z = act_fwd<FA>(o.z); o.w = act_fwd<FA>(o.w); }
                *reinterpret_cast<float4*>(Cs + (n + i) * TM + mg * 4) = o;
            }
        }
    }
}

// Ds[k][m] = ( sum_n W[k][n] * Ys[n][m] ) * act'(Hs[k][m])        (dY·Wᵀ then TanhGrad / ReluGrad; GRAPH:20925-23699)
template <int TM, int ACT>
__device__ __forceinline__ void tile_bwd_dx(const float* __restrict__ Ys, int N, const float* __restrict__ W, int K,
                                            const float* __restrict__ Hs, float* __restrict__ Ds) {
    constexpr int MG = TM / 4, KGS = NT / MG;
    const int mg = threadIdx.x % MG, kg0 = threadIdx.x / MG;
    const int kgroups = (K + 3) >> 2;
    const bool vec = (N & 3) == 0;
    for (int kg = kg0; kg < kgroups; kg += KGS) {
        const int k = kg << 2;
        int kr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) kr[i] = min(k + i, K - 1);
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (vec) {
            for (int n = 0; n < N; n += 4) {
                float4 y[4], w[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) y[q] = *reinterpret_cast<const float4*>(Ys + (n + q) * TM + mg * 4);
#pragma unroll
                for (int i = 0; i < 4; ++i) w[i] = __ldg(reinterpret_cast<const float4*>(W + (size_t)kr[i] * N + n));
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float wv[4] = {w[i].x, w[i].y, w[i].z, w[i].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        acc[i][0] = fmaf(wv[q], y[q].x, acc[i][0]);
                        acc[i][1] = fmaf(wv[q], y[q].y, acc[i][1]);
                        acc[i][2] = fmaf(wv[q], y[q].z, acc[i][2]);
                        acc[i][3] = fmaf(wv[q], y[q].w, acc[i][3]);
                    }
                }
            }
        } else {
            for (int n = 0; n < N; ++n) {
                const float4 y = *reinterpret_cast<const float4*>(Ys + n * TM + mg * 4);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float wv = __ldg(W + (size_t)kr[i] * N + n);
                    acc[i][0] = fmaf(wv, y.x, acc[i][0]);
                    acc[i][1] = fmaf(wv, y.y, acc[i][1]);
                    acc[i][2] = fmaf(wv, y.z, acc[i][2]);
                    acc[i][3] = fmaf(wv, y.w, acc[i][3]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (k + i < K) {
                const float4 h = *reinterpret_cast<const float4*>(Hs + (k + i) * TM + mg * 4);
                float4 o;
                o.x = acc[i][0] * act_dfac<ACT>(h.x);
                o.y = acc[i][1] * act_dfac<ACT>(h.y);
                o.z = acc[i][2] * act_dfac<ACT>(h.z);
                o.w = acc[i][3] * act_dfac<ACT>(h.w);
                *reinterpret_cast<float4*>(Ds + (k + i) * TM + mg * 4) = o;
            }
        }
    }
}

// G[k][n] (+)= sum_m As[k][m] * Ys[n][m]      (Xᵀ·dY weight gradient of this tile) -> global partial slab
template <int TM>
__device__ __forceinline__ void tile_dw(const float* __restrict__ As, int K, const float* __restrict__ Ys, int N,
                                        float* __restrict__ G, bool accumulate) {
    constexpr int MG = TM / 4;
    const int kgroups = (K + 3) >> 2, ngroups = (N + 3) >> 2;
    for (int tt = threadIdx.x; tt < kgroups * ngroups; tt += NT) {
        const int kg = tt / ngroups, ng = tt - kg * ngroups;
        const int k = kg << 2, n = ng << 2;
        int kr[4], nr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            kr[i] = min(k + i, K - 1) * TM;
            nr[i] = min(n + i, N - 1) * TM;
        }
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 2
        for (int it = 0; it < MG; ++it) {
            const int m4 = ((it + ng) % MG) * 4;  // skewed start: threads of a warp hit different banks
            float4 a[4], y[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                a[i] = *reinterpret_cast<const float4*>(As + kr[i] + m4);
                y[i] = *reinterpret_cast<const float4*>(Ys + nr[i] + m4);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    acc[i][j] = fmaf(a[i].x, y[j].x, acc[i][j]);
                    acc[i][j] = fmaf(a[i].y, y[j].y, acc[i][j]);
                    acc[i][j] = fmaf(a[i].z, y[j].z, acc[i][j]);
                    acc[i][j] = fmaf(a[i].w, y[j].w, acc[i][j]);
                }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (k + i < K && n + j < N) {
                    float* g = G + (size_t)(k + i) * N + n + j;
                    *g = accumulate ? (*g + acc[i][j]) : acc[i][j];
                }
    }
}

// G[n] (+)= sum_m Ys[n][m]   (bias / logstd gradients)
template <int TM>
__device__ __forceinline__ void tile_rowsum(const float* __restrict__ Ys, int N, float* __restrict__ G, bool accumulate) {
    for (int n = threadIdx.x; n < N; n += NT) {
        float s = 0.f;
        for (int it = 0; it < TM; ++it) s += Ys[n * TM + ((it + n) % TM)];
        G[n] = accumulate ? (G[n] + s) : s;
    }
}

// transposed, gathered tile load: dst[k][m] = src[rows[m]][k]
template <int TM>
__device__ __forceinline__ void tile_load_rows(const float* __restrict__ src, int width, const int* __restrict__ rows,
                                               int nvalid, float* __restrict__ dst) {
    for (int e = threadIdx.x; e < TM * width; e += NT) {
        const int m = e / width, k = e - m * width;
        dst[k * TM + m] = (m < nvalid) ? __ldg(src + (size_t)rows[m] * width + k) : 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
struct PolicyArgs {
    NetDims d;
    const float* params;
    const float* obs;  // [n][O] (already normalised)
    int n;
    uint32_t md_lo;    // MultiDiscrete head: slice-start mask (md_sample), bits 0-31 here and 32-63 in md_hi, both in padding
    const float* eps;  // optional [n][A]; when NULL Philox noise for (seed, env_id0+i, *step_ctr)
    uint64_t seed;
    uint32_t env_id0;
    uint32_t md_hi;
    const uint32_t* step_ctr;
    float* action;   // [n][A] or NULL
    float* value;    // [n] or NULL
    float* neglogp;  // [n] or NULL
    // optional rollout stores for step t (time-major slabs)
    float* obs_store;    // [n][O]
    float* act_store;    // [n][A]
    float* val_store;    // [n]
    float* nlp_store;    // [n]
    const float* dones_in;  // [n] done flag of the previous env step (runner.hpp:110)
    float* dones_store;     // [n]
    int mode;  // 0: step (pi + V + sample), 1: value only, 2: mean only (deterministic action)
    // action masks of a Discrete / MultiDiscrete head (device_common.cuh): [n] words, bit j = logit j allowed, or NULL (all allowed);
    // mask_store: rollout slab of step t that receives them, or NULL
    const uint64_t* mask;
    uint64_t* mask_store;
};
// the slice-start mask of a MultiDiscrete head from its two halves
__host__ __device__ __forceinline__ uint64_t md_starts(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

__device__ __forceinline__ void store_neglogp(const PolicyArgs& a, int row, float nl) {
    if (a.neglogp) a.neglogp[row] = nl;
    if (a.nlp_store) a.nlp_store[row] = nl;
}

// Gaussian policy step of env `row` (mode 0) on a thread-per-row kernel: act_j = mu_j + exp(logstd_j) e_j with e_j from
// a.eps, or from Philox stream (seed, env, *step_ctr, block j/4, PPO_TAG_ACTION), and neglogp.  logstd(j), mean(j) return
// logstd_j and mu_j; put(j, act) stores the action.  A by reference: a runtime width is read from the kernel parameter
// where it is used (a copy held in a register changes the generated code of the kernels); a compile-time width unrolls.
template <class LS, class MU, class PUT>
__device__ __forceinline__ void gauss_policy_row(const PolicyArgs& a, int row, const int& A, LS logstd, MU mean, PUT put) {
    const uint32_t step = a.eps ? 0u : *a.step_ctr;
    float ss = 0.f, sl = 0.f;
#pragma unroll
    for (int j0 = 0; j0 < A; j0 += 4) {
        float e4[4];
        if (!a.eps) normal4(a.seed, a.env_id0 + (uint32_t)row, step, (uint32_t)(j0 >> 2), PPO_TAG_ACTION, e4);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < A) {
                const float ls = logstd(j);
                const float sd = expf(ls);  // logstd_b = mean*0 + logstd; std = exp (GRAPH:5098-5779)
                const float e = a.eps ? a.eps[(size_t)row * A + j] : e4[q];
                float z2;
                put(j, gauss_sample(mean(j), sd, e, z2));
                ss = __fadd_rn(ss, z2);
                sl = __fadd_rn(sl, ls);
            }
        }
    }
    store_neglogp(a, row, gauss_neglogp_rn(ss, sl, A));
}

// the action mask word of env `row` (all ones without masks), stored into the rollout slab when the step records one
__device__ __forceinline__ uint64_t policy_mask_word(const PolicyArgs& a, int row) {
    const uint64_t m = a.mask ? a.mask[row] : ~0ull;
    if (a.mask_store) a.mask_store[row] = m;
    return m;
}

// Categorical policy step of env `row` (logits l[j * ld]): the index as fp32 in one column, sampled (mode 0; a.eps: [n][A]
// uniforms when given) or argmax (mode 2), over the logits the row's mask allows
__device__ __forceinline__ void cat_policy_row(const PolicyArgs& a, int row, const float* l, int ld) {
    const uint64_t m = policy_mask_word(a, row);
    const int j = a.mode == 0 ? cat_sample(l, ld, a.d.A, a.eps ? a.eps + (size_t)row * a.d.A : nullptr, a.seed, a.env_id0 + (uint32_t)row,
                                           a.eps ? 0u : *a.step_ctr, m)
                              : cat_argmax(l, ld, a.d.A, m);
    if (a.action) a.action[row] = (float)j;
    if (a.act_store) a.act_store[row] = (float)j;
    if (a.mode == 0) store_neglogp(a, row, cat_neglogp(l, ld, a.d.A, j, m));
}

// MultiDiscrete policy step: k indices in k columns, sampled per slice (mode 0, neglogp their sum) or argmax per slice (mode 2)
__device__ __forceinline__ void md_policy_row(const PolicyArgs& a, int row, const float* l, int ld) {
    const uint64_t starts = md_starts(a.md_lo, a.md_hi);
    const int k = __popcll((long long)starts);
    const uint64_t m = policy_mask_word(a, row);
    auto put = [&](int i, int j) {
        if (a.action) a.action[(size_t)row * k + i] = (float)j;
        if (a.act_store) a.act_store[(size_t)row * k + i] = (float)j;
    };
    if (a.mode == 0) {
        float nlp = 0.f;
        int s0 = 0;
        md_sample(l, ld, a.d.A, starts, a.eps ? a.eps + (size_t)row * a.d.A : nullptr, a.seed, a.env_id0 + (uint32_t)row, a.eps ? 0u : *a.step_ctr,
                  [&](int i, int j) {
                      put(i, j);
                      const int s1 = md_slice_end(starts, s0, a.d.A);
                      nlp += cat_neglogp(l + s0 * ld, ld, s1 - s0, j, m >> s0);
                      s0 = s1;
                  },
                  m);
        store_neglogp(a, row, nlp);
    } else {
        for (int i = 0, s0 = 0; s0 < a.d.A; ++i) {
            const int s1 = md_slice_end(starts, s0, a.d.A);
            put(i, cat_argmax(l + s0 * ld, ld, s1 - s0, m >> s0));
            s0 = s1;
        }
    }
}

// MultiBinary policy step: A columns of 0 / 1, sampled (mode 0, with neglogp) or round(sigmoid(l)) (mode 2; TF's Round is half to
// even, so l = 0 gives 0)
__device__ __forceinline__ void bern_policy_row(const PolicyArgs& a, int row, const float* l, int ld) {
    const int n = a.d.A;
    auto put = [&](int j, float x) {
        if (a.action) a.action[(size_t)row * n + j] = x;
        if (a.act_store) a.act_store[(size_t)row * n + j] = x;
    };
    if (a.mode == 0) {
        float nlp = 0.f;
        bern_sample(l, ld, n, a.eps ? a.eps + (size_t)row * n : nullptr, a.seed, a.env_id0 + (uint32_t)row, a.eps ? 0u : *a.step_ctr,
                    [&](int j, float x) {
                        put(j, x);
                        nlp += bern_sce(l[j * ld], x);
                    });
        store_neglogp(a, row, nlp);
    } else {
        for (int j = 0; j < n; ++j) put(j, bern_sigmoid(l[j * ld]) > 0.5f ? 1.f : 0.f);
    }
}

// the policy step of a head without logstd (modes 0 and 2), logits l[j * ld]; the actions go straight to their rows
template <int HEAD>
__device__ __forceinline__ void head_policy_row(const PolicyArgs& a, int row, const float* l, int ld) {
    if constexpr (HEAD == HEAD_DISCRETE) cat_policy_row(a, row, l, ld);
    else if constexpr (HEAD == HEAD_MULTI_DISCRETE) md_policy_row(a, row, l, ld);
    else bern_policy_row(a, row, l, ld);
}

template <int TM>
__host__ __device__ inline size_t policy_smem_floats(const NetDims& d) {
    return (size_t)(d.O + d.H1 + d.H2 + d.A + 1) * TM + (size_t)d.A * (TM + 1);
}

template <int TM, int ACT, int HEAD>
__global__ void __launch_bounds__(NT) policy_tile_kernel(const PolicyArgs a) {
    extern __shared__ __align__(16) float smem[];
    const NetDims& d = a.d;
    float* Xs = smem;
    float* H1s = Xs + d.O * TM;
    float* H2s = H1s + d.H1 * TM;
    float* MU = H2s + d.H2 * TM;
    float* Vs = MU + d.A * TM;
    float* Ac = Vs + TM;  // [A][TM+1] actions staged for a coalesced write-out
    const float* p = a.params;
    const int tid = threadIdx.x;
    const int ntiles = (a.n + TM - 1) / TM;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int r0 = tile * TM, nv = min(TM, a.n - r0);
        for (int e = tid; e < TM * d.O; e += NT) {
            const int m = e / d.O, k = e - m * d.O;
            const float x = (m < nv) ? a.obs[(size_t)(r0 + m) * d.O + k] : 0.f;
            Xs[k * TM + m] = x;
            if (a.obs_store && m < nv) a.obs_store[(size_t)(r0 + m) * d.O + k] = x;
        }
        __syncthreads();
        if (a.mode != 1) {
            tile_fwd<TM, ACT>(Xs, d.O, p + d.off[T_PI_FC0_W], p + d.off[T_PI_FC0_B], d.H1, H1s);
            __syncthreads();
            tile_fwd<TM, ACT>(H1s, d.H1, p + d.off[T_PI_FC1_W], p + d.off[T_PI_FC1_B], d.H2, H2s);
            __syncthreads();
            tile_fwd<TM, ACT_NONE>(H2s, d.H2, p + d.off[T_PI_W], p + d.off[T_PI_B], d.A, MU);
            __syncthreads();
        }
        if (a.mode != 2) {
            tile_fwd<TM, ACT>(Xs, d.O, p + d.off[T_VF_FC0_W], p + d.off[T_VF_FC0_B], d.H1, H1s);
            __syncthreads();
            tile_fwd<TM, ACT>(H1s, d.H1, p + d.off[T_VF_FC1_W], p + d.off[T_VF_FC1_B], d.H2, H2s);
            __syncthreads();
            tile_fwd<TM, ACT_NONE>(H2s, d.H2, p + d.off[T_VF_W], p + d.off[T_VF_B], 1, Vs);
            __syncthreads();
        }
        if (tid < nv) {
            const int m = tid, row = r0 + m;
            if (a.mode != 2) {
                const float v = Vs[m];
                if (a.value) a.value[row] = v;
                if (a.val_store) a.val_store[row] = v;
            }
            if (HEAD != HEAD_BOX && a.mode != 1) {
                head_policy_row<HEAD>(a, row, MU + m, TM);
            } else if (a.mode == 0) {
                const float* logstd = p + d.off[T_LOGSTD];
                gauss_policy_row(a, row, d.A, [&](int j) { return __ldg(logstd + j); }, [&](int j) { return MU[j * TM + m]; },
                                 [&](int j, float act) { Ac[j * (TM + 1) + m] = act; });
            } else if (a.mode == 2) {
                for (int j = 0; j < d.A; ++j) Ac[j * (TM + 1) + m] = MU[j * TM + m];  // mean + 0.0 (GRAPH:6046-6076)
            }
            if (a.dones_store) a.dones_store[row] = a.dones_in[row];
        }
        __syncthreads();
        if (HEAD == HEAD_BOX && a.mode != 1) {  // a head without logstd stored its actions above
            for (int e = tid; e < nv * d.A; e += NT) {
                const int m = e / d.A, j = e - m * d.A;
                const float act = Ac[j * (TM + 1) + m];
                if (a.action) a.action[(size_t)(r0 + m) * d.A + j] = act;
                if (a.act_store) a.act_store[(size_t)(r0 + m) * d.A + j] = act;
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
struct TrainArgs {
    NetDims d;
    const float* params;
    const float *obs, *act, *ret, *val, *nlp;  // rollout buffers (physical rows)
    const int* gather;                          // [slots] physical row per minibatch slot, or NULL (identity)
    const float2* mbstats;                      // (mean, denom) of this minibatch's advantages, or NULL with adv_direct
    const float* adv_direct;                    // already-normalised advantages per slot (ppo_loss_grad), or NULL
    int slot0, count;                           // this rank processes slots [slot0, slot0+count)
    float invB;                                 // 1 / (global minibatch size)
    uint32_t md_lo;                             // MultiDiscrete head: slice-start mask (see PolicyArgs), in padding
    const UpdateScalars* sc;                    // cliprange, cliprange_vf of this update (device)
    int vf_mode;                                // VF_CLIP_*
    float ent_coef, vf_coef;
    uint32_t md_hi;
    float* partial;  // [gridDim.x][PS]
    int PS;
    long long* prof;  // optional [2][32] phase timestamps of CTA 0 of each tower (U family, PPO_UMMA_PROF=1)
    const uint64_t* mask;  // action masks of a Discrete / MultiDiscrete head by physical row (as act), or NULL (all allowed)
};
// the MultiDiscrete slice mask fills padding; the action-mask pointers are appended, so every earlier field keeps its offset
static_assert(sizeof(PolicyArgs) == 240 && sizeof(TrainArgs) == 232, "PolicyArgs / TrainArgs changed size");

// floats of one stored action: the action vector (Box), the index of a categorical head, the k indices of a MultiDiscrete head,
// the A bits of a MultiBinary head
template <int HEAD>
__device__ __forceinline__ int act_cols(const TrainArgs& a) {
    return HEAD == HEAD_DISCRETE ? 1 : HEAD == HEAD_MULTI_DISCRETE ? __popcll((long long)md_starts(a.md_lo, a.md_hi)) : a.d.A;
}

// the action mask word of the sample at physical row `row` (all ones without masks; a MultiBinary head has none)
template <int HEAD>
__device__ __forceinline__ uint64_t train_mask_word(const TrainArgs& a, int row) {
    if constexpr (HEAD == HEAD_DISCRETE || HEAD == HEAD_MULTI_DISCRETE) return a.mask ? a.mask[row] : ~0ull;
    else return ~0ull;
}

// one sample's train terms of a head without logstd over n logits l[j * ld]: neglogp of the stored action (act[j * ald]) and
// entropy H, the clipped surrogate of pg_term, and the logits overwritten with dL/dl (ent_w = ent_coef / B); m: the sample's mask word
template <int HEAD>
__device__ __forceinline__ PgTerm head_train_term(const TrainArgs& a, float* l, int ld, int n, const float* act, int ald, float adv, float oldn,
                                                  float cr, float invB, float ent_w, float& H, uint64_t m) {
    if constexpr (HEAD == HEAD_DISCRETE) return cat_train_term(l, ld, n, (int)act[0], adv, oldn, cr, invB, ent_w, H, m);
    else if constexpr (HEAD == HEAD_MULTI_DISCRETE) return md_train_term(l, ld, n, md_starts(a.md_lo, a.md_hi), act, ald, adv, oldn, cr, invB, ent_w, H, m);
    else return bern_train_term(l, ld, n, act, ald, adv, oldn, cr, invB, ent_w, H);
}

// This CTA's loss sums -> columns P.. of its slab (L = slab + P), the warps combined in a fixed order through s_red
// (5 * NTH / 32 floats).  Entropy column: a head without logstd: the sum of H / B (x world, see UpdateScalars) over the CTA's
// samples; a Box head's box_entropy of the pre-update logstd (logstd(j) loads logstd_j), in CTA 0 only.  A by reference as in
// gauss_policy_row.
template <int NTH, int HEAD, class LS>
__device__ __forceinline__ void store_loss_columns(float* L, float l_pg, float l_vf, float l_kl, float l_cf, float l_ent, float* s_red,
                                                   LS logstd, const int& A) {
    const int tid = threadIdx.x;
    constexpr int NL = HEAD != HEAD_BOX ? 5 : 4;
    float v4[NL];
    v4[0] = l_pg; v4[1] = l_vf; v4[2] = l_kl; v4[3] = l_cf;
    if (HEAD != HEAD_BOX) v4[NL - 1] = l_ent;
#pragma unroll
    for (int q = 0; q < NL; ++q) v4[q] = warp_sum(v4[q]);
    if ((tid & 31) == 0) {
#pragma unroll
        for (int q = 0; q < NL; ++q) s_red[(tid >> 5) * NL + q] = v4[q];
    }
    __syncthreads();
    if (tid == 0) {
        float t[NL];
        for (int q = 0; q < NL; ++q) t[q] = 0.f;
        for (int w = 0; w < NTH / 32; ++w)
            for (int q = 0; q < NL; ++q) t[q] += s_red[w * NL + q];
        L[L_PG] = t[0]; L[L_VF] = t[1]; L[L_KL] = t[2]; L[L_CLIP] = t[3];
        float ent = 0.f;
        if (HEAD != HEAD_BOX) ent = t[NL - 1];
        else if (blockIdx.x == 0) ent = box_entropy(logstd, A);
        L[L_ENT] = ent;
        L[5] = 0.f; L[6] = 0.f; L[7] = 0.f;
    }
}

template <int TM>
__host__ __device__ inline size_t train_smem_floats(const NetDims& d) {
    return (size_t)(d.O + 2 * d.A + 2 * d.H1 + 2 * d.H2) * TM + 5 * (size_t)TM + 64;
}

template <int TM, int ACT, int HEAD>
__global__ void __launch_bounds__(NT) train_tile_kernel(const TrainArgs a) {
    extern __shared__ __align__(16) float smem[];
    const NetDims& d = a.d;
    float* Xs = smem;
    float* Ac = Xs + d.O * TM;
    float* H1s = Ac + d.A * TM;
    float* H2s = H1s + d.H1 * TM;
    float* MU = H2s + d.H2 * TM;
    float* D2 = MU + d.A * TM;
    float* D1 = D2 + d.H2 * TM;
    float* s_adv = D1 + d.H1 * TM;
    float* s_ret = s_adv + TM;
    float* s_oldn = s_ret + TM;
    float* s_oldv = s_oldn + TM;
    int* s_row = reinterpret_cast<int*>(s_oldv + TM);
    float* s_red = reinterpret_cast<float*>(s_row + TM);  // 64 floats

    const float* p = a.params;
    const int tid = threadIdx.x;
    float* my = a.partial + (size_t)blockIdx.x * a.PS;
    const int ntiles = (a.count + TM - 1) / TM;
    const float cr = a.sc->cliprange, vr = vf_clip_range(a.vf_mode, cr, a.sc->cliprange_vf);
    float l_pg = 0.f, l_vf = 0.f, l_kl = 0.f, l_cf = 0.f, l_ent = 0.f;
    bool acc = false;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int s0 = a.slot0 + tile * TM;
        const int nv = min(TM, a.slot0 + a.count - s0);
        uint64_t mw = ~0ull;  // thread tid's sample: its action mask word
        if (tid < TM) {
            float adv = 0.f, r = 0.f, on = 0.f, ov = 0.f;
            int row = 0;
            if (tid < nv) {
                row = a.gather ? a.gather[s0 + tid] : (s0 + tid);
                mw = train_mask_word<HEAD>(a, row);
                r = a.ret[row];
                ov = a.val[row];
                on = a.nlp[row];
                if (a.adv_direct) {
                    adv = a.adv_direct[s0 + tid];
                } else {  // advs = (returns - values - mean) / (sqrt(var) + 1e-8)  (ppo2.hpp:401-406)
                    const float2 st = *a.mbstats;
                    adv = __fdiv_rn(__fsub_rn(__fsub_rn(r, ov), st.x), st.y);
                }
            }
            s_adv[tid] = adv; s_ret[tid] = r; s_oldn[tid] = on; s_oldv[tid] = ov; s_row[tid] = row;
        }
        __syncthreads();
        tile_load_rows<TM>(a.obs, d.O, s_row, nv, Xs);
        tile_load_rows<TM>(a.act, act_cols<HEAD>(a), s_row, nv, Ac);
        __syncthreads();

        // ---------------- pi tower ----------------
        tile_fwd<TM, ACT>(Xs, d.O, p + d.off[T_PI_FC0_W], p + d.off[T_PI_FC0_B], d.H1, H1s);
        __syncthreads();
        tile_fwd<TM, ACT>(H1s, d.H1, p + d.off[T_PI_FC1_W], p + d.off[T_PI_FC1_B], d.H2, H2s);
        __syncthreads();
        tile_fwd<TM, ACT_NONE>(H2s, d.H2, p + d.off[T_PI_W], p + d.off[T_PI_B], d.A, MU);
        __syncthreads();
        if (HEAD != HEAD_BOX && tid < TM) {  // a thread per sample over the A logits; MU becomes dL/dlogits
            const int m = tid;
            float* l = MU + m;
            if (m < nv) {
                float H;
                const PgTerm t = head_train_term<HEAD>(a, l, TM, d.A, Ac + m, TM, s_adv[m], s_oldn[m], cr, a.invB, a.ent_coef * a.invB, H, mw);
                l_pg += t.pg;
                l_kl += t.kl;
                l_cf += t.cf;
                l_ent += H * (a.invB * a.sc->world);
            } else {
                for (int j = 0; j < d.A; ++j) l[j * TM] = 0.f;
            }
        } else if (tid < TM) {
            const int m = tid;
            const float* logstd = p + d.off[T_LOGSTD];
            float g_nlp = 0.f;
            if (m < nv) {
                float ss = 0.f, sl = 0.f;
                for (int j = 0; j < d.A; ++j) {
                    const float ls = __ldg(logstd + j);
                    const float z = (Ac[j * TM + m] - MU[j * TM + m]) / expf(ls);
                    ss += z * z;
                    sl += ls;
                }
                const PgTerm t = pg_term(s_adv[m], s_oldn[m], gauss_neglogp(ss, sl, d.A), cr, a.invB);
                l_pg += t.pg;
                l_kl += t.kl;
                l_cf += t.cf;
                g_nlp = t.g_nlp;
            }
            for (int j = 0; j < d.A; ++j) {
                const float sd = expf(__ldg(logstd + j));
                const float z = (Ac[j * TM + m] - MU[j * TM + m]) / sd;
                Ac[j * TM + m] = g_nlp * (1.f - z * z);  // d nlp / d logstd_j contribution
                MU[j * TM + m] = g_nlp * (-z / sd);      // dL/dmu
            }
        }
        __syncthreads();
        tile_dw<TM>(H2s, d.H2, MU, d.A, my + d.off[T_PI_W], acc);
        tile_rowsum<TM>(MU, d.A, my + d.off[T_PI_B], acc);
        if (HEAD == HEAD_BOX) tile_rowsum<TM>(Ac, d.A, my + d.off[T_LOGSTD], acc);
        tile_bwd_dx<TM, ACT>(MU, d.A, p + d.off[T_PI_W], d.H2, H2s, D2);
        __syncthreads();
        tile_dw<TM>(H1s, d.H1, D2, d.H2, my + d.off[T_PI_FC1_W], acc);
        tile_rowsum<TM>(D2, d.H2, my + d.off[T_PI_FC1_B], acc);
        tile_bwd_dx<TM, ACT>(D2, d.H2, p + d.off[T_PI_FC1_W], d.H1, H1s, D1);
        __syncthreads();
        tile_dw<TM>(Xs, d.O, D1, d.H1, my + d.off[T_PI_FC0_W], acc);
        tile_rowsum<TM>(D1, d.H1, my + d.off[T_PI_FC0_B], acc);
        __syncthreads();

        // ---------------- value tower ----------------
        tile_fwd<TM, ACT>(Xs, d.O, p + d.off[T_VF_FC0_W], p + d.off[T_VF_FC0_B], d.H1, H1s);
        __syncthreads();
        tile_fwd<TM, ACT>(H1s, d.H1, p + d.off[T_VF_FC1_W], p + d.off[T_VF_FC1_B], d.H2, H2s);
        __syncthreads();
        tile_fwd<TM, ACT_NONE>(H2s, d.H2, p + d.off[T_VF_W], p + d.off[T_VF_B], 1, MU);
        __syncthreads();
        if (tid < TM) {
            const int m = tid;
            float dv = 0.f;
            if (m < nv) {
                l_vf += value_loss_term(a.vf_mode, vr, MU[m], s_oldv[m], s_ret[m], a.vf_coef, a.invB, dv);  // GRAPH:10213-10305, 14975-15142
            }
            MU[m] = dv;
        }
        __syncthreads();
        tile_dw<TM>(H2s, d.H2, MU, 1, my + d.off[T_VF_W], acc);
        tile_rowsum<TM>(MU, 1, my + d.off[T_VF_B], acc);
        tile_bwd_dx<TM, ACT>(MU, 1, p + d.off[T_VF_W], d.H2, H2s, D2);
        __syncthreads();
        tile_dw<TM>(H1s, d.H1, D2, d.H2, my + d.off[T_VF_FC1_W], acc);
        tile_rowsum<TM>(D2, d.H2, my + d.off[T_VF_FC1_B], acc);
        tile_bwd_dx<TM, ACT>(D2, d.H2, p + d.off[T_VF_FC1_W], d.H1, H1s, D1);
        __syncthreads();
        tile_dw<TM>(Xs, d.O, D1, d.H1, my + d.off[T_VF_FC0_W], acc);
        tile_rowsum<TM>(D1, d.H1, my + d.off[T_VF_FC0_B], acc);
        __syncthreads();
        acc = true;
    }

    // loss sums of this CTA -> columns P.. of its slab (threads >= TM hold zeros)
    store_loss_columns<NT, HEAD>(my + d.P, l_pg, l_vf, l_kl, l_cf, l_ent, s_red, [ls = p + d.off[T_LOGSTD]](int j) { return __ldg(ls + j); }, d.A);
    // loss = pg_loss - entropy*ent_coef + vf_loss*vf_coef: d(-ent_coef*entropy)/dlogstd_j = -ent_coef, added once
    // (a.ent_coef is already divided by the number of ranks whose slabs get summed)
    if (HEAD == HEAD_BOX && blockIdx.x == 0 && tid < d.A) my[d.off[T_LOGSTD] + tid] -= a.ent_coef;  // same thread wrote it in tile_rowsum
}

}  // namespace ppo
