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
    const float* eps;  // optional [n][A]; when NULL Philox noise for (seed, env_id0+i, *step_ctr)
    uint64_t seed;
    uint32_t env_id0;
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
};

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
            if (HEAD == HEAD_DISCRETE && a.mode != 1) {  // the index as fp32, one column; eps: [n][A] uniforms when given
                const float* l = MU + m;
                const int j = a.mode == 0 ? cat_sample(l, TM, d.A, a.eps ? a.eps + (size_t)row * d.A : nullptr, a.seed,
                                                       a.env_id0 + (uint32_t)row, a.eps ? 0u : *a.step_ctr)
                                          : cat_argmax(l, TM, d.A);
                if (a.action) a.action[row] = (float)j;
                if (a.act_store) a.act_store[row] = (float)j;
                if (a.mode == 0) {
                    const float nl = cat_neglogp(l, TM, d.A, j);
                    if (a.neglogp) a.neglogp[row] = nl;
                    if (a.nlp_store) a.nlp_store[row] = nl;
                }
            } else if (a.mode == 0) {
                const float* logstd = p + d.off[T_LOGSTD];
                const uint32_t step = a.eps ? 0u : *a.step_ctr;
                float ss = 0.f, sl = 0.f;
                for (int j0 = 0; j0 < d.A; j0 += 4) {
                    float e4[4];
                    if (!a.eps) normal4(a.seed, a.env_id0 + (uint32_t)row, step, (uint32_t)(j0 >> 2), PPO_TAG_ACTION, e4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j = j0 + q;
                        if (j < d.A) {
                            const float ls = __ldg(logstd + j);
                            const float sd = expf(ls);  // logstd_b = mean*0 + logstd; std = exp (GRAPH:5098-5779)
                            const float e = a.eps ? a.eps[(size_t)row * d.A + j] : e4[q];
                            const float mu = MU[j * TM + m];
                            const float act = __fadd_rn(mu, __fmul_rn(sd, e));  // GRAPH:5992-6019
                            const float z = __fdiv_rn(__fsub_rn(act, mu), sd);
                            ss = __fadd_rn(ss, __fmul_rn(z, z));
                            sl = __fadd_rn(sl, ls);
                            Ac[j * (TM + 1) + m] = act;
                        }
                    }
                }
                // 0.5*sum(z^2) + 0.5*log(2pi)*float(A) + sum(logstd)   (GRAPH:6103-6672)
                const float nl = __fadd_rn(__fadd_rn(__fmul_rn(0.5f, ss), __fmul_rn(PPO_HALF_LOG_2PI, (float)d.A)), sl);
                if (a.neglogp) a.neglogp[row] = nl;
                if (a.nlp_store) a.nlp_store[row] = nl;
            } else if (a.mode == 2) {
                for (int j = 0; j < d.A; ++j) Ac[j * (TM + 1) + m] = MU[j * TM + m];  // mean + 0.0 (GRAPH:6046-6076)
            }
            if (a.dones_store) a.dones_store[row] = a.dones_in[row];
        }
        __syncthreads();
        if (HEAD == HEAD_BOX && a.mode != 1) {  // a categorical head stored its index above
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
    const UpdateScalars* sc;                    // cliprange, cliprange_vf of this update (device)
    int vf_mode;                                // VF_CLIP_*
    float ent_coef, vf_coef;
    float* partial;  // [gridDim.x][PS]
    int PS;
    long long* prof;  // optional [2][32] phase timestamps of CTA 0 of each tower (U family, PPO_UMMA_PROF=1)
};

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
    const float lo = 1.f - cr, hi = 1.f + cr;
    float l_pg = 0.f, l_vf = 0.f, l_kl = 0.f, l_cf = 0.f, l_ent = 0.f;
    bool acc = false;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int s0 = a.slot0 + tile * TM;
        const int nv = min(TM, a.slot0 + a.count - s0);
        if (tid < TM) {
            float adv = 0.f, r = 0.f, on = 0.f, ov = 0.f;
            int row = 0;
            if (tid < nv) {
                row = a.gather ? a.gather[s0 + tid] : (s0 + tid);
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
        tile_load_rows<TM>(a.act, HEAD == HEAD_DISCRETE ? 1 : d.A, s_row, nv, Ac);
        __syncthreads();

        // ---------------- pi tower ----------------
        tile_fwd<TM, ACT>(Xs, d.O, p + d.off[T_PI_FC0_W], p + d.off[T_PI_FC0_B], d.H1, H1s);
        __syncthreads();
        tile_fwd<TM, ACT>(H1s, d.H1, p + d.off[T_PI_FC1_W], p + d.off[T_PI_FC1_B], d.H2, H2s);
        __syncthreads();
        tile_fwd<TM, ACT_NONE>(H2s, d.H2, p + d.off[T_PI_W], p + d.off[T_PI_B], d.A, MU);
        __syncthreads();
        if (HEAD == HEAD_DISCRETE && tid < TM) {  // a thread per sample over the A logits; MU becomes dL/dlogits
            const int m = tid;
            float* l = MU + m;
            if (m < nv) {
                const int ai = (int)Ac[m];
                float mx;
                const float z = cat_partition(l, TM, d.A, mx);
                const float nlp = logf(z) - (l[ai * TM] - mx);
                const float H = cat_entropy(l, TM, d.A, mx, z);
                const float adv = s_adv[m], oldn = s_oldn[m];
                const float ratio = expf(oldn - nlp);
                const float pg1 = -adv * ratio;
                const float pg2 = -adv * fmaxf(fminf(ratio, hi), lo);
                const bool take1 = pg1 >= pg2;
                l_pg += take1 ? pg1 : pg2;
                const float dn = nlp - oldn;
                l_kl += dn * dn;
                l_cf += (fabsf(ratio - 1.f) > cr) ? 1.f : 0.f;
                l_ent += H * (a.invB * a.sc->world);
                cat_dlogits(l, TM, d.A, ai, mx, z, H, take1 ? (adv * ratio) * a.invB : 0.f, a.ent_coef * a.invB);
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
                const float nlp = (0.5f * ss + PPO_HALF_LOG_2PI * (float)d.A) + sl;  // GRAPH:9428-9997
                const float adv = s_adv[m], oldn = s_oldn[m];
                const float ratio = expf(oldn - nlp);                                 // GRAPH:10423-10447
                const float pg1 = -adv * ratio;
                const float pg2 = -adv * fmaxf(fminf(ratio, hi), lo);                 // clip_by_value = max(min(x,hi),lo)
                const bool take1 = pg1 >= pg2;                                        // ties -> unclipped branch (GRAPH:12609-12776)
                l_pg += take1 ? pg1 : pg2;
                const float dn = nlp - oldn;
                l_kl += dn * dn;
                l_cf += (fabsf(ratio - 1.f) > cr) ? 1.f : 0.f;
                g_nlp = take1 ? (adv * ratio) * a.invB : 0.f;
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
    constexpr int NL = HEAD == HEAD_DISCRETE ? 5 : 4;
    float v4[NL];
    v4[0] = l_pg; v4[1] = l_vf; v4[2] = l_kl; v4[3] = l_cf;
    if (HEAD == HEAD_DISCRETE) v4[NL - 1] = l_ent;
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
        for (int w = 0; w < NT / 32; ++w)
            for (int q = 0; q < NL; ++q) t[q] += s_red[w * NL + q];
        float* L = my + d.P;
        L[L_PG] = t[0]; L[L_VF] = t[1]; L[L_KL] = t[2]; L[L_CLIP] = t[3];
        float ent = 0.f;
        if (HEAD == HEAD_DISCRETE) {
            ent = t[NL - 1];  // sum of H / B (x world, see UpdateScalars) over this CTA's samples
        } else if (blockIdx.x == 0) {
            // entropy = sum_j(logstd_j + 0.5*log(2*pi*e)) with the pre-update weights (GRAPH:10021-10180)
            const float* logstd = p + d.off[T_LOGSTD];
            for (int j = 0; j < d.A; ++j) ent += __ldg(logstd + j) + PPO_HALF_LOG_2PIE;
        }
        L[L_ENT] = ent;
        L[5] = 0.f; L[6] = 0.f; L[7] = 0.f;
    }
    // loss = pg_loss - entropy*ent_coef + vf_loss*vf_coef: d(-ent_coef*entropy)/dlogstd_j = -ent_coef, added once
    // (a.ent_coef is already divided by the number of ranks whose slabs get summed)
    if (HEAD == HEAD_BOX && blockIdx.x == 0 && tid < d.A) my[d.off[T_LOGSTD] + tid] -= a.ent_coef;  // same thread wrote it in tile_rowsum
}

}  // namespace ppo
