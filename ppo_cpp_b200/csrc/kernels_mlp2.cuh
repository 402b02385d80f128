// "F family": fused MLP kernels with the whole trainable parameter vector staged in shared memory and both
// towers (pi and V) advanced in the same phase.  Requires H1 % 4 == 0, H2 % 4 == 0 and that weights +
// activations of one tile fit in shared memory ([64,64]: 48 KB weights + 147 KB activations).  Everything
// else (e.g. the reference's [4,5] net, [256,256]) goes through the generic T family in kernels_mlp.cuh.
//
// Why: ncu on the T family (profiles/r1_train_v1_*.txt) showed long-scoreboard stalls on weight loads that
// miss L1 (every weight is read once per CTA per layer -> L2 latency chains of depth K/4) and ~20 barrier
// phases per tile.  Here weights are read with LDS (29 cycles), a tile needs 8 phases, and bias gradients
// come out of the dW GEMM through a row of ones appended to every activation matrix.
#pragma once
#include "kernels_mlp.cuh"

namespace ppo {

// thread-subgroup description: local index l in a group of G threads
struct Sub {
    int l, G;
};

// Cs[n][m] = act( sum_k As[k][m] * W[k][n] + b[n] ), W/b in shared memory
template <int TM, int FA>
__device__ __forceinline__ void f_fwd(const float* __restrict__ As, int K, const float* __restrict__ W,
                                      const float* __restrict__ b, int N, float* __restrict__ Cs, Sub s) {
    constexpr int MG = TM / 4;
    const int ngroups = (N + 3) >> 2;
    const bool vec = ((N & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
    for (int tile = s.l; tile < MG * ngroups; tile += s.G) {
        const int mg = tile % MG, ng = tile / MG;
        const int n = ng << 2;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (vec) {
#pragma unroll 8
            for (int k = 0; k < K; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(As + k * TM + mg * 4);
                const float4 w = *reinterpret_cast<const float4*>(W + k * N + n);
                const float av[4] = {a.x, a.y, a.z, a.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(wv[i], av[j], acc[i][j]);
            }
        } else {
#pragma unroll 4
            for (int k = 0; k < K; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(As + k * TM + mg * 4);
                const float av[4] = {a.x, a.y, a.z, a.w};
                float wv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) wv[i] = W[k * N + min(n + i, N - 1)];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(wv[i], av[j], acc[i][j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (n + i < N) {
                const float bb = b[n + i];
                float4 o;
                o.x = acc[i][0] + bb; o.y = acc[i][1] + bb; o.z = acc[i][2] + bb; o.w = acc[i][3] + bb;
                if (FA != ACT_NONE) { o.x = act_fwd<FA>(o.x); o.y = act_fwd<FA>(o.y); o.z = act_fwd<FA>(o.z); o.w = act_fwd<FA>(o.w); }
                *reinterpret_cast<float4*>(Cs + (n + i) * TM + mg * 4) = o;
            }
        }
    }
}

// Ds[k][m] = ( sum_n W[k][n] * Ys[n][m] ) * act'(Hs[k][m]), W in shared memory
template <int TM, int ACT>
__device__ __forceinline__ void f_bwd_dx(const float* __restrict__ Ys, int N, const float* __restrict__ W, int K,
                                         const float* __restrict__ Hs, float* __restrict__ Ds, Sub s) {
    constexpr int MG = TM / 4;
    const int kgroups = (K + 3) >> 2;
    const bool vec = ((N & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
    for (int tile = s.l; tile < MG * kgroups; tile += s.G) {
        const int mg = tile % MG, kg = tile / MG;
        const int k = kg << 2;
        int kr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) kr[i] = min(k + i, K - 1) * N;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (vec) {
#pragma unroll 2
            for (int n = 0; n < N; n += 4) {
                float4 y[4], w[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) y[q] = *reinterpret_cast<const float4*>(Ys + (n + q) * TM + mg * 4);
#pragma unroll
                for (int i = 0; i < 4; ++i) w[i] = *reinterpret_cast<const float4*>(W + kr[i] + n);
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
#pragma unroll 2
            for (int n = 0; n < N; ++n) {
                const float4 y = *reinterpret_cast<const float4*>(Ys + n * TM + mg * 4);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float wv = W[kr[i] + n];
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

// Gw[k][n] (+)= sum_m As[k][m] * Ys[n][m] for k < K; row K of As is all ones, so "k == K" yields the bias
// gradient Gb[n] (+)= sum_m Ys[n][m].  As has K+1 rows.
template <int TM>
__device__ __forceinline__ void f_dw(const float* __restrict__ As, int K, const float* __restrict__ Ys, int N,
                                     float* __restrict__ Gw, float* __restrict__ Gb, bool accumulate, Sub s) {
    constexpr int MG = TM / 4;
    const int K1 = K + 1;
    const int kgroups = (K1 + 3) >> 2, ngroups = (N + 3) >> 2;
    for (int tt = s.l; tt < kgroups * ngroups; tt += s.G) {
        const int kg = tt / ngroups, ng = tt - kg * ngroups;
        const int k = kg << 2, n = ng << 2;
        int kr[4], nr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            kr[i] = min(k + i, K1 - 1) * TM;
            nr[i] = min(n + i, N - 1) * TM;
        }
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 2
        for (int it = 0; it < MG; ++it) {
            const int m4 = ((it + ng + kg) % MG) * 4;  // skewed start: threads of a warp hit different banks
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
                if (k + i < K1 && n + j < N) {
                    float* g = (k + i < K) ? (Gw + (size_t)(k + i) * N + n + j) : (Gb + n + j);
                    *g = accumulate ? (*g + acc[i][j]) : acc[i][j];
                }
    }
}

// smem layout of one tile (floats).  Activation matrices carry one extra row of ones (bias-gradient trick).
struct FLayout {
    int w, xs, ac, mu, vs, h1[2], h2[2], d2[2], d1[2], adv, ret, oldn, oldv, rows, red, sd, total;
    __host__ __device__ void init(const NetDims& d, int TM, bool train) {
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        w = take(d.P + 4);
        xs = take((d.O + 1) * TM);
        ac = take(d.A * (TM + (train ? 0 : 1)));
        mu = take(d.A * TM);
        vs = take(TM);
        for (int t = 0; t < 2; ++t) {
            h1[t] = take((d.H1 + 1) * TM);
            h2[t] = take((d.H2 + 1) * TM);
            if (train) {
                d2[t] = take(d.H2 * TM);
                d1[t] = take(d.H1 * TM);
            } else {
                d2[t] = d1[t] = 0;
            }
        }
        adv = take(TM); ret = take(TM); oldn = take(TM); oldv = take(TM); rows = take(TM);
        red = take(8 * TM);  // per-sample partial sums of the loss stage / block reductions
        sd = take(2 * d.A);  // exp(logstd), logstd
        total = o;
    }
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// stage the trainable parameter vector into shared memory (16-byte async copies; params is 256-byte aligned
// and has at least 3 floats of q-head behind P, so rounding the length up to a multiple of 4 stays in bounds)
template <int NTH>
__device__ __forceinline__ void stage_weights(float* sW, const float* __restrict__ params, int P) {
    const int n4 = (P + 3) >> 2;
    for (int i = threadIdx.x; i < n4; i += NTH) cp_async16(sW + i * 4, params + i * 4);
}

// ------------------------------------------------------------------------------------------------ train
template <int TM, int NTH, int ACT, int HEAD>
__global__ void __launch_bounds__(NTH, 1) train_fused_kernel(const TrainArgs a) {
    extern __shared__ __align__(16) float smem[];
    const NetDims& d = a.d;
    FLayout L;
    L.init(d, TM, true);
    float* sW = smem + L.w;
    float* Xs = smem + L.xs;
    float* Ac = smem + L.ac;
    float* MU = smem + L.mu;
    float* Vs = smem + L.vs;
    float* s_adv = smem + L.adv;
    float* s_ret = smem + L.ret;
    float* s_oldn = smem + L.oldn;
    float* s_oldv = smem + L.oldv;
    int* s_row = reinterpret_cast<int*>(smem + L.rows);
    float* s_red = smem + L.red;
    float* s_sd = smem + L.sd;
    const int tid = threadIdx.x;
    constexpr int HALF = NTH / 2;
    const int tw = tid / HALF;               // tower handled by this thread: 0 = pi, 1 = V
    const Sub half{tid % HALF, HALF};
    const Sub all{tid, NTH};
    float* H1 = smem + L.h1[tw];
    float* H2 = smem + L.h2[tw];
    float* D2 = smem + L.d2[tw];
    float* D1 = smem + L.d1[tw];
    float* my = a.partial + (size_t)blockIdx.x * a.PS;
    const int ntiles = (a.count + TM - 1) / TM;
    const float cr = a.sc->cliprange, vr = vf_clip_range(a.vf_mode, cr, a.sc->cliprange_vf);
    const float lo = 1.f - cr, hi = 1.f + cr;

    stage_weights<NTH>(sW, a.params, d.P);
    // rows of ones behind every activation matrix (bias gradients fall out of the dW GEMM)
    for (int m = tid; m < TM; m += NTH) {
        Xs[d.O * TM + m] = 1.f;
        for (int t = 0; t < 2; ++t) {
            smem[L.h1[t] + d.H1 * TM + m] = 1.f;
            smem[L.h2[t] + d.H2 * TM + m] = 1.f;
        }
    }
    float l_pg = 0.f, l_vf = 0.f, l_kl = 0.f, l_cf = 0.f, l_ent = 0.f;
    bool acc = false;
    bool first = true;

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
        for (int e = tid; e < TM * d.O; e += NTH) {
            const int m = e / d.O, k = e - m * d.O;
            Xs[k * TM + m] = (m < nv) ? __ldg(a.obs + (size_t)s_row[m] * d.O + k) : 0.f;
        }
        const int AW = HEAD == HEAD_DISCRETE ? 1 : d.A;  // stored action width
        for (int e = tid; e < TM * AW; e += NTH) {
            const int m = e / AW, j = e - m * AW;
            Ac[j * TM + m] = (m < nv) ? __ldg(a.act + (size_t)s_row[m] * AW + j) : 0.f;
        }
        if (first) {
            cp_async_wait_all();
            first = false;
        }
        __syncthreads();
        if (HEAD == HEAD_BOX && tid < d.A && tile == (int)blockIdx.x) {
            const float ls = sW[d.off[T_LOGSTD] + tid];
            s_sd[tid] = expf(ls);
            s_sd[d.A + tid] = ls;
        }

        // ---- forward, both towers at once
        f_fwd<TM, ACT>(Xs, d.O, sW + d.off[tw ? T_VF_FC0_W : T_PI_FC0_W], sW + d.off[tw ? T_VF_FC0_B : T_PI_FC0_B], d.H1, H1, half);
        __syncthreads();
        f_fwd<TM, ACT>(H1, d.H1, sW + d.off[tw ? T_VF_FC1_W : T_PI_FC1_W], sW + d.off[tw ? T_VF_FC1_B : T_PI_FC1_B], d.H2, H2, half);
        __syncthreads();
        if (tw == 0) f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_PI_W], sW + d.off[T_PI_B], d.A, MU, half);
        else f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_VF_W], sW + d.off[T_VF_B], 1, Vs, half);
        __syncthreads();

        // ---- loss stage.  Thread (m, jg) handles actions j = jg, jg + JG, ... of sample m.
        constexpr int JG = (NTH / TM) < 8 ? (NTH / TM) : 8;
        const int m = tid % TM, jg = tid / TM;
        if (HEAD == HEAD_DISCRETE) {  // a thread per sample over the A logits; MU becomes dL/dlogits, Vs dL/dv
            if (jg == 0) {
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
                    float dv;
                    l_vf += value_loss_term(a.vf_mode, vr, Vs[m], s_oldv[m], s_ret[m], a.vf_coef, a.invB, dv);
                    Vs[m] = dv;
                } else {
                    for (int j = 0; j < d.A; ++j) l[j * TM] = 0.f;
                    Vs[m] = 0.f;
                }
            }
        } else {
        if (jg < JG) {
            float ss = 0.f;
            for (int j = jg; j < d.A; j += JG) {
                const float z = (Ac[j * TM + m] - MU[j * TM + m]) / s_sd[j];
                ss += z * z;
            }
            s_red[jg * TM + m] = ss;
        }
        __syncthreads();
        float g_nlp = 0.f;
        if (jg < JG) {
            if (m < nv) {
                float ss = 0.f, sl = 0.f;
                for (int q = 0; q < JG; ++q) ss += s_red[q * TM + m];
                for (int j = 0; j < d.A; ++j) sl += s_sd[d.A + j];
                const float nlp = (0.5f * ss + PPO_HALF_LOG_2PI * (float)d.A) + sl;  // GRAPH:9428-9997
                const float adv = s_adv[m], oldn = s_oldn[m];
                const float ratio = expf(oldn - nlp);                                 // GRAPH:10423-10447
                const float pg1 = -adv * ratio;
                const float pg2 = -adv * fmaxf(fminf(ratio, hi), lo);                 // clip_by_value = max(min(x,hi),lo)
                const bool take1 = pg1 >= pg2;                                        // ties -> unclipped branch
                g_nlp = take1 ? (adv * ratio) * a.invB : 0.f;
                if (jg == 0) {
                    l_pg += take1 ? pg1 : pg2;
                    const float dn = nlp - oldn;
                    l_kl += dn * dn;
                    l_cf += (fabsf(ratio - 1.f) > cr) ? 1.f : 0.f;
                    float dv;
                    l_vf += value_loss_term(a.vf_mode, vr, Vs[m], s_oldv[m], s_ret[m], a.vf_coef, a.invB, dv);  // GRAPH:10213-10400
                    Vs[m] = dv;
                }
            } else if (jg == 0) {
                Vs[m] = 0.f;
            }
            for (int j = jg; j < d.A; j += JG) {
                const float sd = s_sd[j];
                const float z = (Ac[j * TM + m] - MU[j * TM + m]) / sd;
                Ac[j * TM + m] = g_nlp * (1.f - z * z);  // d nlp / d logstd_j contribution
                MU[j * TM + m] = g_nlp * (-z / sd);      // dL/dmu
            }
        }
        }
        __syncthreads();

        // ---- backward: heads
        if (tw == 0) {
            f_bwd_dx<TM, ACT>(MU, d.A, sW + d.off[T_PI_W], d.H2, H2, D2, half);
            f_dw<TM>(H2, d.H2, MU, d.A, my + d.off[T_PI_W], my + d.off[T_PI_B], acc, half);
        } else {
            f_bwd_dx<TM, ACT>(Vs, 1, sW + d.off[T_VF_W], d.H2, H2, D2, half);
            f_dw<TM>(H2, d.H2, Vs, 1, my + d.off[T_VF_W], my + d.off[T_VF_B], acc, half);
            // logstd gradient = row sums of Ac: ones-row trick with K = 0 (As = the ones row of Xs)
            if (HEAD == HEAD_BOX) f_dw<TM>(Xs + d.O * TM, 0, Ac, d.A, my + d.off[T_LOGSTD], my + d.off[T_LOGSTD], acc, half);
        }
        __syncthreads();
        // ---- backward: hidden layer 1
        f_dw<TM>(H1, d.H1, D2, d.H2, my + d.off[tw ? T_VF_FC1_W : T_PI_FC1_W], my + d.off[tw ? T_VF_FC1_B : T_PI_FC1_B], acc, half);
        f_bwd_dx<TM, ACT>(D2, d.H2, sW + d.off[tw ? T_VF_FC1_W : T_PI_FC1_W], d.H1, H1, D1, half);
        __syncthreads();
        // ---- backward: hidden layer 0
        f_dw<TM>(Xs, d.O, D1, d.H1, my + d.off[tw ? T_VF_FC0_W : T_PI_FC0_W], my + d.off[tw ? T_VF_FC0_B : T_PI_FC0_B], acc, half);
        __syncthreads();
        acc = true;
    }
    if (first) cp_async_wait_all();

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
        for (int w = 0; w < NTH / 32; ++w)
            for (int q = 0; q < NL; ++q) t[q] += s_red[w * NL + q];
        float* Lp = my + d.P;
        Lp[L_PG] = t[0]; Lp[L_VF] = t[1]; Lp[L_KL] = t[2]; Lp[L_CLIP] = t[3];
        float ent = 0.f;
        if (HEAD == HEAD_DISCRETE) ent = t[NL - 1];  // sum of H / B (x world, see UpdateScalars) over this CTA's samples
        else if (blockIdx.x == 0)
            for (int j = 0; j < d.A; ++j) ent += sW[d.off[T_LOGSTD] + j] + PPO_HALF_LOG_2PIE;  // GRAPH:10021-10180
        Lp[L_ENT] = ent;
        Lp[5] = 0.f; Lp[6] = 0.f; Lp[7] = 0.f;
    }
    __syncthreads();
    // d(-ent_coef*entropy)/dlogstd_j = -ent_coef, once (a.ent_coef is pre-divided by the number of ranks)
    if (HEAD == HEAD_BOX && blockIdx.x == 0 && tid < d.A) my[d.off[T_LOGSTD] + tid] -= a.ent_coef;
}

// ------------------------------------------------------------------------------------------------ policy
template <int TM, int NTH, int ACT, int HEAD>
__global__ void __launch_bounds__(NTH) policy_fused_kernel(const PolicyArgs a) {
    extern __shared__ __align__(16) float smem[];
    const NetDims& d = a.d;
    FLayout L;
    L.init(d, TM, false);
    float* sW = smem + L.w;
    float* Xs = smem + L.xs;
    float* Ac = smem + L.ac;  // [A][TM+1]
    float* MU = smem + L.mu;
    float* Vs = smem + L.vs;
    const int tid = threadIdx.x;
    constexpr int HALF = NTH / 2;
    const int tw = tid / HALF;
    const Sub half{tid % HALF, HALF};
    float* H1 = smem + L.h1[tw];
    float* H2 = smem + L.h2[tw];
    const int ntiles = (a.n + TM - 1) / TM;
    stage_weights<NTH>(sW, a.params, d.P);
    bool first = true;
    const bool do_pi = a.mode != 1, do_v = a.mode != 2;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int r0 = tile * TM, nv = min(TM, a.n - r0);
        for (int e = tid; e < TM * d.O; e += NTH) {
            const int m = e / d.O, k = e - m * d.O;
            const float x = (m < nv) ? a.obs[(size_t)(r0 + m) * d.O + k] : 0.f;
            Xs[k * TM + m] = x;
            if (a.obs_store && m < nv) a.obs_store[(size_t)(r0 + m) * d.O + k] = x;
        }
        if (first) {
            cp_async_wait_all();
            first = false;
        }
        __syncthreads();
        if ((tw == 0 && do_pi) || (tw == 1 && do_v))
            f_fwd<TM, ACT>(Xs, d.O, sW + d.off[tw ? T_VF_FC0_W : T_PI_FC0_W], sW + d.off[tw ? T_VF_FC0_B : T_PI_FC0_B], d.H1, H1, half);
        __syncthreads();
        if ((tw == 0 && do_pi) || (tw == 1 && do_v))
            f_fwd<TM, ACT>(H1, d.H1, sW + d.off[tw ? T_VF_FC1_W : T_PI_FC1_W], sW + d.off[tw ? T_VF_FC1_B : T_PI_FC1_B], d.H2, H2, half);
        __syncthreads();
        if (tw == 0 && do_pi) f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_PI_W], sW + d.off[T_PI_B], d.A, MU, half);
        if (tw == 1 && do_v) f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_VF_W], sW + d.off[T_VF_B], 1, Vs, half);
        __syncthreads();
        if (tid < nv) {
            const int m = tid, row = r0 + m;
            if (do_v) {
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
                const float* logstd = sW + d.off[T_LOGSTD];
                const uint32_t step = a.eps ? 0u : *a.step_ctr;
                float ss = 0.f, sl = 0.f;
                for (int j0 = 0; j0 < d.A; j0 += 4) {
                    float e4[4];
                    if (!a.eps) normal4(a.seed, a.env_id0 + (uint32_t)row, step, (uint32_t)(j0 >> 2), PPO_TAG_ACTION, e4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j = j0 + q;
                        if (j < d.A) {
                            const float ls = logstd[j];
                            const float sd = expf(ls);
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
                const float nl = __fadd_rn(__fadd_rn(__fmul_rn(0.5f, ss), __fmul_rn(PPO_HALF_LOG_2PI, (float)d.A)), sl);
                if (a.neglogp) a.neglogp[row] = nl;
                if (a.nlp_store) a.nlp_store[row] = nl;
            } else if (a.mode == 2) {
                for (int j = 0; j < d.A; ++j) Ac[j * (TM + 1) + m] = MU[j * TM + m];
            }
            if (a.dones_store) a.dones_store[row] = a.dones_in[row];
        }
        __syncthreads();
        if (HEAD == HEAD_BOX && do_pi) {  // a categorical head stored its index above
            for (int e = tid; e < nv * d.A; e += NTH) {
                const int m = e / d.A, j = e - m * d.A;
                const float act = Ac[j * (TM + 1) + m];
                if (a.action) a.action[(size_t)(r0 + m) * d.A + j] = act;
                if (a.act_store) a.act_store[(size_t)(r0 + m) * d.A + j] = act;
            }
        }
        __syncthreads();
    }
    if (first) cp_async_wait_all();
}

}  // namespace ppo
