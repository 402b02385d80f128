// "S family": train kernel for the reference's own tiny networks (the shipped graph is MLP [4,5], 334 trainable
// parameters; SURVEY §3.4) — one THREAD per sample, everything in registers.
//
// Replaces the loss / autodiff sub-graph of one PPO2::_train_step (ppo2/ppo2.hpp:430-470, GRAPH:6889-23699); math and
// TF tie-breaking rules are those of SURVEY §3.5b, identical to the tile kernels.
//
// Why a separate family: a [4,5] layer is a 4x5 matrix — the tile kernels (4x4 register tiles over a 64-sample tile,
// one __syncthreads per layer) leave 250 of 256 threads idle in most phases and reach 1 % of the HBM roofline on the
// C5 buffer (profiles/r1_v4_c5_microbench.jsonl).  Here
//   * the parameter vector sits in shared memory and is read with LDS.128 broadcasts (one load per 4 FMAs),
//   * a thread loads its gathered observation / action rows (2 x 72 B), runs both towers forward, the loss, and the
//     hand-derived backward pass out of registers (all loops unrolled at compile time: dims are template parameters),
//   * the P per-sample gradient contributions are summed over the 32 samples of a warp by a transpose through shared
//     memory, 32 parameters at a time: lane l ends up with the warp's sum of contribution l.  Each lane therefore owns
//     P/32 accumulators (11 for [4,5]) for the whole grid-stride loop,
//   * warps are combined through shared memory in a fixed order and the CTA writes one slab of the usual layout, so the
//     cooperative reduce + clip + Adam kernel is shared with the other families.
#pragma once
#include "kernels_mlp.cuh"

namespace ppo {
namespace small {

constexpr int NTH = 128;

// v[0..31] per lane  ->  returns (in every lane l) the sum over the 32 lanes of their v[l], through a per-warp
// [32][TR_LD] shared-memory tile: 32 conflict-free scalar stores (lane-consecutive addresses), 8 LDS.128 of the lane's
// own row (row stride 36 floats: the 8 lanes of a quarter-warp hit disjoint bank groups), 32 adds in a fixed order.
// (A shuffle butterfly needs 31 SHFL + 62 FSEL + warp-sync bookkeeping per 32 values: 2.5x the instructions.)
constexpr int TR_LD = 36;
__device__ __forceinline__ float transpose_reduce32(const float (&v)[32], float* tile, int lane) {
    __syncwarp();  // previous readers of the tile are done
#pragma unroll
    for (int i = 0; i < 32; ++i) tile[i * TR_LD + lane] = v[i];
    __syncwarp();
    const float4* row = reinterpret_cast<const float4*>(tile + lane * TR_LD);
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 t = row[q];
        s += t.x;
        s += t.y;
        s += t.z;
        s += t.w;
    }
    return s;
}

template <int O, int A, int H1, int H2>
struct Dims {
    // offsets of the 13 trainable tensors in the flat parameter vector (device_common.cuh order)
    static constexpr int PI0W = 0, PI0B = PI0W + O * H1, VF0W = PI0B + H1, VF0B = VF0W + O * H1, PI1W = VF0B + H1,
                         PI1B = PI1W + H1 * H2, VF1W = PI1B + H2, VF1B = VF1W + H1 * H2, VFW = VF1B + H2, VFB = VFW + H2,
                         PIW = VFB + 1, PIB = PIW + H2 * A, LS = PIB + A, P = LS + A;
    static constexpr int GROUPS = (P + 31) / 32;
};

// Per-thread accumulators of a CTA's share of a minibatch
template <int GROUPS>
struct SmallAcc {
    float accg[GROUPS];
    float l_pg, l_vf, l_kl, l_cf;
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int g = 0; g < GROUPS; ++g) accg[g] = 0.f;
        l_pg = l_vf = l_kl = l_cf = 0.f;
    }
};

// One warp tile (32 samples, one per lane): forward, loss, backward; the per-parameter contributions summed over the warp into acc
template <int O, int A, int H1, int H2, int ACT>
__device__ __forceinline__ void small_warp_tile(const TrainArgs& a, const float* __restrict__ sW, int slot, bool valid, const float2* mbstats,
                                                const float (&sd)[A], const float (&isd)[A], float sum_ls,
                                                SmallAcc<Dims<O, A, H1, H2>::GROUPS>& acc, float* tile, int lane) {
    using D = Dims<O, A, H1, H2>;
    float (&accg)[D::GROUPS] = acc.accg;
    float &l_pg = acc.l_pg, &l_vf = acc.l_vf, &l_kl = acc.l_kl, &l_cf = acc.l_cf;
    (void)sd;
    {
        float x[O], act[A];
        float adv = 0.f, R = 0.f, oldn = 0.f, oldv = 0.f;
        {
            const long row = valid ? (long)(a.gather ? __ldg(a.gather + slot) : slot) : 0;
            const float2* xs = reinterpret_cast<const float2*>(a.obs + row * O);
            const float2* as = reinterpret_cast<const float2*>(a.act + row * A);
#pragma unroll
            for (int k = 0; k < O / 2; ++k) {
                const float2 v = valid ? __ldg(xs + k) : make_float2(0.f, 0.f);
                x[2 * k] = v.x;
                x[2 * k + 1] = v.y;
            }
#pragma unroll
            for (int j = 0; j < A / 2; ++j) {
                const float2 v = valid ? __ldg(as + j) : make_float2(0.f, 0.f);
                act[2 * j] = v.x;
                act[2 * j + 1] = v.y;
            }
            if (valid) {
                R = __ldg(a.ret + row);
                oldv = __ldg(a.val + row);
                oldn = __ldg(a.nlp + row);
                if (a.adv_direct) {
                    adv = __ldg(a.adv_direct + slot);
                } else {  // advs = (returns - values - mean) / (sqrt(var) + 1e-8)  (ppo2.hpp:401-406)
                    const float2 st = __ldg(mbstats);
                    adv = __fdiv_rn(__fsub_rn(__fsub_rn(R, oldv), st.x), st.y);
                }
            }
        }
        // ---- forward, both towers (GRAPH:6889-9187)
        float h1[H1], g1[H1], h2[H2], g2[H2], mu[A];
#pragma unroll
        for (int n = 0; n < H1; ++n) {
            float sp = 0.f, sv = 0.f;
#pragma unroll
            for (int k = 0; k < O; ++k) {
                sp = fmaf(x[k], sW[D::PI0W + k * H1 + n], sp);
                sv = fmaf(x[k], sW[D::VF0W + k * H1 + n], sv);
            }
            h1[n] = act_fwd<ACT>(sp + sW[D::PI0B + n]);
            g1[n] = act_fwd<ACT>(sv + sW[D::VF0B + n]);
        }
#pragma unroll
        for (int n = 0; n < H2; ++n) {
            float sp = 0.f, sv = 0.f;
#pragma unroll
            for (int k = 0; k < H1; ++k) {
                sp = fmaf(h1[k], sW[D::PI1W + k * H2 + n], sp);
                sv = fmaf(g1[k], sW[D::VF1W + k * H2 + n], sv);
            }
            h2[n] = act_fwd<ACT>(sp + sW[D::PI1B + n]);
            g2[n] = act_fwd<ACT>(sv + sW[D::VF1B + n]);
        }
        float v = 0.f;
#pragma unroll
        for (int k = 0; k < H2; ++k) v = fmaf(g2[k], sW[D::VFW + k], v);
        v += sW[D::VFB];
#pragma unroll
        for (int j = 0; j < A; ++j) {
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < H2; ++k) s = fmaf(h2[k], sW[D::PIW + k * A + j], s);
            mu[j] = s + sW[D::PIB + j];
        }
        // ---- loss stage (GRAPH:9428-11446) and dL/dmu, dL/dlogstd contributions, dL/dv
        float dmu[A], dls[A], dv = 0.f;
        {
            float z[A], ss = 0.f;
#pragma unroll
            for (int j = 0; j < A; ++j) {
                z[j] = (act[j] - mu[j]) * isd[j];
                ss += z[j] * z[j];
            }
            float g_nlp = 0.f;
            if (valid) {
                // the clip ranges are loaded where they are used: kept live across the loop they cost the epoch kernel spills
                const float cr = a.sc->cliprange;
                const PgTerm t = pg_term(adv, oldn, gauss_neglogp(ss, sum_ls, A), cr, a.invB);
                g_nlp = t.g_nlp;
                l_pg += t.pg;
                l_kl += t.kl;
                l_cf += t.cf;
                const float vr = vf_clip_range(a.vf_mode, cr, a.sc->cliprange_vf);
                l_vf += value_loss_term(a.vf_mode, vr, v, oldv, R, a.vf_coef, a.invB, dv);  // GRAPH:10213-10400
            }
#pragma unroll
            for (int j = 0; j < A; ++j) {
                dmu[j] = g_nlp * (-z[j] * isd[j]);
                dls[j] = g_nlp * (1.f - z[j] * z[j]);
            }
        }
        // ---- backward through the towers (TanhGrad(y, dy) = dy * (1 - y^2), ReluGrad = dy * (y > 0))
        float dp2[H2], dg2[H2], dp1[H1], dg1[H1];
#pragma unroll
        for (int k = 0; k < H2; ++k) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < A; ++j) s = fmaf(dmu[j], sW[D::PIW + k * A + j], s);
            dp2[k] = s * act_dfac<ACT>(h2[k]);
            dg2[k] = dv * sW[D::VFW + k] * act_dfac<ACT>(g2[k]);
        }
#pragma unroll
        for (int k = 0; k < H1; ++k) {
            float sp = 0.f, sv = 0.f;
#pragma unroll
            for (int n = 0; n < H2; ++n) {
                sp = fmaf(dp2[n], sW[D::PI1W + k * H2 + n], sp);
                sv = fmaf(dg2[n], sW[D::VF1W + k * H2 + n], sv);
            }
            dp1[k] = sp * act_dfac<ACT>(h1[k]);
            dg1[k] = sv * act_dfac<ACT>(g1[k]);
        }
        // ---- per-sample gradient contributions, 32 parameters at a time, summed over the warp's 32 samples
#pragma unroll
        for (int g = 0; g < D::GROUPS; ++g) {
            float c[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int idx = 32 * g + i;  // compile-time constant after unrolling
                float val = 0.f;
                if (idx < D::PI0B) val = x[(idx - D::PI0W) / H1] * dp1[(idx - D::PI0W) % H1];
                else if (idx < D::VF0W) val = dp1[idx - D::PI0B];
                else if (idx < D::VF0B) val = x[(idx - D::VF0W) / H1] * dg1[(idx - D::VF0W) % H1];
                else if (idx < D::PI1W) val = dg1[idx - D::VF0B];
                else if (idx < D::PI1B) val = h1[(idx - D::PI1W) / H2] * dp2[(idx - D::PI1W) % H2];
                else if (idx < D::VF1W) val = dp2[idx - D::PI1B];
                else if (idx < D::VF1B) val = g1[(idx - D::VF1W) / H2] * dg2[(idx - D::VF1W) % H2];
                else if (idx < D::VFW) val = dg2[idx - D::VF1B];
                else if (idx < D::VFB) val = g2[idx - D::VFW] * dv;
                else if (idx < D::PIW) val = dv;
                else if (idx < D::PIB) val = h2[(idx - D::PIW) / A] * dmu[(idx - D::PIW) % A];
                else if (idx < D::LS) val = dmu[idx - D::PIB];
                else if (idx < D::P) val = dls[idx - D::LS];
                c[i] = val;
            }
            accg[g] += transpose_reduce32(c, tile, lane);
        }
    }
}

template <int O, int A, int H1, int H2, int ACT>
__global__ void __launch_bounds__(NTH) train_small_kernel(const TrainArgs a) {
    using D = Dims<O, A, H1, H2>;
    static_assert(O % 2 == 0 && A % 2 == 0, "rows are read as float2");
    __shared__ __align__(16) float sW[(D::P + 3 + 4) & ~3];
    __shared__ float s_part[NTH / 32][D::GROUPS * 32 + 4];
    __shared__ __align__(16) float s_tile[NTH / 32][32 * TR_LD];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < D::P; i += NTH) sW[i] = __ldg(a.params + i);
    __syncthreads();

    float sd[A], isd[A];
    float sum_ls = 0.f;
#pragma unroll
    for (int j = 0; j < A; ++j) {
        const float ls = sW[D::LS + j];
        sd[j] = expf(ls);
        isd[j] = 1.f / sd[j];
        sum_ls += ls;
    }
    SmallAcc<D::GROUPS> acc;
    acc.clear();

    const int nwarp_tiles = (a.count + 31) / 32;
    for (int wt = blockIdx.x * (NTH / 32) + warp; wt < nwarp_tiles; wt += gridDim.x * (NTH / 32)) {
        const int slot = a.slot0 + wt * 32 + lane;
        const bool valid = wt * 32 + lane < a.count;
        small_warp_tile<O, A, H1, H2, ACT>(a, sW, slot, valid, a.mbstats, sd, isd, sum_ls, acc, s_tile[warp], lane);
    }
    float (&accg)[D::GROUPS] = acc.accg;
    const float l_pg = acc.l_pg, l_vf = acc.l_vf, l_kl = acc.l_kl, l_cf = acc.l_cf;

    // ---- CTA combine (fixed order over the warps) -> slab
    float* my = a.partial + (size_t)blockIdx.x * a.PS;
#pragma unroll
    for (int g = 0; g < D::GROUPS; ++g) s_part[warp][32 * g + lane] = accg[g];
    float v4[4] = {l_pg, l_vf, l_kl, l_cf};
#pragma unroll
    for (int q = 0; q < 4; ++q) v4[q] = warp_sum(v4[q]);
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) s_part[warp][D::GROUPS * 32 + q] = v4[q];
    }
    __syncthreads();
    for (int i = tid; i < D::P; i += NTH) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < NTH / 32; ++w) s += s_part[w][i];
        // d(-ent_coef*entropy)/dlogstd_j = -ent_coef, once (a.ent_coef is pre-divided by the number of ranks)
        if (blockIdx.x == 0 && i >= D::LS) s -= a.ent_coef;
        my[i] = s;
    }
    if (tid == 0) {
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        for (int w = 0; w < NTH / 32; ++w)
            for (int q = 0; q < 4; ++q) t[q] += s_part[w][D::GROUPS * 32 + q];
        float* Lp = my + D::P;
        Lp[L_PG] = t[0]; Lp[L_VF] = t[1]; Lp[L_KL] = t[2]; Lp[L_CLIP] = t[3];
        float ent = 0.f;
        if (blockIdx.x == 0) ent = box_entropy([&](int j) { return sW[D::LS + j]; }, A);
        Lp[L_ENT] = ent;
        Lp[5] = 0.f; Lp[6] = 0.f; Lp[7] = 0.f;
    }
}

// Policy step of the S family (MlpPolicy::step / value / deterministic action, policies.hpp:33-77): one THREAD per env, parameters in
// shared memory (LDS.128 broadcasts), the env's observation row in registers, the same accumulation order as the tile kernels
// (k ascending from 0, bias added last, act_fwd) so that actions / values / neglogp are bit-identical to every other forward path.
// Observation rows come in and action rows go out through a shared-memory tile, so global accesses are contiguous per warp.
// (policy_tile_kernel, which served this net before, spends 12 M warp instructions on 65 536 envs: 4x4 register tiles over layers
// that are 4 and 5 wide leave most threads of a phase idle — 37 us per step against 7; profiles/r2_small_kernels_ncu.txt.)
template <int O, int A, int H1, int H2, int ACT>
__global__ void __launch_bounds__(NTH) policy_small_kernel(const PolicyArgs a) {
    using D = Dims<O, A, H1, H2>;
    constexpr int XL = O + 1 + ((O + 1) % 2 == 0 ? 1 : 0);  // odd row strides: a lane reading its own row hits its own bank
    constexpr int AL = A + 1 + ((A + 1) % 2 == 0 ? 1 : 0);
    __shared__ __align__(16) float sW[(D::P + 3 + 4) & ~3];
    __shared__ float sX[NTH * XL];
    __shared__ float sA[NTH * AL];
    const int tid = threadIdx.x;
    for (int i = tid; i < D::P; i += NTH) sW[i] = __ldg(a.params + i);
    const int ntiles = (a.n + NTH - 1) / NTH;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int r0 = tile * NTH, nv = min(NTH, a.n - r0);
        __syncthreads();  // parameters staged (first tile) / previous tile's action rows written out
        {
            const float* src = a.obs + (size_t)r0 * O;
            float* dst = a.obs_store ? a.obs_store + (size_t)r0 * O : nullptr;
            for (int e = tid; e < nv * O; e += NTH) {
                const float x = src[e];
                sX[(e / O) * XL + (e % O)] = x;
                if (dst) dst[e] = x;
            }
        }
        __syncthreads();
        if (tid < nv) {
            const int row = r0 + tid;
            float x[O];
#pragma unroll
            for (int k = 0; k < O; ++k) x[k] = sX[tid * XL + k];
            float mu[A];
            if (a.mode != 1) {
                float h1[H1], h2[H2];
#pragma unroll
                for (int n = 0; n < H1; ++n) {
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < O; ++k) s = fmaf(sW[D::PI0W + k * H1 + n], x[k], s);
                    h1[n] = act_fwd<ACT>(s + sW[D::PI0B + n]);
                }
#pragma unroll
                for (int n = 0; n < H2; ++n) {
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < H1; ++k) s = fmaf(sW[D::PI1W + k * H2 + n], h1[k], s);
                    h2[n] = act_fwd<ACT>(s + sW[D::PI1B + n]);
                }
#pragma unroll
                for (int j = 0; j < A; ++j) {
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < H2; ++k) s = fmaf(sW[D::PIW + k * A + j], h2[k], s);
                    mu[j] = s + sW[D::PIB + j];
                }
            }
            if (a.mode != 2) {
                float g1[H1], g2[H2];
#pragma unroll
                for (int n = 0; n < H1; ++n) {
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < O; ++k) s = fmaf(sW[D::VF0W + k * H1 + n], x[k], s);
                    g1[n] = act_fwd<ACT>(s + sW[D::VF0B + n]);
                }
#pragma unroll
                for (int n = 0; n < H2; ++n) {
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < H1; ++k) s = fmaf(sW[D::VF1W + k * H2 + n], g1[k], s);
                    g2[n] = act_fwd<ACT>(s + sW[D::VF1B + n]);
                }
                float v = 0.f;
#pragma unroll
                for (int k = 0; k < H2; ++k) v = fmaf(sW[D::VFW + k], g2[k], v);
                v += sW[D::VFB];
                if (a.value) a.value[row] = v;
                if (a.val_store) a.val_store[row] = v;
            }
            if (a.mode == 0) {
                gauss_policy_row(a, row, A, [&](int j) { return sW[D::LS + j]; }, [&](int j) { return mu[j]; },
                                 [&](int j, float act) { sA[tid * AL + j] = act; });
            } else if (a.mode == 2) {
#pragma unroll
                for (int j = 0; j < A; ++j) sA[tid * AL + j] = mu[j];  // mean + 0.0 (GRAPH:6046-6076)
            }
            if (a.dones_store) a.dones_store[row] = a.dones_in[row];
        }
        __syncthreads();
        if (a.mode != 1) {
            float* o1 = a.action ? a.action + (size_t)r0 * A : nullptr;
            float* o2 = a.act_store ? a.act_store + (size_t)r0 * A : nullptr;
            for (int e = tid; e < nv * A; e += NTH) {
                const float act = sA[(e / A) * AL + (e % A)];
                if (o1) o1[e] = act;
                if (o2) o2[e] = act;
            }
        }
    }
}

// Epoch kernel of the S family for minibatches that ONE CTA handles (the reference's own C1 shape: 2048 transitions in 32
// minibatches of 64): all minibatches of an epoch in one launch of one CTA — parameters and Adam moments live in shared memory,
// per minibatch: warp tiles -> fixed-order combine of the warps -> sum of squares -> clip -> TF ApplyAdam in place -> next
// minibatch.  No grid barrier, no slab, no second kernel: a launch pair per minibatch (train_small_kernel + cooperative
// reduce / Adam) cost 12 us per step, 3.9 of C1's 9.4 ms per update.  Single GPU only (there is no exchange in here).
struct SmallEpochArgs {
    int M, B;                // minibatches of this launch, slots per minibatch
    const float2* mbstats;   // [M]
    float* loss_rows;        // [M][5]
    AdamArgs adam;           // canonical params / m / v, lr, betas, eps, clip_norm, beta powers in / out, invB, gnorm_out
};
template <int O, int A, int H1, int H2, int ACT>
__global__ void __launch_bounds__(NTH) train_small_epoch_kernel(const TrainArgs a, const SmallEpochArgs ep) {
    using D = Dims<O, A, H1, H2>;
    constexpr int PP = (D::P + 3 + 4) & ~3;
    __shared__ __align__(16) float sW[PP];
    __shared__ float sM[PP], sV[PP];
    __shared__ float s_part[NTH / 32][D::GROUPS * 32 + 4];
    __shared__ __align__(16) float s_tile[NTH / 32][32 * TR_LD];
    __shared__ double s_q[NTH / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const AdamArgs& ad = ep.adam;
    for (int i = tid; i < D::P; i += NTH) {
        sW[i] = __ldcg(ad.params + i);
        sM[i] = __ldcg(ad.m + i);
        sV[i] = __ldcg(ad.v + i);
    }
    float b1p = ad.bpow_in[0], b2p = ad.bpow_in[1];
    const int nwarp_tiles = (a.count + 31) / 32;
    __syncthreads();
    for (int mb = 0; mb < ep.M; ++mb) {
        float sd[A], isd[A];
        float sum_ls = 0.f;
#pragma unroll
        for (int j = 0; j < A; ++j) {
            const float ls = sW[D::LS + j];
            sd[j] = expf(ls);
            isd[j] = 1.f / sd[j];
            sum_ls += ls;
        }
        SmallAcc<D::GROUPS> acc;
        acc.clear();
        for (int wt = warp; wt < nwarp_tiles; wt += NTH / 32) {
            const int slot = mb * ep.B + a.slot0 + wt * 32 + lane;
            const bool valid = wt * 32 + lane < a.count;
            small_warp_tile<O, A, H1, H2, ACT>(a, sW, slot, valid, ep.mbstats + mb, sd, isd, sum_ls, acc, s_tile[warp], lane);
        }
        // ---- combine the warps in a fixed order (as train_small_kernel), gradient of parameter i in thread i % NTH
#pragma unroll
        for (int g = 0; g < D::GROUPS; ++g) s_part[warp][32 * g + lane] = acc.accg[g];
        float v4[4] = {acc.l_pg, acc.l_vf, acc.l_kl, acc.l_cf};
#pragma unroll
        for (int q = 0; q < 4; ++q) v4[q] = warp_sum(v4[q]);
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) s_part[warp][D::GROUPS * 32 + q] = v4[q];
        }
        __syncthreads();
        constexpr int PT = (D::P + NTH - 1) / NTH;
        float g[PT];
        double q = 0.0;
#pragma unroll
        for (int u = 0; u < PT; ++u) {
            const int i = tid + u * NTH;
            float sum = 0.f;
            if (i < D::P) {
#pragma unroll
                for (int w = 0; w < NTH / 32; ++w) sum += s_part[w][i];
                if (i >= D::LS) sum -= a.ent_coef;  // d(-ent_coef*entropy)/dlogstd_j = -ent_coef
                q += (double)sum * (double)sum;
            }
            g[u] = sum;
        }
        q = warp_sum(q);
        if (lane == 0) s_q[warp] = q;
        float lsum[4] = {0.f, 0.f, 0.f, 0.f};
        if (tid == 0) {
            for (int w = 0; w < NTH / 32; ++w)
                for (int k = 0; k < 4; ++k) lsum[k] += s_part[w][D::GROUPS * 32 + k];
        }
        __syncthreads();  // s_q complete; s_part and sW have been read
        double ss = 0.0;
#pragma unroll
        for (int w = 0; w < NTH / 32; ++w) ss += s_q[w];
        float gnorm;
        const float scale = clip_scale(ss, ad.clip_norm, gnorm);
        if (tid == 0) {
            const float L[5] = {lsum[0], lsum[1], box_entropy([&](int j) { return sW[D::LS + j]; }, A), lsum[2], lsum[3]};  // entropy: the parameters before this step
            loss_row(ep.loss_rows + (size_t)mb * 5, L, ad.invB, ad.inv_world);
            *ad.gnorm_out = gnorm;
        }
        __syncthreads();  // thread 0 has read logstd before it moves
        // ---- TF ApplyAdam, in place in shared memory
        const float alpha = adam_alpha(ad.sc->lr, b1p, b2p);
#pragma unroll
        for (int u = 0; u < PT; ++u) {
            const int i = tid + u * NTH;
            if (i < D::P) {
                float m = sM[i], v = sV[i];
                adam_moments(__fmul_rn(g[u], scale), m, v, ad.beta1, ad.beta2);
                sM[i] = m;
                sV[i] = v;
                sW[i] = adam_param(sW[i], m, v, alpha, ad.eps);
            }
        }
        b1p = __fmul_rn(b1p, ad.beta1);
        b2p = __fmul_rn(b2p, ad.beta2);
        __syncthreads();  // the new parameters are in place
    }
    for (int i = tid; i < D::P; i += NTH) {
        ad.params[i] = sW[i];
        ad.m[i] = sM[i];
        ad.v[i] = sV[i];
    }
    if (tid == 0) {
        ad.bpow_out[0] = b1p;
        ad.bpow_out[1] = b2p;
    }
}

}  // namespace small
}  // namespace ppo
