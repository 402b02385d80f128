// "R family": the whole synthetic-env rollout (Runner::run + set_returns, ppo2/runner.hpp:56-191) as ONE persistent
// cooperative kernel.
//
// The per-step chain of the reference — MlpPolicy::step (policies.hpp:33-46), env.step, EnvNormalize::step
// (env_normalize.hpp:64-92) — is a sequence of tiny dependent operations; launched as separate kernels it is pure
// launch latency (4 launches x n_steps, profiles/r1_v3_launches_summary.txt: 2.3 ms of an 11.3 ms update at C3).
// Here a CTA owns TM envs (x tiles-per-CTA) for the whole rollout:
//   * the parameter vector is staged into shared memory ONCE per rollout (cp.async, 16 B), activations live in shared
//     memory feature-major, env state / running returns / normalised observations stay in shared memory across steps;
//   * the only cross-CTA dependency of a step is the VecNormalize batch moment (RunningStatistics::update,
//     running_statistics.hpp:26-35): per-CTA fp64 partial sums -> one grid barrier -> every CTA sums the partials in
//     the same fixed order and performs the Chan merge redundantly (bit-identical in every CTA, no second barrier);
//   * bootstrap value and the GAE reverse scan (runner.hpp:159-191) run in the same kernel: a CTA only needs the
//     rewards / values / dones of its own envs.
// Arithmetic is the same as the step-by-step kernels (policy_*_kernel, synth_env_step_kernel, norm_*_kernel,
// gae_kernel): same Philox counters, same fp32 operation order, fp64 moment sums around the same pivot.
#pragma once
#include <cooperative_groups.h>

#include "kernels_misc.cuh"
#include "kernels_mlp2.cuh"

namespace ppo {

struct RolloutArgs {
    NetDims d;
    const float* params;
    int n, T, tpc;  // envs of this rank, steps, tiles per CTA
    uint64_t seed;
    uint32_t env_id0;
    uint32_t* step_ctr;
    SynthEnv env;
    NormStats st;
    float* ret;  // [n] discounted return accumulator of EnvNormalize
    float norm_gamma, clip_obs, clip_rew, eps;
    int norm_obs, norm_reward, upd_obs, upd_ret;
    double* partial;  // [2][gridDim.x][2*(D+1)]
    float *cur_obs, *cur_dones, *last_values;
    // time-major rollout slabs of this rank, row t = 0; one step further = n rows
    float *obs_store, *act_store, *val_store, *nlp_store, *dones_store, *rew_store, *urew_store, *ret_store;
    float gamma, lam;
    unsigned *bar_ctr, *bar_gen;  // grid barrier (sync_prims.cuh), device-resident generation
    int n_global;                 // envs over all ranks (rows of one VecNormalize batch)
    PeerMailbox mbox;             // multi-GPU: per-step exchange of the batch moments over NVLink P2P stores
    unsigned* mbox_seq;
    // multi-GPU: the five train inputs (obs, actions, values, neglogp, returns) are stored into EVERY rank's buffers
    // (byte offsets inside the IPC-mapped arena mbox.base[r]; rows of this rank start at row_off) — the rollout kernel
    // performs the allgather of the rollout as it goes.  world == 1: the *_store pointers below are used.
    size_t off_obs, off_act, off_val, off_nlp, off_ret;
    size_t row_off;
    unsigned* done_seq;  // sequence number of the end-of-rollout cross-rank barrier
    // host-env mode (h_actions != NULL; Runner::run against a host env, runner.hpp:116-129): instead of the synthetic env the
    // CTA writes its actions into mapped pinned host memory, raises its flag, and polls the host's flag for the env's answer
    // (raw observation, reward, done in mapped pinned memory).  One kernel for the whole rollout: no launch, no stream
    // synchronisation and no cudaMemcpy per env step — per step it costs one PCIe write, one host poll, one PCIe read.
    float* h_actions;             // [n][A]   device -> host (step t at h_actions + t * h_act_stride)
    size_t h_act_stride;          // 0: one buffer reused every step; n * A: the caller's [n_steps][n][A] array, written in place
    const float *h_obs, *h_rew, *h_done;  // [n][O], [n], [n]   host -> device
    unsigned* h_act_flag;         // [gridDim.x]: t + 1 once this CTA's actions of step t are in h_actions
    const unsigned* h_obs_flag;   // t + 1 once the env's answer to step t is in place; PPO_HOST_ENV_ABORT = stop
    unsigned* host_err;           // set when the host never answered (bounded wait)
    // Observations through the copy engine WITHOUT a flag copy behind them (h_obs is a device staging buffer): the kernel keeps the
    // first word of every 32-byte sector of the buffer at a sentinel bit pattern (a NaN with a payload no env produces) between steps
    // and waits until the sectors of ITS rows carry something else — a DMA write of a sector is atomic, so whatever order the copy
    // engine works in, a CTA goes on exactly when its slice has landed (and does not wait for the rest of the copy).  h_obs_flag then
    // only carries the abort.
    int h_sentinel;
    // A single env (<= 30 observation dims): both directions as LL words in mapped memory — actions [A] and the env's answer
    // [obs D | reward | done], each an 8-byte (value, t + 1) word.  No fence and no flag on either side, and the kernel's poll of the
    // answer IS the read of the answer: one PCIe round trip instead of flag poll + payload read.  sequence 0xffffffff = abort.
    uint2* h_act_ll;
    const uint2* h_ans_ll;
    long long* prof;  // optional [32] phase timestamps of CTA 0 during env step 1 (PPO_ROLLOUT_PROF=1)
};

#define R_PROF()                                                                              \
    do {                                                                                      \
        if (a.prof && blockIdx.x == 0 && tid == 0 && t == 1 && prof_i < 32) a.prof[prof_i++] = clock64(); \
    } while (0)

constexpr int R_TM = 32, R_NTH = 256;
constexpr int R_SOLO_CHUNK = 32;  // env steps whose noise is drawn ahead in the single-env path
// shared memory of the single-env path behind RLayout: [2 buffers][2 kinds][R_SOLO_CHUNK][4 * ceil(D / 4)] floats
__host__ __device__ inline size_t rollout_solo_noise_bytes(int D) { return (size_t)2 * 2 * R_SOLO_CHUNK * 4 * ((D + 3) / 4) * sizeof(float) + 16; }
constexpr unsigned PPO_HOST_ENV_ABORT = 0xffffffffu;
constexpr unsigned PPO_OBS_SENTINEL = 0xffc0ffeeu;  // quiet NaN, payload 0x40ffee

// rank r's copy of THIS rank's slab of a train-input buffer (row t = 0), or the local slab on a single GPU
__device__ __forceinline__ float* rslab(const RolloutArgs& a, int r, size_t off, int width, float* local) {
    return a.mbox.world > 1 ? reinterpret_cast<float*>(a.mbox.base[r] + off) + a.row_off * width : local;
}

struct RLayout {
    FLayout f;
    int obs, state, raw, ret, dn, tenv, res, rew, done, lastv, z2, mean, var, inv, misc, csum, total_bytes;
    __host__ __device__ void init(const NetDims& d, int tpc) {
        f.init(d, R_TM, false);
        int o = f.total;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        obs = take(tpc * d.O * R_TM);
        state = take(tpc * d.O * R_TM);
        raw = take(tpc * d.O * R_TM);
        ret = take(tpc * R_TM); dn = take(tpc * R_TM); tenv = take(tpc * R_TM); res = take(tpc * R_TM);
        rew = take(tpc * R_TM); done = take(tpc * R_TM); lastv = take(tpc * R_TM);
        z2 = take(d.A * R_TM);
        mean = take(d.O + 1); var = take(d.O + 1); inv = take(d.O + 1); misc = take(8);
        o = (o + 1) & ~1;  // 8-byte alignment for the doubles
        csum = o;
        o += 2 * (2 * (d.O + 1) + 2);  // doubles: column sums, obs_count, ret_count
        total_bytes = o * 4;
    }
};

// Forward pass of ONE env by one warp with the layer widths known at compile time (the reference's [4,5] net and the [64,64] default):
// lane l owns output units l, l + 32, ... of [pi tower | V tower]; fully unrolled, so the loads of a chain are issued ahead of its fmaf
// sequence (k ascending, as f_fwd).  With run-time widths the same loops took ~70 cycles per k-step.
template <int O, int H1, int H2, int A, int TM, int ACT>
__device__ __forceinline__ void solo_forward(const float* __restrict__ sW, const NetDims& d, const float* __restrict__ OBS, float* H1p, float* H1v,
                                             float* H2p, float* H2v, float* MU, float* Vs, int lane) {
#pragma unroll
    for (int i = 0; i < (2 * H1 + 31) / 32; ++i) {
        const int o = lane + 32 * i;
        if (o < 2 * H1) {
            const bool vt = o >= H1;
            const int n = vt ? o - H1 : o;
            const float* w = sW + d.off[vt ? T_VF_FC0_W : T_PI_FC0_W] + n;
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < O; ++k) acc = fmaf(w[k * H1], OBS[k * TM], acc);
            (vt ? H1v : H1p)[n * TM] = act_fwd<ACT>(acc + sW[d.off[vt ? T_VF_FC0_B : T_PI_FC0_B] + n]);
        }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < (2 * H2 + 31) / 32; ++i) {
        const int o = lane + 32 * i;
        if (o < 2 * H2) {
            const bool vt = o >= H2;
            const int n = vt ? o - H2 : o;
            const float* w = sW + d.off[vt ? T_VF_FC1_W : T_PI_FC1_W] + n;
            const float* hin = vt ? H1v : H1p;
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < H1; ++k) acc = fmaf(w[k * H2], hin[k * TM], acc);
            (vt ? H2v : H2p)[n * TM] = act_fwd<ACT>(acc + sW[d.off[vt ? T_VF_FC1_B : T_PI_FC1_B] + n]);
        }
    }
    __syncwarp();
    static_assert(A + 1 <= 32, "one lane per head output");
    if (lane < A + 1) {
        const bool vh = lane == A;
        const int N = vh ? 1 : A, n = vh ? 0 : lane;
        const float* w = sW + d.off[vh ? T_VF_W : T_PI_W] + n;
        const float* hin = vh ? H2v : H2p;
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < H2; ++k) acc = fmaf(w[k * N], hin[k * TM], acc);
        if (vh) Vs[0] = acc + sW[d.off[T_VF_B]];
        else MU[n * TM] = acc + sW[d.off[T_PI_B] + n];
    }
    __syncwarp();
}

template <int ACT>
__global__ void __launch_bounds__(R_NTH) rollout_persistent_kernel(const RolloutArgs a) {
    extern __shared__ __align__(16) float smem[];
    const NetDims& d = a.d;
    constexpr int TM = R_TM, NTH = R_NTH;
    const int O = d.O, A = d.A, D = d.O;
    RLayout L;
    L.init(d, a.tpc);
    float* sW = smem + L.f.w;
    float* Ac = smem + L.f.ac;  // [A][TM+1]
    float* MU = smem + L.f.mu;
    float* Vs = smem + L.f.vs;
    float* OBS = smem + L.obs;      // [tpc][O][TM] normalised observation, feature-major (the policy's input)
    float* S = smem + L.state;      // [tpc][TM][D] env state
    float* RAW = smem + L.raw;      // [tpc][TM][D] raw observation of this step
    float* RET = smem + L.ret;
    float* DN = smem + L.dn;
    uint32_t* TENV = reinterpret_cast<uint32_t*>(smem + L.tenv);
    uint32_t* RES = reinterpret_cast<uint32_t*>(smem + L.res);
    float* REW = smem + L.rew;
    float* DONE = smem + L.done;
    float* LASTV = smem + L.lastv;
    float* Z2 = smem + L.z2;        // [A][TM]
    float* s_mean = smem + L.mean;  // [D] obs mean, [D] = ret mean
    float* s_var = smem + L.var;
    float* s_inv = smem + L.inv;
    double* csum = reinterpret_cast<double*>(smem + L.csum);  // [2*(D+1)] then obs_count, ret_count
    double* s_cnt = csum + 2 * (D + 1);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int HALF = NTH / 2;
    const int tw = tid / HALF;
    const Sub half{tid % HALF, HALF};
    float* H1 = smem + L.f.h1[tw];
    float* H2 = smem + L.f.h2[tw];
    const int ntiles = (a.n + TM - 1) / TM;
    const int tile0 = blockIdx.x * a.tpc;
    const int my_tiles = max(0, min(a.tpc, ntiles - tile0));
    const int nblk = (D + 3) >> 2;  // Philox blocks of 4 dims
    const uint32_t step0 = *a.step_ctr;
    const bool merge = a.upd_obs || a.upd_ret;
    GridBarrier bar{a.bar_ctr, gridDim.x, *a.bar_gen};
    const int world = a.mbox.world;
    const bool host_env = a.h_actions != nullptr;
    __shared__ int s_abort;
    if (tid == 0) s_abort = 0;
    const unsigned seq0 = world > 1 ? *a.mbox_seq : 0u;
    const unsigned dseq0 = world > 1 ? *a.done_seq : 0u;

    // ---- one-time: weights, running statistics, per-env state
    stage_weights<NTH>(sW, a.params, d.P);
    if (tid < D) {
        s_mean[tid] = a.st.obs_mean[tid];
        s_var[tid] = a.st.obs_var[tid];
    } else if (tid == D) {
        s_mean[D] = *a.st.ret_mean;
        s_var[D] = *a.st.ret_var;
        s_cnt[0] = *a.st.obs_count;
        s_cnt[1] = *a.st.ret_count;
    }
    for (int tl = 0; tl < my_tiles; ++tl) {
        const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
        for (int e = tid; e < TM * D; e += NTH) {
            const int m = e / D, k = e - m * D;
            const bool ok = m < nv;
            OBS[(tl * O + k) * TM + m] = ok ? a.cur_obs[(size_t)(r0 + m) * O + k] : 0.f;
            S[(tl * TM + m) * D + k] = ok ? a.env.state[(size_t)(r0 + m) * D + k] : 0.f;
        }
        if (tid < TM) {
            const bool ok = tid < nv;
            RET[tl * TM + tid] = ok ? a.ret[r0 + tid] : 0.f;
            DN[tl * TM + tid] = ok ? a.cur_dones[r0 + tid] : 0.f;
            TENV[tl * TM + tid] = ok ? a.env.t_env[r0 + tid] : 0u;
            RES[tl * TM + tid] = ok ? a.env.resets[r0 + tid] : 0u;
        }
    }
    if (a.h_actions != nullptr && a.h_sentinel) {  // no copy of the env's answer is under way before the first actions went out
        for (int tl = 0; tl < my_tiles; ++tl) {
            const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
            unsigned* dst = reinterpret_cast<unsigned*>(const_cast<float*>(a.h_obs) + (size_t)r0 * D);
            for (int i = tid; i < ((nv * D + 7) >> 3); i += NTH) dst[8 * i] = PPO_OBS_SENTINEL;
        }
    }
    cp_async_wait_all();
    bar.sync();  // every CTA has read the launch-time state (step counter, barrier generation, sequence number)

    const float* logstd = sW + d.off[T_LOGSTD];
    const uint2 ekey = make_uint2((uint32_t)a.env.seed, (uint32_t)(a.env.seed >> 32));

    int prof_i = 0;
    // ---------------------------------------------------------------------------------------------------- one env
    // The reference's own shape (C1: a single env, 2048 steps) is ONE chain of tiny dependent operations per env step; with the
    // tile machinery above (256 threads, a __syncthreads behind every stage, Philox + Box-Muller twice per step on five threads)
    // it took 15 k cycles per step.  Here warp 0 walks the chain alone (thread per output unit, __syncwarp between the stages,
    // the same fp32 operations in the same order as f_fwd / the tile code: bit-identical results) and the other seven warps
    // draw the Gaussian noise of the NEXT 32 env steps meanwhile (it depends on the counters only).
    const bool solo_env = a.n == 1 && gridDim.x == 1 && world == 1;
    if (solo_env) {
        constexpr int CH = R_SOLO_CHUNK;
        const int NB = 4 * nblk;                                   // noise values per step and kind
        float* NZ = smem + ((L.total_bytes + 15) / 16) * 4;        // [2 buffers][2 kinds][CH][NB] behind the tile layout
        const uint32_t gid = a.env.env_id0;
        const uint32_t te0 = TENV[0];
        auto draw_chunk = [&](int c) {  // warps 1..7: noise of steps [c * CH, (c + 1) * CH)
            float* dst = NZ + (size_t)(c & 1) * 2 * CH * NB;
            const int per_kind = CH * nblk, total = host_env ? per_kind : 2 * per_kind;
            for (int e = tid - 32; e < total; e += NTH - 32) {
                const int kind = e / per_kind, r = e - kind * per_kind, s = r / nblk, blk = r - s * nblk, t = c * CH + s;
                if (t >= a.T) continue;
                float x4[4];
                if (kind == 0) normal4(a.seed, a.env_id0, step0 + (uint32_t)t, (uint32_t)blk, PPO_TAG_ACTION, x4);
                else normal4(a.env.seed, gid, te0 + (uint32_t)t, (uint32_t)blk, PPO_TAG_ENVNOISE, x4);
                float* o = dst + ((size_t)kind * CH + s) * NB + blk * 4;
                o[0] = x4[0]; o[1] = x4[1]; o[2] = x4[2]; o[3] = x4[3];
            }
        };
        if (warp > 0) draw_chunk(0);
        __syncthreads();
        // constants of the rollout (the generic loop recomputes them per step with the same operations)
        float sl_c = 0.f;  // sum of logstd in action order (GRAPH:6103-6672)
        for (int j = 0; j < A; ++j) sl_c = __fadd_rn(sl_c, logstd[j]);
        const int nH1 = d.H1, nH2 = d.H2;
        const float *W0p = sW + d.off[T_PI_FC0_W], *W0v = sW + d.off[T_VF_FC0_W], *B0p = sW + d.off[T_PI_FC0_B], *B0v = sW + d.off[T_VF_FC0_B];
        const float *W1p = sW + d.off[T_PI_FC1_W], *W1v = sW + d.off[T_VF_FC1_W], *B1p = sW + d.off[T_PI_FC1_B], *B1v = sW + d.off[T_VF_FC1_B];
        const float *WHp = sW + d.off[T_PI_W], *WHv = sW + d.off[T_VF_W];
        float *H1p = smem + L.f.h1[0], *H1v = smem + L.f.h1[1], *H2p = smem + L.f.h2[0], *H2v = smem + L.f.h2[1];
        // sigma_j of this lane's actions (the generic loop takes expf(logstd[j]) per step: the same value)
        float sd_l[2];
        sd_l[0] = lane < A ? expf(logstd[lane]) : 1.f;
        sd_l[1] = lane + 32 < A ? expf(logstd[lane + 32]) : 1.f;
        for (int c = 0; c * CH < a.T; ++c) {
            if (warp > 0) {
                draw_chunk(c + 1);
            } else {
                const float* na = NZ + (size_t)(c & 1) * 2 * CH * NB;
                const float* ne = na + (size_t)CH * NB;
                for (int s = 0; s < CH && c * CH + s < a.T; ++s) {
                    const int t = c * CH + s;
                    R_PROF();  // step start
                    // -- store the observation the policy acts on (runner.hpp:75-78)
                    for (int k = lane; k < O; k += 32) a.obs_store[(size_t)t * O + k] = OBS[k * TM];
                    // -- MlpPolicy::step, both towers: lane per output unit, k ascending as f_fwd
                    if (O == 18 && A == 18 && nH1 == 4 && nH2 == 5) {
                        solo_forward<18, 4, 5, 18, TM, ACT>(sW, d, OBS, H1p, H1v, H2p, H2v, MU, Vs, lane);
                    } else if (O == 18 && A == 18 && nH1 == 64 && nH2 == 64) {
                        solo_forward<18, 64, 64, 18, TM, ACT>(sW, d, OBS, H1p, H1v, H2p, H2v, MU, Vs, lane);
                    } else {
                    for (int o = lane; o < 2 * nH1; o += 32) {
                        const bool vt = o >= nH1;
                        const int n = vt ? o - nH1 : o;
                        const float* w = (vt ? W0v : W0p) + n;
                        float acc = 0.f;
#pragma unroll 6
                        for (int k = 0; k < O; ++k) acc = fmaf(w[k * nH1], OBS[k * TM], acc);
                        (vt ? H1v : H1p)[n * TM] = act_fwd<ACT>(acc + (vt ? B0v : B0p)[n]);
                    }
                    __syncwarp();
                    for (int o = lane; o < 2 * nH2; o += 32) {
                        const bool vt = o >= nH2;
                        const int n = vt ? o - nH2 : o;
                        const float* w = (vt ? W1v : W1p) + n;
                        const float* hin = vt ? H1v : H1p;
                        float acc = 0.f;
#pragma unroll 4
                        for (int k = 0; k < nH1; ++k) acc = fmaf(w[k * nH2], hin[k * TM], acc);
                        (vt ? H2v : H2p)[n * TM] = act_fwd<ACT>(acc + (vt ? B1v : B1p)[n]);
                    }
                    __syncwarp();
                    for (int o = lane; o < A + 1; o += 32) {
                        const bool vh = o == A;
                        const int N = vh ? 1 : A, n = vh ? 0 : o;
                        const float* w = (vh ? WHv : WHp) + n;
                        const float* hin = vh ? H2v : H2p;
                        float acc = 0.f;
#pragma unroll 4
                        for (int k = 0; k < nH2; ++k) acc = fmaf(w[k * N], hin[k * TM], acc);
                        if (vh) Vs[0] = acc + sW[d.off[T_VF_B]];
                        else MU[n * TM] = acc + sW[d.off[T_PI_B] + n];
                    }
                    __syncwarp();
                    }
                    R_PROF();  // forward done
                    // -- Gaussian sample (GRAPH:5894-6019)
                    for (int j = lane, jj = 0; j < A; j += 32, ++jj) {
                        const float sd = jj ? sd_l[1] : sd_l[0];  // (A <= 32 + 32; asserted by the host: obs_dim == act_dim <= 32)
                        float z2;
                        const float act = gauss_sample(MU[j * TM], sd, na[s * NB + j], z2);
                        Ac[j * (TM + 1)] = act;
                        Z2[j * TM] = z2;
                        a.act_store[(size_t)t * A + j] = act;
                        if (host_env) {
                            if (a.h_act_ll) ll_store(a.h_act_ll + j, __float_as_uint(act), (unsigned)t + 1u);
                            else a.h_actions[(size_t)t * a.h_act_stride + j] = act;
                        }
                    }
                    __syncwarp();
                    if (lane == 0) {  // neglogp (GRAPH:6103-6672): sequential sum in action order
                        float ss = 0.f;
                        for (int j = 0; j < A; ++j) ss = __fadd_rn(ss, Z2[j * TM]);
                        a.nlp_store[t] = gauss_neglogp_rn(ss, sl_c, A);
                        a.val_store[t] = Vs[0];
                        a.dones_store[t] = DN[0];  // done flag of the previous env step (runner.hpp:110)
                    }
                    R_PROF();  // sample + stores issued
                    if (host_env && a.h_ans_ll) {
                        // -- the env's answer: lane k polls word k (the actions left as LL words above)
                        const unsigned want = (unsigned)t + 1u;
                        uint2 w = make_uint2(0u, want);
                        bool gone = false;
                        if (lane < D + 2) {
                            const unsigned long long t0 = globaltimer_ns();
                            unsigned spins = 0;
                            while (true) {
                                w = ll_load(a.h_ans_ll + lane);
                                if (w.y == want) break;
                                if (w.y == PPO_HOST_ENV_ABORT) { gone = true; break; }
                                if (((++spins) & 0xffu) == 0u && globaltimer_ns() - t0 > 120000000000ull) {  // 120 s: the host is gone
                                    *a.host_err = 1u;
                                    gone = true;
                                    break;
                                }
                            }
                        }
                        if (__any_sync(0xffffffffu, gone)) {
                            if (lane == 0) s_abort = 1;
                            break;
                        }
                        if (lane < D) RAW[lane] = __uint_as_float(w.x);
                        else if (lane == D) REW[0] = __uint_as_float(w.x);
                        else if (lane == D + 1) DONE[0] = __uint_as_float(w.x);
                        __syncwarp();
                        if (lane == 0) RET[0] = __fadd_rn(__fmul_rn(RET[0], a.norm_gamma), REW[0]);  // env_normalize.hpp:71
                    } else if (host_env) {
                        // -- actions to the host, the env's answer back (mapped pinned memory, one flag each way)
                        __syncwarp();
                        unsigned v = 0u;
                        if (lane == 0) {
                            __threadfence_system();
                            st_release_sys(a.h_act_flag, (unsigned)t + 1u);
                            const unsigned long long t0 = globaltimer_ns();
                            unsigned spins = 0;
                            while ((v = *reinterpret_cast<const volatile unsigned*>(a.h_obs_flag)) != (unsigned)t + 1u && v != PPO_HOST_ENV_ABORT) {
                                if (((++spins) & 0xffu) == 0u && globaltimer_ns() - t0 > 120000000000ull) {  // 120 s: the host is gone
                                    *a.host_err = 1u;
                                    v = PPO_HOST_ENV_ABORT;
                                    break;
                                }
                            }
                            __threadfence_system();
                        }
                        v = __shfl_sync(0xffffffffu, v, 0);
                        if (v == PPO_HOST_ENV_ABORT) {
                            if (lane == 0) s_abort = 1;
                            break;
                        }
                        for (int k = lane; k < D; k += 32) RAW[k] = __ldcv(a.h_obs + k);
                        if (lane == 0) {
                            REW[0] = __ldcv(a.h_rew);
                            DONE[0] = __ldcv(a.h_done);
                        }
                        __syncwarp();
                        if (lane == 0) RET[0] = __fadd_rn(__fmul_rn(RET[0], a.norm_gamma), REW[0]);  // env_normalize.hpp:71
                    } else {
                        // -- synthetic env step (SURVEY §8d)
                        const uint32_t te = te0 + (uint32_t)t;
                        const bool dn = ((te + 1u) % 334u) == 0u;
                        for (int k = lane; k < D; k += 32) {
                            const float sk = S[k];
                            float ac = Ac[k * (TM + 1)];
                            ac = ac < -1.f ? -1.f : (ac > 1.f ? 1.f : ac);
                            float sn = __fadd_rn(__fadd_rn(__fmul_rn(0.9f, sk), __fmul_rn(0.1f, ac)), __fmul_rn(0.01f, ne[s * NB + k]));
                            if (k == 0) REW[0] = __fsub_rn(sn, sk);
                            if (dn) {
                                const uint4 w = philox4x32_10(make_uint4(gid, RES[0], (uint32_t)(k >> 2), PPO_TAG_ENVRESET), ekey);
                                const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
                                sn = __fmul_rn(0.1f, __fsub_rn(__fmul_rn(2.0f, u32_to_unit(wv[k & 3])), 1.0f));
                            }
                            S[k] = sn;
                            RAW[k] = sn;
                        }
                        __syncwarp();
                        if (lane == 0) {
                            DONE[0] = dn ? 1.f : 0.f;
                            TENV[0] = te + 1u;
                            if (dn) RES[0] += 1u;
                            RET[0] = __fadd_rn(__fmul_rn(RET[0], a.norm_gamma), REW[0]);  // env_normalize.hpp:71
                        }
                    }
                    __syncwarp();
                    R_PROF();  // env step done
                    // -- RunningStatistics::update with a batch of one row (fp64 around the running mean, as the tile code) + Chan merge
                    if (merge && lane <= D) {
                        const int cidx = lane;
                        const bool is_ret = cidx == D;
                        const double x = is_ret ? (double)RET[0] : (double)RAW[cidx] - (double)s_mean[cidx];
                        double ps = 0.0, pq = 0.0;
                        ps += x;
                        pq += x * x;
                        if (is_ret ? a.upd_ret : a.upd_obs) {
                            const double rows = (double)a.n_global;  // = 1: x / 1.0 is x, the divisions can go
                            const double pv = is_ret ? 0.0 : (double)s_mean[cidx];
                            const double m1 = ps;
                            const double mean_d = pv + m1;
                            double var_d = pq - m1 * m1;
                            if (var_d < 0.0) var_d = 0.0;
                            float mm = s_mean[cidx], vv = s_var[cidx];
                            chan_merge(mm, vv, s_cnt[is_ret ? 1 : 0], (float)mean_d, (float)var_d, rows);
                            s_mean[cidx] = mm;
                            s_var[cidx] = vv;
                        }
                    }
                    __syncwarp();
                    if (merge && lane == 0) {
                        if (a.upd_obs) s_cnt[0] = (double)a.n_global + s_cnt[0];
                        if (a.upd_ret) s_cnt[1] = (double)a.n_global + s_cnt[1];
                    }
                    R_PROF();  // merged
                    if (lane <= D) s_inv[lane] = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(s_var[lane], a.eps)));
                    __syncwarp();
                    // -- EnvNormalize::step post-processing (env_normalize.hpp:74-91)
                    for (int k = lane; k < D; k += 32) {
                        float x = RAW[k];
                        if (a.norm_obs) {
                            x = __fmul_rn(__fsub_rn(x, s_mean[k]), s_inv[k]);
                            x = fminf(fmaxf(x, -a.clip_obs), a.clip_obs);
                        }
                        OBS[k * TM] = x;
                    }
                    if (lane == 0) {
                        const float raw = REW[0];
                        float r = raw;
                        if (a.norm_reward) {
                            r = __fmul_rn(raw, s_inv[D]);
                            r = fminf(fmaxf(r, -a.clip_rew), a.clip_rew);
                        }
                        const float dn2 = DONE[0];
                        RET[0] = __fmul_rn(RET[0], __fsub_rn(1.0f, dn2));
                        DN[0] = dn2;
                        a.rew_store[t] = r;
                        a.urew_store[t] = raw;
                    }
                    __syncwarp();
                    R_PROF();  // applied
                }
            }
            __syncthreads();  // next chunk's noise drawn, this chunk's steps done
            if (s_abort) break;
        }
    } else
    for (int t = 0; t < a.T; ++t) {
        const uint32_t step = step0 + (uint32_t)t;
        R_PROF();  // step start
        double ps = 0.0, pq = 0.0;  // this thread's column partial over the CTA's envs (threads 0..D)
        const float pivot = (tid < D) ? s_mean[tid] : 0.f;
        // host-env mode runs the tile loop twice: pass 0 = policy step of every tile + actions to the host, then the
        // exchange with the host, pass 1 = the env's answer of every tile + moments
        for (int pass = 0; pass < (host_env ? 2 : 1); ++pass) {
        if (pass == 1) {
            __syncthreads();  // every action store of this CTA has been issued
            if (a.h_sentinel) {
                if (tid == 0) {
                    __threadfence_system();
                    st_release_sys(a.h_act_flag + blockIdx.x, (unsigned)t + 1u);
                }
                // wait for the first word of every sector of this CTA's rows to change (all its tiles; sectors start at multiples of
                // 8 floats of the buffer: a tile's rows start at a multiple of TM * D * 4 = 32 * D * 4 bytes)
                int gone = 0;
                const unsigned long long t0 = globaltimer_ns();
                for (int tl = 0; tl < my_tiles && !gone; ++tl) {
                    const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
                    const unsigned* src = reinterpret_cast<const unsigned*>(a.h_obs + (size_t)r0 * D);
                    const int nsec = (nv * D + 7) >> 3;
                    for (int i = tid; i < nsec && !gone; i += NTH) {
                        unsigned spins = 0;
                        while (__ldcv(src + 8 * i) == PPO_OBS_SENTINEL) {
                            if (((++spins) & 0x3fu) == 0u) {
                                if (__ldcv(a.h_obs_flag) == PPO_HOST_ENV_ABORT) { gone = 1; break; }
                                if (globaltimer_ns() - t0 > 120000000000ull) {  // 120 s: the host is gone
                                    *a.host_err = 1u;
                                    gone = 1;
                                    break;
                                }
                            }
                        }
                    }
                }
                const int any_gone = __syncthreads_or(gone);
                if (tid == 0) s_abort = any_gone;
                __syncthreads();
                if (s_abort) break;
            } else {
            if (tid == 0) {
                __threadfence_system();
                st_release_sys(a.h_act_flag + blockIdx.x, (unsigned)t + 1u);
                const unsigned long long t0 = globaltimer_ns();
                unsigned v, spins = 0;
                while ((v = *reinterpret_cast<const volatile unsigned*>(a.h_obs_flag)) != (unsigned)t + 1u && v != PPO_HOST_ENV_ABORT) {
                    if (((++spins) & 0xffu) == 0u && globaltimer_ns() - t0 > 120000000000ull) {  // 120 s: the host is gone
                        *a.host_err = 1u;
                        v = PPO_HOST_ENV_ABORT;
                        break;
                    }
                }
                s_abort = (v == PPO_HOST_ENV_ABORT) ? 1 : 0;
                __threadfence_system();
            }
            __syncthreads();
            if (s_abort) break;
            }
        }
        for (int tl = 0; tl < my_tiles; ++tl) {
            const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
            float* Xs = OBS + tl * O * TM;
            if (pass == 0) {
            // -- store the observation the policy acts on (runner.hpp:75-78)
            for (int r = 0; r < world; ++r) {
                float* dst = rslab(a, r, a.off_obs, O, a.obs_store) + ((size_t)t * a.n + r0) * O;
                for (int e = tid; e < nv * O; e += NTH) {
                    const int m = e / O, k = e - m * O;
                    dst[e] = Xs[k * TM + m];
                }
            }
            // -- MlpPolicy::step: both towers in the same phase
            f_fwd<TM, ACT>(Xs, O, sW + d.off[tw ? T_VF_FC0_W : T_PI_FC0_W], sW + d.off[tw ? T_VF_FC0_B : T_PI_FC0_B], d.H1, H1, half);
            __syncthreads();
            f_fwd<TM, ACT>(H1, d.H1, sW + d.off[tw ? T_VF_FC1_W : T_PI_FC1_W], sW + d.off[tw ? T_VF_FC1_B : T_PI_FC1_B], d.H2, H2, half);
            __syncthreads();
            if (tw == 0) f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_PI_W], sW + d.off[T_PI_B], A, MU, half);
            else f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_VF_W], sW + d.off[T_VF_B], 1, Vs, half);
            __syncthreads();
            R_PROF();  // forward done
            // -- Gaussian sample (GRAPH:5894-6019): thread (m, blk) draws 4 actions
            for (int e = tid; e < TM * nblk; e += NTH) {
                const int m = e % TM, blk = e / TM;
                if (m < nv) {
                    float e4[4];
                    normal4(a.seed, a.env_id0 + (uint32_t)(r0 + m), step, (uint32_t)blk, PPO_TAG_ACTION, e4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j = blk * 4 + q;
                        if (j < A) {
                            float z2;
                            Ac[j * (TM + 1) + m] = gauss_sample(MU[j * TM + m], expf(logstd[j]), e4[q], z2);
                            Z2[j * TM + m] = z2;
                        }
                    }
                }
            }
            __syncthreads();
            if (tid < nv) {  // neglogp (GRAPH:6103-6672): sequential sums in action order, as the step kernels
                const int m = tid, row = r0 + m;
                float ss = 0.f, sl = 0.f;
                for (int j = 0; j < A; ++j) {
                    ss = __fadd_rn(ss, Z2[j * TM + m]);
                    sl = __fadd_rn(sl, logstd[j]);
                }
                const float nl = gauss_neglogp_rn(ss, sl, A);
                const size_t idx = (size_t)t * a.n + row;
                for (int r = 0; r < world; ++r) {
                    rslab(a, r, a.off_nlp, 1, a.nlp_store)[idx] = nl;
                    rslab(a, r, a.off_val, 1, a.val_store)[idx] = Vs[m];
                }
                a.dones_store[idx] = DN[tl * TM + m];  // done flag of the previous env step (runner.hpp:110)
            }
            for (int r = 0; r < world; ++r) {
                float* dst = rslab(a, r, a.off_act, A, a.act_store) + ((size_t)t * a.n + r0) * A;
                for (int e = tid; e < nv * A; e += NTH) {
                    const int m = e / A, j = e - m * A;
                    dst[e] = Ac[j * (TM + 1) + m];
                }
            }
            R_PROF();  // sample + stores issued
            }  // pass 0
            if (host_env) {
                if (pass == 0) {  // actions of this tile -> the host's array (clipping is the env's business, hexapod_env.hpp:140)
                    // 16-byte stores: over PCIe a warp's 512 contiguous bytes travel as two full 256-byte packets (4-byte stores: 128-byte
                    // packets; measured 27 us per env step for the 295 KB of 4096 envs)
                    float* dst = a.h_actions + (size_t)t * a.h_act_stride + (size_t)r0 * A;
                    const int ne = nv * A;
                    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                        for (int e4 = tid; e4 < (ne >> 2); e4 += NTH) {
                            float v[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int e = 4 * e4 + i, m = e / A, j = e - m * A;
                                v[i] = Ac[j * (TM + 1) + m];
                            }
                            *reinterpret_cast<float4*>(dst + 4 * e4) = make_float4(v[0], v[1], v[2], v[3]);
                        }
                        for (int e = (ne & ~3) + tid; e < ne; e += NTH) {
                            const int m = e / A, j = e - m * A;
                            dst[e] = Ac[j * (TM + 1) + m];
                        }
                    } else {
                        for (int e = tid; e < ne; e += NTH) {
                            const int m = e / A, j = e - m * A;
                            dst[e] = Ac[j * (TM + 1) + m];
                        }
                    }
                    __syncthreads();  // Ac is reused by the next tile
                    continue;
                }
                // the env's answer (mapped host memory, read past every cache: the same addresses carry new data every step)
                for (int e = tid; e < nv * D; e += NTH) RAW[tl * TM * D + e] = __ldcv(a.h_obs + (size_t)r0 * D + e);
                if (tid < nv) {
                    REW[tl * TM + tid] = __ldcv(a.h_rew + r0 + tid);
                    DONE[tl * TM + tid] = __ldcv(a.h_done + r0 + tid);
                }
                __syncthreads();
                if (a.h_sentinel) {  // the rows are in shared memory: the sectors wait for the next step's copy again
                    unsigned* dst = reinterpret_cast<unsigned*>(const_cast<float*>(a.h_obs) + (size_t)r0 * D);
                    for (int i = tid; i < ((nv * D + 7) >> 3); i += NTH) dst[8 * i] = PPO_OBS_SENTINEL;
                }
                if (tid < nv) RET[tl * TM + tid] = __fadd_rn(__fmul_rn(RET[tl * TM + tid], a.norm_gamma), REW[tl * TM + tid]);  // env_normalize.hpp:71
                __syncthreads();
            } else {
            // -- synthetic env step (SURVEY §8d): thread (m, blk) advances 4 state dims
            for (int e = tid; e < TM * nblk; e += NTH) {
                const int m = e % TM, blk = e / TM;
                if (m < nv) {
                    const uint32_t gid = a.env.env_id0 + (uint32_t)(r0 + m);
                    const uint32_t te = TENV[tl * TM + m];
                    const bool dn = ((te + 1u) % 334u) == 0u;
                    float xi[4];
                    normal4(a.env.seed, gid, te, (uint32_t)blk, PPO_TAG_ENVNOISE, xi);
                    float* st = S + (tl * TM + m) * D;
                    float* rw = RAW + (tl * TM + m) * D;
                    uint4 w = make_uint4(0, 0, 0, 0);
                    if (dn) w = philox4x32_10(make_uint4(gid, RES[tl * TM + m], (uint32_t)blk, PPO_TAG_ENVRESET), ekey);
                    const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int k = blk * 4 + q;
                        if (k < D) {
                            const float sk = st[k];
                            float ac = Ac[k * (TM + 1) + m];
                            ac = ac < -1.f ? -1.f : (ac > 1.f ? 1.f : ac);
                            float sn = __fadd_rn(__fadd_rn(__fmul_rn(0.9f, sk), __fmul_rn(0.1f, ac)), __fmul_rn(0.01f, xi[q]));
                            if (k == 0) REW[tl * TM + m] = __fsub_rn(sn, sk);
                            if (dn) sn = __fmul_rn(0.1f, __fsub_rn(__fmul_rn(2.0f, u32_to_unit(wv[q])), 1.0f));
                            st[k] = sn;
                            rw[k] = sn;
                        }
                    }
                    if (blk == 0) DONE[tl * TM + m] = dn ? 1.f : 0.f;
                }
            }
            __syncthreads();
            if (tid < nv) {
                const int m = tid;
                TENV[tl * TM + m] += 1u;
                if (DONE[tl * TM + m] != 0.f) RES[tl * TM + m] += 1u;
                RET[tl * TM + m] = __fadd_rn(__fmul_rn(RET[tl * TM + m], a.norm_gamma), REW[tl * TM + m]);  // env_normalize.hpp:71
            }
            __syncthreads();
            }  // synthetic env
            R_PROF();  // env step done
            // -- batch moments of this tile (fp64 around the running mean), accumulated over the CTA's tiles
            if (merge) {
                if (tid < D) {
                    for (int m = 0; m < nv; ++m) {
                        const double x = (double)RAW[(tl * TM + m) * D + tid] - (double)pivot;
                        ps += x;
                        pq += x * x;
                    }
                } else if (tid == D) {
                    for (int m = 0; m < nv; ++m) {
                        const double r = (double)RET[tl * TM + m];
                        ps += r;
                        pq += r * r;
                    }
                }
            }
        }
        }  // passes
        if (s_abort) break;  // host-env mode: the env aborted (every CTA sees the same flag at the same step)
        if (merge) {
            // -- RunningStatistics::update over ALL envs: partials -> grid barrier -> fixed-order total in every CTA
            // partial layout [parity][column][cta]: the totals below read 32 consecutive CTAs per load instruction
            const bool solo = gridDim.x == 1 && world == 1;  // one CTA holds every env (C1 / C2 shapes): its partials ARE the totals
            double* mine = a.partial + (size_t)(t & 1) * 2 * (D + 1) * gridDim.x + blockIdx.x;
            if (solo) {
                if (tid <= D) {
                    csum[tid] = ps;
                    csum[D + 1 + tid] = pq;
                }
            } else if (tid <= D) {
                mine[(size_t)tid * gridDim.x] = ps;
                mine[(size_t)(D + 1 + tid) * gridDim.x] = pq;
            }
            R_PROF();  // partial moments written
            if (!solo) bar.sync();
            R_PROF();  // grid barrier passed
            const double* all = a.partial + (size_t)(t & 1) * 2 * (D + 1) * gridDim.x;
            if (!solo && (world == 1 || blockIdx.x == 0)) {
                // warp w sums columns w, w+8, ...: lane partials over the CTAs (independent loads, 5 columns x 4 in flight),
                // then a butterfly — the same order in every CTA, so every CTA gets the same bits
                constexpr int CPW = 5;  // columns per warp: 8 warps x 5 >= 2*(D+1) for D <= 19
                double acc[CPW];
#pragma unroll
                for (int i = 0; i < CPW; ++i) acc[i] = 0.0;
#pragma unroll 4
                for (int b0 = 0; b0 < (int)gridDim.x; b0 += 32) {
                    double x[CPW];
#pragma unroll
                    for (int i = 0; i < CPW; ++i) {
                        const int c = warp + (NTH / 32) * i;
                        x[i] = (c < 2 * (D + 1) && b0 + lane < (int)gridDim.x) ? __ldcg(all + (size_t)c * gridDim.x + b0 + lane) : 0.0;
                    }
#pragma unroll
                    for (int i = 0; i < CPW; ++i) acc[i] += x[i];
                }
#pragma unroll
                for (int i = 0; i < CPW; ++i) {
                    const int c = warp + (NTH / 32) * i;
                    const double v = warp_sum(acc[i]);
                    if (lane == 0 && c < 2 * (D + 1)) csum[c] = v;
                }
                for (int c = (NTH / 32) * CPW + warp; c < 2 * (D + 1); c += NTH / 32) {  // D > 19: remaining columns
                    double v = 0.0;
                    for (int b = lane; b < (int)gridDim.x; b += 32) v += __ldcg(all + (size_t)c * gridDim.x + b);
                    v = warp_sum(v);
                    if (lane == 0) csum[c] = v;
                }
            }
            __syncthreads();
            if (world > 1) {
                // CTA 0 publishes this rank's totals to every rank; every CTA then adds the `world` slots in rank order
                const unsigned seq = seq0 + (unsigned)t + 1u;
                // (LL words: 4 bytes of data + seq in one 8-byte store, no fence, the receivers poll the payload)
                if (blockIdx.x == 0 && tid < 2 * (D + 1)) {
                    const unsigned long long bits = (unsigned long long)__double_as_longlong(csum[tid]);
                    for (int dst = 0; dst < world; ++dst) {
                        uint2* sl = a.mbox.ll_slot(dst, seq, a.mbox.rank) + 2 * tid;
                        ll_store(sl, (unsigned)bits, seq);
                        ll_store(sl + 1, (unsigned)(bits >> 32), seq);
                    }
                }
                __syncthreads();  // CTA 0: csum has been read before it is overwritten below
                if (tid < 2 * (D + 1)) {
                    double v = 0.0;
                    for (int s0 = 0; s0 < world; s0 += 4) {  // four ranks' words in flight together, added in rank order
                        unsigned long long w[4];
                        a.mbox.ll_wait4_pair(seq, (size_t)(2 * tid), s0, w);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (s0 + k < world) v += __longlong_as_double((long long)w[k]);
                    }
                    csum[tid] = v;
                }
                __syncthreads();
            }
            R_PROF();  // totals
            if (tid <= D) {
                const int c = tid;
                const bool is_ret = c == D;
                if (is_ret ? a.upd_ret : a.upd_obs) {
                    const double rows = (double)a.n_global;
                    const double pv = is_ret ? 0.0 : (double)s_mean[c];
                    const double m1 = csum[c] / rows;
                    const double mean_d = pv + m1;
                    double var_d = csum[D + 1 + c] / rows - m1 * m1;
                    if (var_d < 0.0) var_d = 0.0;
                    float mm = s_mean[c], vv = s_var[c];
                    chan_merge(mm, vv, s_cnt[is_ret ? 1 : 0], (float)mean_d, (float)var_d, rows);
                    s_mean[c] = mm;
                    s_var[c] = vv;
                }
            }
            __syncthreads();
            if (tid == 0) {
                if (a.upd_obs) s_cnt[0] = (double)a.n_global + s_cnt[0];
                if (a.upd_ret) s_cnt[1] = (double)a.n_global + s_cnt[1];
            }
        }
        R_PROF();  // merged
        if (tid <= D) s_inv[tid] = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(s_var[tid], a.eps)));
        __syncthreads();
        // -- EnvNormalize::step post-processing (env_normalize.hpp:74-91)
        for (int tl = 0; tl < my_tiles; ++tl) {
            const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
            for (int e = tid; e < TM * D; e += NTH) {
                const int m = e / D, k = e - m * D;
                float x = RAW[(tl * TM + m) * D + k];
                if (a.norm_obs) {
                    x = __fmul_rn(__fsub_rn(x, s_mean[k]), s_inv[k]);
                    x = fminf(fmaxf(x, -a.clip_obs), a.clip_obs);
                }
                OBS[(tl * O + k) * TM + m] = (m < nv) ? x : 0.f;
            }
            if (tid < nv) {
                const int m = tid;
                const float raw = REW[tl * TM + m];
                float r = raw;
                if (a.norm_reward) {
                    r = __fmul_rn(raw, s_inv[D]);
                    r = fminf(fmaxf(r, -a.clip_rew), a.clip_rew);
                }
                const float dn = DONE[tl * TM + m];
                RET[tl * TM + m] = __fmul_rn(RET[tl * TM + m], __fsub_rn(1.0f, dn));
                DN[tl * TM + m] = dn;
                const size_t idx = (size_t)t * a.n + r0 + m;
                a.rew_store[idx] = r;
                a.urew_store[idx] = raw;
            }
        }
        __syncthreads();
        R_PROF();  // applied
    }

    // ---- bootstrap value (runner.hpp:161-166) + GAE (runner.hpp:174-190) + state write-back
    for (int tl = 0; tl < my_tiles; ++tl) {
        const int r0 = (tile0 + tl) * TM, nv = min(TM, a.n - r0);
        float* Xs = OBS + tl * O * TM;
        if (tw == 1) f_fwd<TM, ACT>(Xs, O, sW + d.off[T_VF_FC0_W], sW + d.off[T_VF_FC0_B], d.H1, H1, half);
        __syncthreads();
        if (tw == 1) f_fwd<TM, ACT>(H1, d.H1, sW + d.off[T_VF_FC1_W], sW + d.off[T_VF_FC1_B], d.H2, H2, half);
        __syncthreads();
        if (tw == 1) f_fwd<TM, ACT_NONE>(H2, d.H2, sW + d.off[T_VF_W], sW + d.off[T_VF_B], 1, Vs, half);
        __syncthreads();
        if (tid < nv) LASTV[tl * TM + tid] = Vs[tid];
        for (int e = tid; e < nv * D; e += NTH) {
            const int m = e / D, k = e - m * D;
            a.cur_obs[(size_t)r0 * O + e] = Xs[k * TM + m];
            a.env.state[(size_t)r0 * D + e] = S[(tl * TM + m) * D + k];
        }
        __syncthreads();
    }
    for (int e = tid; e < my_tiles * TM; e += NTH) {
        const int tl = e / TM, m = e - tl * TM;
        const int row = (tile0 + tl) * TM + m;
        if (row >= a.n) continue;
        a.ret[row] = RET[e];
        a.cur_dones[row] = DN[e];
        a.env.t_env[row] = TENV[e];
        a.env.resets[row] = RES[e];
        a.last_values[row] = LASTV[e];
        const float gl = __fmul_rn(a.gamma, a.lam);
        float last = 0.f, nextv = LASTV[e], nextnt = 1.0f - DN[e];
#pragma unroll 8
        for (int t = a.T - 1; t >= 0; --t) {
            const size_t idx = (size_t)t * a.n + row;
            const float v = a.val_store[idx];
            const float delta = __fsub_rn(__fadd_rn(a.rew_store[idx], __fmul_rn(a.gamma, __fmul_rn(nextv, nextnt))), v);
            last = __fadd_rn(delta, __fmul_rn(gl, __fmul_rn(nextnt, last)));
            const float rt = __fadd_rn(last, v);
            for (int r = 0; r < world; ++r) rslab(a, r, a.off_ret, 1, a.ret_store)[idx] = rt;
            nextv = v;
            nextnt = 1.0f - a.dones_store[idx];
        }
    }
    if (world > 1) {
        // every rank's rows must have landed in every rank's buffers before anybody trains on them: system-scope fence
        // per CTA, local grid barrier, then CTA 0 trades "rollout complete" flags with the peers
        __syncthreads();
        if (tid == 0) __threadfence_system();
        bar.sync();
        if (blockIdx.x == 0 && tid == 0) {
            a.mbox.signal_all(PPO_MBOX_DONE_CHANNEL, dseq0 + 1u);
            a.mbox.wait_all(PPO_MBOX_DONE_CHANNEL, dseq0 + 1u);
            *a.done_seq = dseq0 + 1u;
        }
    }
    if (blockIdx.x == 0) {
        if (tid < D) {
            a.st.obs_mean[tid] = s_mean[tid];
            a.st.obs_var[tid] = s_var[tid];
        } else if (tid == D) {
            *a.st.ret_mean = s_mean[D];
            *a.st.ret_var = s_var[D];
            *a.st.obs_count = s_cnt[0];
            *a.st.ret_count = s_cnt[1];
            *a.step_ctr = step0 + (uint32_t)a.T;
            *a.bar_gen = bar.gen;
            if (world > 1 && merge) *a.mbox_seq = seq0 + (unsigned)a.T;
        }
    }
}

}  // namespace ppo
