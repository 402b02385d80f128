// Device-side helpers shared by all kernels: network layout, Philox4x32-10, Box-Muller.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ppo {

// Tensor indices in the flat parameter vector (graph gradient order, GRAPH:23738-24074, then q head).
enum TensorId {
    T_PI_FC0_W, T_PI_FC0_B, T_VF_FC0_W, T_VF_FC0_B, T_PI_FC1_W, T_PI_FC1_B, T_VF_FC1_W, T_VF_FC1_B,
    T_VF_W, T_VF_B, T_PI_W, T_PI_B, T_LOGSTD, T_Q_W, T_Q_B, T_COUNT
};

// Policy head (ppo_action_space in ppo_core.h): Box -> diagonal Gaussian with model/pi/logstd, Discrete(A) -> categorical over
// A logits.  Uniform per core, a template parameter of the kernels that evaluate it.
enum { HEAD_BOX = 0, HEAD_DISCRETE = 1 };

struct NetDims {
    int O, A, H1, H2;      // A: width of the policy output (action dimensions, or logits of a categorical head)
    int off[T_COUNT + 1];  // off[T_Q_W] = P (trainable), off[T_COUNT] = total
    int P, Pq;
    // a categorical head has no logstd: T_LOGSTD has size 0, every other offset stays in graph gradient order
    __host__ void init(int o, int a, int h1, int h2, int head = HEAD_BOX) {
        O = o; A = a; H1 = h1; H2 = h2;
        const int ls = head == HEAD_DISCRETE ? 0 : A;
        const int sz[T_COUNT] = {O * H1, H1, O * H1, H1, H1 * H2, H2, H1 * H2, H2, H2, 1, H2 * A, A, ls, H2 * A, A};
        off[0] = 0;
        for (int i = 0; i < T_COUNT; ++i) off[i + 1] = off[i] + sz[i];
        P = off[T_Q_W];
        Pq = off[T_COUNT];
    }
};

// columns appended to every per-CTA partial gradient slab: loss sums
enum { L_PG = 0, L_VF = 1, L_ENT = 2, L_KL = 3, L_CLIP = 4, L_PAD = 8 };

// Per-update scalars of one core in device memory.  Written on the core's stream before each update (a one-thread
// kernel, so the host never waits); the train kernels and the Adam steps read them there, so the captured update
// graphs do not depend on their values and a learning-rate / clip-range schedule replays the same graphs.
// world: number of ranks whose gradient slabs get summed (the categorical head's per-sample entropy column is scaled by it, so
// that the reduce kernels' 1 / world_size leaves the minibatch mean)
struct UpdateScalars {
    float lr, cliprange, cliprange_vf, world;
};

// Value-function loss of Stable-Baselines' PPO2 (ppo_vf_clip in ppo_core.h); uniform per launch
enum { VF_CLIP_SHARED = 0, VF_CLIP_NONE = 1, VF_CLIP_SEPARATE = 2 };

__host__ __device__ __forceinline__ float vf_clip_range(int mode, float cliprange, float cliprange_vf) {
    return mode == VF_CLIP_SEPARATE ? cliprange_vf : cliprange;
}

// One sample's value loss (GRAPH:10213-10400): returns max(l1, l2) with l1 = (v - R)^2, l2 = (vc - R)^2,
// vc = old_v + clip(v - old_v, -range, range), and sets dv = dL/dv = vf_coef * 0.5/B * d max(l1, l2)/dv.
// TF's tie rules: Maximum's gradient goes to l1 on l1 >= l2, clip_by_value's passes on -range <= v - old_v <= range.
// VF_CLIP_NONE is vc = v exactly (not an infinite range: old_v + (v - old_v) is not v in fp32, and the tie would
// then fall on either branch by rounding), so l2 == l1 and the tie takes the unclipped branch.
__device__ __forceinline__ float value_loss_term(int mode, float range, float v, float oldv, float R, float vf_coef, float invB, float& dv) {
    const bool none = mode == VF_CLIP_NONE;
    const float dvo = v - oldv;
    const float vc = none ? v : oldv + fmaxf(fminf(dvo, range), -range);
    const float l1 = (v - R) * (v - R), l2 = (vc - R) * (vc - R);
    const bool tk = l1 >= l2;
    const bool inr = none || ((dvo <= range) && (dvo >= -range));
    dv = vf_coef * 0.5f * invB * (tk ? 2.f * (v - R) : (inr ? 2.f * (vc - R) : 0.f));
    return tk ? l1 : l2;
}

// Hidden-layer activation of the MLP (ppo_activation in ppo_core.h); uniform per core, a template parameter of every kernel
// that evaluates it, so each activation compiles to its own code.  The derivative is taken from the OUTPUT h, as a factor:
// TanhGrad (1 - h^2) and ReluGrad (h > 0: a unit whose pre-activation is exactly 0 gets no gradient, as TF's
// gradients * (features > 0)).
enum { ACT_TANH = 0, ACT_RELU = 1, ACT_NONE = 2 };  // ACT_NONE: the linear heads of the tile forward helpers

template <int ACT>
__device__ __forceinline__ float act_fwd(float x) {
    if (ACT == ACT_NONE) return x;
    if (ACT == ACT_RELU) return x < 0.f ? 0.f : x;
    return tanhf(x);
}
template <int ACT>
__device__ __forceinline__ float act_dfac(float h) {
    if (ACT == ACT_RELU) return h > 0.f ? 1.f : 0.f;
    return 1.f - h * h;
}

// 0.5*log(2*pi), 0.5*log(2*pi*e) as the fp32 constants baked in the graph (GRAPH:6103-6672, 10021-10180)
#define PPO_HALF_LOG_2PI 0.9189385175704956f
#define PPO_HALF_LOG_2PIE 1.4189385175704956f

#define PPO_TAG_ACTION 0x50504F32u    // "PPO2": action noise stream
#define PPO_TAG_CATEG 0x43415431u     // "CAT1": uniforms of the categorical head's Gumbel-max sample
#define PPO_TAG_ENVNOISE 0x454E5631u  // "ENV1": synthetic env process noise
#define PPO_TAG_ENVRESET 0x52535431u  // "RST1": synthetic env reset state

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// Philox4x32-10 (Salmon et al., SC'11) — the generator TF's RandomStandardNormal uses (SURVEY §3.5c).
__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// TF's Uint32ToFloat: 23 mantissa bits -> [0,1)
__device__ __forceinline__ float u32_to_unit(uint32_t x) { return __uint_as_float((x & 0x7fffffu) | 0x3f800000u) - 1.0f; }

// Box-Muller on two 32-bit words, TF-style (u1 clamped to 1e-7); full-precision logf/sinf/cosf.
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, float& n0, float& n1) {
    float u1 = fmaxf(u32_to_unit(w0), 1.0e-7f);
    const float u2 = u32_to_unit(w1);
    const float r = sqrtf(-2.0f * logf(u1));
    const float th = 6.2831853071795864769f * u2;
    float s, c;
    sincosf(th, &s, &c);
    n0 = r * s;
    n1 = r * c;
}

// N(0,1) block `blk` (4 values) of stream (seed, a, b, tag)
__device__ __forceinline__ void normal4(uint64_t seed, uint32_t a, uint32_t b, uint32_t blk, uint32_t tag, float out[4]) {
    const uint4 w = philox4x32_10(make_uint4(a, b, blk, tag), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    box_muller(w.x, w.y, out[0], out[1]);
    box_muller(w.z, w.w, out[2], out[3]);
}

// ---- categorical head (Stable-Baselines' CategoricalProbabilityDistribution) of one sample: logits l[j * ld], j < n
// sample = argmax_j (l_j - log(-log(u_j))), u uniform in [0, 1) from stream (seed, env, step, block j/4, PPO_TAG_CATEG) or given;
// u = 0 gives -inf and is never taken; ties go to the first index (TF's ArgMax)
__device__ __forceinline__ int cat_sample(const float* l, int ld, int n, const float* u_given, uint64_t seed, uint32_t env, uint32_t step) {
    float best = -__int_as_float(0x7f800000);
    int bi = 0;
    for (int j0 = 0; j0 < n; j0 += 4) {
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (!u_given) w = philox4x32_10(make_uint4(env, step, (uint32_t)(j0 >> 2), PPO_TAG_CATEG), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < n) {
                const float u = u_given ? u_given[j] : u32_to_unit(wv[q]);
                const float g = l[j * ld] - logf(-logf(u));
                if (g > best) { best = g; bi = j; }
            }
        }
    }
    return bi;
}
// deterministic action: argmax_j l_j, first index on ties
__device__ __forceinline__ int cat_argmax(const float* l, int ld, int n) {
    int bi = 0;
    for (int j = 1; j < n; ++j)
        if (l[j * ld] > l[bi * ld]) bi = j;
    return bi;
}
// max shift and partition: mx = max_j l_j, returns z = sum_j exp(l_j - mx)
__device__ __forceinline__ float cat_partition(const float* l, int ld, int n, float& mx) {
    mx = l[0];
    for (int j = 1; j < n; ++j) mx = fmaxf(mx, l[j * ld]);
    float z = 0.f;
    for (int j = 0; j < n; ++j) z += expf(l[j * ld] - mx);
    return z;
}
// neglogp(a) = log z - (l_a - mx), as softmax_cross_entropy_with_logits_v2
__device__ __forceinline__ float cat_neglogp(const float* l, int ld, int n, int a) {
    float mx;
    const float z = cat_partition(l, ld, n, mx);
    return logf(z) - (l[a * ld] - mx);
}
// entropy H = sum_j p_j (log z - a0_j), a0 = l - mx, p = exp(a0) / z (CategoricalProbabilityDistribution.entropy)
__device__ __forceinline__ float cat_entropy(const float* l, int ld, int n, float mx, float z) {
    const float lz = logf(z);
    float h = 0.f;
    for (int j = 0; j < n; ++j) {
        const float a0 = l[j * ld] - mx;
        h += (expf(a0) / z) * (lz - a0);
    }
    return h;
}
// overwrites the logits with dL/dl_j = g_nlp (p_j - [j == a]) + ent_w p_j (log p_j + H): the pg term through neglogp (TF's
// softmax - labels) and -ent_coef/B * dH/dl_j with ent_w = ent_coef / B
__device__ __forceinline__ void cat_dlogits(float* l, int ld, int n, int a, float mx, float z, float H, float g_nlp, float ent_w) {
    const float lz = logf(z);
    for (int j = 0; j < n; ++j) {
        const float a0 = l[j * ld] - mx;
        const float p = expf(a0) / z;
        l[j * ld] = g_nlp * (p - (j == a ? 1.f : 0.f)) + ent_w * p * ((a0 - lz) + H);
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ppo
