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

// Policy head (ppo_action_space in ppo_core.h, same values): Box -> diagonal Gaussian with model/pi/logstd, Discrete(A) ->
// categorical over A logits, MultiDiscrete(nvec) -> k categoricals over slices of the A = sum(nvec) logits, MultiBinary(A) -> A
// Bernoullis.  Uniform per core, a template parameter of the kernels that evaluate it.
enum { HEAD_BOX = 0, HEAD_DISCRETE = 1, HEAD_MULTI_DISCRETE = 2, HEAD_MULTI_BINARY = 3 };

struct NetDims {
    int O, A, H1, H2;      // A: width of the policy output (action dimensions, or logits of a categorical head)
    int off[T_COUNT + 1];  // off[T_Q_W] = P (trainable), off[T_COUNT] = total
    int P, Pq;
    // only a Gaussian head has a logstd: otherwise T_LOGSTD has size 0, every other offset stays in graph gradient order
    __host__ void init(int o, int a, int h1, int h2, int head = HEAD_BOX) {
        O = o; A = a; H1 = h1; H2 = h2;
        const int ls = head == HEAD_BOX ? A : 0;
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

// One sample's clipped surrogate (GRAPH:10423-10447, 12609-12776): pg = max(-adv r, -adv clip(r, 1 - cr, 1 + cr)) with
// r = exp(oldneglogp - neglogp), its approxkl (dn^2) and clipfrac terms, and g_nlp = dL/dneglogp = adv r / B on the unclipped
// branch, 0 on the clipped one.  clip_by_value = max(min(x, hi), lo); ties go to the unclipped branch.
struct PgTerm {
    float pg, kl, cf, g_nlp;
};
__device__ __forceinline__ PgTerm pg_term(float adv, float oldn, float nlp, float cr, float invB) {
    const float ratio = expf(oldn - nlp);
    const float pg1 = -adv * ratio;
    const float pg2 = -adv * fmaxf(fminf(ratio, 1.f + cr), 1.f - cr);
    const bool take1 = pg1 >= pg2;
    const float dn = nlp - oldn;
    return {take1 ? pg1 : pg2, dn * dn, (fabsf(ratio - 1.f) > cr) ? 1.f : 0.f, take1 ? (adv * ratio) * invB : 0.f};
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

// Diagonal Gaussian neglogp = 0.5*sum(z^2) + 0.5*log(2pi)*float(A) + sum(logstd) from the finished sums ss = sum(z^2),
// sl = sum(logstd).  Two roundings: the train kernels' form may contract (GRAPH:9428-9997); the policy step's is
// _rn throughout (GRAPH:6103-6672), as are its sample and z^2 (gauss_sample).
__device__ __forceinline__ float gauss_neglogp(float ss, float sl, int A) { return (0.5f * ss + PPO_HALF_LOG_2PI * (float)A) + sl; }
__device__ __forceinline__ float gauss_neglogp_rn(float ss, float sl, int A) {
    return __fadd_rn(__fadd_rn(__fmul_rn(0.5f, ss), __fmul_rn(PPO_HALF_LOG_2PI, (float)A)), sl);
}
// act = mu + sd * e (GRAPH:5992-6019); z2 = ((act - mu) / sd)^2
__device__ __forceinline__ float gauss_sample(float mu, float sd, float e, float& z2) {
    const float act = __fadd_rn(mu, __fmul_rn(sd, e));
    const float z = __fdiv_rn(__fsub_rn(act, mu), sd);
    z2 = __fmul_rn(z, z);
    return act;
}
// entropy = sum_j(logstd_j + 0.5*log(2*pi*e)) (GRAPH:10021-10180); logstd(j) loads logstd_j
template <class LS>
__device__ __forceinline__ float box_entropy(LS logstd, int A) {
    float ent = 0.f;
    for (int j = 0; j < A; ++j) ent += logstd(j) + PPO_HALF_LOG_2PIE;
    return ent;
}

#define PPO_TAG_ACTION 0x50504F32u    // "PPO2": action noise stream
#define PPO_TAG_CATEG 0x43415431u     // "CAT1": uniforms of the categorical head's Gumbel-max sample
#define PPO_TAG_BERN 0x42455231u      // "BER1": uniforms of the Bernoulli head's sample
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
// Action masks (sb3-contrib's MaskableCategorical): m is the sample's mask word, bit j set = logit j allowed; every helper works
// over the allowed logits S only, as if the forbidden ones were -inf.  m = ~0 (no mask) is the arithmetic of the unmasked head,
// in the same order.  S must not be empty (the callers check the masks they are handed).
// first allowed index of m (0 for m = ~0)
__device__ __forceinline__ int cat_first(uint64_t m) { return __ffsll((long long)m) - 1; }
__device__ __forceinline__ bool cat_allowed(uint64_t m, int j) { return (m >> j) & 1ull; }
// sample = argmax_{j in S} (l_j - log(-log(u_j))), u uniform in [0, 1) from stream (seed, env, step, block j/4, PPO_TAG_CATEG) or
// given; u = 0 gives -inf and is never taken (unless it is all S has); ties go to the first index (TF's ArgMax)
__device__ __forceinline__ int cat_sample(const float* l, int ld, int n, const float* u_given, uint64_t seed, uint32_t env, uint32_t step,
                                          uint64_t m = ~0ull) {
    float best = -__int_as_float(0x7f800000);
    int bi = cat_first(m);
    for (int j0 = 0; j0 < n; j0 += 4) {
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (!u_given) w = philox4x32_10(make_uint4(env, step, (uint32_t)(j0 >> 2), PPO_TAG_CATEG), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < n && cat_allowed(m, j)) {
                const float u = u_given ? u_given[j] : u32_to_unit(wv[q]);
                const float g = l[j * ld] - logf(-logf(u));
                if (g > best) { best = g; bi = j; }
            }
        }
    }
    return bi;
}
// deterministic action: argmax_{j in S} l_j, first index on ties
__device__ __forceinline__ int cat_argmax(const float* l, int ld, int n, uint64_t m = ~0ull) {
    int bi = cat_first(m);
    for (int j = bi + 1; j < n; ++j)
        if (cat_allowed(m, j) && l[j * ld] > l[bi * ld]) bi = j;
    return bi;
}
// max shift and partition: mx = max_{j in S} l_j, returns z = sum_{j in S} exp(l_j - mx)
__device__ __forceinline__ float cat_partition(const float* l, int ld, int n, float& mx, uint64_t m = ~0ull) {
    const int f = cat_first(m);
    mx = l[f * ld];
    for (int j = f + 1; j < n; ++j)
        if (cat_allowed(m, j)) mx = fmaxf(mx, l[j * ld]);
    float z = 0.f;
    for (int j = f; j < n; ++j)
        if (cat_allowed(m, j)) z += expf(l[j * ld] - mx);
    return z;
}
// neglogp(a) = log z - (l_a - mx), as softmax_cross_entropy_with_logits_v2
__device__ __forceinline__ float cat_neglogp(const float* l, int ld, int n, int a, uint64_t m = ~0ull) {
    float mx;
    const float z = cat_partition(l, ld, n, mx, m);
    return logf(z) - (l[a * ld] - mx);
}
// entropy H = sum_{j in S} p_j (log z - a0_j), a0 = l - mx, p = exp(a0) / z (CategoricalProbabilityDistribution.entropy; sb3-contrib's
// where(mask, p log p, 0))
__device__ __forceinline__ float cat_entropy(const float* l, int ld, int n, float mx, float z, uint64_t m = ~0ull) {
    const float lz = logf(z);
    float h = 0.f;
    for (int j = 0; j < n; ++j) {
        if (!cat_allowed(m, j)) continue;
        const float a0 = l[j * ld] - mx;
        h += (expf(a0) / z) * (lz - a0);
    }
    return h;
}
// overwrites the logits with dL/dl_j = g_nlp (p_j - [j == a]) + ent_w p_j (log p_j + H) for j in S: the pg term through neglogp (TF's
// softmax - labels) and -ent_coef/B * dH/dl_j with ent_w = ent_coef / B; exactly 0 for a forbidden j (torch.where blocks it)
__device__ __forceinline__ void cat_dlogits(float* l, int ld, int n, int a, float mx, float z, float H, float g_nlp, float ent_w, uint64_t m = ~0ull) {
    const float lz = logf(z);
    for (int j = 0; j < n; ++j) {
        if (!cat_allowed(m, j)) {
            l[j * ld] = 0.f;
            continue;
        }
        const float a0 = l[j * ld] - mx;
        const float p = expf(a0) / z;
        l[j * ld] = g_nlp * (p - (j == a ? 1.f : 0.f)) + ent_w * p * ((a0 - lz) + H);
    }
}
// one sample's categorical train terms: neglogp(a) and entropy H of the logits, the clipped surrogate of pg_term, and the
// logits overwritten with dL/dl_j (cat_dlogits, ent_w = ent_coef / B)
__device__ __forceinline__ PgTerm cat_train_term(float* l, int ld, int n, int a, float adv, float oldn, float cr, float invB, float ent_w,
                                                 float& H, uint64_t m = ~0ull) {
    float mx;
    const float z = cat_partition(l, ld, n, mx, m);
    const float nlp = logf(z) - (l[a * ld] - mx);
    H = cat_entropy(l, ld, n, mx, z, m);
    const PgTerm t = pg_term(adv, oldn, nlp, cr, invB);
    cat_dlogits(l, ld, n, a, mx, z, H, t.g_nlp, ent_w, m);
    return t;
}

// ---- MultiDiscrete head (MultiCategoricalProbabilityDistribution): k categoricals side by side over slices of the n <= 64
// logits, given as a mask of slice starts (bit j set: a slice starts at logit j; bit 0 always set, k = popcount); an action is
// one index per slice, within the slice.  The categorical helpers above, per slice; the action mask m is over all n logits (the
// slice that starts at s0 sees m >> s0).
// end of the slice that starts at s0: the next start, or n
__device__ __forceinline__ int md_slice_end(uint64_t starts, int s0, int n) {
    const uint64_t rest = s0 >= 63 ? 0ull : starts & (~0ull << (s0 + 1));
    return rest ? __ffsll((long long)rest) - 1 : n;
}
// sample: Gumbel-max per slice over the uniforms of the flat logit index (the categorical stream, so MultiDiscrete([n]) draws
// what Discrete(n) draws); put(i, index) receives slice i's index once the slice is finished
template <class PUT>
__device__ __forceinline__ void md_sample(const float* l, int ld, int n, uint64_t starts, const float* u_given, uint64_t seed, uint32_t env,
                                          uint32_t step, PUT put, uint64_t m = ~0ull) {
    float best = -__int_as_float(0x7f800000);
    int i = 0, s0 = 0, bi = cat_first(m);
    for (int j0 = 0; j0 < n; j0 += 4) {
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (!u_given) w = philox4x32_10(make_uint4(env, step, (uint32_t)(j0 >> 2), PPO_TAG_CATEG), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < n) {
                if (j > 0 && ((starts >> j) & 1ull)) {  // slice i done; ties stayed on its first allowed index
                    put(i++, bi - s0);
                    s0 = j;
                    bi = cat_first(m & (~0ull << j));
                    best = -__int_as_float(0x7f800000);
                }
                if (cat_allowed(m, j)) {
                    const float u = u_given ? u_given[j] : u32_to_unit(wv[q]);
                    const float g = l[j * ld] - logf(-logf(u));
                    if (g > best) { best = g; bi = j; }
                }
            }
        }
    }
    put(i, bi - s0);
}
// one sample's MultiDiscrete train terms: neglogp = sum_i neglogp_i(a_i) (TF's add_n in slice order), H = sum_i H_i, the
// clipped surrogate of pg_term, and the logits overwritten with dL/dl: slice i as cat_dlogits with its own entropy H_i.
// act[i * ald]: slice i's index
__device__ __forceinline__ PgTerm md_train_term(float* l, int ld, int n, uint64_t starts, const float* act, int ald, float adv, float oldn,
                                                float cr, float invB, float ent_w, float& H, uint64_t m = ~0ull) {
    float nlp = 0.f;
    H = 0.f;
    for (int i = 0, s0 = 0; s0 < n; ++i) {
        const int s1 = md_slice_end(starts, s0, n);
        const float* s = l + s0 * ld;
        const uint64_t ms = m >> s0;
        float mx;
        const float z = cat_partition(s, ld, s1 - s0, mx, ms);
        nlp += logf(z) - (s[(int)act[i * ald] * ld] - mx);
        H += cat_entropy(s, ld, s1 - s0, mx, z, ms);
        s0 = s1;
    }
    const PgTerm t = pg_term(adv, oldn, nlp, cr, invB);
    for (int i = 0, s0 = 0; s0 < n; ++i) {
        const int s1 = md_slice_end(starts, s0, n);
        float* s = l + s0 * ld;
        const uint64_t ms = m >> s0;
        float mx;
        const float z = cat_partition(s, ld, s1 - s0, mx, ms);
        cat_dlogits(s, ld, s1 - s0, (int)act[i * ald], mx, z, cat_entropy(s, ld, s1 - s0, mx, z, ms), t.g_nlp, ent_w, ms);
        s0 = s1;
    }
    return t;
}

// ---- MultiBinary head (BernoulliProbabilityDistribution) of one sample: logits l[j * ld], j < n, an action of n columns 0 / 1
__device__ __forceinline__ float bern_sigmoid(float l) { return 1.f / (1.f + expf(-l)); }
// TF's sigmoid_cross_entropy_with_logits: sce(l, z) = max(l, 0) - l z + log1p(exp(-|l|))
__device__ __forceinline__ float bern_sce(float l, float z) { return fmaxf(l, 0.f) - l * z + log1pf(expf(-fabsf(l))); }
// sample x_j = [u_j < sigmoid(l_j)], u uniform in [0, 1) from stream (seed, env, step, block j/4, PPO_TAG_BERN) or given;
// put(j, x_j)
template <class PUT>
__device__ __forceinline__ void bern_sample(const float* l, int ld, int n, const float* u_given, uint64_t seed, uint32_t env, uint32_t step, PUT put) {
    for (int j0 = 0; j0 < n; j0 += 4) {
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (!u_given) w = philox4x32_10(make_uint4(env, step, (uint32_t)(j0 >> 2), PPO_TAG_BERN), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < n) put(j, (u_given ? u_given[j] : u32_to_unit(wv[q])) < bern_sigmoid(l[j * ld]) ? 1.f : 0.f);
        }
    }
}
// neglogp(x) = sum_j sce(l_j, x_j); x[j * xld]
__device__ __forceinline__ float bern_neglogp(const float* l, int ld, int n, const float* x, int xld) {
    float s = 0.f;
    for (int j = 0; j < n; ++j) s += bern_sce(l[j * ld], x[j * xld]);
    return s;
}
// one sample's MultiBinary train terms: neglogp(x), the entropy H = sum_j sce(l_j, sigmoid(l_j)), the clipped surrogate of
// pg_term, and the logits overwritten with dL/dl_j = g_nlp (s_j - x_j) + ent_w l_j s_j (1 - s_j), s = sigmoid(l): Stable-Baselines
// does not stop the gradient through the entropy's labels, so dH/dl = -l s (1 - s)
__device__ __forceinline__ PgTerm bern_train_term(float* l, int ld, int n, const float* x, int xld, float adv, float oldn, float cr,
                                                  float invB, float ent_w, float& H) {
    const float nlp = bern_neglogp(l, ld, n, x, xld);
    H = 0.f;
    for (int j = 0; j < n; ++j) H += bern_sce(l[j * ld], bern_sigmoid(l[j * ld]));
    const PgTerm t = pg_term(adv, oldn, nlp, cr, invB);
    for (int j = 0; j < n; ++j) {
        const float v = l[j * ld], s = bern_sigmoid(v);
        l[j * ld] = t.g_nlp * (s - x[j * xld]) + ent_w * v * s * (1.f - s);
    }
    return t;
}

// ---- gradient step: clip_by_global_norm (GRAPH:24102-25392) and TF 1.14 ApplyAdam (GRAPH:25426-31383: epsilon outside the
// sqrt, not bias-corrected), every operation rounded as written
// scale = clip * min(1/||g||, 1/clip), NaN when ||g|| is not finite (GRAPH:24493-24543); ss: sum of squares, gnorm = ||g||
__device__ __forceinline__ float clip_scale(double ss, float clip_norm, float& gnorm) {
    gnorm = (float)sqrt(ss);
    const float inv = __fdiv_rn(1.0f, gnorm), invc = __fdiv_rn(1.0f, clip_norm);
    float scale = __fmul_rn(clip_norm, fminf(inv, invc));
    if (!isfinite(gnorm)) scale = __int_as_float(0x7fc00000);
    return scale;
}
// step size lr * sqrt(1 - beta2^t) / (1 - beta1^t) from the beta powers before this step
__device__ __forceinline__ float adam_alpha(float lr, float b1p, float b2p) {
    return __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.0f, b2p))), __fsub_rn(1.0f, b1p));
}
// moments m, v of one parameter updated in place with its clipped gradient g
__device__ __forceinline__ void adam_moments(float g, float& m, float& v, float beta1, float beta2) {
    m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), __fsub_rn(1.0f, beta1)));
    v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), __fsub_rn(1.0f, beta2)));
}
// the parameter p after the step, from its updated moments
__device__ __forceinline__ float adam_param(float p, float m, float v, float alpha, float eps) {
    return __fsub_rn(p, __fdiv_rn(__fmul_rn(m, alpha), __fadd_rn(__fsqrt_rn(v), eps)));
}
// the step's loss row [5]: pg, vf, entropy, approxkl, clipfrac from the summed loss columns L[L_PG .. L_CLIP]
__device__ __forceinline__ void loss_row(float* row, const float* L, float invB, float inv_world) {
    row[0] = L[L_PG] * invB;
    row[1] = 0.5f * (L[L_VF] * invB);
    row[2] = L[L_ENT] * inv_world;
    row[3] = 0.5f * (L[L_KL] * invB);
    row[4] = L[L_CLIP] * invB;
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
