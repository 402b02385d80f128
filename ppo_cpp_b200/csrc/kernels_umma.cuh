// "U family": tcgen05 (5th-gen tensor core) train kernel for the [64,64] MLP (H1 == H2 == 64, obs/act widths as template parameters, 18/18 instantiated).
//
// Replaces the loss / autodiff sub-graph of one PPO2::_train_step (ppo2/ppo2.hpp:430-470, GRAPH:6889-23699) for a
// minibatch; math and TF tie-breaking rules are those of SURVEY §3.5b, identical to train_fused_kernel.
//
// Mapping to the hardware
//   * one CTA = one tower (blockIdx.y: 0 = pi, 1 = V) of one tile of 128 samples (= the 128 TMEM lanes); the towers
//     share nothing but the advantage / return inputs, so a minibatch of 8192 samples is 64 tiles x 2 towers = 128 CTAs.
//   * every GEMM of the forward and the hand-derived backward pass runs on tcgen05.mma (kind::f16, fp16 operands,
//     fp32 accumulators in TMEM).  fp32 parity (1e-5) is kept by splitting every fp32 operand x into TWO fp16 pieces
//     x = hi + lo (11 + 11 mantissa bits; lo is exact down to fp16's subnormal step 2^-24) and issuing the three
//     products hi*hi, hi*lo, lo*hi (the dropped lo*lo is < 2^-22 relative).  Round 1 used three bf16 pieces and six
//     products: twice the tensor-pipe time and 1.5x the shared-memory traffic for the same accuracy.  fp16 has a 5-bit
//     exponent, so the operands must be O(1): observations are clipped to +-10 by VecNormalize, activations are tanh
//     outputs (ReLU outputs get their own scale, see PW_H_RELU), weights are O(1), and the BACKWARD tensors (which carry the 1/B of the batch mean, ~1e-4) are scaled by
//     a power of two S with S/B in [1/16, 1/8) — exact in fp32 — and the weight gradients are multiplied by 1/S when
//     they leave TMEM.  |x| * S/B > 65504 (a per-sample dL/dmu beyond ~5e5 / B) would overflow to inf and surface as a
//     non-finite global norm (NaN update, as the graph's IsFinite select does for any non-finite gradient).
//     kind::tf32 was measured first (tools/probe/umma_probe*.cu): it silently produces zeros for MN-major operands on
//     sm_100a, and the dW GEMMs need MN-major views; kind::f16 supports both.
//   * operands live in shared memory as [rows][64 bf16] blocks in the canonical SWIZZLE_128B layout, so the SAME bytes
//     serve as K-major operand (forward: act x W, backward: dY x W^T) and as MN-major operand (dW = act^T x dY, reduced
//     over the 128 samples of the tile).  The back-propagated dP2 / dP1 have their own blocks, so the weight-gradient
//     GEMMs (which still read H2 / H1) never sit on the tile's critical path: they run on the tensor pipe while the CUDA
//     cores do the next epilogue, and one commit at the end of the tile collects them.
//   * the gathered observation rows of a tile (the minibatch slice of ppo2.hpp:291-307, 72 bytes each at a shuffled row index) come in
//     through the TMA engine: one cp.async.bulk per row into a shared-memory staging row (a 16-byte aligned 80-byte window around the
//     row), all 128 completing on one mbarrier; the persistent kernel issues them behind its arrival at the grid barrier of the previous
//     minibatch, so they land during the gradient step, and the fp16 split reads them out of shared memory.
//   * bias gradients and the logstd gradient are column sums over samples: one extra N=8 MMA against a block whose
//     first row is ones.  The V head (N = 1) is a dot product in the epilogue; its weight gradient is again an N=8 MMA.
//   * weight gradients accumulate in TMEM across the tiles a CTA processes and are written once to the CTA's slab.
//   * the epilogues (tanh, loss, tanh', bf16 splitting) run on 8 warps: warp w owns TMEM lanes 32*(w&3).. and the
//     32-column half (w>>2) of a 64-wide accumulator; activations stay in registers between forward and backward.
//   * accuracy: the tensor core truncates (RZ) at every accumulation, a bias that grows with the number of MMAs chained
//     into one accumulator and that the value loss amplifies (v - R cancels over the batch).  The leading product p0p0
//     therefore accumulates alone, the two small cross products go to a second TMEM accumulator (2^-11 of the
//     magnitude, so 2^-11 of the truncation error) and the epilogue adds the two in fp32 (round to nearest).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "kernels_misc.cuh"
#include "kernels_mlp2.cuh"

namespace ppo {
namespace umma {

// Operand blocks sit high in fp16's range (an fp16 lo piece below 2^-14 is subnormal: values whose hi piece is below ~0.25
// would lose relative accuracy): weights max in [2^8, 2^9), activations and the ones block times 2^8, observations times 2^5
// (|obs| <= clip_obs = 10), back-propagated tensors times S and renormalised by 2^-8 after every product with a weight block.
// ReLU activations are unbounded, so their blocks (and the ones block with them) hold H * 2^PW_H_RELU = H itself: exact as
// two pieces for H >= 2^-3, an absolute error <= 2^-25 below that, and H up to fp16's 65504.  A larger activation becomes
// inf and surfaces as a non-finite global norm (a NaN update), as an overflowing backward tensor does.
constexpr int PW_W = 8, PW_H = 8, PW_X = 5, PW_H_RELU = 0;
template <int ACT>
constexpr int pw_h() { return ACT == ACT_RELU ? PW_H_RELU : PW_H; }
constexpr int TM = 128;   // samples per tile
constexpr int NTH = 256;  // threads per CTA
constexpr int HID = 64;   // hidden width handled by this family

// ---- shared memory map (bytes from a 1024-aligned base)
constexpr int NP = 2;                           // fp16 pieces per fp32 operand value
constexpr uint32_t ACT_PIECE = TM * 128;        // [128 x 64] fp16 = 16 KB
constexpr uint32_t ACT_BLOCK = NP * ACT_PIECE;  // both pieces
constexpr uint32_t W0_PIECE = 32 * 128;         // [32 x 64] fp16 (rows: O inputs, bias row, zero padding)
constexpr uint32_t W1_PIECE = 64 * 128;         // [64 x 64]
constexpr uint32_t WP_PIECE = 64 * 128;         // [64 x 64], columns >= A are zero
constexpr uint32_t ROW8_PIECE = 2 * 1024;       // [8 x 128] fp16, K-major operand over the 128 samples
constexpr uint32_t ROW16_BLOCK = 4 * 1024;      // [16 x 128] fp16 K-major: per 64-sample half 16 rows of 128 B (rows 0..7 | rows 8..15)
constexpr uint32_t OFF_H1 = 0;
constexpr uint32_t OFF_H2 = OFF_H1 + ACT_BLOCK;
constexpr uint32_t OFF_Y = OFF_H2 + ACT_BLOCK;  // X' (obs + ones column)
constexpr uint32_t OFF_D2 = OFF_Y + ACT_BLOCK;  // dP2 = dL/d(pre-activation of layer 1)
constexpr uint32_t OFF_D1 = OFF_D2 + ACT_BLOCK; // [dMU | dLS] (pi tower), then dP1
constexpr uint32_t OFF_W0 = OFF_D1 + ACT_BLOCK;
constexpr uint32_t OFF_W1 = OFF_W0 + NP * W0_PIECE;
constexpr uint32_t OFF_WP = OFF_W1 + NP * W1_PIECE;   // pi head weights; the V tower keeps its dv rows here
constexpr uint32_t OFF_ONES = OFF_WP + NP * WP_PIECE;
constexpr uint32_t OFF_F32 = OFF_ONES + ROW16_BLOCK;  // fp32 vectors
constexpr uint32_t F32_B1 = 0, F32_BH = 64, F32_WV = 96, F32_SD = 160, F32_LS = 192, F32_MISC = 224, F32_PV = 256,
                   F32_DV = 512, F32_RED = 640, F32_ISD = 704, F32_COUNT = 736;
constexpr uint32_t OFF_BAR = OFF_F32 + F32_COUNT * 4;
// Staging rows of the bulk copies (cp.async.bulk, the TMA engine) that bring the gathered observation rows of a tile in: one
// 16-byte aligned window per sample row.  A row of O floats starts 8-byte aligned, so its window starts 0 or 8 bytes below it
// and spans round16(4 O + 8) bytes at most (80 for O = 18).
constexpr uint32_t OFF_STG = OFF_BAR + 64;
constexpr uint32_t stg_row_bytes(int O) { return (uint32_t)((4 * O + 8 + 15) & ~15); }
constexpr uint32_t SMEM_BYTES = OFF_STG + TM * stg_row_bytes(18) + 1024;  // + alignment slack; the widths instantiated are 18 / 18

// ---- TMEM columns: every accumulator has a twin ("+ XC") for the small cross products
constexpr uint32_t ACC_WORK = 0, ACC_WORK_C = 64;  // Z1, Z2, MU (first 32 columns), dH2, dH1
// Weight-gradient accumulators (M = 64: row r in TMEM lane 32 * (r >> 4) + (r & 15)), TWO instructions per k-step: the B operand with
// its pieces side by side ([Q_hi | Q_lo], N = 128 / 96 / 16: the piece stride is the atom stride of the descriptor) gives the leading
// product in columns [0, 64) and hi x lo in columns [64, ..); the second instruction adds P_lo x Q_hi to the cross columns.
// Column sums (M = 128: row r in lane r), ONE instruction per k-step: [P_hi ; P_lo] x ones -> rows < 64 hi sums, rows >= 64 lo sums.
// (Stacking P for the big gradients too — one instruction per k-step — was measured: the lo x hi rows then sit in other lanes than
// the rows they belong to and the flush pays more for bringing them together than the 24 instructions saved.)
constexpr uint32_t ACC_DWP = 128 /* N = 96 (pi) | 16 (V) */, ACC_CS = 224 /* N = 16 */, ACC_DW1 = 240 /* N = 128 */, ACC_DB1 = 368 /* N = 16 */,
                   ACC_DW0 = 384 /* N = 96 */, TMEM_COLS = 512;

// 2^k for -126 <= k <= 127 (the exponents of the block floating point scheme stay within +-100)
__device__ __forceinline__ float pow2f(int k) { return __int_as_float((k + 127) << 23); }
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of the 16-byte chunk j (8 bf16 columns) of row r inside a SWIZZLE_128B [R x 64] bf16 block
__device__ __forceinline__ uint32_t chunk_off(int r, int j) { return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((j ^ (r & 7)) << 4)); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;  // SWIZZLE_128B
    return d;
}
// instruction descriptor: D = f32 (bits 4-5 = 1), A = B = fp16 (format fields 7-9 / 10-12 = 0)
__device__ __forceinline__ uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// One operand of a GEMM: descriptor of piece 0 / k-step 0 plus strides (in 16-byte units).
// k-step ks (16 elements of K) sits at (ks >> 2) * k_hi + (ks & 3) * k_lo.
struct Operand {
    uint64_t desc;
    uint32_t piece, k_lo, k_hi;
};
// K-major view (mn = row, k = column) of a [rows x (64 * nblk)] block
__device__ __forceinline__ Operand op_kmajor(uint32_t base, uint32_t piece_bytes, int rows) {
    return Operand{make_desc(base, 16, 1024), piece_bytes >> 4, 32 >> 4, (uint32_t)((rows >> 3) * 1024) >> 4};
}
// MN-major view (k = row, mn = column) of a [rows x 64] block: one k-step = 16 rows = 2 KB
__device__ __forceinline__ Operand op_mnmajor(uint32_t base, uint32_t piece_bytes, int rows) {
    return Operand{make_desc(base, (uint32_t)((rows >> 3) * 1024), 1024), piece_bytes >> 4, 2048 >> 4, 8192 >> 4};
}

__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// ---- bf16 x 3 flavour of the operand helpers, used by the W family (kernels_wide.cuh): three bf16 pieces per fp32 value,
// six products.  Activations of a wide layer are not bounded the way the U family's fp16 scheme needs.
__device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
    return make_idesc(M, N, a_mn, b_mn) | (1u << 7) | (1u << 10);  // A = B = bf16
}
__device__ __forceinline__ void split_pair3(float x0, float x1, uint32_t& p0, uint32_t& p1, uint32_t& p2) {
    __nv_bfloat162 b = __floats2bfloat162_rn(x0, x1);
    p0 = *reinterpret_cast<uint32_t*>(&b);
    const float r0 = x0 - __uint_as_float(p0 << 16), r1 = x1 - __uint_as_float(p0 & 0xffff0000u);
    b = __floats2bfloat162_rn(r0, r1);
    p1 = *reinterpret_cast<uint32_t*>(&b);
    const float s0 = r0 - __uint_as_float(p1 << 16), s1 = r1 - __uint_as_float(p1 & 0xffff0000u);
    b = __floats2bfloat162_rn(s0, s1);
    p2 = *reinterpret_cast<uint32_t*>(&b);
}
__device__ __forceinline__ void store_chunk3(uint8_t* block, uint32_t piece_bytes, uint32_t off, const float* x) {
    uint4 q0, q1, q2;
    split_pair3(x[0], x[1], q0.x, q1.x, q2.x);
    split_pair3(x[2], x[3], q0.y, q1.y, q2.y);
    split_pair3(x[4], x[5], q0.z, q1.z, q2.z);
    split_pair3(x[6], x[7], q0.w, q1.w, q2.w);
    *reinterpret_cast<uint4*>(block + off) = q0;
    *reinterpret_cast<uint4*>(block + piece_bytes + off) = q1;
    *reinterpret_cast<uint4*>(block + 2 * piece_bytes + off) = q2;
}

// D (+)= A * B with split operands: the leading product goes to `dm`, the cross products to `dc`.
// NPB == 2: both operands in two pieces, three products; NPB == 1: B is exact in fp16 (ones), two products.
template <int NPB, int KSTEPS>
__device__ __forceinline__ void issue_gemm(uint32_t dm, uint32_t dc, const Operand& A, const Operand& B, uint32_t idesc, bool accumulate) {
    const uint32_t acc0 = accumulate ? 1u : 0u;
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
        const uint64_t a = A.desc + (uint64_t)((ks >> 2) * A.k_hi + (ks & 3) * A.k_lo);
        const uint64_t b = B.desc + (uint64_t)((ks >> 2) * B.k_hi + (ks & 3) * B.k_lo);
        const uint32_t acc = ks ? 1u : acc0;
        mma_f16(dm, a, b, idesc, acc);
        if (NPB == 2) {
            mma_f16(dc, a, b + B.piece, idesc, acc);
            mma_f16(dc, a + A.piece, b, idesc, 1u);
        } else {
            mma_f16(dc, a + A.piece, b, idesc, acc);
        }
    }
}

// D (+)= A * B for a GEMM whose result an epilogue waits for, in TWO instructions per k-step instead of three: the two pieces of
// B sit one piece stride apart, which is exactly the stride between two 64-wide (MN-major view) / 64-row (K-major view) atoms
// of the same descriptor, so ONE instruction with N doubled to 128 computes A_hi * [B_hi | B_lo] -> columns [0, 64) (leading
// product, alone in its accumulator) and [64, 128) (cross product); the second adds A_lo * B_hi to the cross columns.  The
// tensor pipe spends ~45 cycles per instruction of these shapes whatever N is, so instructions are what counts.
template <int KSTEPS>
__device__ __forceinline__ void issue_gemm_wide(uint32_t dwork, const Operand& A, const Operand& B, uint32_t idesc_n128, uint32_t idesc_cross) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
        const uint64_t a = A.desc + (uint64_t)((ks >> 2) * A.k_hi + (ks & 3) * A.k_lo);
        const uint64_t b = B.desc + (uint64_t)((ks >> 2) * B.k_hi + (ks & 3) * B.k_lo);
        mma_f16(dwork, a, b, idesc_n128, ks ? 1u : 0u);
        mma_f16(dwork + 64u, a + A.piece, b, idesc_cross, 1u);
    }
}

// weight gradient, two instructions per k-step (see the TMEM map): A_hi x [B_hi | B_lo] -> d, A_lo x B_hi -> d + cross_col
template <int KSTEPS>
__device__ __forceinline__ void issue_gemm_dw(uint32_t d, uint32_t cross_col, const Operand& A, const Operand& B, uint32_t idesc_wide, uint32_t idesc_cross,
                                              bool accumulate) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
        const uint64_t a = A.desc + (uint64_t)((ks >> 2) * A.k_hi + (ks & 3) * A.k_lo);
        const uint64_t b = B.desc + (uint64_t)((ks >> 2) * B.k_hi + (ks & 3) * B.k_lo);
        mma_f16(d, a, b, idesc_wide, (ks || accumulate) ? 1u : 0u);
        mma_f16(d + cross_col, a + A.piece, b, idesc_cross, 1u);
    }
}
// column sums, one instruction per k-step: both pieces of A stacked as M = 128
template <int KSTEPS>
__device__ __forceinline__ void issue_gemm_stacked(uint32_t d, const Operand& A, const Operand& B, uint32_t idesc, bool accumulate) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
        const uint64_t a = A.desc + (uint64_t)((ks >> 2) * A.k_hi + (ks & 3) * A.k_lo);
        const uint64_t b = B.desc + (uint64_t)((ks >> 2) * B.k_hi + (ks & 3) * B.k_lo);
        mma_f16(d, a, b, idesc, (ks || accumulate) ? 1u : 0u);
    }
}

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

#define PPO_TMEM_LD32(taddr, r)                                                                                                        \
    asm volatile(                                                                                                                      \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                                      \
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];" \
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),      \
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),         \
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),         \
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])                                                                           \
        : "r"(taddr))
#define PPO_TMEM_LD8(taddr, r)                                                      \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" \
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) \
                 : "r"(taddr))

// v[0..32) = main + cross accumulator: 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32_sum(uint32_t tmain, uint32_t tcross, float* v) {
    uint32_t r[32], s[32];
    PPO_TMEM_LD32(tmain, r);
    PPO_TMEM_LD32(tcross, s);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(s[i]);
}
#define PPO_TMEM_LD16(taddr, r)                                                                                                       \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"              \
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), \
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])                                        \
                 : "r"(taddr))
// the same 16 columns at a time: half the live temporaries (the epilogues of the tile loop sit at the register limit)
__device__ __forceinline__ void tmem_ld16_sum(uint32_t tmain, uint32_t tcross, float* v) {
    uint32_t r[16], s[16];
    PPO_TMEM_LD16(tmain, r);
    PPO_TMEM_LD16(tcross, s);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(s[i]);
}
__device__ __forceinline__ void tmem_ld8_sum(uint32_t tmain, uint32_t tcross, float* v) {
    uint32_t r[8], s[8];
    PPO_TMEM_LD8(tmain, r);
    PPO_TMEM_LD8(tcross, s);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(s[i]);
}

// tanh for the activation epilogues (issue-bound: 32 per thread and layer): 1 - 2 / (1 + 2^(2 log2(e) x)) on the two MUFU units,
// x - x^3/3 + 2 x^5/15 below |x| = 1/16 where the exponential form loses relative accuracy.  11 instructions against tanhf's 17;
// max abs error 2.3e-7, max relative error 2.1e-6 over [-12, 12] (tanhf: 1.0e-7 / 1.9e-7) — inside the 1e-5 parity bar, checked by
// the gradient tests against the fp64 oracle and the executed graph.
__device__ __forceinline__ float tanh_epi(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    const float big = fmaf(-2.0f, r, 1.0f);
    const float x2 = x * x;
    const float small = fmaf(x * x2, fmaf(x2, 0.13333333f, -0.33333333f), x);
    return fabsf(x) < 0.0625f ? small : big;
}
template <int ACT>
__device__ __forceinline__ float act_epi(float x) {
    if (ACT == ACT_RELU) return act_fwd<ACT_RELU>(x);
    return tanh_epi(x);
}
// x0, x1 -> two packed fp16 pairs hi, lo with x = hi + lo (x0 in the low half = lower address)
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t& p0, uint32_t& p1) {
    const __half2 h = __floats2half2_rn(x0, x1);
    p0 = *reinterpret_cast<const uint32_t*>(&h);
    const float2 f = __half22float2(h);
    const __half2 l = __floats2half2_rn(x0 - f.x, x1 - f.y);
    p1 = *reinterpret_cast<const uint32_t*>(&l);
}
// eight consecutive columns (one 16-byte chunk) -> the two pieces of a block
__device__ __forceinline__ void store_chunk(uint8_t* block, uint32_t piece_bytes, uint32_t off, const float* x) {
    uint4 q0, q1;
    split_pair(x[0], x[1], q0.x, q1.x);
    split_pair(x[2], x[3], q0.y, q1.y);
    split_pair(x[4], x[5], q0.z, q1.z);
    split_pair(x[6], x[7], q0.w, q1.w);
    *reinterpret_cast<uint4*>(block + off) = q0;
    *reinterpret_cast<uint4*>(block + piece_bytes + off) = q1;
}
// 32 consecutive columns [32 * half, 32 * half + 32) of row r of an activation block
__device__ __forceinline__ void store_row32(uint8_t* block, int r, int half, const float* x, float scale = 1.f) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] = x[8 * j + i] * scale;
        store_chunk(block, ACT_PIECE, chunk_off(r, 4 * half + j), y);
    }
}

// Observation rows of a tile travel global -> shared memory as bulk copies (one per gathered row, issued by the thread that owns the
// sample, all completing on one mbarrier), so the gather of ppo2.hpp:291-307 costs no register and no LSU round trip on the
// tile's critical path: the split into fp16 pieces reads the landed rows out of shared memory.
template <int O>
struct ObsStage {
    static constexpr uint32_t ROW = stg_row_bytes(O);
    // issued by the 128 threads gh == 0 (the mbarrier expects 128 arrivals per tile); rows that do not exist only arrive
    static __device__ __forceinline__ void issue(const float* __restrict__ obs, long grow, bool valid, uint32_t stg_row, uint32_t bar) {
        if (valid) {
            const uint64_t addr = (uint64_t)(obs + grow * O);
            const uint32_t off = (uint32_t)(addr & 15u);
            const uint32_t bytes = (off + 4u * O + 15u) & ~15u;  // never past the 16-byte block that holds the row's last float
            uint64_t st;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 %0, [%1], %2;" : "=l"(st) : "r"(bar), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stg_row),
                         "l"(addr - off), "r"(bytes), "r"(bar)
                         : "memory");
        } else {
            uint64_t st;
            asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(st) : "r"(bar) : "memory");
        }
    }
    // the landed row of this thread (columns [16h, 16h+16)) -> registers: kept apart from the split so that the compiler can weave the
    // split into whatever runs between the two (the weight blocks: with the wait and the split in one piece behind them it was 1.2 k cycles)
    float2 x[8];
    __device__ __forceinline__ void load(const uint8_t* stg, const float* __restrict__ obs, long grow, bool valid, int r, int h) {
        const uint32_t off = (uint32_t)((uint64_t)(obs + grow * O) & 15u);
        const float2* src = reinterpret_cast<const float2*>(stg + (uint32_t)r * ROW + off);  // rows are 8-byte aligned (O even)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = 16 * h + 2 * i;
            x[i] = (valid && c < O) ? src[c >> 1] : make_float2(0.f, 0.f);
        }
    }
    // X' = [obs | 1 | 0 ...] of row r, columns [16h, 16h+16): the ones column folds the layer-0 bias into the GEMM and yields its gradient
    __device__ __forceinline__ void store(uint8_t* Y, int r, int h) const {
        float v[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            v[2 * i] = x[i].x * (float)(1 << PW_X);
            v[2 * i + 1] = x[i].y * (float)(1 << PW_X);
        }
        if (O >= 16 * h && O < 16 * h + 16) v[O - 16 * h] = (float)(1 << PW_X);
        store_chunk(Y, ACT_PIECE, chunk_off(r, 2 * h), v);
        store_chunk(Y, ACT_PIECE, chunk_off(r, 2 * h + 1), v + 8);
    }
};

// Persistent variant (PERSIST = true): ONE cooperative launch runs all the minibatches of an epoch.  Per minibatch:
// weights re-staged from the (just updated) fp32 parameters -> tiles -> slabs | grid barrier | column reduce (+ peer
// mailbox allreduce) + sum of squares | grid barrier | clip + Adam | grid barrier.  TMEM, mbarriers and the constant
// operand blocks are set up once per epoch; 2 kernel launches per minibatch become 3 grid barriers.
struct EpochArgs {
    int M;                  // minibatches in this launch
    int B;                  // slots per (global) minibatch
    int rank_off;           // this rank processes slots [k*B + rank_off, k*B + rank_off + count)
    const float2* mbstats;  // [M]
    float* loss_rows;       // [M][5]
    ReduceAdamArgs ra;
};

// phase stamps of CTA 0 of each tower: the stand-alone kernel writes a.prof[tower][0..32), the persistent kernel stamps
// minibatch 2 only (steady state) into a.prof[64 + 48 * tower ..)
// per-CTA timeline of minibatch 2 (global timer, ns): a.prof[256 + (tower * gridDim.x + blockIdx.x) * 8 + i]
#define UMMA_TL(i)                                                                                               \
    do {                                                                                                         \
        if (PERSIST && a.prof && tid == 0 && prof_on) a.prof[256 + (tower * gridDim.x + blockIdx.x) * 8 + (i)] = (long long)globaltimer_ns(); \
    } while (0)
#define UMMA_PROF()                                                                                              \
    do {                                                                                                         \
        if (a.prof && blockIdx.x == 0 && tid == 0 && prof_on && prof_i < (PERSIST ? 48 : 32))                     \
            a.prof[(PERSIST ? 64 + tower * 48 : tower * 32) + prof_i++] = clock64();                              \
    } while (0)

// MODE 0: one minibatch per launch (slabs are reduced by another kernel).  MODE 1: persistent epoch, three grid barriers per
// minibatch.  (A barrier-free variant — every cross-CTA hand-over an LL word polled by its consumer — was built and measured
// in round 2: 7.22 ms per C3 update against 6.97 ms; each dependent global hop costs ~0.8 us either way and the LL slabs
// double the bytes of the largest exchange.  profiles/r2_u_family_ll_experiment.txt; not kept.)
template <int O, int A, int MODE, int ACT>
__global__ void __launch_bounds__(NTH, 1) train_umma_kernel(const TrainArgs a, const EpochArgs ep) {
    constexpr bool PERSIST = MODE != 0;
    static_assert(O % 2 == 0 && O >= 2 && O <= 30 && A % 2 == 0 && A >= 2 && A <= 32, "unsupported obs/act width");
    static_assert(OFF_STG + TM * stg_row_bytes(O) + 1024 <= SMEM_BYTES, "staging rows of this obs width do not fit SMEM_BYTES");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    const NetDims& d = a.d;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform by construction
    const int q = warp & 3, half = warp >> 2;                // TMEM lane quarter / column half
    const int row = q * 32 + lane;                           // sample row of this thread in the epilogues
    const int tower = blockIdx.y;                            // 0 = pi, 1 = V
    int prof_i = 0;
    bool prof_on = !PERSIST;
    UMMA_PROF();  // kernel entry

    uint8_t* sH1 = smem + OFF_H1;
    uint8_t* sH2 = smem + OFF_H2;
    uint8_t* sY = smem + OFF_Y;
    float* f32 = reinterpret_cast<float*>(smem + OFF_F32);
    // barD: the bulk copies of a tile's observation rows (128 arrivals + their bytes);
    // barA: the GEMM the next epilogue waits for; barB: the MMAs that read [dMU | dLS] out of Y (pi tower, before X' returns
    // there); barC: everything a tile issued (weight gradients included), waited once at the tile's end
    const uint32_t barA = sbase + OFF_BAR, barB = barA + 8, barC = barA + 16, barD = barA + 24;
    const uint8_t* sStg = smem + OFF_STG;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 32);
    uint8_t* sD2 = smem + OFF_D2;
    uint8_t* sD1 = smem + OFF_D1;
    const int ntiles = (a.count + TM - 1) / TM;

    // ---------------------------------------------------------------- inputs of the first tile (latency overlaps the setup)
    // Thread (gr = tid & 127, gh = tid >> 7) stages half of observation row gr; for column half 0, gr == row.
    const int gr = tid & 127, gh = tid >> 7;
    ObsStage<O> xin;
    long grow = 0;
    bool gvalid = false;
    float s_ret = 0.f, s_oldn = 0.f, s_oldv = 0.f;  // per-sample scalars (threads of column half 0)
    int cur_slot0 = PERSIST ? ep.rank_off : a.slot0;
    const float2* cur_mbstats = PERSIST ? ep.mbstats : a.mbstats;
    // input staging is split so that the two dependent global round trips (gather index -> rows) can be issued early and
    // consumed late: load_index, then load_rows (addresses need the index), the arithmetic happens at the tile's start
    float s_advd = 0.f;
    float2 s_st = make_float2(0.f, 1.f);
    int in_s0 = 0;
    auto load_index = [&](int tile) {
        in_s0 = cur_slot0 + tile * TM;
        const int nv = min(TM, cur_slot0 + a.count - in_s0);
        gvalid = tile < ntiles && gr < nv;
        grow = gvalid ? (long)(a.gather ? __ldg(a.gather + in_s0 + gr) : (in_s0 + gr)) : 0;
    };
    auto load_rows = [&]() {
        if (gh == 0) ObsStage<O>::issue(a.obs, grow, gvalid, sbase + OFF_STG + (uint32_t)gr * ObsStage<O>::ROW, barD);
        s_ret = s_oldn = s_oldv = s_advd = 0.f;
        if (gh == 0 && gvalid) {
            s_ret = __ldg(a.ret + grow);
            s_oldv = __ldg(a.val + grow);
            s_oldn = __ldg(a.nlp + grow);
            if (a.adv_direct) s_advd = __ldg(a.adv_direct + in_s0 + gr);
            else s_st = __ldg(cur_mbstats);
        }
    };
    auto load_inputs = [&](int tile) {
        load_index(tile);
        load_rows();
    };
    load_index(blockIdx.x);  // the rows follow once the mbarrier of their bulk copies exists

    // ---------------------------------------------------------------- one-time setup
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(barA));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(barB));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(barC));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(barD), "n"(TM));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // constant operand blocks: the V tower's dv rows (row 0 is rewritten per tile, rows 1..7 stay zero) and the ones block
    // (row 0 of each 8-row group = 2^PW_H = 256.0 = fp16 0x5C00, the scale of the activation blocks; rows 1..7 = 0;
    // ReLU: 2^PW_H_RELU = 1.0 = fp16 0x3C00)
    if (tower != 0)
        for (int i = tid; i < (int)ROW16_BLOCK / 16; i += NTH) reinterpret_cast<uint4*>(smem + OFF_WP)[i] = make_uint4(0, 0, 0, 0);
    if (tid < (int)ROW16_BLOCK / 16) {  // per 64-sample half: 128 chunks of 16 B, the first 8 are row 0
        const uint32_t v = ((tid & 127) < 8) ? (ACT == ACT_RELU ? 0x3C003C00u : 0x5C005C00u) : 0u;
        reinterpret_cast<uint4*>(smem + OFF_ONES)[tid] = make_uint4(v, v, v, v);
    }
    // persistent state: grid barrier generation, mailbox sequence number, Adam's beta powers (every CTA tracks them)
    GridBarrier bar{PERSIST ? ep.ra.bar_ctr : nullptr, 2u * gridDim.x, PERSIST ? *ep.ra.bar_gen : 0u};
    unsigned mseq = (PERSIST && ep.ra.mbox.world > 1) ? *ep.ra.mbox_seq : 0u;
    float b1p = PERSIST ? ep.ra.adam.bpow_in[0] : 0.f, b2p = PERSIST ? ep.ra.adam.bpow_in[1] : 0.f;
    unsigned sqseq = (PERSIST && ep.ra.sq_ll) ? *ep.ra.sq_seq : 0u;  // sequence number of the sum-of-squares LL exchange
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);

    // operand views
    const Operand opY_k = op_kmajor(sbase + OFF_Y, ACT_PIECE, TM);      // X' / dMU as A (m = sample)
    const Operand opY_mn = op_mnmajor(sbase + OFF_Y, ACT_PIECE, TM);    // X' / [dMU|dLS] reduced over samples
    const Operand opH1_k = op_kmajor(sbase + OFF_H1, ACT_PIECE, TM);
    const Operand opH1_mn = op_mnmajor(sbase + OFF_H1, ACT_PIECE, TM);
    const Operand opH2_k = op_kmajor(sbase + OFF_H2, ACT_PIECE, TM);
    const Operand opH2_mn = op_mnmajor(sbase + OFF_H2, ACT_PIECE, TM);
    const Operand opD2_k = op_kmajor(sbase + OFF_D2, ACT_PIECE, TM);
    const Operand opD2_mn = op_mnmajor(sbase + OFF_D2, ACT_PIECE, TM);
    const Operand opD1_mn = op_mnmajor(sbase + OFF_D1, ACT_PIECE, TM);
    const Operand opD1_k = op_kmajor(sbase + OFF_D1, ACT_PIECE, TM);    // [dMU | dLS] as A (pi tower, until dP1 takes the block)
    const Operand opW0_f = op_mnmajor(sbase + OFF_W0, W0_PIECE, 32);    // forward: B(n = out, k = in)
    const Operand opW1_f = op_mnmajor(sbase + OFF_W1, W1_PIECE, 64);
    const Operand opW1_b = op_kmajor(sbase + OFF_W1, W1_PIECE, 64);     // backward: B(n = in, k = out)
    const Operand opWP_f = op_mnmajor(sbase + OFF_WP, WP_PIECE, 64);
    const Operand opWP_b = op_kmajor(sbase + OFF_WP, WP_PIECE, 64);
    const Operand opDV = op_kmajor(sbase + OFF_WP, 0, 16);              // V tower: row 0 = dv_hi, row 8 = dv_lo over the samples
    const Operand opONES = op_kmajor(sbase + OFF_ONES, 0, 16);          // row 0 = ones, the rest zero
    const uint32_t id_f64 = make_idesc(128, 64, 0, 1);    // act(K-major) x W(MN view), N = 64
    const uint32_t id_f128 = make_idesc(128, 128, 0, 1);  // ... x [W_hi | W_lo], N = 128
    const uint32_t id_b128 = make_idesc(128, 128, 0, 0);  // dY(K-major) x [W_hi ; W_lo] (K-major view), N = 128
    const uint32_t id_f32 = make_idesc(128, 32, 0, 1);    // head forward, N = 32
    const uint32_t id_b64 = make_idesc(128, 64, 0, 0);    // dY(K-major) x W(K-major view)
    const uint32_t id_w128 = make_idesc(64, 128, 1, 1);   // dY_hi^T x [act_hi | act_lo] over samples
    const uint32_t id_w96 = make_idesc(64, 96, 1, 1);     // ... x [B_hi (64 columns) | B_lo (32 columns)]
    const uint32_t id_w64 = make_idesc(64, 64, 1, 1);     // dY_lo^T x act_hi
    const uint32_t id_w32 = make_idesc(64, 32, 1, 1);
    const uint32_t id_v16 = make_idesc(64, 16, 1, 0);     // V head: H2_hi^T x [dv_hi ; dv_lo] (K-major [16 x 128] B)
    const uint32_t id_v8 = make_idesc(64, 8, 1, 0);       // H2_lo^T x dv_hi
    const uint32_t id_s16 = make_idesc(128, 16, 1, 0);    // column sums: MN-major [A_hi ; A_lo] x K-major ones

    const float cr = a.sc->cliprange, vr = vf_clip_range(a.vf_mode, cr, a.sc->cliprange_vf);
    // the backward tensors (which carry the 1/B of the batch mean) are stored times a power of two so that they are O(1) as
    // fp16 operands (see the header); exponents are chosen per minibatch when the weights are staged
    int invB_exp;
    (void)frexpf(a.invB, &invB_exp);  // invB = m * 2^e, m in [0.5, 1)
    int k_w0 = 0, k_w1 = 0, k_hd = 0, n_s = 0;
    uint32_t phA = 0, phB = 0, phC = 0, phD = 0;
    float l_0, l_1, l_2, l_dbv;  // pi: pg, kl, clipfrac sums; V: vf sum, dbv (per minibatch)
    bool accw;
    float h1r[32], h2r[32];

    const int n_mb = PERSIST ? ep.M : 1;
#define LDW(p) (PERSIST ? __ldcg(p) : __ldg(p))  // the persistent kernel re-reads parameters that it updates itself
    for (int mb = 0; mb < n_mb; ++mb) {
        if (PERSIST) {
            prof_on = mb == 2;
            UMMA_PROF();  // start of the stamped minibatch
            UMMA_TL(0);
        }
        {
            // weights -> two fp16 pieces in the SWIZZLE_128B operand layout; all global loads are issued before the first use
            // (Measured and not kept: reading one of 4 / 16 / 64 replicas written by the Adam step instead of the one vector that 64 CTAs
            // fetch at the same moment — 7.07 / 7.08 / 7.27 ms per update against 7.22 on the same box, no hot-line effect worth the
            // stores.  Issuing the weight-gradient GEMMs from warps 1 and 2 behind warp 0's critical GEMM: the time moved from the
            // dH2 / dH1 waits to the wait at the tile's end — the tensor pipe needs ~45 cycles per tcgen05.mma of these shapes (152 per
            // tile), whoever issues them.  A ninth, issue-only warp: three warps on one SM sub-partition cap the kernel at 168 registers.)
            const float* P = a.params;
            const float* W1 = P + d.off[tower ? T_VF_FC1_W : T_PI_FC1_W];
            const float* W0 = P + d.off[tower ? T_VF_FC0_W : T_PI_FC0_W];
            const float* B0 = P + d.off[tower ? T_VF_FC0_B : T_PI_FC0_B];
            float4 w1v[2][2], w0v[2];
            float wpv[8];
            constexpr int WPI_LD = (HID * A + NTH - 1) / NTH;
            float wpf[WPI_LD];
            float b1 = 0.f, wv = 0.f, ls = 0.f, bh = 0.f, bv = 0.f;
            {
    #pragma unroll
            for (int i = 0; i < 2; ++i) {  // W1: 64 rows x 8 chunks = 512 tasks
                const int e = tid + NTH * i, r = e >> 3, j = e & 7;
                w1v[i][0] = LDW(reinterpret_cast<const float4*>(W1 + r * HID + 8 * j));
                w1v[i][1] = LDW(reinterpret_cast<const float4*>(W1 + r * HID + 8 * j + 4));
            }
            {  // W0': rows < O weights, row O bias, rows up to 31 zero: 32 rows x 8 chunks = 256 tasks
                const int r = tid >> 3, j = tid & 7;
                const float* src = r < O ? (W0 + r * HID + 8 * j) : (B0 + 8 * j);
                const bool nz = r <= O;
                w0v[0] = nz ? LDW(reinterpret_cast<const float4*>(src)) : make_float4(0.f, 0.f, 0.f, 0.f);
                w0v[1] = nz ? LDW(reinterpret_cast<const float4*>(src + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
    #pragma unroll
            for (int k = 0; k < 8; ++k) wpv[k] = 0.f;
            // Wpi [64 x A].  Persistent kernel: read as the flat run of 64 A floats it is (thread t takes t, t + 256, ...: a warp
            // instruction is 128 contiguous bytes) and dealt out through shared memory behind the maxima's barrier.  Each thread
            // fetching the 8 columns of its own chunk with scalar loads (the rows are only 4-byte aligned: the tensor starts at an
            // odd offset) is 8 L2 requests per sector from every one of the 64 pi CTAs at the same moment right after a grid
            // barrier: the parameters of the pi tower arrived 1.4 k cycles after those of the V tower (C3 train phase 6.44 ->
            // 6.14 ms).  The stand-alone kernel keeps the per-chunk loads: there the flat variant measured 16.4 us against 15.0.
            if (tower == 0) {
                if (PERSIST) {
    #pragma unroll
                    for (int i = 0; i < WPI_LD; ++i) {
                        const int e = tid + NTH * i;
                        wpf[i] = e < HID * A ? LDW(P + d.off[T_PI_W] + e) : 0.f;
                    }
                } else {
                    const int r = tid >> 2, j = tid & 3;
                    const float* src = P + d.off[T_PI_W] + r * A + 8 * j;
    #pragma unroll
                    for (int k = 0; k < 8; ++k) wpv[k] = (8 * j + k < A) ? LDW(src + k) : 0.f;
                }
            }
            if (tid < HID) {
                b1 = LDW(P + d.off[tower ? T_VF_FC1_B : T_PI_FC1_B] + tid);
                wv = LDW(P + d.off[T_VF_W] + tid);
            }
            if (tid < 32) {
                ls = tid < A ? LDW(P + d.off[T_LOGSTD] + tid) : 0.f;
                bh = tid < A ? LDW(P + d.off[T_PI_B] + tid) : 0.f;
                bv = LDW(P + d.off[T_VF_B]);
            }
            }
            // first tile of the launch: bulk copies of the gathered observation rows + the per-sample scalars, behind the parameter loads
            // (the gather index they need has been in flight since the kernel's entry; later minibatches issue theirs at barrier 1)
            if (mb == 0) load_rows();
            float* xw = reinterpret_cast<float*>(sD2);  // the idle dP2 block is the exchange buffer of Wpi (read back behind the maxima's barrier)
            if (PERSIST && tower == 0) {
    #pragma unroll
                for (int i = 0; i < WPI_LD; ++i)
                    if (tid + NTH * i < HID * A) xw[tid + NTH * i] = wpf[i];
            }
            // ---- block floating point: every weight matrix is stored times a power of two that brings its largest entry into
            // [1, 2) (exact in fp32; undone in the fp32 epilogues), so that both fp16 pieces of the entries that matter are
            // normal numbers whatever the scale of the matrix (the policy head starts at 1e-3, GRAPH:4843).  The same powers
            // of two ride along the backward pass (dH2 = dMU * (Wpi * 2^k)^T ...) and keep dP2 / dP1 at O(1) as well.
            {
                float mx[4] = {0.f, 0.f, 0.f, -3.0e38f};
                mx[0] = fmaxf(fmaxf(fmaxf(fabsf(w0v[0].x), fabsf(w0v[0].y)), fmaxf(fabsf(w0v[0].z), fabsf(w0v[0].w))),
                              fmaxf(fmaxf(fabsf(w0v[1].x), fabsf(w0v[1].y)), fmaxf(fabsf(w0v[1].z), fabsf(w0v[1].w))));
    #pragma unroll
                for (int i = 0; i < 2; ++i)
    #pragma unroll
                    for (int h = 0; h < 2; ++h)
                        mx[1] = fmaxf(mx[1], fmaxf(fmaxf(fabsf(w1v[i][h].x), fabsf(w1v[i][h].y)), fmaxf(fabsf(w1v[i][h].z), fabsf(w1v[i][h].w))));
                if (tower == 0) {
                    if (PERSIST) {
    #pragma unroll
                        for (int i = 0; i < WPI_LD; ++i) mx[2] = fmaxf(mx[2], fabsf(wpf[i]));  // (entries past the tensor's end are 0)
                    } else {
    #pragma unroll
                        for (int k = 0; k < 8; ++k) mx[2] = fmaxf(mx[2], fabsf(wpv[k]));
                    }
                } else if (tid < HID) {
                    mx[2] = fabsf(wv);
                }
                if (tid < A) mx[3] = -ls;  // max(-logstd) = -min(logstd)
    #pragma unroll
                for (int k = 0; k < 4; ++k)
    #pragma unroll
                    for (int o = 16; o > 0; o >>= 1) mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
                if (lane == 0) {
    #pragma unroll
                    for (int k = 0; k < 4; ++k) f32[F32_RED + warp * 4 + k] = mx[k];
                }
                __syncthreads();
                UMMA_PROF();  // parameters arrived, maxima exchanged
                mbar_wait(barD, phD); phD ^= 1;  // the observation rows of the first tile have landed (persistent kernel: a gradient step ago)
                xin.load(sStg, a.obs, grow, gvalid, gr, gh);
                if (PERSIST && tower == 0) {  // Wpi -> chunks 0..3 of every row (columns >= A zero): 256 tasks
                    const int r = tid >> 2, j = tid & 3;
    #pragma unroll
                    for (int k = 0; k < 8; ++k) wpv[k] = (8 * j + k < A) ? xw[r * A + 8 * j + k] : 0.f;
                }
    #pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float m = f32[F32_RED + k];
                    for (int w = 1; w < NTH / 32; ++w) m = fmaxf(m, f32[F32_RED + w * 4 + k]);
                    mx[k] = m;
                }
                auto pow2_to_unit = [](float m) {  // k with m * 2^k in [1, 2); 0 for a zero / non-finite matrix
                    const int ef = (__float_as_int(m) >> 23) & 0xff;  // m = f * 2^(ef - 126), f in [0.5, 1) (subnormals clamp below)
                    if (!(m > 0.f) || ef == 0xff) return 0;
                    return max(-24, min(24, 127 - ef));
                };
                k_w0 = pow2_to_unit(mx[0]) + PW_W;  // block = W * 2^k, max in [2^8, 2^9)
                k_w1 = pow2_to_unit(mx[1]) + PW_W;
                k_hd = pow2_to_unit(mx[2]) + PW_W;
                const int e_sig = ((__float_as_int(expf(-mx[3])) >> 23) & 0xff) - 126;  // sigma_min = f * 2^e, f in [0.5, 1)
                const int k_sig = max(-24, min(8, e_sig - 1));                           // 2^k_sig <= sigma_min
                // backward scale S = 2^n_s: pi  S * invB / sigma_min in (4, 16];  V  S * invB in [32, 64)
                n_s = tower == 0 ? (-invB_exp + k_sig + 4) : (-invB_exp + 6);
            }
            const float s_w0 = pow2f(k_w0), s_w1 = pow2f(k_w1), s_hd = pow2f(k_hd);
            // ---- consume
    #pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int e = tid + NTH * i, r = e >> 3, j = e & 7;
                const float x[8] = {w1v[i][0].x * s_w1, w1v[i][0].y * s_w1, w1v[i][0].z * s_w1, w1v[i][0].w * s_w1,
                                    w1v[i][1].x * s_w1, w1v[i][1].y * s_w1, w1v[i][1].z * s_w1, w1v[i][1].w * s_w1};
                store_chunk(smem + OFF_W1, W1_PIECE, chunk_off(r, j), x);
            }
            {
                const int r = tid >> 3, j = tid & 7;
                const float x[8] = {w0v[0].x * s_w0, w0v[0].y * s_w0, w0v[0].z * s_w0, w0v[0].w * s_w0,
                                    w0v[1].x * s_w0, w0v[1].y * s_w0, w0v[1].z * s_w0, w0v[1].w * s_w0};
                store_chunk(smem + OFF_W0, W0_PIECE, chunk_off(r, j), x);
            }
            if (tower == 0) {
                const int r = tid >> 2, j = tid & 3;
    #pragma unroll
                for (int k = 0; k < 8; ++k) wpv[k] *= s_hd;
                store_chunk(smem + OFF_WP, WP_PIECE, chunk_off(r, j), wpv);
            }
            if (tid < HID) {
                f32[F32_B1 + tid] = b1;
                f32[F32_WV + tid] = wv;
            }
            if (tid < 32) {
                f32[F32_BH + tid] = bh;
                f32[F32_LS + tid] = ls;
                f32[F32_SD + tid] = expf(ls);
                f32[F32_ISD + tid] = 1.f / expf(ls);
                const float sl = warp_sum(ls);  // lanes >= A contribute 0
                if (tid == 0) {
                    f32[F32_MISC + 0] = bv;
                    f32[F32_MISC + 1] = sl;
                }
            }
        }
        UMMA_PROF();  // weight blocks written
        // epilogue factors of this minibatch (exact powers of two)
        constexpr int PWH = pw_h<ACT>();
        const float u_w0 = pow2f(-k_w0 - PW_X), u_w1 = pow2f(-k_w1 - PWH), u_hd = pow2f(-k_hd - PWH);
        const float s_hd_v = pow2f(k_hd - PW_W);                 // V tower: dP2 = dv * (wv 2^kh) (1 - g2^2), kh = k_hd - PW_W
        const float S_b = pow2f(n_s);                            // backward tensors are stored times S_b
        constexpr float RENORM = 1.0f / (float)(1 << PW_W);      // after a product with a weight block (W * 2^(kh + PW_W))
        constexpr float H_SCALE = (float)(1 << PWH);             // activation blocks hold H * 2^PWH
        const float un_hd = pow2f(-n_s - PWH);                                // dWpi, column sums (ones = 2^PWH), dWv
        const float un_w1 = pow2f(-n_s - (k_hd - PW_W) - PWH);                 // dW1, db1
        const float un_w0 = pow2f(-n_s - (k_hd - PW_W) - (k_w1 - PW_W) - PW_X);  // dW0' (bias column: the ones of X' are 2^PW_X)
        xin.store(sY, gr, gh);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        UMMA_PROF();  // setup done, X' of the first tile staged
        UMMA_TL(1);
        l_0 = l_1 = l_2 = l_dbv = 0.f;
        accw = false;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // inputs of this tile (the registers are refilled with the next tile's before the end of the loop);
        // gr == row for both column halves, so grow is the rollout row of this thread's sample
        const float c_ret = s_ret, c_oldn = s_oldn, c_oldv = s_oldv;
        // advs = (returns - values - mean) / (sqrt(var) + 1e-8)  (ppo2.hpp:401-406)
        const float c_adv = (gh == 0 && gvalid) ? (a.adv_direct ? s_advd : __fdiv_rn(__fsub_rn(__fsub_rn(s_ret, s_oldv), s_st.x), s_st.y)) : 0.f;
        const long c_grow = grow;
        const bool valid = gvalid;

        // ---- layer 0: Z1 = X' * W0'  (bias through the ones column)
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_gemm_wide<2>(tmem + ACC_WORK, opY_k, opW0_f, id_f128, id_f64);
                umma_commit(barA);
            }
            __syncwarp();
        }
        mbar_wait(barA, phA); phA ^= 1;
        tc_fence_after();
        UMMA_PROF();
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {  // 16 columns at a time
            float v[16];
            tmem_ld16_sum(tlane + ACC_WORK + 32 * half + 16 * hh, tlane + ACC_WORK_C + 32 * half + 16 * hh, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) h1r[16 * hh + j] = act_epi<ACT>(v[j] * u_w0);
        }
        store_row32(sH1, row, half, h1r, H_SCALE);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        UMMA_PROF();

        // ---- layer 1: Z2 = H1 * W1
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_gemm_wide<4>(tmem + ACC_WORK, opH1_k, opW1_f, id_f128, id_f64);
                umma_commit(barA);
            }
            __syncwarp();
        }
        // pi tower: the action row of the sample (both column halves need all of it for the loss stage)
        float2 act2[A / 2];
        if (tower == 0) {
            const float2* src = reinterpret_cast<const float2*>(a.act + c_grow * A);
#pragma unroll
            for (int i = 0; i < A / 2; ++i) act2[i] = valid ? __ldg(src + i) : make_float2(0.f, 0.f);
        }
        mbar_wait(barA, phA); phA ^= 1;
        tc_fence_after();
        UMMA_PROF();
        {
            float pv = 0.f;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {  // 16 columns at a time
                float v[16];
                tmem_ld16_sum(tlane + ACC_WORK + 32 * half + 16 * hh, tlane + ACC_WORK_C + 32 * half + 16 * hh, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int jj = 16 * hh + j;
                    h2r[jj] = act_epi<ACT>(fmaf(v[j], u_w1, f32[F32_B1 + 32 * half + jj]));
                    pv = fmaf(h2r[jj], f32[F32_WV + 32 * half + jj], pv);
                }
            }
            store_row32(sH2, row, half, h2r, H_SCALE);
            if (tower == 1) f32[F32_PV + half * TM + row] = pv;
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        UMMA_PROF();

        if (tower == 0) {
            // ---- pi head: MU = H2 * Wpi
            if (warp == 0) {
                tc_fence_after();
                if (elect_one()) {
                    issue_gemm_wide<4>(tmem + ACC_WORK, opH2_k, opWP_f, id_f128, id_f32);
                    umma_commit(barA);
                }
                __syncwarp();
            }
            mbar_wait(barA, phA); phA ^= 1;
            tc_fence_after();
            UMMA_PROF();
            {
                // loss stage (GRAPH:9428-11446).  Both column halves evaluate the sample's scalars; half 0 then emits
                // dL/dmu (columns 0..31 of Y), half 1 the logstd contributions (columns 32..63) — both times S_b.
                float z[32];
                float ss = 0.f;
                {
                    float mu[32];
                    tmem_ld32_sum(tlane + ACC_WORK, tlane + ACC_WORK_C, mu);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        z[j] = 0.f;
                        if (j < A) {
                            const float aj = (j & 1) ? act2[j >> 1].y : act2[j >> 1].x;
                            z[j] = (aj - fmaf(mu[j], u_hd, f32[F32_BH + j])) * f32[F32_ISD + j];  // (a - mu) / sigma
                            ss += z[j] * z[j];
                        }
                    }
                }
                float g_nlp = 0.f;
                // the scalars live in the threads of column half 0; half 1 gets them through shared memory
                if (half == 0) {
                    f32[F32_PV + row] = c_adv;
                    f32[F32_PV + TM + row] = c_oldn;
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                const float adv = f32[F32_PV + row], oldn = f32[F32_PV + TM + row];
                if (valid) {
                    const float nlp = gauss_neglogp(ss, f32[F32_MISC + 1], A);
                    g_nlp = pg_term(adv, oldn, nlp, cr, a.invB).g_nlp * S_b;
                    if (half == 0) {
                        // the same pg_term (merged with the one above), so that its loss terms are evaluated in this branch
                        // only: one call ahead of the branch was tried and changes this kernel's instruction mix
                        const PgTerm t = pg_term(adv, oldn, nlp, cr, a.invB);
                        l_0 += t.pg;
                        l_1 += t.kl;
                        l_2 += t.cf;
                    }
                }
                if (half == 0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) z[j] = (j < A) ? g_nlp * (-z[j] * f32[F32_ISD + j]) : 0.f;  // dL/dmu
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) z[j] = (j < A) ? g_nlp * (1.f - z[j] * z[j]) : 0.f;  // d nlp / d logstd_j
                }
                store_row32(sD1, row, half, z);  // (the dP1 block is free until the end of the tile; X' stays in its own)
            }
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            UMMA_PROF();
            // ---- backward through the head: dH2 = dMU * Wpi^T (the epilogue below waits for it); behind it, off the
            // critical path: dWpi += H2^T * dMU ; column sums of [dMU | dLS]
            if (warp == 0) {
                tc_fence_after();
                if (elect_one()) {
                    issue_gemm_wide<2>(tmem + ACC_WORK, opD1_k, opWP_b, id_b128, id_b64);
                    umma_commit(barA);
                    issue_gemm_dw<8>(tmem + ACC_DWP, 64u, opH2_mn, opD1_mn, id_w96, id_w32, accw);
                    issue_gemm_stacked<8>(tmem + ACC_CS, opD1_mn, opONES, id_s16, accw);
                    umma_commit(barB);
                }
                __syncwarp();
            }
            mbar_wait(barA, phA); phA ^= 1;
            tc_fence_after();
            UMMA_PROF();
            float v[32];
            tmem_ld32_sum(tlane + ACC_WORK + 32 * half, tlane + ACC_WORK_C + 32 * half, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= act_dfac<ACT>(h2r[j]) * RENORM;
            store_row32(sD2, row, half, v);  // dP2 (its own block: the dWpi GEMM may still be reading H2)
        } else {
            // ---- V head (GRAPH:10213-10400): value, clipped value loss and dL/dv on the CUDA cores
            if (half == 0) {
                float dv = 0.f;
                if (valid) {
                    const float v = (f32[F32_PV + row] + f32[F32_PV + TM + row]) + f32[F32_MISC + 0];
                    l_0 += value_loss_term(a.vf_mode, vr, v, c_oldv, c_ret, a.vf_coef, a.invB, dv);
                    l_dbv += dv;
                    dv *= S_b;  // as an operand: times S
                }
                f32[F32_DV + row] = dv;
                uint32_t p0, p1;
                split_pair(dv, 0.f, p0, p1);
                const uint32_t o = (uint32_t)((row >> 6) * 2048 + (((row & 63) >> 3) << 4) + (row & 7) * 2);  // row 0 (hi) / row 8 (lo) of the [16 x 128] block
                *reinterpret_cast<uint16_t*>(smem + OFF_WP + o) = (uint16_t)p0;
                *reinterpret_cast<uint16_t*>(smem + OFF_WP + 1024 + o) = (uint16_t)p1;
            }
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            UMMA_PROF();
            // dWv += H2^T * dv (off the critical path; collected by barC)
            if (warp == 0) {
                tc_fence_after();
                if (elect_one()) issue_gemm_dw<8>(tmem + ACC_DWP, 8u, opH2_mn, opDV, id_v16, id_v8, accw);
                __syncwarp();
            }
            const float dvr = f32[F32_DV + row];
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = dvr * (f32[F32_WV + 32 * half + j] * s_hd_v) * act_dfac<ACT>(h2r[j]);
            UMMA_PROF();
            store_row32(sD2, row, half, v);  // dP2
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        UMMA_PROF();

        // ---- hidden layer 1 backward: dH1 = dP2 * W1^T (waited for); behind it dW1^T += dP2^T * H1 ; db1 += colsum(dP2)
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_gemm_wide<4>(tmem + ACC_WORK, opD2_k, opW1_b, id_b128, id_b64);
                umma_commit(barA);
                issue_gemm_dw<8>(tmem + ACC_DW1, 64u, opD2_mn, opH1_mn, id_w128, id_w64, accw);
                issue_gemm_stacked<8>(tmem + ACC_DB1, opD2_mn, opONES, id_s16, accw);
            }
            __syncwarp();
        }
        mbar_wait(barA, phA); phA ^= 1;
        // pi tower: dP1 goes where [dMU | dLS] sat; barB says the MMAs that read those (issued two phases ago) have completed
        if (tower == 0) {
            mbar_wait(barB, phB); phB ^= 1;
        }
        tc_fence_after();
        UMMA_PROF();
        {
            float v[32];
            tmem_ld32_sum(tlane + ACC_WORK + 32 * half, tlane + ACC_WORK_C + 32 * half, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= act_dfac<ACT>(h1r[j]) * RENORM;
            store_row32(sD1, row, half, v);  // dP1
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        UMMA_PROF();
        // ---- layer 0 backward: dW0'^T += dP1^T * X'   (column O of the result is the bias gradient)
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_gemm_dw<8>(tmem + ACC_DW0, 64u, opD1_mn, opY_mn, id_w96, id_w32, accw);
                umma_commit(barC);
            }
            __syncwarp();
        }
        accw = true;
        const bool more = tile + (int)gridDim.x < ntiles;
        if (more) load_inputs(tile + gridDim.x);
        mbar_wait(barC, phC); phC ^= 1;  // every MMA of this tile has completed: all operand blocks are free again
        tc_fence_after();
        UMMA_PROF();
        if (more) {
            mbar_wait(barD, phD); phD ^= 1;
            xin.load(sStg, a.obs, grow, gvalid, gr, gh);
            xin.store(sY, gr, gh);
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
        }
    }

    if (PERSIST && mb + 1 < n_mb) {  // gather index of the next minibatch's first tile: in flight during the flush
        cur_slot0 = (mb + 1) * ep.B + ep.rank_off;
        cur_mbstats = ep.mbstats + mb + 1;
        load_index(blockIdx.x);
    }
    UMMA_TL(2);  // tiles done
    // ---------------------------------------------------------------- flush the weight gradients of this CTA
    // (Gathering the entries in shared memory in slab order and storing them as float4 from 32 lanes instead of 4-byte stores from the
    // 16 lanes that hold an accumulator row was measured: 3.4 k -> 4.0 k cycles; the accumulator reads and the un-scaling are the cost.)
    float* my = a.partial + (size_t)blockIdx.x * a.PS;
    auto put = [&](int col, float val) { my[col] = val; };
    // M = 64 accumulators: row r of D sits in TMEM lane 32 * (r >> 4) + (r & 15); the column sums (M = 128: row r in lane r) have their
    // lo parts in the upper lane quarters: those warps park them in shared memory for the warps that own the rows
    const int r64 = q * 16 + lane;
    const bool has = lane < 16;
    float* S4 = f32 + F32_PV;  // [db1 lo 64 | head lo 64] (the per-sample scratch of the tiles is free)
    if (!accw) {  // no tile for this CTA: write zeros
        if (tower == 0) {
            for (int i = tid; i < d.H1 * O + d.H1; i += NTH) put(d.off[T_PI_FC0_W] + i, 0.f);
            for (int i = tid; i < d.H1 * d.H2 + d.H2; i += NTH) put(d.off[T_PI_FC1_W] + i, 0.f);
            for (int i = tid; i < d.H2 * A + 2 * A; i += NTH) put(d.off[T_PI_W] + i, 0.f);
        } else {
            for (int i = tid; i < d.H1 * O + d.H1; i += NTH) put(d.off[T_VF_FC0_W] + i, 0.f);
            for (int i = tid; i < d.H1 * d.H2 + d.H2; i += NTH) put(d.off[T_VF_FC1_W] + i, 0.f);
            for (int i = tid; i < d.H2; i += NTH) put(d.off[T_VF_W] + i, 0.f);  // vf/b comes with the loss sums below
        }
    } else {
        float v[32];
        uint32_t r8[8];
        if (half == 1 && q >= 2) {  // lo parts of the column sums (rows 64 + 32 (q - 2) + lane)
            PPO_TMEM_LD8(tlane + ACC_DB1, r8);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            S4[(q - 2) * 32 + lane] = __uint_as_float(r8[0]);
            if (tower == 0) {
                PPO_TMEM_LD8(tlane + ACC_CS, r8);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                S4[64 + (q - 2) * 32 + lane] = __uint_as_float(r8[0]);
            }
        }
        // dW1^T[j][k] -> W1[k][j]
        tmem_ld32_sum(tlane + ACC_DW1 + 32 * half, tlane + ACC_DW1 + 64 + 32 * half, v);
        if (has) {
            const int g = d.off[tower ? T_VF_FC1_W : T_PI_FC1_W];
#pragma unroll
            for (int k = 0; k < 32; ++k) put(g + (32 * half + k) * HID + r64, v[k] * un_w1);
        }
        if (half == 0) {
            // dW0'^T[j][k]: k < O -> W0[k][j], k == O -> b0[j]
            tmem_ld32_sum(tlane + ACC_DW0, tlane + ACC_DW0 + 64, v);
            if (has) {
                const int g = d.off[tower ? T_VF_FC0_W : T_PI_FC0_W], gb = d.off[tower ? T_VF_FC0_B : T_PI_FC0_B];
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    if (k < O) put(g + k * HID + r64, v[k] * un_w0);
                    else if (k == O) put(gb + r64, v[k] * un_w0);
                }
            }
        } else {
            if (tower == 0) {
                // dWpi[k][j]
                tmem_ld32_sum(tlane + ACC_DWP, tlane + ACC_DWP + 64, v);
                if (has) {
                    const int g = d.off[T_PI_W] + r64 * A;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < A) put(g + j, v[j] * un_hd);
                }
            } else {
                uint32_t r2[8];
                PPO_TMEM_LD8(tlane + ACC_DWP, r8);      // x dv_hi
                PPO_TMEM_LD8(tlane + ACC_DWP + 8, r2);  // x dv_lo, + H2_lo x dv_hi
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (has) put(d.off[T_VF_W] + r64, (__uint_as_float(r8[0]) + __uint_as_float(r2[0])) * un_hd);
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the four warps of this column half: the lo sums are parked
            if (q < 2) {  // hi parts: row 32 q + lane
                const int rr = q * 32 + lane;
                PPO_TMEM_LD8(tlane + ACC_DB1, r8);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                put(d.off[tower ? T_VF_FC1_B : T_PI_FC1_B] + rr, (__uint_as_float(r8[0]) + S4[rr]) * un_w1);
                if (tower == 0) {
                    // column sums of [dMU | dLS]: rows < A -> dbpi, rows 32 .. 32 + A -> dlogstd
                    PPO_TMEM_LD8(tlane + ACC_CS, r8);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    const float cs = (__uint_as_float(r8[0]) + S4[64 + rr]) * un_hd;
                    if (rr < A) put(d.off[T_PI_B] + rr, cs);
                    // d(-ent_coef*entropy)/dlogstd_j = -ent_coef, once (a.ent_coef is pre-divided by the number of ranks)
                    if (rr >= 32 && rr < 32 + A) put(d.off[T_LOGSTD] + rr - 32, cs - (blockIdx.x == 0 ? a.ent_coef : 0.f));
                }
            }
        }
    }
    // ---- loss sums
    {
        float v4[4] = {l_0, l_1, l_2, l_dbv};
#pragma unroll
        for (int k = 0; k < 4; ++k) v4[k] = warp_sum(v4[k]);
        __syncthreads();
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) f32[F32_RED + warp * 4 + k] = v4[k];
        }
        __syncthreads();
        if (tid == 0) {
            float t[4] = {0.f, 0.f, 0.f, 0.f};
            for (int w = 0; w < NTH / 32; ++w)
                for (int k = 0; k < 4; ++k) t[k] += f32[F32_RED + w * 4 + k];
            const int Lp = d.P;
            if (tower == 0) {
                put(Lp + L_PG, t[0]); put(Lp + L_KL, t[1]); put(Lp + L_CLIP, t[2]);
                float ent = 0.f;
                if (blockIdx.x == 0) ent = box_entropy([&](int j) { return f32[F32_LS + j]; }, A);
                put(Lp + L_ENT, ent);
                put(Lp + 5, 0.f); put(Lp + 6, 0.f); put(Lp + 7, 0.f);
            } else {
                put(Lp + L_VF, t[0]);
                put(d.off[T_VF_B], accw ? t[3] : 0.f);
            }
        }
    }
    UMMA_PROF();
        if (PERSIST) {
            // slabs complete -> reduce (+ allreduce) -> global norm -> Adam -> parameters visible to every CTA
            tc_fence_before();  // orders this minibatch's tcgen05.ld before the next minibatch's MMAs (barriers below)
            UMMA_TL(3);  // flushed
            bar.arrive();
            // next minibatch's first tile (index issued before the flush): 128 bulk copies are ~0.3 us of issue, so they go out
            // after this CTA's arrival at the barrier, while the others still come in, and land during the gradient step
            if (mb + 1 < n_mb) load_rows();
            bar.wait();
            UMMA_PROF();  // barrier 1 passed
            UMMA_TL(4);
            ++mseq;
            // (the combine buffer of the gradient step is the H1 block: every MMA that read it has completed, the next writer is the
            // H1 epilogue of the next minibatch, two grid barriers away)
            reduce_adam_device<true>(ep.ra, (int)(blockIdx.y * gridDim.x + blockIdx.x), (int)(2 * gridDim.x), bar, mseq, b1p, b2p,
                                     ep.loss_rows + (size_t)mb * 5,
                                     (a.prof && blockIdx.x == 0 && mb == 2) ? a.prof + 160 + tower * 8 : nullptr, ++sqseq,
                                     reinterpret_cast<float*>(sH1));
            b1p = __fmul_rn(b1p, ep.ra.adam.beta1);
            b2p = __fmul_rn(b2p, ep.ra.adam.beta2);
            UMMA_PROF();  // reduce + partials + Adam done
            UMMA_TL(5);
            bar.sync();
            tc_fence_after();
            UMMA_PROF();  // barrier 3 passed
            UMMA_TL(6);
        }
    }  // minibatches
#undef LDW
    if (PERSIST && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) {
        ep.ra.adam.bpow_out[0] = b1p;
        ep.ra.adam.bpow_out[1] = b2p;
        *ep.ra.bar_gen = bar.gen;
        if (ep.ra.mbox.world > 1) *ep.ra.mbox_seq = mseq;
        if (ep.ra.sq_ll) *ep.ra.sq_seq = sqseq;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
}
#undef UMMA_PROF
#undef UMMA_TL

}  // namespace umma
}  // namespace ppo
