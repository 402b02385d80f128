// "W family": layer-wise tcgen05 train path for wide hidden layers (H1 == H2 == H, H a multiple of 128; [256,256] is
// BASELINE.json's C4 net).  Same math as train_tile_kernel (loss / autodiff sub-graph of PPO2::_train_step,
// ppo2/ppo2.hpp:430-470, GRAPH:6889-23699; tie-breaking rules of SURVEY §3.5b).
//
// Why layer-wise: one 128-sample tile of a 256-wide activation is 192 KB as a split-bf16 MMA operand, so the fused
// one-CTA-per-tile scheme of the U family ([64,64], kernels_umma.cuh) cannot keep two activations plus the weights in
// shared memory, and a 256 x 256 weight gradient is all of TMEM.  Here every layer of forward and backward is one
// GEMM over the whole minibatch; activations travel between the GEMMs as *operand images* in global memory (L2 /
// HBM): the bytes are already laid out as the SWIZZLE_128B shared-memory blocks the tensor core reads, two fp16
// pieces per fp32 value (x = hi + lo, three products per fp32 product, block floating point exactly as in the U family:
// every weight matrix times a power of two that brings its largest entry into [1, 2), the backward tensors times a power
// of two S, all undone in fp32 epilogues — see kernels_umma.cuh; round 1 used three bf16 pieces and six products: twice
// the tensor-pipe time and 1.5x the operand traffic), so a GEMM stage is
// filled by plain bulk copies (cp.async.bulk, the non-tensor TMA path) with no address arithmetic per element.
//   image of a [rows x 64k] matrix: [tile of 128 rows][piece 0..1][column block of 64][16 KB block]
//   block: row r, 16-byte chunk j (8 bf16) at (r >> 3) * 1024 + (r & 7) * 128 + ((j ^ (r & 7)) << 4)
// The same block serves as K-major operand (forward: act x W, backward: dY x W^T) and as MN-major operand
// (weight gradients: act^T x dY reduced over the samples).
//
// Kernels (one minibatch = 9 launches + reduce + Adam, all captured in the update's CUDA graph):
//   wide_prep_weights_kernel   fp32 parameters -> weight images (W0' with the bias as an extra input row, W1, heads)
//   wide_gather_kernel         minibatch rows of the rollout buffer -> X' image (obs | 1)
//   wgemm_kernel               persistent, warp-specialised (bulk-copy producer / MMA issuer / 8 epilogue warps),
//                              2-stage shared-memory ring, double-buffered TMEM accumulators (main + cross product)
//       mode FWD   C = A(K-major image) x W(MN-major view)      Z1, Z2, head
//       mode BWD   C = A(K-major image) x W^T(K-major view)     dH2, dH1
//       mode DW    slab[kgroup] = A^T(MN-major) x B(MN-major) over a range of samples (split-K): dW1, dWhead, dW0'
//       epilogues: fp32 result | H = tanh(acc + b) -> image | dP = acc * (1 - H^2) -> image + column sums (bias gradient)
//                  | heads -> policy / value losses per sample, dL/dmu, dL/dlogstd terms, dL/dv -> dY image + per-warp sums
//   wide_fold_kernel           per-tile column / loss sums -> slab 0 (zeros in the other slabs)
// The slabs then go through the same reduce (+ cross-GPU exchange) + global-norm clip + Adam kernel as every family.
#pragma once
#include "kernels_umma.cuh"

namespace ppo {
namespace wide {

using umma::chunk_off;
using umma::smem_u32;

constexpr int TM = 128;            // samples per tile
constexpr int GEMM_NTH = 320;      // warp 0: producer, warp 1: MMA issuer, warps 2..9: epilogue (two per TMEM lane quarter)
constexpr uint32_t BLK16 = 16384;  // [128 x 64] bf16 block
constexpr uint32_t BLK8 = 8192;    // [64 x 64]
constexpr int NPW = 2;             // fp16 pieces per fp32 value
constexpr uint32_t STAGE_A = NPW * BLK16, STAGE_B = NPW * BLK16, STAGE = STAGE_A + STAGE_B;
constexpr int NSTAGE = 3;          // 64 KB per stage
// per-tower scale table (floats, written by wide_prep_weights_kernel every time the weight images are rebuilt)
constexpr int SC_STRIDE = 16;
enum { SC_S_W0 = 0, SC_U_W0, SC_S_W1, SC_U_W1, SC_S_HD, SC_U_HD, SC_S_B, SC_UN_HD, SC_UN_W1, SC_UN_W0, SC_UNC_B1, SC_UNC_B0, SC_COUNT };
// Operand images sit high in fp16's range: an fp16 lo piece below 2^-14 is subnormal (absolute step 2^-24), so a value
// whose hi piece is below ~0.25 loses relative accuracy — with matrices scaled to a maximum of 1..2 most entries sat
// there and a cancelling sum over 5000 samples (a bias gradient) came out at 1.07e-5.  Powers of two again:
//   weights  max in [2^8, 2^9)   activations H * 2^8   observations X' * 2^5 (|obs| <= clip_obs = 10)
//   back-propagated tensors times S (pi: S / (B sigma_min) in (4, 16], V: S / B in [32, 64)), renormalised by 2^-8 after
//   every product with a weight image.  fp16 overflows at 65504: headroom of 2^6 .. 2^7 over the typical magnitude.
// ReLU activations are unbounded: their images hold H * 2^PW_H_RELU = H (umma::pw_h), exact as two pieces for H >= 2^-3,
// an absolute error <= 2^-25 below that, H up to 65504; beyond it inf, a non-finite global norm and a NaN update.
constexpr int PW_W = 8, PW_X = 5;
using umma::pw_h;
constexpr uint32_t EPI_STAGE = 4096;  // per epilogue warp: 32 rows x 128 B of an image block, staged for a bulk store
constexpr uint32_t GEMM_SMEM = NSTAGE * STAGE + 128 + 8 * EPI_STAGE + 1024;  // + barriers + epilogue staging + alignment slack
constexpr int COLPART = 64;        // floats per tile written by the loss kernel
constexpr int CP_DBPI = 0, CP_DLS = 18, CP_DBV = 36, CP_PG = 37, CP_VF = 38, CP_KL = 39, CP_CLIP = 40;

// byte geometry of the images for hidden width H and NT tiles
struct Geom {
    int H, nb, NT, Bpad;
    size_t act_piece, act_tile, act_tower;  // activation images [tower][tile][piece][nb][16 KB]
    size_t x_tile;                          // X' image [tile][piece][16 KB]
    size_t dy_tile, dy_tower;               // dY image [tower][tile][piece][16 KB]
    size_t w0_piece, w0_tower;              // [tower][piece][nb][4 KB]  (32 input rows x 64 outputs)
    size_t w1_piece, w1_tower;              // [tower][piece][co][ri][8 KB]
    size_t wh_piece, wh_tower;              // [tower][piece][ri][8 KB]  (64 inputs x 64 head columns)
    size_t z_tower, mu_tower;               // fp32 results, in floats
    int cap;
    // ntiles tiles in use; the tower strides come from the allocation's capacity, so that a region never changes owner
    __host__ void init(int h, int ntiles, int cap_tiles) {
        H = h; nb = h / 64; NT = ntiles; Bpad = ntiles * TM;
        act_piece = (size_t)nb * BLK16; act_tile = NPW * act_piece; act_tower = (size_t)cap_tiles * act_tile;
        x_tile = NPW * (size_t)BLK16;
        dy_tile = NPW * (size_t)BLK16; dy_tower = (size_t)cap_tiles * dy_tile;
        w0_piece = (size_t)nb * 4096; w0_tower = NPW * w0_piece;
        w1_piece = (size_t)nb * nb * BLK8; w1_tower = NPW * w1_piece;
        wh_piece = (size_t)nb * BLK8; wh_tower = NPW * wh_piece;
        z_tower = (size_t)cap_tiles * TM * h;
        mu_tower = (size_t)cap_tiles * TM * 64;
        cap = cap_tiles;
    }
};

enum { MODE_FWD = 0, MODE_BWD = 1, MODE_DW = 2 };
enum { DW_W1 = 0, DW_HEAD = 1, DW_W0 = 2 };
enum { EPI_STORE = 0, EPI_ACT = 1, EPI_DACT = 2, EPI_LOSS = 3 };  // fp32 result | act(acc + b) -> image | acc * act'(H) -> image (+ column sums) | heads -> losses -> dY image

struct DwProb {
    const uint8_t* A; size_t a_tower, a_tile, a_piece;  // M side: image whose features become the rows of the result
    const uint8_t* B; size_t b_tower, b_tile, b_piece;  // N side
    int m_blks, n_blks, n_tile, kind, task0, ntasks;
};

struct GemmArgs {
    int mode, ntasks;
    // FWD / BWD
    const uint8_t* A; size_t a_tower, a_tile, a_piece;
    int kblocks, ksteps;
    const uint8_t* B; size_t b_tower, b_piece, b_kb, b_g;
    uint32_t b_bytes;
    int n_tile, n_blks, m_tiles;
    float* C; size_t c_tower; int ldc;
    // fused epilogues (FWD / BWD): activation images [tower][tile][piece][nb][16 KB]
    int epi;
    const float* P; int bias_off[2];          // EPI_ACT: bias per tower (offset into P, or -1)
    uint8_t* img_out;
    size_t img_tower, img_tile, img_piece;
    float* colsum; int cap;                   // EPI_DACT: [tower][tile * 4 + lane quarter][H] partial column sums, or NULL
    float* gbuf;                              // act'(H) (1 - H^2 / H > 0) as fp32, [tower][tile][column][128 rows]: written by EPI_ACT, read by EPI_DACT
    TrainArgs ta;                             // EPI_LOSS: the minibatch (gather list, rollout buffers, advantage statistics)
    uint8_t* dY; size_t dy_tower, dy_tile;    // EPI_LOSS: head gradients image [tower][tile][piece][16 KB]
    float* colloss;                           // EPI_LOSS: [tile * 4 + lane quarter][COLPART] per-warp sums
    const float* sc;                          // per-tower scale table (SC_*), block floating point of the fp16 operands
    int sc_fwd;                               // FWD / EPI_STORE: table entry that undoes the weight scaling of this GEMM (SC_U_*)
    // DW
    DwProb dw[3];
    int n_dw, KG, HT;     // split-K groups, half tiles (64 samples) in the minibatch
    float* partial; int PS;
    int H, O, A_dim;
    int off_w1[2], off_w0[2], off_b0[2], off_piw, off_vfw;
};

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }

// mbarrier wait with a time bound: a pipeline bug must end in an error, not in a hung GPU
__device__ __forceinline__ void mbar_wait_b(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    long long t0 = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (!done && (spin & 0xfffu) == 0xfffu) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000LL) __trap();  // ~2 s
        }
    }
}

// x[c] summed over the 32 lanes, for 32 columns at once (31 shuffles): lane l returns the sum of column l.  Fixed order.
__device__ __forceinline__ float colsum32(float (&x)[32], int lane) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < o; ++i) {
            const float send = up ? x[i] : x[i + o];
            const float keep = up ? x[i + o] : x[i];
            x[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    return x[0];
}

struct Task {
    int tower, m, n, kg, prob;
};

__device__ __forceinline__ Task decode_task(const GemmArgs& g, int t) {
    Task k{};
    if (g.mode != MODE_DW) {
        k.n = t % g.n_blks; t /= g.n_blks;
        k.m = t % g.m_tiles; t /= g.m_tiles;
        k.tower = t;
    } else {
        int p = 0;
        while (p + 1 < g.n_dw && t >= g.dw[p + 1].task0) ++p;
        const DwProb& P = g.dw[p];
        t -= P.task0;
        k.prob = p;
        k.kg = t % g.KG; t /= g.KG;
        k.n = t % P.n_blks; t /= P.n_blks;
        k.m = t % P.m_blks; t /= P.m_blks;
        k.tower = t;
    }
    return k;
}

template <int ACT>
__global__ void __launch_bounds__(GEMM_NTH, 1) wgemm_kernel(const GemmArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar0 = sbase + NSTAGE * STAGE;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + NSTAGE * STAGE + 112);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
#define BAR_FULL(s) (bar0 + 8u * (s))
#define BAR_EMPTY(s) (bar0 + 32u + 8u * (s))
#define BAR_ACCFULL(b) (bar0 + 64u + 8u * (b))
#define BAR_ACCEMPTY(b) (bar0 + 80u + 8u * (b))
    static_assert(NSTAGE <= 4, "barrier block holds four stages");
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(BAR_FULL(s)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(BAR_EMPTY(s)));
        }
        for (int b = 0; b < 2; ++b) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(BAR_ACCFULL(b)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 8;" ::"r"(BAR_ACCEMPTY(b)));
        }
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();
    const uint32_t tmem = *s_tmem;
    const bool dwm = g.mode == MODE_DW;

    if (warp == 0) {
        // ------------------------------------------------------------ producer: bulk copies global image -> stage
        if (umma::elect_one()) {
            uint32_t it = 0;
            for (int t = blockIdx.x; t < g.ntasks; t += gridDim.x) {
                const Task k = decode_task(g, t);
                int kb0 = 0, kb1 = g.kblocks;
                if (dwm) {
                    kb0 = (int)(((long long)k.kg * g.HT) / g.KG);
                    kb1 = (int)(((long long)(k.kg + 1) * g.HT) / g.KG);
                }
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1u;
                    mbar_wait_b(BAR_EMPTY(s), ph ^ 1u);
                    const uint32_t sA = sbase + s * STAGE, sB = sA + STAGE_A;
                    if (!dwm) {
                        const int NG = g.mode == MODE_FWD ? g.n_tile / 64 : 1;
                        mbar_expect_tx(BAR_FULL(s), (uint32_t)NPW * (BLK16 + (uint32_t)NG * g.b_bytes));
                        const uint8_t* a = g.A + k.tower * g.a_tower + (size_t)k.m * g.a_tile + (size_t)kb * BLK16;
                        const uint8_t* b = g.B + k.tower * g.b_tower + (size_t)kb * g.b_kb;
#pragma unroll
                        for (int p = 0; p < NPW; ++p) {
                            bulk_g2s(sA + p * BLK16, a + p * g.a_piece, BLK16, BAR_FULL(s));
                            for (int q = 0; q < NG; ++q)
                                bulk_g2s(sB + (uint32_t)(p * NG + q) * g.b_bytes, b + p * g.b_piece + (size_t)(k.n * NG + q) * g.b_g, g.b_bytes, BAR_FULL(s));
                        }
                    } else {
                        const DwProb& P = g.dw[k.prob];
                        const int NG = P.n_tile / 64, tile = kb >> 1, sh = kb & 1;
                        mbar_expect_tx(BAR_FULL(s), (uint32_t)NPW * (2u + (uint32_t)NG) * BLK8);
                        const uint8_t* a = P.A + k.tower * P.a_tower + (size_t)tile * P.a_tile + (size_t)sh * BLK8;
                        const uint8_t* b = P.B + k.tower * P.b_tower + (size_t)tile * P.b_tile + (size_t)sh * BLK8;
#pragma unroll
                        for (int p = 0; p < NPW; ++p) {
                            for (int q = 0; q < 2; ++q)
                                bulk_g2s(sA + (uint32_t)(p * 2 + q) * BLK8, a + p * P.a_piece + (size_t)(k.m * 2 + q) * BLK16, BLK8, BAR_FULL(s));
                            for (int q = 0; q < NG; ++q)
                                bulk_g2s(sB + (uint32_t)(p * NG + q) * BLK8, b + p * P.b_piece + (size_t)(k.n * NG + q) * BLK16, BLK8, BAR_FULL(s));
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        if (umma::elect_one()) {
            uint32_t it = 0, tc = 0;
            for (int t = blockIdx.x; t < g.ntasks; t += gridDim.x, ++tc) {
                const Task k = decode_task(g, t);
                int kb0 = 0, kb1 = g.kblocks, n_tile = g.n_tile, ksteps = g.ksteps;
                if (dwm) {
                    kb0 = (int)(((long long)k.kg * g.HT) / g.KG);
                    kb1 = (int)(((long long)(k.kg + 1) * g.HT) / g.KG);
                    n_tile = g.dw[k.prob].n_tile;
                    ksteps = 4;
                }
                const int NG = n_tile / 64;
                // operand geometry in the stage (16-byte units)
                uint32_t a_lbo, a_piece, a_ks, b_lbo, b_piece, b_ks;
                int a_mn, b_mn;
                if (g.mode == MODE_FWD) {
                    a_mn = 0; a_lbo = 16; a_piece = BLK16 >> 4; a_ks = 2;
                    b_mn = 1; b_lbo = g.b_bytes; b_piece = (uint32_t)(NG * g.b_bytes) >> 4; b_ks = 2048 >> 4;
                } else if (g.mode == MODE_BWD) {
                    a_mn = 0; a_lbo = 16; a_piece = BLK16 >> 4; a_ks = 2;
                    b_mn = 0; b_lbo = 16; b_piece = g.b_bytes >> 4; b_ks = 2;
                } else {
                    a_mn = 1; a_lbo = BLK8; a_piece = (2 * BLK8) >> 4; a_ks = 2048 >> 4;
                    b_mn = 1; b_lbo = BLK8; b_piece = (uint32_t)(NG * BLK8) >> 4; b_ks = 2048 >> 4;
                }
                const uint32_t idesc = umma::make_idesc(128, n_tile, a_mn, b_mn);  // fp16 operands
                const uint32_t ab = tc & 1u, aph = (tc >> 1) & 1u;
                mbar_wait_b(BAR_ACCEMPTY(ab), aph ^ 1u);
                umma::tc_fence_after();
                const uint32_t dm = tmem + ab * 256u, dc = dm + 128u;
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1u;
                    mbar_wait_b(BAR_FULL(s), ph);
                    umma::tc_fence_after();
                    const uint32_t sA = sbase + s * STAGE, sB = sA + STAGE_A;
                    const uint64_t ad = umma::make_desc(sA, a_lbo, 1024), bd = umma::make_desc(sB, b_lbo, 1024);
#pragma unroll 4
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint64_t a = ad + (uint64_t)(ks * a_ks), b = bd + (uint64_t)(ks * b_ks);
                        const uint32_t acc = (kb > kb0 || ks > 0) ? 1u : 0u;
                        umma::mma_f16(dm, a, b, idesc, acc);              // hi * hi -> main accumulator
                        umma::mma_f16(dc, a, b + b_piece, idesc, acc);    // hi * lo, lo * hi -> cross accumulator
                        umma::mma_f16(dc, a + a_piece, b, idesc, 1u);
                    }
                    umma::umma_commit(BAR_EMPTY(s));  // the stage is free once these MMAs have read it
                }
                umma::umma_commit(BAR_ACCFULL(ab));
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue: TMEM -> result
        // warp (2 + e): TMEM lane quarter q = warp & 3 (the quarter a warp may read), column half e >> 2 of the tile.
        // Image epilogues: a warp owns 32 rows x 64 columns = one contiguous 4 KB slice of a [128 x 64] image block per
        // piece; it is assembled in shared memory (same swizzle, conflict-free) and leaves as ONE bulk store - storing the
        // 16-byte chunks from the row-per-thread TMEM layout costs 32 L1 requests per instruction and was the bound.
        const int q = warp & 3, half = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
        uint8_t* stg = smem + NSTAGE * STAGE + 128 + (uint32_t)(warp - 2) * EPI_STAGE;
        const uint32_t stg_u32 = smem_u32(stg);
        uint32_t tc = 0;
        for (int t = blockIdx.x; t < g.ntasks; t += gridDim.x, ++tc) {
            const Task k = decode_task(g, t);
            const uint32_t ab = tc & 1u, aph = (tc >> 1) & 1u;
            float v[64];
            if (!dwm && g.epi == EPI_LOSS && half == 1) {  // the heads fit in the first 32 columns: these warps only release the buffer
                mbar_wait_b(BAR_ACCFULL(ab), aph);
                umma::tc_fence_after();
                umma::tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR_ACCEMPTY(ab));
                continue;
            }
            if (!dwm && g.epi != EPI_STORE) {
                uint8_t* out_base;
                size_t out_piece;
                if (g.epi == EPI_LOSS) {
                    // ---- losses and head gradients of this warp's 32 samples (GRAPH:9428-11446, 10213-10400): the accumulator
                    // holds mu - b (pi tower, columns 0..A-1) or v - b (V tower, column 0); the sample's inputs are requested
                    // before the accumulator is waited for
                    constexpr int A = 18;
                    const TrainArgs& a = g.ta;
                    const NetDims& d = a.d;
                    const float* P = a.params;
                    const int grow = k.m * TM + row;
                    const bool valid = grow < a.count;
                    float ret = 0.f, oldv = 0.f, oldn = 0.f, adv = 0.f, act[A];
#pragma unroll
                    for (int j = 0; j < A; ++j) act[j] = 0.f;
                    if (valid) {
                        const long src = a.gather ? (long)__ldg(a.gather + a.slot0 + grow) : (long)(a.slot0 + grow);
                        ret = __ldg(a.ret + src);
                        oldv = __ldg(a.val + src);
                        if (k.tower == 0) {
                            oldn = __ldg(a.nlp + src);
#pragma unroll
                            for (int j = 0; j < A; ++j) act[j] = __ldg(a.act + src * A + j);
                            if (a.adv_direct) adv = __ldg(a.adv_direct + a.slot0 + grow);
                            else {  // advs = (returns - values - mean) / (sqrt(var) + 1e-8)  (ppo2.hpp:401-406)
                                const float2 st = __ldg(a.mbstats);
                                adv = __fdiv_rn(__fsub_rn(__fsub_rn(ret, oldv), st.x), st.y);
                            }
                        }
                    }
                    mbar_wait_b(BAR_ACCFULL(ab), aph);
                    umma::tc_fence_after();
                    float mu[32];
                    umma::tmem_ld32_sum(tlane + ab * 256u, tlane + ab * 256u + 128u, mu);
                    umma::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(BAR_ACCEMPTY(ab));
#pragma unroll
                    for (int i = 0; i < 64; ++i) v[i] = 0.f;
                    float* cl = g.colloss + ((size_t)k.m * 4 + q) * COLPART;
                    const float u_hd = __ldg(g.sc + k.tower * SC_STRIDE + SC_U_HD);  // the head image is W * 2^k
                    const float S_b = __ldg(g.sc + k.tower * SC_STRIDE + SC_S_B);    // the dY image carries dL/dy * S
                    if (k.tower == 0) {
                        float l_pg = 0.f, l_kl = 0.f, l_cf = 0.f;
                        if (valid) {
                            const float cr = a.sc->cliprange;
                            float z[A], isd[A];
                            float ss = 0.f, sl = 0.f;
#pragma unroll
                            for (int j = 0; j < A; ++j) {
                                const float ls = __ldg(P + d.off[T_LOGSTD] + j);
                                isd[j] = 1.f / expf(ls);
                                z[j] = (act[j] - fmaf(mu[j], u_hd, __ldg(P + d.off[T_PI_B] + j))) * isd[j];
                                ss += z[j] * z[j];
                                sl += ls;
                            }
                            const PgTerm t = pg_term(adv, oldn, gauss_neglogp(ss, sl, A), cr, a.invB);
                            l_pg = t.pg;
                            l_kl = t.kl;
                            l_cf = t.cf;
                            const float g_nlp = t.g_nlp;
#pragma unroll
                            for (int j = 0; j < A; ++j) {
                                v[j] = g_nlp * (-z[j] * isd[j]);        // dL/dmu_j
                                v[32 + j] = g_nlp * (1.f - z[j] * z[j]);  // dL/dlogstd_j term
                            }
                        }
                        float w32[32];
#pragma unroll
                        for (int i = 0; i < 32; ++i) w32[i] = v[i];
                        const float s0 = colsum32(w32, lane);
#pragma unroll
                        for (int i = 0; i < 32; ++i) w32[i] = v[32 + i];
                        const float s1 = colsum32(w32, lane);
                        if (lane < A) {
                            cl[CP_DBPI + lane] = s0;
                            cl[CP_DLS + lane] = s1;
                        }
                        const float t1 = warp_sum(l_pg), t3 = warp_sum(l_kl), t4 = warp_sum(l_cf);
                        if (lane == 0) { cl[CP_PG] = t1; cl[CP_KL] = t3; cl[CP_CLIP] = t4; }
#pragma unroll
                        for (int i = 0; i < 64; ++i) v[i] *= S_b;  // the column sums above are of the unscaled values
                    } else {
                        float dv = 0.f, l_vf = 0.f;
                        if (valid) {
                            const float vv = fmaf(mu[0], u_hd, __ldg(P + d.off[T_VF_B]));
                            const float vr = vf_clip_range(a.vf_mode, a.sc->cliprange, a.sc->cliprange_vf);
                            l_vf = value_loss_term(a.vf_mode, vr, vv, oldv, ret, a.vf_coef, a.invB, dv);
                        }
                        v[0] = dv * S_b;
                        const float t0 = warp_sum(dv), t2 = warp_sum(l_vf);
                        if (lane == 0) { cl[CP_DBV] = t0; cl[CP_VF] = t2; }
                    }
                    out_base = g.dY + k.tower * g.dy_tower + (size_t)k.m * g.dy_tile + (size_t)q * EPI_STAGE;
                    out_piece = BLK16;
                } else {
                // ---- H = act(acc + b) or dP = acc * act'(H), 64 columns = column block cb of the layer
                const int col0 = k.n * g.n_tile + 64 * half;
                const size_t boff = k.tower * g.img_tower + (size_t)k.m * g.img_tile + (size_t)(col0 >> 6) * BLK16 + (size_t)q * EPI_STAGE;
                float* gp = g.gbuf + (((size_t)k.tower * g.cap + k.m) * g.H + col0) * TM + row;
                float gr[64];
                if (g.epi == EPI_DACT) {  // requested before the accumulator is waited for
#pragma unroll
                    for (int i = 0; i < 64; ++i) gr[i] = __ldg(gp + (size_t)i * TM);
                }
                mbar_wait_b(BAR_ACCFULL(ab), aph);
                umma::tc_fence_after();
                const uint32_t dm = tlane + ab * 256u + 64u * half, dc = dm + 128u;
                umma::tmem_ld32_sum(dm, dc, v);
                umma::tmem_ld32_sum(dm + 32, dc + 32, v + 32);
                umma::tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR_ACCEMPTY(ab));  // the accumulator is in registers: the MMA warp may go on
                if (g.epi == EPI_ACT) {
                    const int ob = g.bias_off[k.tower];
                    const float u_w = __ldg(g.sc + k.tower * SC_STRIDE + g.sc_fwd);  // the weight image is W * 2^k
#pragma unroll
                    for (int i = 0; i < 64; ++i) {
                        v[i] = act_fwd<ACT>(ob >= 0 ? fmaf(v[i], u_w, __ldg(g.P + ob + col0 + i)) : v[i] * u_w);
                        if (g.gbuf) gp[(size_t)i * TM] = act_dfac<ACT>(v[i]);  // kept for the backward pass (training only)
                        v[i] *= (float)(1 << pw_h<ACT>());                    // the image holds H * 2^pw_h
                    }
                } else {  // TanhGrad / ReluGrad (GRAPH:20925-23699)
#pragma unroll
                    for (int i = 0; i < 64; ++i) v[i] *= gr[i] * (1.0f / (float)(1 << PW_W));  // renormalised: the weight image was W * 2^(k + PW_W)
                    if (g.colsum) {  // bias gradient: column sums over this warp's 32 rows
                        float* cs = g.colsum + (((size_t)k.tower * g.cap + k.m) * 4 + q) * g.H + col0 + lane;
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            float w32[32];
#pragma unroll
                            for (int i = 0; i < 32; ++i) w32[i] = v[32 * hh + i];
                            cs[32 * hh] = colsum32(w32, lane);
                        }
                    }
                }
                out_base = g.img_out + boff;
                out_piece = g.img_piece;
                }
                // two fp16 pieces, one after the other through the staging slice: hi = fp16(x), lo = fp16(x - hi)
#pragma unroll 1
                for (int p = 0; p < NPW; ++p) {
                    if (p) {
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        uint4 pk;
                        uint32_t* w4 = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const __half2 h2 = __floats2half2_rn(v[8 * j + 2 * i], v[8 * j + 2 * i + 1]);
                            w4[i] = *reinterpret_cast<const uint32_t*>(&h2);
                            const float2 f2 = __half22float2(h2);
                            v[8 * j + 2 * i] -= f2.x;
                            v[8 * j + 2 * i + 1] -= f2.y;
                        }
                        *reinterpret_cast<uint4*>(stg + chunk_off(lane, j)) = pk;
                    }
                    umma::fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out_base + (size_t)p * out_piece),
                                     "r"(stg_u32), "r"(EPI_STAGE)
                                     : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                }
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncwarp();
                continue;
            }
            mbar_wait_b(BAR_ACCFULL(ab), aph);
            umma::tc_fence_after();
            const uint32_t dm = tlane + ab * 256u, dc = dm + 128u;
            if (!dwm) {  // EPI_STORE: fp32 result
                const int ncols = g.n_tile >> 1, cbeg = half * ncols;
                const float u_w = __ldg(g.sc + k.tower * SC_STRIDE + g.sc_fwd);
                float* dst = g.C + k.tower * g.c_tower + ((size_t)k.m * TM + row) * g.ldc + (size_t)k.n * g.n_tile;
                for (int c0 = cbeg; c0 < cbeg + ncols; c0 += 32) {
                    umma::tmem_ld32_sum(dm + c0, dc + c0, v);
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        reinterpret_cast<float4*>(dst + c0)[i] = make_float4(v[4 * i] * u_w, v[4 * i + 1] * u_w, v[4 * i + 2] * u_w, v[4 * i + 3] * u_w);
                }
            } else {
                const DwProb& P = g.dw[k.prob];
                float* slab = g.partial + (size_t)k.kg * g.PS;
                const int r = k.m * TM + row;  // feature index of the M side
                // the back-propagated operands carry S (and the powers of two of the weight images they went through)
                const float un = __ldg(g.sc + k.tower * SC_STRIDE + (P.kind == DW_W1 ? SC_UN_W1 : (P.kind == DW_HEAD ? SC_UN_HD : SC_UN_W0)));
                if (P.kind == DW_W1) {  // dW1[k_in = r][n_out]
                    const int ncols = P.n_tile >> 1, cbeg = half * ncols;
                    for (int c0 = cbeg; c0 < cbeg + ncols; c0 += 32) {
                        umma::tmem_ld32_sum(dm + c0, dc + c0, v);
                        float* dst = slab + g.off_w1[k.tower] + (size_t)r * g.H + (size_t)k.n * P.n_tile + c0;
#pragma unroll
                        for (int i = 0; i < 32; ++i) dst[i] = v[i] * un;  // slabs are PS floats apart (odd): no vector stores
                    }
                } else if (half == 0) {  // heads and X' use the first 32 columns only
                    umma::tmem_ld32_sum(dm, dc, v);
                    if (P.kind == DW_HEAD) {  // pi: dWpi[r][j]; V: dwv[r]
                        if (k.tower == 0) {
                            float* dst = slab + g.off_piw + (size_t)r * g.A_dim;
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < g.A_dim) dst[j] = v[j] * un;
                        } else {
                            slab[g.off_vfw + r] = v[0] * un;
                        }
                    } else {  // dW0'^T[n_out = r][k_in = j]: j < O weights, j == O bias
                        float* dw = slab + g.off_w0[k.tower] + r;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (j < g.O) dw[(size_t)j * g.H] = v[j] * un;
                            else if (j == g.O) slab[g.off_b0[k.tower] + r] = v[j] * un;
                    }
                }
            }
            umma::tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR_ACCEMPTY(ab));
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
#undef BAR_FULL
#undef BAR_EMPTY
#undef BAR_ACCFULL
#undef BAR_ACCEMPTY
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
}

// ------------------------------------------------------------------------------------------------ elementwise kernels
struct WideBufs {
    Geom G;
    uint8_t *X, *H1, *H2, *dP2, *dP1, *dY;  // images
    uint8_t *W0, *W1, *WH;                  // weight images
    float *G1, *G2, *MU;                    // G: 1 - H^2 per layer, fp32 [2][cap][H][128]; MU: fp32 head results [2][cap * 128 x 64]
    float *colloss;                         // [cap * 4][COLPART]: per (tile, lane quarter) sums of the loss stage
    float *colb1;                           // [2][cap * 4][H]: per (tile, lane quarter) column sums of dP2
    float *colb0;                           // ... and of dP1 (layer-0 bias gradient: fp32 sums of the unsplit values, not the ones row of X')
    float *pmax;                            // [WMAX_BLOCKS][8]: per-block |max| of the six weight matrices, max(-logstd)
    float *sc;                              // [2][SC_STRIDE]: the scale table of the current weight images (SC_*)
};

// |max| of every weight matrix that becomes an operand image (block floating point), max(-logstd) for the backward scale.
// Categories: tower * 3 + {W0' (weights and bias row), W1, head}; 6 = -logstd.  Per-block partials, no atomics.
constexpr int WMAX_BLOCKS = 296;
__global__ void __launch_bounds__(256) wide_absmax_kernel(const float* __restrict__ P, const NetDims d, float* __restrict__ pmax) {
    __shared__ float red[8][8];
    float mx[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) mx[k] = k == 6 ? -3.0e38f : 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.P; i += gridDim.x * blockDim.x) {
        int t = 0;
        while (i >= d.off[t + 1]) ++t;
        const float x = __ldg(P + i);
        int cat = -1;
        switch (t) {
            case T_PI_FC0_W: case T_PI_FC0_B: cat = 0; break;
            case T_PI_FC1_W: cat = 1; break;
            case T_PI_W: cat = 2; break;
            case T_VF_FC0_W: case T_VF_FC0_B: cat = 3; break;
            case T_VF_FC1_W: cat = 4; break;
            case T_VF_W: cat = 5; break;
            case T_LOGSTD: cat = 6; break;
            default: break;
        }
#pragma unroll
        for (int k = 0; k < 7; ++k)
            if (cat == k) mx[k] = fmaxf(mx[k], k == 6 ? -x : fabsf(x));
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        if (lane == 0) red[warp][k] = mx[k];
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float m = red[0][threadIdx.x];
        for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w][threadIdx.x]);
        pmax[blockIdx.x * 8 + threadIdx.x] = m;
    }
}
// k with m * 2^k in [1, 2); 0 for a zero / non-finite matrix
__device__ __forceinline__ int pow2_to_unit(float m) {
    int e = 0;
    if (!(m > 0.f) || !isfinite(m)) return 0;
    (void)frexpf(m, &e);
    return max(-24, min(24, 1 - e));
}

// fp32 parameters -> weight images.  One thread per 16-byte chunk.
template <int ACT>
__global__ void wide_prep_weights_kernel(const float* __restrict__ P, const NetDims d, const WideBufs w, float invB) {
    const Geom& G = w.G;
    const int nb = G.nb, H = G.H;
    // scale table: every block folds the partial maxima (the same numbers in the same order everywhere), block 0 publishes
    __shared__ float s_sc[2][SC_STRIDE];
    __shared__ float s_max[8];
    if (threadIdx.x < 8) {
        float m = w.pmax[threadIdx.x];
        for (int b = 1; b < WMAX_BLOCKS; ++b) m = fmaxf(m, w.pmax[b * 8 + threadIdx.x]);
        s_max[threadIdx.x] = m;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        const int t = threadIdx.x;
        const float m_w0 = s_max[3 * t], m_w1 = s_max[3 * t + 1], m_hd = s_max[3 * t + 2], neg_ls_max = s_max[6];
        const int k_w0 = pow2_to_unit(m_w0) + PW_W, k_w1 = pow2_to_unit(m_w1) + PW_W, k_hd = pow2_to_unit(m_hd) + PW_W;  // image = W * 2^k
        int e_b = 0, e_sig = 0;
        (void)frexpf(invB, &e_b);                                   // invB = m * 2^e, m in [0.5, 1)
        (void)frexpf(expf(-neg_ls_max), &e_sig);                    // sigma_min = f * 2^e
        const int k_sig = max(-24, min(8, e_sig - 1));
        const int n_s = t == 0 ? (-e_b + k_sig + 4) : (-e_b + 6);   // pi: S * invB / sigma_min in (4, 16]; V: S * invB in [32, 64)
        // the backward chain renormalises by 2^-PW_W after each weight image, so dP2 carries S * 2^kh, dP1 S * 2^(kh + k1)
        const int kh = k_hd - PW_W, k1 = k_w1 - PW_W;
        constexpr int PW_H = pw_h<ACT>();  // activation images hold H * 2^PW_H
        float* r = s_sc[t];
        r[SC_S_W0] = ldexpf(1.f, k_w0); r[SC_U_W0] = ldexpf(1.f, -k_w0 - PW_X);   // layer 0: acc = (X' 2^PW_X)(W0' 2^k)
        r[SC_S_W1] = ldexpf(1.f, k_w1); r[SC_U_W1] = ldexpf(1.f, -k_w1 - PW_H);   // layer 1: acc = (H1 2^PW_H)(W1 2^k)
        r[SC_S_HD] = ldexpf(1.f, k_hd); r[SC_U_HD] = ldexpf(1.f, -k_hd - PW_H);
        r[SC_S_B] = ldexpf(1.f, n_s);
        r[SC_UN_HD] = ldexpf(1.f, -n_s - PW_H);                 // dWhead = (H2 2^PW_H)^T (dY S)
        r[SC_UN_W1] = ldexpf(1.f, -n_s - kh - PW_H);            // dW1 = (H1 2^PW_H)^T (dP2 S 2^kh)
        r[SC_UN_W0] = ldexpf(1.f, -n_s - kh - k1 - PW_X);       // dW0' = (dP1 S 2^(kh+k1))^T (X' 2^PW_X)
        r[SC_UNC_B1] = ldexpf(1.f, -n_s - kh);                  // column sums of dP2
        r[SC_UNC_B0] = ldexpf(1.f, -n_s - kh - k1);             // column sums of dP1
        if (blockIdx.x == 0)
            for (int i = 0; i < SC_COUNT; ++i) w.sc[t * SC_STRIDE + i] = r[i];
    }
    __syncthreads();
    const int n_w0 = 2 * nb * 32 * 8, n_w1 = 2 * nb * nb * 64 * 8, n_wh = 2 * nb * 64 * 8;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_w0 + n_w1 + n_wh; e += gridDim.x * blockDim.x) {
        float x[8];
        uint8_t* dst;
        size_t piece;
        float scale;
        if (e < n_w0) {
            int t = e;
            const int j = t & 7; t >>= 3;
            const int r = t & 31; t >>= 5;
            const int nbk = t % nb, tower = t / nb;
            const float* W0 = P + d.off[tower ? T_VF_FC0_W : T_PI_FC0_W];
            const float* B0 = P + d.off[tower ? T_VF_FC0_B : T_PI_FC0_B];
            const int n = nbk * 64 + 8 * j;
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = r < d.O ? __ldg(W0 + (size_t)r * H + n + i) : (r == d.O ? __ldg(B0 + n + i) : 0.f);
            dst = w.W0 + tower * G.w0_tower + (size_t)nbk * 4096 + chunk_off(r, j);
            piece = G.w0_piece;
            scale = s_sc[tower][SC_S_W0];
        } else if (e < n_w0 + n_w1) {
            int t = e - n_w0;
            const int j = t & 7; t >>= 3;
            const int r = t & 63; t >>= 6;
            const int ri = t % nb; t /= nb;
            const int co = t % nb, tower = t / nb;
            const float* W1 = P + d.off[tower ? T_VF_FC1_W : T_PI_FC1_W] + (size_t)(ri * 64 + r) * H + co * 64 + 8 * j;
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = __ldg(W1 + i);
            dst = w.W1 + tower * G.w1_tower + (size_t)(co * nb + ri) * BLK8 + chunk_off(r, j);
            piece = G.w1_piece;
            scale = s_sc[tower][SC_S_W1];
        } else {
            int t = e - n_w0 - n_w1;
            const int j = t & 7; t >>= 3;
            const int r = t & 63; t >>= 6;
            const int ri = t % nb, tower = t / nb;
            const int k = ri * 64 + r;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = 8 * j + i;
                x[i] = tower == 0 ? (c < d.A ? __ldg(P + d.off[T_PI_W] + (size_t)k * d.A + c) : 0.f) : (c == 0 ? __ldg(P + d.off[T_VF_W] + k) : 0.f);
            }
            dst = w.WH + tower * G.wh_tower + (size_t)ri * BLK8 + chunk_off(r, j);
            piece = G.wh_piece;
            scale = s_sc[tower][SC_S_HD];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] *= scale;
        umma::store_chunk(dst, (uint32_t)piece, 0, x);
    }
}

// minibatch rows -> X' image: [obs | 1 | 0 ...]; rows past the minibatch are zero (they then contribute nothing:
// the loss kernel masks them and every gradient flows through dY).  Only the chunks that can be non-zero are written.
__global__ void wide_gather_kernel(const TrainArgs a, const WideBufs w) {
    const Geom& G = w.G;
    const int O = a.d.O, nj = O / 8 + 1;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < G.Bpad * nj; e += gridDim.x * blockDim.x) {
        const int row = e / nj, j = e % nj;
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = 0.f;
        if (row < a.count) {
            const long src = a.gather ? (long)__ldg(a.gather + a.slot0 + row) : (long)(a.slot0 + row);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = 8 * j + i;
                x[i] = (c < O ? __ldg(a.obs + src * O + c) : (c == O ? 1.f : 0.f)) * (float)(1 << PW_X);
            }
        }
        umma::store_chunk(w.X + (size_t)(row >> 7) * G.x_tile, BLK16, chunk_off(row & 127, j), x);
    }
}

// ---- policy step on the W family (MlpPolicy::step/value/get_deterministic_action, policies.hpp:33-77): the three
// forward GEMMs above, then one thread per env: Gaussian sample (Philox or given noise), neglogp, value, rollout stores
__global__ void wide_policy_gather_kernel(const float* __restrict__ obs, int n, float* __restrict__ obs_store, int O, const WideBufs w) {
    const Geom& G = w.G;
    const int nj = O / 8 + 1;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < G.Bpad * nj; e += gridDim.x * blockDim.x) {
        const int row = e / nj, j = e % nj;
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = 8 * j + i;
            x[i] = 0.f;
            if (row < n) {
                if (c < O) {
                    const float ob = __ldg(obs + (size_t)row * O + c);
                    if (obs_store) obs_store[(size_t)row * O + c] = ob;
                    x[i] = ob * (float)(1 << PW_X);
                } else if (c == O) x[i] = (float)(1 << PW_X);
            }
        }
        umma::store_chunk(w.X + (size_t)(row >> 7) * G.x_tile, BLK16, chunk_off(row & 127, j), x);
    }
}

__global__ void wide_policy_head_kernel(const PolicyArgs a, const WideBufs w) {
    const NetDims& d = a.d;
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= a.n) return;
    const float* p = a.params;
    if (a.mode != 2) {
        const float v = w.MU[w.G.mu_tower + (size_t)row * 64] + __ldg(p + d.off[T_VF_B]);
        if (a.value) a.value[row] = v;
        if (a.val_store) a.val_store[row] = v;
    }
    const float* mu = w.MU + (size_t)row * 64;
    if (a.mode == 0) {
        const float* logstd = p + d.off[T_LOGSTD];
        gauss_policy_row(a, row, d.A, [&](int j) { return __ldg(logstd + j); }, [&](int j) { return mu[j] + __ldg(p + d.off[T_PI_B] + j); },
                         [&](int j, float act) {
                             if (a.action) a.action[(size_t)row * d.A + j] = act;
                             if (a.act_store) a.act_store[(size_t)row * d.A + j] = act;
                         });
    } else if (a.mode == 2) {
        for (int j = 0; j < d.A; ++j) {
            const float m = mu[j] + __ldg(p + d.off[T_PI_B] + j);  // mean + 0.0 (GRAPH:6046-6076)
            if (a.action) a.action[(size_t)row * d.A + j] = m;
            if (a.act_store) a.act_store[(size_t)row * d.A + j] = m;
        }
    }
    if (a.dones_store) a.dones_store[row] = a.dones_in[row];
}

// per-tile sums -> slab 0; the same columns of the other slabs are zero (the GEMMs own every weight column of every slab).
// One warp per output column: lanes stride over the tiles, fixed-order butterfly in double.
__global__ void wide_fold_kernel(const TrainArgs a, const WideBufs w, int nslabs) {
    const Geom& G = w.G;
    const NetDims& d = a.d;
    const int H = G.H, A = d.A, lane = threadIdx.x & 31;
    const int n = 2 * H + 2 * A + 1 + L_PAD + 2 * H;
    for (int e0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; e0 < n; e0 += (gridDim.x * blockDim.x) >> 5) {
        double t = 0.0;
        int col;
        const float* src = nullptr;
        size_t stride = 0;
        const bool is_b0 = e0 >= 2 * H + 2 * A + 1 + L_PAD;
        const int e = is_b0 ? 0 : e0;
        if (is_b0) {
            const int i = e0 - (2 * H + 2 * A + 1 + L_PAD), tower = i / H, c = i % H;
            src = w.colb0 + (size_t)tower * G.cap * 4 * H + c; stride = H;
            col = d.off[tower ? T_VF_FC0_B : T_PI_FC0_B] + c;
        } else if (e < 2 * H) {
            const int tower = e / H, c = e % H;
            src = w.colb1 + (size_t)tower * G.cap * 4 * H + c; stride = H;
            col = d.off[tower ? T_VF_FC1_B : T_PI_FC1_B] + c;
        } else if (e < 2 * H + 2 * A + 1) {
            const int c = e - 2 * H;  // colloss columns 0 .. 2A: dbpi, dlogstd, dbv
            src = w.colloss + c; stride = COLPART;
            col = c < A ? d.off[T_PI_B] + c : (c < 2 * A ? d.off[T_LOGSTD] + c - A : d.off[T_VF_B]);
        } else {
            const int l = e - (2 * H + 2 * A + 1);
            col = d.P + l;
            const int sc = l == L_PG ? CP_PG : l == L_VF ? CP_VF : l == L_KL ? CP_KL : l == L_CLIP ? CP_CLIP : -1;
            if (sc >= 0) { src = w.colloss + sc; stride = COLPART; }
        }
        const int nsrc = 4 * G.NT;  // one entry per (tile, TMEM lane quarter = epilogue warp)
        if (src)
            for (int i = lane; i < nsrc; i += 32) t += (double)src[(size_t)i * stride];
        t = warp_sum(t);
        if (is_b0) t *= (double)__ldg(w.sc + ((e0 - (2 * H + 2 * A + 1 + L_PAD)) / H) * SC_STRIDE + SC_UNC_B0);  // column sums of dP1
        else if (e < 2 * H) t *= (double)__ldg(w.sc + (e / H) * SC_STRIDE + SC_UNC_B1);  // column sums of dP2 = dL/dz2 * S * 2^k_head
        if (lane == 0) {
            if (!is_b0 && e >= 2 * H + A && e < 2 * H + 2 * A) t -= (double)a.ent_coef;  // d(-ent_coef * entropy)/dlogstd_j (ent_coef is pre-divided by the world size)
            if (!is_b0 && col == d.P + L_ENT)  // every rank adds it; the Adam kernel scales the summed row by 1 / world_size
                for (int j = 0; j < A; ++j) t += (double)(__ldg(a.params + d.off[T_LOGSTD] + j) + PPO_HALF_LOG_2PIE);
            a.partial[col] = (float)t;
            for (int s = 1; s < nslabs; ++s) a.partial[(size_t)s * a.PS + col] = 0.f;
        }
    }
}

}  // namespace wide
}  // namespace ppo
