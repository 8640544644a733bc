// infer_hmma.cuh -- the SMALL-BATCH variant of the fused MAMuZeroNet.recurrent_inference kernel (sm_100a).
//
// Same computation and same descriptor as infer_fused.cuh (config/smac/model.py:562-574 + core/config.py:430-499 +
// mcts_sampled.py:158-161); different decomposition.  tcgen05.mma needs a tile of 128 token rows per CTA (M = 64 only
// fills 16 lanes of each TMEM quadrant), so the 3m configuration of BASELINE.json (1024 roots x 3 agents = 3072 rows)
// occupies 26 of the 148 SMs and every one of them walks the 25-stage dependency chain of its tile at
// ~3.6 us per stage (TMEM round trip, MMA-warp hand-off, commit -> wait latency): 88 us per launch, tensor pipe 2 % busy.
// The search is bound by that LATENCY (one launch per simulation), not by tensor throughput.  This kernel trades
// peak tensor rate for parallelism and a short chain:
//   * 32-row tiles (floor(32/N) whole roots)  -> 103 CTAs for 3m instead of 26;
//   * warp-level mma.sync.m16n8k16 (bf16 x bf16 -> fp32): accumulators and the fp32 residual stream stay in REGISTERS,
//     the epilogue of a stage runs on the fragments it just computed -- no TMEM load, no issuer warp, no commit;
//     operand fragments of step k+1 are loaded (ldmatrix) before the MMAs of step k are issued;
//   * a stage costs one or two 256-thread barriers; q, k, v are one pass over the activations; the three output heads
//     share two stages (20 GEMM stages instead of 25) and their barrier phases;
//   * weights stream from L2 through the same 3-slot bulk-TMA ring (a dedicated producer warp), row-major with an
//     8-element pad so that ldmatrix is bank-conflict free.
// The weights (0.9 MB) are re-read from L2 once per CTA, so above a few hundred tiles the tcgen05 kernel wins;
// mazero_b200/fused.py::use_small picks by batch size.
#pragma once
#include <cuda_bf16.h>

#include "../../include/maz_infer.h"
#include "umma.cuh"

namespace maz {
namespace hmma {

using namespace umma;

constexpr int H = 128, NHEAD = 8, HD = 16, GH = 64, PH = 32, SUP = 11, NLAYER = 3;
constexpr int NCHUNK = MAZ_INFER_NCHUNK, NSLOT = 3;
constexpr int TM = 32;                       // token rows per CTA
#ifndef MAZ_HMMA_NQ
#define MAZ_HMMA_NQ 4
#endif
constexpr int NQ = MAZ_HMMA_NQ;              // column groups: a warp owns 16 rows x (128 / NQ) columns of a 128-wide stage
constexpr int NT = H / NQ / 8;               // n8 tiles per warp in a 128-wide stage
constexpr int GT = GH / NQ / 8;              // n8 tiles per warp and half (gc | nn) of a stacked graph-net GEMM
constexpr int CW = H / NQ, FW = GH / NQ;     // columns / graph features per warp
static_assert(NQ == 4 || NQ == 8, "NQ");
constexpr int NCONS = 64 * NQ, NTHREADS = NCONS + 32;   // 2*NQ compute warps + 1 producer warp
constexpr int PAD = 8;                       // bf16 elements of row padding (16 bytes: ldmatrix rows land in distinct banks)
constexpr int LDA = (H + PAD) * 2;           // bytes per activation row
constexpr int LDQ = (3 * H + PAD) * 2;       // bytes per q|k|v row
constexpr int LDP = (PH + PAD) * 2;          // bytes per policy-hidden row
constexpr int LDO = (48 + PAD) * 2;          // bytes per one-hot row (sized for the largest KA)
constexpr int LDG = GH + 4;                  // floats per graph-sum row
constexpr int LDV = GH + 4;                  // floats per row of the padded copy of a 11 x 64 head
constexpr uint32_t SLOT_BYTES = 128 * (H + PAD) * 2;
#ifndef MAZ_HMMA_PIECE
#define MAZ_HMMA_PIECE 4352
#endif
constexpr uint32_t PIECE = MAZ_HMMA_PIECE;   // bytes per bulk-copy request (16 weight rows)
// k-loop unrolling of the GEMM stages: 2 keeps the double-buffered fragment indices compile-time and the code small (the kernel
// runs ~25 different stages once per simulation: its instruction footprint, not its loop overhead, is what costs)
#ifndef MAZ_GEMM_UNROLL
#define MAZ_GEMM_UNROLL 2
#endif
constexpr int GEMM_UNROLL = MAZ_GEMM_UNROLL;

// ---- shared-memory map (compile-time offsets from the dynamic base: every access is a plain LDS / STS) -------------
constexpr uint32_t OFF_X = 0;                                    // activation tile X        [TM][LDA]
constexpr uint32_t OFF_T = OFF_X + TM * LDA;                     // activation tile T        [TM][LDA]
constexpr uint32_t OFF_HH = OFF_T + TM * LDA;                    // parent hidden state h    [TM][LDA] (kept for fc_dynamic)
constexpr uint32_t OFF_ONE = OFF_HH + TM * LDA;                  // one-hot joint action     [TM][LDO]
constexpr uint32_t OFF_PH = OFF_ONE + TM * LDO;                  // policy hidden            [TM][LDP]
constexpr uint32_t OFF_Q = OFF_PH + TM * LDP;                    // q|k|v rows (layers) / fp32 scratch of the heads
constexpr uint32_t OFF_STAT = OFF_Q + TM * LDQ;                  // row statistics, 3 sets   [3][TM][NQ] float2
constexpr uint32_t STAT_SET = TM * NQ * 8;                       // bytes per set
constexpr uint32_t OFF_VP = OFF_STAT + 3 * TM * NQ * 8;           // padded reward / value head weights [2][SUP][LDV] fp32
constexpr uint32_t OFF_ROW = OFF_VP + 2 * SUP * LDV * 4;         // row table                [TM] RowInfo
constexpr uint32_t OFF_W = ((OFF_ROW + TM * 16 + 127) / 128) * 128;   // weight ring         [NSLOT][SLOT_BYTES]
constexpr uint32_t OFF_P = OFF_W + NSLOT * SLOT_BYTES;           // fp32 parameters (d.vec)
// fp32 scratch inside the Q region (heads only), in floats
constexpr int G_R = 0, G_V = TM * LDG;                           // graph sums of the reward / value GNN   [TM][LDG]
constexpr int Y_R = 0, Y_V = TM * GH;                            // layer-2 features (fp32, in the X + T tiles) [TM][GH]
constexpr int PL0 = 2 * TM * LDG;                                // policy logits                          [TM][48]
static_assert((PL0 + TM * 48) * 4 <= TM * LDQ, "heads scratch must fit in the q|k|v region");
static_assert(2 * TM * GH * 4 <= 2 * TM * LDA, "layer-2 features must fit in the X + T tiles");
// The WIDE variant (template argument W = true, 48 < KA <= 128) keeps this map.  The one-hot tile region holds one int per row
// (the row's action, -1 = none) and the one-hot MMA operand is built in registers (gemm_onehot); the policy logits, [TM][128]
// fp32, go to the X + T tiles once the layer-2 features there have been consumed (stage_heads2).
constexpr int KA_NARROW = 48, KA_WIDE = 128;
static_assert(TM * 4 <= TM * LDO, "wide variant: the row actions must fit in the one-hot tile region");
static_assert(TM * KA_WIDE * 4 <= 2 * TM * LDA, "wide variant: the policy logits must fit in the X + T tiles");

using Desc = ::maz_infer_desc;

struct RowInfo { int root, agent, valid, r0; };   // r0 = first row of my root inside the tile

// whole roots per 32-row tile (the persistent search kernel owns fewer roots per CTA than fit: one warp per tree)
__device__ __forceinline__ int tile_rpt(const Desc &d) { return d.roots_per_tile > 0 ? d.roots_per_tile : TM / d.N; }

// The per-simulation pointers: constants of the descriptor for the one-step kernel, advanced per simulation by the
// persistent whole-search kernel (search_persist.cuh).
struct SimIo {
    // the exchange arrays between the tree step and the network: indexed by (root - root0).  Global memory with root0 = 0 for the
    // one-step kernel; the persistent kernel keeps its CTA's slice of them in SHARED memory (root0 = the CTA's first root).
    const int *idx_x;      // (B,) pool index of the parent
    const int *actions;    // (B,N) joint action, or (B,1) tree action when the joint action is assembled here
    float *reward, *value, *probs, *beta;
    int root0;
    // global memory, indexed by the root
    float *next_hidden;    // (B, N*H)
    int *greedy;           // (B,N) or NULL
    float *logits_out;     // (B,N,A) or NULL
};
__device__ __forceinline__ SimIo io_from_desc(const Desc &d)
{
    return SimIo{d.idx_x, d.actions, d.reward, d.value, d.probs, d.beta, 0, d.next_hidden, d.greedy, d.logits_out};
}

__host__ __device__ inline size_t smem_bytes(int vec_floats) { return (size_t)OFF_P + (size_t)vec_floats * 4 + 128; }

#define HSM_DECL extern __shared__ __align__(128) uint8_t hsm[]
__device__ __forceinline__ uint32_t sbase()
{
    HSM_DECL;
    return smem_u32(hsm);
}

// ---- tensor-core primitives ------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t (&r)[4])
{
    // (no "memory" clobber: every shared-memory write that a ldmatrix reads is separated from it by a bar.sync / mbarrier
    //  wait, which are compiler barriers and, like this, volatile; a clobber here would spill by-reference accumulators)
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float a, float b)
{
    __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&p);
}
__device__ __forceinline__ void sts32(uint32_t saddr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }
// parameters (d.vec): written once by the bulk copy before any stage function runs, read-only afterwards
__device__ __forceinline__ float2 ldp2(uint32_t saddr)
{
    float2 v;
    asm("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ float4 lds4v(uint32_t saddr)   // ordered with the barriers (scratch produced by other threads)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}

// who am I inside the 2*NQ compute warps: warp = nq*2 + mt; the warp owns rows [16*mt, +16) and, of a 128-wide stage,
// columns [CW*nq, +CW) as NT n8 tiles.  Fragment element acc[nt][2*hf + j] = (row 16*mt + g + 8*hf, col n0 + 8*nt + 2*t + j).
struct Thr {
    int lane, warp, g, t, mt, nq, rA, rB;
    uint32_t a_off, w_off;      // per-lane parts of the ldmatrix row addresses
    __device__ __forceinline__ Thr()
    {
        const int tid = threadIdx.x;
        lane = tid & 31; warp = tid >> 5; g = lane >> 2; t = lane & 3; mt = warp & 1; nq = warp >> 1;
        rA = 16 * mt + g; rB = rA + 8;
        a_off = (uint32_t)(16 * mt + (lane & 7) + ((lane >> 3) & 1) * 8);   // activation row; k offset (lane>>4)*16 bytes
        w_off = (uint32_t)((lane & 7) + (lane >> 4) * 8);                   // weight row inside a pair of n8 tiles; k offset ((lane>>3)&1)*16
    }
    __device__ __forceinline__ uint32_t a_addr(uint32_t tile, int lda) const { return tile + a_off * lda + (uint32_t)(lane >> 4) * 16u; }
    __device__ __forceinline__ uint32_t w_addr(uint32_t slot, int ldw, int n0) const
    {
        return slot + (uint32_t)(n0 + w_off) * ldw + (uint32_t)((lane >> 3) & 1) * 16u;
    }
};

// acc[NT] (+)= A[16 rows x 16*KS] * W[n0 .. n0+8*NT)^T, fully unrolled, operands of step k+1 in flight during the MMAs of step k
template <int NT, int KS>
__device__ __forceinline__ void gemm_fixed(float (&acc)[NT][4], const Thr &th, uint32_t a_tile, int lda, uint32_t w_slot, int ldw, int n0)
{
    const uint32_t aa = th.a_addr(a_tile, lda), wa = th.w_addr(w_slot, ldw, n0);
    uint32_t a[2][4], b[2][NT / 2][4];
    ldsm4(aa, a[0]);
#pragma unroll
    for (int p = 0; p < NT / 2; ++p) ldsm4(wa + (uint32_t)(16 * p) * ldw, b[0][p]);
#pragma unroll GEMM_UNROLL
    for (int ks = 0; ks < KS; ++ks) {
        const int cur = ks & 1, nxt = cur ^ 1;
        if (ks + 1 < KS) {
            ldsm4(aa + 32u * (ks + 1), a[nxt]);
#pragma unroll
            for (int p = 0; p < NT / 2; ++p) ldsm4(wa + (uint32_t)(16 * p) * ldw + 32u * (ks + 1), b[nxt][p]);
        }
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) {
            mma16816(acc[2 * p], a[cur], b[cur][p][0], b[cur][p][1]);
            mma16816(acc[2 * p + 1], a[cur], b[cur][p][2], b[cur][p][3]);
        }
    }
}
// the same with a run-time K (the one-hot operand of the narrow variant: K = KA in {16, 32, 48})
template <int NT>
__device__ __forceinline__ void gemm_rt(float (&acc)[NT][4], const Thr &th, uint32_t a_tile, int lda, uint32_t w_slot, int ldw, int n0, int K)
{
    const uint32_t aa = th.a_addr(a_tile, lda), wa = th.w_addr(w_slot, ldw, n0);
#pragma unroll 1
    for (int k0 = 0; k0 < K; k0 += 16) {
        uint32_t a[4], b[NT / 2][4];
        ldsm4(aa + 2u * k0, a);
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) ldsm4(wa + (uint32_t)(16 * p) * ldw + 2u * k0, b[p]);
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) {
            mma16816(acc[2 * p], a, b[p][0], b[p][1]);
            mma16816(acc[2 * p + 1], a, b[p][2], b[p][3]);
        }
    }
}
// the same product for the wide variant: the A operand is the one-hot matrix of the row actions actA (row th.rA) and actB (row
// th.rB), built in registers -- fragment word i holds rows rA (i even) / rB (i odd), columns k0 + 2t (+8 for i >= 2) and +1
template <int NT>
__device__ __forceinline__ void gemm_onehot(float (&acc)[NT][4], const Thr &th, int actA, int actB, uint32_t w_slot, int ldw, int n0, int K)
{
    const uint32_t wa = th.w_addr(w_slot, ldw, n0);
#pragma unroll 1
    for (int k0 = 0; k0 < K; k0 += 16) {
        const int c = k0 + 2 * th.t;
        uint32_t a[4], b[NT / 2][4];
        a[0] = pack2(c == actA ? 1.f : 0.f, c + 1 == actA ? 1.f : 0.f);
        a[1] = pack2(c == actB ? 1.f : 0.f, c + 1 == actB ? 1.f : 0.f);
        a[2] = pack2(c + 8 == actA ? 1.f : 0.f, c + 9 == actA ? 1.f : 0.f);
        a[3] = pack2(c + 8 == actB ? 1.f : 0.f, c + 9 == actB ? 1.f : 0.f);
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) ldsm4(wa + (uint32_t)(16 * p) * ldw + 2u * k0, b[p]);
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) {
            mma16816(acc[2 * p], a, b[p][0], b[p][1]);
            mma16816(acc[2 * p + 1], a, b[p][2], b[p][3]);
        }
    }
}
// acc += [h | onehot(a)] one-hot part: the one-hot tile (narrow) or the row actions (wide)
template <bool W, int NT>
__device__ __forceinline__ void gemm_action(float (&acc)[NT][4], const Thr &th, uint32_t sb, uint32_t w_slot, int ldw, int n0, int K)
{
    if constexpr (W) {
        const int actA = __float_as_int(lds1v(sb + OFF_ONE + 4u * th.rA)), actB = __float_as_int(lds1v(sb + OFF_ONE + 4u * th.rB));
        gemm_onehot<NT>(acc, th, actA, actB, w_slot, ldw, n0, K);
    } else {
        gemm_rt<NT>(acc, th, sb + OFF_ONE, LDO, w_slot, ldw, n0, K);
    }
}

// ---- weight ring ---------------------------------------------------------------------------------------------------------
// one chunk = several bulk copies on the same mbarrier (16 weight rows each)
__device__ __forceinline__ void issue_chunk(const Desc &d, int k, int slot, uint64_t *bar_full)
{
    HSM_DECL;
    const uint32_t nbytes = (d.dbg_flags & 4) ? 16u : d.chunk_bytes[k];   // profiling: tiny copies
    const uint8_t *src = reinterpret_cast<const uint8_t *>(d.wpk) + d.chunk_off[k];
    uint8_t *dst = hsm + OFF_W + (size_t)slot * SLOT_BYTES;
    mbar_expect_tx(&bar_full[slot], nbytes);
    for (uint32_t o = 0; o < nbytes; o += PIECE) {
        const uint32_t n = (nbytes - o < PIECE) ? (nbytes - o) : PIECE;
        bulk_g2s(dst + o, src + o, n, &bar_full[slot]);
    }
}

// Consumer side (a dedicated producer warp keeps the ring full: produce_weights).
struct Ring {
    uint64_t *full, *empty;
    int c;
    __device__ __forceinline__ uint32_t acquire(int ahead = 0)
    {
        const int cc = c + ahead, s = cc % NSLOT;
        mbar_wait(&full[s], (cc / NSLOT) & 1);
        return sbase() + OFF_W + (uint32_t)s * SLOT_BYTES;
    }
    __device__ __forceinline__ void release(int lane, int n = 1)
    {
        __syncwarp();
        if (lane == 0)
            for (int i = 0; i < n; ++i) mbar_arrive(&empty[(c + i) % NSLOT]);
        c += n;
    }
};

__device__ __forceinline__ void cta_sync() { named_bar_sync(1, NCONS); }

template <int NT>
__device__ __forceinline__ void zero(float (&acc)[NT][4])
{
#pragma unroll
    for (int i = 0; i < NT; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
}
template <int NT>
__device__ __forceinline__ void copy(float (&dst)[NT][4], const float (&src)[NT][4])
{
#pragma unroll
    for (int i = 0; i < NT; ++i) { dst[i][0] = src[i][0]; dst[i][1] = src[i][1]; dst[i][2] = src[i][2]; dst[i][3] = src[i][3]; }
}

// acc += bias[c] (fp32 parameters at shared address `b`), c = column of the fragment element
template <int NT>
__device__ __forceinline__ void add_bias(float (&acc)[NT][4], const Thr &th, uint32_t b, int n0)
{
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const float2 v = ldp2(b + 4u * (n0 + 8 * nt + 2 * th.t));
        acc[nt][0] += v.x; acc[nt][1] += v.y; acc[nt][2] += v.x; acc[nt][3] += v.y;
    }
}
// fragment -> bf16 activation tile at shared address `tile` (row stride ld bytes), columns n0 + ...
template <int NT>
__device__ __forceinline__ void store_tile(uint32_t tile, int ld, const Thr &th, int n0, const float (&acc)[NT][4])
{
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const int c = n0 + 8 * nt + 2 * th.t;
        sts32(tile + (uint32_t)th.rA * ld + 2u * c, pack2(acc[nt][0], acc[nt][1]));
        sts32(tile + (uint32_t)th.rB * ld + 2u * c, pack2(acc[nt][2], acc[nt][3]));
    }
}
template <int NT>
__device__ __forceinline__ void relu(float (&acc)[NT][4])
{
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        acc[nt][0] = fmaxf(acc[nt][0], 0.f); acc[nt][1] = fmaxf(acc[nt][1], 0.f);
        acc[nt][2] = fmaxf(acc[nt][2], 0.f); acc[nt][3] = fmaxf(acc[nt][3], 0.f);
    }
}

// (sum, sum of squares) of rows rA / rB over this warp's NT tiles, reduced over the quad; lane t == 0 writes slot nq of
// `stat` ([TM][NQ] float2, shared address).  After a cta_sync, stats_read gives (mean, rstd) over the whole row.
template <int NT>
__device__ __forceinline__ void stats_write(const float (&v)[NT][4], const Thr &th, uint32_t stat)
{
    float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        s0 += v[nt][0] + v[nt][1]; q0 += v[nt][0] * v[nt][0] + v[nt][1] * v[nt][1];
        s1 += v[nt][2] + v[nt][3]; q1 += v[nt][2] * v[nt][2] + v[nt][3] * v[nt][3];
    }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o); q0 += __shfl_xor_sync(0xffffffffu, q0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o);
    }
    if (th.t == 0) {
        sts2f(stat + (uint32_t)(th.rA * NQ + th.nq) * 8u, s0, q0);
        sts2f(stat + (uint32_t)(th.rB * NQ + th.nq) * 8u, s1, q1);
    }
}
__device__ __forceinline__ void stats_read(uint32_t stat, int row, float inv_width, float &mean, float &rstd)
{
    float4 v[NQ / 2];
#pragma unroll
    for (int i = 0; i < NQ / 2; ++i) v[i] = lds4v(stat + (uint32_t)row * (NQ * 8u) + 16u * i);
    float s = 0.f, q = 0.f;
#pragma unroll
    for (int i = 0; i < NQ / 2; ++i) { s += v[i].x + v[i].z; q += v[i].y + v[i].w; }
    mean = s * inv_width;
    rstd = rsqrtf(fmaxf(q * inv_width - mean * mean, 0.f) + 1e-5f);
}

// LayerNorm(128) with affine on a fragment (bias already added); optional ReLU after.  One cta_sync inside.
__device__ __forceinline__ void layer_norm128(float (&x)[NT][4], const Thr &th, uint32_t gam, uint32_t bet, int n0, bool relu_after)
{
    const uint32_t stat = sbase() + OFF_STAT;
    stats_write<NT>(x, th, stat);
    cta_sync();
    float mA, sA, mB, sB;
    stats_read(stat, th.rA, 1.f / H, mA, sA);
    stats_read(stat, th.rB, 1.f / H, mB, sB);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const int c = n0 + 8 * nt + 2 * th.t;
        const float2 gg = ldp2(gam + 4u * c), bb = ldp2(bet + 4u * c);
        x[nt][0] = (x[nt][0] - mA) * sA * gg.x + bb.x; x[nt][1] = (x[nt][1] - mA) * sA * gg.y + bb.y;
        x[nt][2] = (x[nt][2] - mB) * sB * gg.x + bb.x; x[nt][3] = (x[nt][3] - mB) * sB * gg.y + bb.y;
    }
    if (relu_after) relu<NT>(x);
}

__device__ __forceinline__ RowInfo row_info(int r)
{
    uint32_t a, b, c, e;
    lds4u(sbase() + OFF_ROW + 16u * r, a, b, c, e);
    RowInfo ri;
    ri.root = (int)a; ri.agent = (int)b; ri.valid = (int)c; ri.r0 = (int)e;
    return ri;
}

// ---- stages (not inlined: the kernel is one long straight line, small code keeps the instruction cache warm) ----------
// fp32 pool rows -> bf16 tile HH; one-hot joint action -> tile One (wide variant: the row's action).  Thread (row = tid/8, 16
// columns each).
template <bool W>
static __device__ __noinline__ void stage_gather(const Desc &d, const SimIo io)
{
    HSM_DECL;
    const int tid = threadIdx.x, r = tid >> 3, part = tid & 7;
    if (tid >= TM * 8) return;
    const RowInfo ri = row_info(r);
    uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int action = -1;
    if (ri.valid) {
        const int ix = io.idx_x ? __ldcg(io.idx_x + ri.root) : 0;
        if (d.greedy_pool == nullptr || d.cur < 0)
            action = __ldcg(io.actions + (size_t)ri.root * d.N + ri.agent);
        else if (ri.agent == d.cur)                   // sequential-agent mode (mcts_sampled.py:116-147): the tree's action,
            action = __ldcg(io.actions + ri.root);
        else if (ri.agent < d.cur)                    // ... the earlier agents' chosen actions,
            action = d.factor ? __ldcg(d.factor + (size_t)ri.root * d.N + ri.agent) : 0;
        else                                          // ... argmax_a prediction(parent).policy for the later agents
            action = __ldcg(d.greedy_pool + ((size_t)ix * d.B + ri.root) * d.N + ri.agent);
        const float *h = d.pool + ((size_t)ix * d.B + ri.root) * (size_t)(d.N * H) + (size_t)ri.agent * H + part * 16;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(h) + i);
            w[2 * i] = pack2(v.x, v.y);
            w[2 * i + 1] = pack2(v.z, v.w);
        }
    }
    uint4 *dst = reinterpret_cast<uint4 *>(hsm + OFF_HH + (size_t)r * LDA + part * 32);
    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    if constexpr (W) {
        if (part == 0) *reinterpret_cast<int *>(hsm + OFF_ONE + (size_t)r * 4) = action;
    } else if (part * 8 < d.KA) {        // 8 one-hot columns per thread
        const int c0 = part * 8;
        uint32_t o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = pack2((c0 + 2 * i == action) ? 1.f : 0.f, (c0 + 2 * i + 1 == action) ? 1.f : 0.f);
        *reinterpret_cast<uint4 *>(hsm + OFF_ONE + (size_t)r * LDO + c0 * 2) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// x0 = relu(W_in [h | onehot] + b) + pos[agent]  -> residual fragment x, bf16 tile X
template <bool W>
static __device__ __noinline__ void stage_inproj(const Desc &d, Ring &ring, float (&xio)[NT][4])
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq, ldo = (d.KA + PAD) * 2;
    float x[NT][4];                  // registers (xio lives in the caller's frame: local memory)
    zero<NT>(x);
    uint32_t w = ring.acquire();
    gemm_fixed<NT, 8>(x, th, sb + OFF_HH, LDA, w, LDA, n0);
    ring.release(th.lane);
    w = ring.acquire();
    gemm_action<W, NT>(x, th, sb, w, ldo, n0, d.KA);
    ring.release(th.lane);
    add_bias<NT>(x, th, sb + OFF_P + 4u * d.o_bin, n0);
    const uint32_t pA = sb + OFF_P + 4u * (d.o_pos + row_info(th.rA).agent * H), pB = sb + OFF_P + 4u * (d.o_pos + row_info(th.rB).agent * H);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const int c = n0 + 8 * nt + 2 * th.t;
        const float2 a = ldp2(pA + 4u * c), b = ldp2(pB + 4u * c);
        x[nt][0] = fmaxf(x[nt][0], 0.f) + a.x; x[nt][1] = fmaxf(x[nt][1], 0.f) + a.y;
        x[nt][2] = fmaxf(x[nt][2], 0.f) + b.x; x[nt][3] = fmaxf(x[nt][3], 0.f) + b.y;
    }
    store_tile<NT>(sb + OFF_X, LDA, th, n0, x);
    copy<NT>(xio, x);
    cta_sync();
}

// q | k | v = X W^T + b  -> bf16 rows in Q (stride LDQ).  ONE pass over the activations: the three weight chunks are
// resident together (all ring slots), the A fragment of a k-step feeds 3*NT MMAs.
static __device__ __noinline__ void stage_qkv(Ring &ring, uint32_t lv)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq;
    float acc[3 * NT][4];
    zero<3 * NT>(acc);
    uint32_t wa[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) wa[i] = th.w_addr(ring.acquire(i), LDA, n0);
    const uint32_t aa = th.a_addr(sb + OFF_X, LDA);
    constexpr int PW = NT / 2, NP = 3 * PW;          // ldmatrix pairs of n8 tiles per weight chunk / in total
    uint32_t a[2][4], b[2][NP][4];
    ldsm4(aa, a[0]);
#pragma unroll
    for (int p = 0; p < NP; ++p) ldsm4(wa[p / PW] + (uint32_t)(16 * (p % PW)) * LDA, b[0][p]);
#pragma unroll GEMM_UNROLL
    for (int ks = 0; ks < 8; ++ks) {
        const int cur = ks & 1, nxt = cur ^ 1;
        if (ks + 1 < 8) {
            ldsm4(aa + 32u * (ks + 1), a[nxt]);
#pragma unroll
            for (int p = 0; p < NP; ++p) ldsm4(wa[p / PW] + (uint32_t)(16 * (p % PW)) * LDA + 32u * (ks + 1), b[nxt][p]);
        }
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            mma16816(acc[2 * p], a[cur], b[cur][p][0], b[cur][p][1]);
            mma16816(acc[2 * p + 1], a[cur], b[cur][p][2], b[cur][p][3]);
        }
    }
    ring.release(th.lane, 3);
#pragma unroll
    for (int which = 0; which < 3; ++which) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const int c = n0 + 8 * nt + 2 * th.t;
            const float2 bv = ldp2(lv + 4u * (which * H + c));
            const float *v = acc[which * NT + nt];
            sts32(sb + OFF_Q + (uint32_t)th.rA * LDQ + 2u * (which * H + c), pack2(v[0] + bv.x, v[1] + bv.y));
            sts32(sb + OFF_Q + (uint32_t)th.rB * LDQ + 2u * (which * H + c), pack2(v[2] + bv.x, v[3] + bv.y));
        }
    }
    cta_sync();
}

__device__ __forceinline__ void unpack16(const uint32_t (&w)[8], float (&f)[16])
{
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        f[2 * i] = __uint_as_float(w[i] << 16);
        f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ void lds32B(uint32_t saddr, uint32_t (&w)[8])
{
    lds4u(saddr, w[0], w[1], w[2], w[3]);
    lds4u(saddr + 16u, w[4], w[5], w[6], w[7]);
}

// scaled dot-product attention over the agents of my root; thread = (row, head).  Output (bf16) -> tile T.
// Small teams: two-phase softmax, every score chain independent; larger teams: one pass, online softmax.
template <int NN>
__device__ __forceinline__ void attention_small(uint32_t qbase, int r0, int hh, const float (&q)[16], float (&o)[16])
{
    float s[NN];
    uint32_t kw[NN][8], vw[NN][8];
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        const uint32_t kr = qbase + (uint32_t)(r0 + j) * LDQ + H * 2 + hh * 32;
        lds32B(kr, kw[j]);
        lds32B(kr + H * 2, vw[j]);
    }
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        float k[16];
        unpack16(kw[j], k);
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int i = 0; i < 16; i += 2) { a += q[i] * k[i]; b += q[i + 1] * k[i + 1]; }
        s[j] = a + b;
    }
    float m = s[0];
#pragma unroll
    for (int j = 1; j < NN; ++j) m = fmaxf(m, s[j]);
    float l = 0.f;
#pragma unroll
    for (int j = 0; j < NN; ++j) { s[j] = __expf(s[j] - m); l += s[j]; }
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < 16; ++i) o[i] = 0.f;
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        float v[16];
        unpack16(vw[j], v);
        const float p = s[j] * inv;
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] += p * v[i];
    }
}

static __device__ __noinline__ void stage_attention(const Desc &d)
{
    const uint32_t sb = sbase(), qbase = sb + OFF_Q;
    const int tid = threadIdx.x, r = tid >> 3, hh = tid & 7;
    if (tid >= TM * NHEAD) {         // warp-uniform: (row, head) pairs fill the first 8 warps
        cta_sync();
        return;
    }
    const RowInfo ri = row_info(r);
    const int N = d.N;
    float q[16], o[16];
    {
        uint32_t w[8];
        lds32B(qbase + (uint32_t)r * LDQ + hh * 32, w);
        unpack16(w, q);
#pragma unroll
        for (int i = 0; i < 16; ++i) q[i] *= 0.25f;              // 1/sqrt(head_dim)
    }
    if (N <= 4) {                  // CTA-uniform
        switch (N) {
            case 1: attention_small<1>(qbase, ri.r0, hh, q, o); break;
            case 2: attention_small<2>(qbase, ri.r0, hh, q, o); break;
            case 3: attention_small<3>(qbase, ri.r0, hh, q, o); break;
            default: attention_small<4>(qbase, ri.r0, hh, q, o); break;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] = 0.f;
        float m = -INFINITY, lsum = 0.f;
#pragma unroll 1
        for (int j = 0; j < N; ++j) {
            const uint32_t kr = qbase + (uint32_t)(ri.r0 + j) * LDQ + H * 2 + hh * 32;
            uint32_t kw[8], vw[8];
            lds32B(kr, kw);
            lds32B(kr + H * 2, vw);
            float k[16], v[16];
            unpack16(kw, k);
            unpack16(vw, v);
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) s += q[i] * k[i];
            const float mn = fmaxf(m, s);
            const float corr = __expf(m - mn), p = __expf(s - mn);
            lsum = lsum * corr + p;
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = o[i] * corr + p * v[i];
            m = mn;
        }
        const float inv = 1.f / lsum;
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] *= inv;
    }
    uint4 a, b;
    a.x = pack2(o[0], o[1]); a.y = pack2(o[2], o[3]); a.z = pack2(o[4], o[5]); a.w = pack2(o[6], o[7]);
    b.x = pack2(o[8], o[9]); b.y = pack2(o[10], o[11]); b.z = pack2(o[12], o[13]); b.w = pack2(o[14], o[15]);
    sts4(sb + OFF_T + (uint32_t)r * LDA + hh * 32, a);
    sts4(sb + OFF_T + (uint32_t)r * LDA + hh * 32 + 16, b);
    cta_sync();
}

// x = LN(x + T W^T + b) * g + be   (post-LN residual block: out-proj / linear2) -> fragment x, bf16 tile X
static __device__ __noinline__ void stage_residual_ln(Ring &ring, float (&xio)[NT][4], uint32_t bias, uint32_t gam, uint32_t bet)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq;
    float x[NT][4];                  // registers (xio lives in the caller's frame: local memory)
    copy<NT>(x, xio);
    const uint32_t w = ring.acquire();
    gemm_fixed<NT, 8>(x, th, sb + OFF_T, LDA, w, LDA, n0);
    ring.release(th.lane);
    add_bias<NT>(x, th, bias, n0);
    layer_norm128(x, th, gam, bet, n0, false);
    store_tile<NT>(sb + OFF_X, LDA, th, n0, x);
    copy<NT>(xio, x);
    cta_sync();
}

// f = relu(X W1^T + b1) -> bf16 tile T
static __device__ __noinline__ void stage_linear_relu(Ring &ring, uint32_t bias)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq;
    float acc[NT][4];
    zero<NT>(acc);
    const uint32_t w = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_X, LDA, w, LDA, n0);
    ring.release(th.lane);
    add_bias<NT>(acc, th, bias, n0);
    relu<NT>(acc);
    store_tile<NT>(sb + OFF_T, LDA, th, n0, acc);
    cta_sync();
}

// fc_dynamic (model.py:262-268): [h | onehot | attn] -> Linear LN ReLU -> Linear LN ReLU -> Linear, + h; next_hidden to
// global (fp32) and to tile T (bf16)
template <bool W>
static __device__ __noinline__ void stage_dynamics(const Desc &d, Ring &ring, const SimIo io)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq, ldo = (d.KA + PAD) * 2;
    const uint32_t dv = sb + OFF_P + 4u * d.o_dyn;
    float acc[NT][4];
    zero<NT>(acc);
    uint32_t w = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_HH, LDA, w, LDA, n0);        // h
    ring.release(th.lane);
    w = ring.acquire();
    gemm_action<W, NT>(acc, th, sb, w, ldo, n0, d.KA);               // one-hot action
    ring.release(th.lane);
    w = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_X, LDA, w, LDA, n0);         // attention output
    ring.release(th.lane);
    add_bias<NT>(acc, th, dv, n0);
    layer_norm128(acc, th, dv + 4u * 128, dv + 4u * 256, n0, true);
    store_tile<NT>(sb + OFF_T, LDA, th, n0, acc);
    cta_sync();
    zero<NT>(acc);
    w = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_T, LDA, w, LDA, n0);
    ring.release(th.lane);
    add_bias<NT>(acc, th, dv + 4u * 384, n0);
    layer_norm128(acc, th, dv + 4u * 512, dv + 4u * 640, n0, true);
    store_tile<NT>(sb + OFF_X, LDA, th, n0, acc);
    cta_sync();
    // the fp32 residual h comes straight from the pool: issue those loads before the last GEMM
    const RowInfo ra = row_info(th.rA), rb = row_info(th.rB);
    float2 hv[2][NT];
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
        const RowInfo &ri = hf ? rb : ra;
        const int ix = (ri.valid && io.idx_x) ? io.idx_x[ri.root - io.root0] : 0;   // (plain load: global or shared)
        const float *hp = d.pool + ((size_t)ix * d.B + (ri.valid ? ri.root : 0)) * (size_t)(d.N * H) + (size_t)ri.agent * H;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
            hv[hf][nt] = ri.valid ? __ldcg(reinterpret_cast<const float2 *>(hp + n0 + 8 * nt + 2 * th.t)) : make_float2(0.f, 0.f);
    }
    zero<NT>(acc);
    w = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_X, LDA, w, LDA, n0);
    ring.release(th.lane);
    add_bias<NT>(acc, th, dv + 4u * 768, n0);
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
        const RowInfo &ri = hf ? rb : ra;
        float *nh = io.next_hidden + (size_t)(ri.valid ? ri.root : 0) * (d.N * H) + (size_t)ri.agent * H;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            acc[nt][2 * hf] += hv[hf][nt].x;
            acc[nt][2 * hf + 1] += hv[hf][nt].y;
            if (ri.valid) *reinterpret_cast<float2 *>(nh + n0 + 8 * nt + 2 * th.t) = make_float2(acc[nt][2 * hf], acc[nt][2 * hf + 1]);
        }
    }
    store_tile<NT>(sb + OFF_T, LDA, th, n0, acc);
    cta_sync();
}

// ---- GraphNetNN layer (model.py:151-163) in barrier phases shared by the reward and the value head --------------------
// The stacked weight rows are interleaved on the host so that warp nq holds, for the FW features f = FW*nq .. +FW-1, tiles
// [0, GT) = gc.lin(x)[f] and tiles [GT, 2*GT) = nn(x)[f].   y = LN(relu(sum_over_agents(gc + b_gc) + nn + b_nn)), no affine.
// phase A: gc + b_gc -> G (fp32, shared);  [cta_sync]  phase B: agent sums, relu, row statistics;  [cta_sync]  phase C: normalise.
__device__ __forceinline__ void gnn_phase_a(const float (&acc)[NT][4], const Thr &th, uint32_t G, uint32_t b)
{
    const int f0 = FW * th.nq + 2 * th.t;
#pragma unroll
    for (int tl = 0; tl < GT; ++tl) {
        const float2 bg = ldp2(b + 4u * (f0 + 8 * tl));
        sts2f(G + 4u * (th.rA * LDG + f0 + 8 * tl), acc[tl][0] + bg.x, acc[tl][1] + bg.y);
        sts2f(G + 4u * (th.rB * LDG + f0 + 8 * tl), acc[tl][2] + bg.x, acc[tl][3] + bg.y);
    }
}
// sums over the NN agent rows of my two roots: all loads are issued before the first add (the loads are volatile and the
// SM issues in order: a load that is consumed right away exposes its full latency)
template <int NN>
__device__ __forceinline__ void agent_sums(uint32_t G, int f0, int r0A, int r0B, float2 (&sa)[GT], float2 (&sc)[GT])
{
    float2 a[NN][GT], c[NN][GT];
#pragma unroll
    for (int j = 0; j < NN; ++j)
#pragma unroll
        for (int tl = 0; tl < GT; ++tl) {
            a[j][tl] = lds2f(G + 4u * ((r0A + j) * LDG + f0 + 8 * tl));
            c[j][tl] = lds2f(G + 4u * ((r0B + j) * LDG + f0 + 8 * tl));
        }
#pragma unroll
    for (int j = 0; j < NN; ++j)
#pragma unroll
        for (int tl = 0; tl < GT; ++tl) {
            sa[tl].x += a[j][tl].x; sa[tl].y += a[j][tl].y; sc[tl].x += c[j][tl].x; sc[tl].y += c[j][tl].y;
        }
}
__device__ __forceinline__ void gnn_phase_b(const float (&acc)[NT][4], const Thr &th, uint32_t G, uint32_t b, uint32_t stat, int N, int r0A,
                                            int r0B, float (&y)[GT][4])
{
    const int f0 = FW * th.nq + 2 * th.t;
    float2 sa[GT], sc[GT];
#pragma unroll
    for (int tl = 0; tl < GT; ++tl) sa[tl] = sc[tl] = make_float2(0.f, 0.f);
    {
        int j = 0;
#pragma unroll 1
        for (; j + 3 <= N; j += 3) agent_sums<3>(G, f0, r0A + j, r0B + j, sa, sc);
#pragma unroll 1
        for (; j < N; ++j) agent_sums<1>(G, f0, r0A + j, r0B + j, sa, sc);
    }
#pragma unroll
    for (int tl = 0; tl < GT; ++tl) {
        const float2 bn = ldp2(b + 4u * (GH + f0 + 8 * tl));
        y[tl][0] = fmaxf(sa[tl].x + acc[GT + tl][0] + bn.x, 0.f); y[tl][1] = fmaxf(sa[tl].y + acc[GT + tl][1] + bn.y, 0.f);
        y[tl][2] = fmaxf(sc[tl].x + acc[GT + tl][2] + bn.x, 0.f); y[tl][3] = fmaxf(sc[tl].y + acc[GT + tl][3] + bn.y, 0.f);
    }
    stats_write<GT>(y, th, stat);
}
__device__ __forceinline__ void gnn_phase_c(const Thr &th, uint32_t stat, float (&y)[GT][4])
{
    float mA, sA, mB, sB;
    stats_read(stat, th.rA, 1.f / GH, mA, sA);
    stats_read(stat, th.rB, 1.f / GH, mB, sB);
#pragma unroll
    for (int tl = 0; tl < GT; ++tl) {
        y[tl][0] = (y[tl][0] - mA) * sA; y[tl][1] = (y[tl][1] - mA) * sA;
        y[tl][2] = (y[tl][2] - mB) * sB; y[tl][3] = (y[tl][3] - mB) * sB;
    }
}

// heads, first layers, ONE stage: reward GNN layer 1 on [next_hidden | onehot], value GNN layer 1 and fc_policy.0 on
// next_hidden.  Outputs: X[:, 0:64] = reward features, X[:, 64:128] = value features, Ph = relu(LN(policy hidden)).
template <bool W>
static __device__ __noinline__ void stage_heads1(const Desc &d, Ring &ring)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq, ldo = (d.KA + PAD) * 2;
    float aR[NT][4], aV[NT][4], aP[2][4];
    zero<NT>(aR); zero<NT>(aV); zero<2>(aP);
    uint32_t w = ring.acquire();
    gemm_fixed<NT, 8>(aR, th, sb + OFF_T, LDA, w, LDA, n0);
    ring.release(th.lane);
    w = ring.acquire();
    gemm_action<W, NT>(aR, th, sb, w, ldo, n0, d.KA);
    ring.release(th.lane);
    w = ring.acquire();
    gemm_fixed<NT, 8>(aV, th, sb + OFF_T, LDA, w, LDA, n0);
    ring.release(th.lane);
    w = ring.acquire();
    if (th.nq < 2) gemm_fixed<2, 8>(aP, th, sb + OFF_T, LDA, w, LDA, 16 * th.nq);   // 32 policy-hidden columns: warps nq = 0, 1
    ring.release(th.lane);
    const uint32_t G = sb + OFF_Q, stat = sb + OFF_STAT, pr = sb + OFF_P + 4u * d.o_rg, pvv = sb + OFF_P + 4u * d.o_vg;
    const uint32_t pp = sb + OFF_P + 4u * d.o_pol;
    // phase A
    gnn_phase_a(aR, th, G + 4u * G_R, pr);
    gnn_phase_a(aV, th, G + 4u * G_V, pvv);
    if (th.nq < 2) add_bias<2>(aP, th, pp, 16 * th.nq);
    stats_write<2>(aP, th, stat + 2 * STAT_SET);          // (warps nq >= 2 contribute zeros)
    cta_sync();
    // phase B
    const int r0A = row_info(th.rA).r0, r0B = row_info(th.rB).r0;
    float yR[GT][4], yV[GT][4];
    gnn_phase_b(aR, th, G + 4u * G_R, pr, stat, d.N, r0A, r0B, yR);
    gnn_phase_b(aV, th, G + 4u * G_V, pvv, stat + STAT_SET, d.N, r0A, r0B, yV);
    if (th.nq < 2) {                                      // policy hidden: relu(LN(acc + b) * g + be) over 32 columns
        float mA, sA, mB, sB;
        stats_read(stat + 2 * STAT_SET, th.rA, 1.f / PH, mA, sA);
        stats_read(stat + 2 * STAT_SET, th.rB, 1.f / PH, mB, sB);
#pragma unroll
        for (int tl = 0; tl < 2; ++tl) {
            const int c = 16 * th.nq + 8 * tl + 2 * th.t;
            const float2 gg = ldp2(pp + 4u * (PH + c)), bb = ldp2(pp + 4u * (2 * PH + c));
            const float v0 = fmaxf((aP[tl][0] - mA) * sA * gg.x + bb.x, 0.f), v1 = fmaxf((aP[tl][1] - mA) * sA * gg.y + bb.y, 0.f);
            const float v2 = fmaxf((aP[tl][2] - mB) * sB * gg.x + bb.x, 0.f), v3 = fmaxf((aP[tl][3] - mB) * sB * gg.y + bb.y, 0.f);
            sts32(sb + OFF_PH + (uint32_t)th.rA * LDP + 2u * c, pack2(v0, v1));
            sts32(sb + OFF_PH + (uint32_t)th.rB * LDP + 2u * c, pack2(v2, v3));
        }
    }
    cta_sync();
    // phase C
    gnn_phase_c(th, stat, yR);
    gnn_phase_c(th, stat + STAT_SET, yV);
    store_tile<GT>(sb + OFF_X, LDA, th, FW * th.nq, yR);
    store_tile<GT>(sb + OFF_X, LDA, th, GH + FW * th.nq, yV);
    cta_sync();
}

// softmax . support -> inv_h (core/config.py:430-442, 463-499) of 11 logits
__device__ __forceinline__ float support_to_scalar(const float (&v)[SUP])
{
    float m = v[0];
#pragma unroll
    for (int k = 1; k < SUP; ++k) m = fmaxf(m, v[k]);
    float s = 0.f, x = 0.f;
#pragma unroll
    for (int k = 0; k < SUP; ++k) {
        const float e = __expf(v[k] - m);
        s += e;
        x += e * (float)(k - 5);
    }
    x /= s;
    const float eps = 0.001f;
    const float r = (sqrtf(1.f + 4.f * eps * (fabsf(x) + 1.f + eps)) - 1.f) / (2.f * eps);
    float out = r * r - 1.f;
    out = (x < 0.f) ? -out : out;
    if (!(out == out)) out = 0.f;
    if (fabsf(out) < eps) out = 0.f;
    return out;
}

// policy outputs from the fp32 logits at shared address PL ([TM][LD]): 8 threads per row (softmax, beta, greedy).  Every thread
// keeps its (at most LD / 8) logits in registers: one batch of loads, two 8-lane reductions, one batch of stores.
template <int LD>
__device__ __forceinline__ void policy_outputs(const Desc &d, const SimIo io, uint32_t PL, long long *hs_clk, int &hs_n)
{
    const int N = d.N, A = d.A, tid = threadIdx.x;
#define HS() \
    if (hs_clk && hs_n < 64) hs_clk[hs_n++] = clock64();
    if (tid < TM * 8) {   // warp-uniform condition
        constexpr int PA = LD / 8;                                     // actions per thread
        const int r = tid >> 3, sub = tid & 7;
        const RowInfo ri = row_info(r);
        const uint32_t lg = PL + 4u * (r * LD);
        float v[PA];
#pragma unroll
        for (int i = 0; i < PA; ++i) v[i] = (sub + 8 * i < A) ? lds1v(lg + 4u * (sub + 8 * i)) : -INFINITY;
        float m = -INFINITY;
        int am = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < PA; ++i)
            if (v[i] > m) { m = v[i]; am = sub + 8 * i; }
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
            const float om = __shfl_xor_sync(0xffffffffu, m, o);
            const int oa = __shfl_xor_sync(0xffffffffu, am, o);
            if (om > m || (om == m && oa < am)) { m = om; am = oa; }
        }
        HS();
        const bool unit_tau = (d.inv_tau == 1.0f);
        float e[PA], eb[PA], s = 0.f, sbeta = 0.f;
#pragma unroll
        for (int i = 0; i < PA; ++i) {
            e[i] = (sub + 8 * i < A) ? __expf(v[i] - m) : 0.f;
            eb[i] = unit_tau ? e[i] : ((sub + 8 * i < A) ? __powf(e[i], d.inv_tau) : 0.f);
            s += e[i];
            sbeta += eb[i];
        }
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            sbeta += __shfl_xor_sync(0xffffffffu, sbeta, o);
        }
        HS();
        if (ri.valid) {
            if (io.greedy && sub == 0) io.greedy[(size_t)ri.root * N + ri.agent] = am;
            const int ta = (d.cur < 0) ? ri.agent : (ri.agent == d.cur ? 0 : -1);
            const float invs = 1.f / s, invb = 1.f / sbeta;
#pragma unroll
            for (int i = 0; i < PA; ++i) {
                const int a = sub + 8 * i;
                if (a < A) {
                    if (io.logits_out) io.logits_out[((size_t)ri.root * N + ri.agent) * A + a] = v[i];
                    if (ta >= 0) {
                        const size_t o = ((size_t)(ri.root - io.root0) * d.Nt + ta) * A + a;
                        io.probs[o] = e[i] * invs;
                        io.beta[o] = eb[i] * invb;
                    }
                }
            }
        }
    }
#undef HS
}

// heads, second layers + outputs, ONE stage: reward / value GNN layer 2 -> mean over agents -> 64->11 head -> scalar;
// fc_policy.3 -> softmax / beta / greedy (mcts_sampled.py:158-161).  The narrow variant stages the policy logits in the q|k|v
// region and computes the policy outputs in phase B; the wide variant keeps its PB logit blocks per warp in registers until
// phase D has consumed the layer-2 features and then uses the X + T tiles (one more barrier).
template <bool W>
static __device__ __noinline__ void stage_heads2(const Desc &d, Ring &ring, const SimIo io, long long *hs_clk)
{
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq, ldg = (GH + PAD) * 2;
    const int N = d.N, tid = threadIdx.x;
    int hs_n = 40;
#define HS() \
    if (hs_clk && hs_n < 64) hs_clk[hs_n++] = clock64();
    HS();
    constexpr int PB = W ? (KA_WIDE / 16 + NQ - 1) / NQ : 1;          // 16-column logit blocks per warp
    float aR[NT][4], aV[NT][4], aP[PB][2][4];
    zero<NT>(aR); zero<NT>(aV);
#pragma unroll
    for (int bk = 0; bk < PB; ++bk) zero<2>(aP[bk]);
    uint32_t w = ring.acquire();
    gemm_fixed<NT, 4>(aR, th, sb + OFF_X, LDA, w, ldg, n0);
    ring.release(th.lane);
    w = ring.acquire();
    gemm_fixed<NT, 4>(aV, th, sb + OFF_X + GH * 2, LDA, w, ldg, n0);
    ring.release(th.lane);
    w = ring.acquire();
    const int pc0 = 16 * th.nq;                                    // policy logit columns [16*nq, +16) (+ 16*NQ*bk) when < NAP
#pragma unroll
    for (int bk = 0; bk < PB; ++bk)
        if (pc0 + NQ * 16 * bk < d.NAP) gemm_fixed<2, 2>(aP[bk], th, sb + OFF_PH, LDP, w, LDP, pc0 + NQ * 16 * bk);
    ring.release(th.lane);
    const uint32_t G = sb + OFF_Q, stat = sb + OFF_STAT, pr = sb + OFF_P + 4u * (d.o_rg + 128), pvv = sb + OFF_P + 4u * (d.o_vg + 128);
    const uint32_t PL = G + 4u * PL0;
    HS();
    // phase A
    gnn_phase_a(aR, th, G + 4u * G_R, pr);
    gnn_phase_a(aV, th, G + 4u * G_V, pvv);
    if (!W && pc0 < d.NAP) {                                       // policy logits + bias -> fp32 scratch [TM][48]
        const uint32_t b2 = sb + OFF_P + 4u * (d.o_pol + 96);
#pragma unroll
        for (int tl = 0; tl < 2; ++tl) {
            const int c = pc0 + 8 * tl + 2 * th.t;
            const float2 bb = ldp2(b2 + 4u * c);
            sts2f(PL + 4u * (th.rA * 48 + c), aP[0][tl][0] + bb.x, aP[0][tl][1] + bb.y);
            sts2f(PL + 4u * (th.rB * 48 + c), aP[0][tl][2] + bb.x, aP[0][tl][3] + bb.y);
        }
    }
    cta_sync();
    HS();
    // phase B
    const int r0A = row_info(th.rA).r0, r0B = row_info(th.rB).r0;
    float yR[GT][4], yV[GT][4];
    gnn_phase_b(aR, th, G + 4u * G_R, pr, stat, N, r0A, r0B, yR);
    gnn_phase_b(aV, th, G + 4u * G_V, pvv, stat + STAT_SET, N, r0A, r0B, yV);
    // the raw (post-ReLU) layer-2 features, fp32 -> Y in the X + T tiles (free since the GEMMs above)
    const uint32_t YB = sb + OFF_X;
#pragma unroll
    for (int tl = 0; tl < GT; ++tl) {
        const int f = FW * th.nq + 8 * tl + 2 * th.t;
        sts2f(YB + 4u * (Y_R + th.rA * GH + f), yR[tl][0], yR[tl][1]);
        sts2f(YB + 4u * (Y_R + th.rB * GH + f), yR[tl][2], yR[tl][3]);
        sts2f(YB + 4u * (Y_V + th.rA * GH + f), yV[tl][0], yV[tl][1]);
        sts2f(YB + 4u * (Y_V + th.rB * GH + f), yV[tl][2], yV[tl][3]);
    }
    HS();
    if constexpr (!W) policy_outputs<KA_NARROW>(d, io, PL, hs_clk, hs_n);
    HS();
    cta_sync();
    HS();
    // phase D: per root and head, the mean over its agents of LayerNorm(y) (no affine: model.py:157,163) -> pooled (fp32) at the
    // start of the G region (nobody reads G any more).  The row statistics are applied on the fly: no separate normalisation
    // phase, no barrier for it.
    const int rpt = tile_rpt(d);
    const uint32_t POOL = G;
    const float invn = 1.f / (float)N;
    for (int i = tid; i < 2 * rpt * (GH / 2); i += NCONS) {
        const int f2 = i & (GH / 2 - 1), rest = i >> 5, kind = rest >= rpt ? 1 : 0, rl = rest - kind * rpt;
        const uint32_t src = YB + 4u * ((kind ? Y_V : Y_R) + (rl * N) * GH + 2 * f2), st = stat + (kind ? STAT_SET : 0u);
        float2 s = make_float2(0.f, 0.f);
        int j = 0;
#pragma unroll 1
        for (; j + 3 <= N; j += 3) {
            float m0, r0, m1, r1, m2, r2;
            stats_read(st, rl * N + j, 1.f / GH, m0, r0);
            stats_read(st, rl * N + j + 1, 1.f / GH, m1, r1);
            stats_read(st, rl * N + j + 2, 1.f / GH, m2, r2);
            const float2 v0 = lds2f(src + 4u * (j * GH)), v1 = lds2f(src + 4u * ((j + 1) * GH)), v2 = lds2f(src + 4u * ((j + 2) * GH));
            s.x += (v0.x - m0) * r0 + (v1.x - m1) * r1 + (v2.x - m2) * r2;
            s.y += (v0.y - m0) * r0 + (v1.y - m1) * r1 + (v2.y - m2) * r2;
        }
#pragma unroll 1
        for (; j < N; ++j) {
            float m0, r0;
            stats_read(st, rl * N + j, 1.f / GH, m0, r0);
            const float2 v = lds2f(src + 4u * (j * GH));
            s.x += (v.x - m0) * r0; s.y += (v.y - m0) * r0;
        }
        sts2f(POOL + 4u * ((kind * rpt + rl) * GH + 2 * f2), s.x * invn, s.y * invn);
    }
    cta_sync();
    HS();
    if constexpr (W) {                                             // the layer-2 features are consumed: logits + bias -> X + T tiles
        const uint32_t b2 = sb + OFF_P + 4u * (d.o_pol + 96);
#pragma unroll
        for (int bk = 0; bk < PB; ++bk) {
            const int pc = pc0 + NQ * 16 * bk;
            if (pc < d.NAP) {
#pragma unroll
                for (int tl = 0; tl < 2; ++tl) {
                    const int c = pc + 8 * tl + 2 * th.t;
                    const float2 bb = ldp2(b2 + 4u * c);
                    sts2f(sb + OFF_X + 4u * (th.rA * KA_WIDE + c), aP[bk][tl][0] + bb.x, aP[bk][tl][1] + bb.y);
                    sts2f(sb + OFF_X + 4u * (th.rB * KA_WIDE + c), aP[bk][tl][2] + bb.x, aP[bk][tl][3] + bb.y);
                }
            }
        }
    }
    // phase E: a half-warp per (root, head): lane k < 11 computes logit k of the 64 -> 11 head (weights from the padded copy:
    // conflict-free float4 rows), the 11 logits meet in the half-warp's first lane by shuffles, which applies
    // softmax . support -> inv_h and stores the scalar.  No barrier, no shared-memory round trip.
    {
        const int hw = tid >> 4, l16 = tid & 15, lane = tid & 31;
        for (int pair = hw; pair < rpt * 2; pair += NCONS / 16) {      // (both half-warps of a warp run the same number of rounds)
            const int rl = pair >> 1, kind = pair & 1;
            float logit = 0.f;
            if (l16 < SUP) {
                const uint32_t pv = POOL + 4u * ((kind * rpt + rl) * GH), vw = sb + OFF_VP + 4u * ((kind * SUP + l16) * LDV);
                float s0 = 0.f, s1 = 0.f;
#pragma unroll
                for (int f = 0; f < GH; f += 32) {          // 8 volatile loads in flight, then the math
                    float4 a[8], wv[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) a[q] = lds4v(pv + 4u * (f + 4 * q));
#pragma unroll
                    for (int q = 0; q < 8; ++q) wv[q] = lds4(vw + 4u * (f + 4 * q));
#pragma unroll
                    for (int q = 0; q < 8; q += 2) {
                        s0 += a[q].x * wv[q].x + a[q].y * wv[q].y + a[q].z * wv[q].z + a[q].w * wv[q].w;
                        s1 += a[q + 1].x * wv[q + 1].x + a[q + 1].y * wv[q + 1].y + a[q + 1].z * wv[q + 1].z + a[q + 1].w * wv[q + 1].w;
                    }
                }
                logit = s0 + s1 + lds1(sb + OFF_P + 4u * ((kind ? d.o_vg : d.o_rg) + 256 + SUP * GH + l16));
            }
            float v[SUP];
#pragma unroll
            for (int k = 0; k < SUP; ++k) v[k] = __shfl_sync(0xffffffffu, logit, (lane & 16) + k);
            const int root = blockIdx.x * rpt + rl;
            if (l16 == 0 && root < d.B) (kind ? io.value : io.reward)[root - io.root0] = support_to_scalar(v);
        }
    }
    HS();
    if constexpr (W) {
        cta_sync();
        policy_outputs<KA_WIDE>(d, io, sb + OFF_X, hs_clk, hs_n);
    }
#undef HS
}

// ---- pieces shared by the one-step kernel below and the persistent whole-search kernel (search_persist.cuh) -----------
__device__ __forceinline__ void setup_rows(const Desc &d)     // threads < TM: the tile's row table
{
    HSM_DECL;
    const int tid = threadIdx.x, N = d.N;
    if (tid < TM) {
        const int rpt = tile_rpt(d), rl = tid / N, agent = tid - rl * N;
        const int root = blockIdx.x * rpt + rl;
        RowInfo ri;
        ri.valid = (rl < rpt) && (root < d.B);
        ri.root = root; ri.agent = (rl < rpt) ? agent : 0;
        ri.r0 = (rl < rpt) ? rl * N : 0;
        reinterpret_cast<RowInfo *>(hsm + OFF_ROW)[tid] = ri;
    }
}

// weight producer (one thread): the fp32 parameter block once, then `rounds` passes over the NCHUNK weight chunks through
// the NSLOT-deep ring (one pass per recurrent_inference; the persistent kernel keeps streaming across simulations, so the
// first chunks of simulation s+1 arrive while the CTA runs the tree step of simulation s)
__device__ __forceinline__ void produce_weights(const Desc &d, uint64_t *bar_full, uint64_t *bar_empty, uint64_t *bar_vec, int rounds)
{
    HSM_DECL;
    mbar_expect_tx(bar_vec, (uint32_t)d.vec_floats * 4u);
    bulk_g2s(hsm + OFF_P, d.vec, (uint32_t)d.vec_floats * 4u, bar_vec);
    const int total = rounds * NCHUNK;
#pragma unroll 1
    for (int c = 0, k = 0; c < total; ++c, k = (k + 1 == NCHUNK) ? 0 : k + 1) {
        const int s = c % NSLOT;
        if (c >= NSLOT) mbar_wait_backoff(&bar_empty[s], ((c / NSLOT) - 1) & 1);
        issue_chunk(d, k, s, bar_full);
    }
}

// padded copies of the two 11 x 64 head matrices (conflict-free float4 rows for the final logits); parameters resident
__device__ __forceinline__ void setup_head_copies(const Desc &d)
{
    const uint32_t sb = sbase();
    for (int i = threadIdx.x; i < 2 * SUP * GH; i += NCONS) {
        const int f = i % GH, rest = i / GH, k = rest % SUP, kind = rest / SUP;
        sts1f(sb + OFF_VP + 4u * ((kind * SUP + k) * LDV + f), lds1v(sb + OFF_P + 4u * ((kind ? d.o_vg : d.o_rg) + 256 + k * GH + f)));
    }
}

// one recurrent_inference of the CTA's tile: every stage after the gather (compute warps; row table, parameters and head
// copies are set up).  `clk` (or NULL): SM-cycle timestamps of the stages, written by thread 0.  W: the wide variant (KA > 48).
template <bool W>
__device__ __forceinline__ void infer_stages(const Desc &d, const SimIo io, Ring &ring, long long *clk)
{
    int ts_n = 2;
#define TS() \
    if (clk && ts_n < 64) clk[ts_n++] = clock64();
    TS();
    float x[NT][4];
    stage_inproj<W>(d, ring, x);
    TS();
    const uint32_t pbase = sbase() + OFF_P;
#pragma unroll 1
    for (int l = 0; l < NLAYER; ++l) {
        const uint32_t lv = pbase + 4u * (d.o_layer + l * 1280);     // bq bk bv bo g1 be1 b1 b2 g2 be2
        stage_qkv(ring, lv);
        TS();
        stage_attention(d);
        TS();
        stage_residual_ln(ring, x, lv + 4u * 384, lv + 4u * 512, lv + 4u * 640);      // x = norm1(x + sa Wo^T + bo)
        TS();
        stage_linear_relu(ring, lv + 4u * 768);                                        // f = relu(linear1(x))
        TS();
        stage_residual_ln(ring, x, lv + 4u * 896, lv + 4u * 1024, lv + 4u * 1152);    // x = norm2(x + linear2(f))
        TS();
    }
    TS();
    stage_dynamics<W>(d, ring, io);
    TS();
    stage_heads1<W>(d, ring);
    TS();
    stage_heads2<W>(d, ring, io, clk);
    TS();
#undef TS
}

#ifndef MAZ_HMMA_NO_KERNEL
template <bool W>
__global__ void __launch_bounds__(NTHREADS, 1) k_recurrent_inference_small(const __grid_constant__ Desc d)
{
    HSM_DECL;
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_vec;
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], NCONS / 32); }
        mbar_init(&bar_vec, 1);
        mbar_fence_init();
    }
    setup_rows(d);
    __syncthreads();

    if (warp == NCONS / 32) {
        if ((tid & 31) == 0) produce_weights(d, bar_full, bar_empty, &bar_vec, 1);
        return;
    }
    // ==================================== compute warps =========================================================
    Ring ring{bar_full, bar_empty, 0};
    long long *clk = (d.dbg_clock != nullptr && blockIdx.x == 0 && tid == 0) ? d.dbg_clock : nullptr;
    if (clk) clk[0] = clock64();
    // PDL: everything above (and the producer warp's parameter / weight streaming, which reads constants only) may overlap the
    // tail of the tree kernel that produces idx_x / actions; wait for it before touching its outputs or the pool.  Only then
    // may the next tree kernel start: its pre-wait section reads tree state that the kernel we waited for was still writing.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const SimIo io = io_from_desc(d);
    stage_gather<W>(d, io);
    if (clk) clk[1] = clock64();
    mbar_wait(&bar_vec, 0);          // parameters resident
    setup_head_copies(d);
    cta_sync();
    infer_stages<W>(d, io, ring, clk);
}
#endif  // MAZ_HMMA_NO_KERNEL

}  // namespace hmma
}  // namespace maz
