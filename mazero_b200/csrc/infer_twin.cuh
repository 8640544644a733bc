// infer_twin.cuh -- the large-batch recurrent_inference kernel, second generation (sm_100a): TWO 128-row tiles in flight per CTA.
//
// Same computation as infer_fused.cuh (config/smac/model.py:562-574 = dynamics :251-282 with attention.py:27-43, prediction
// :335-373, GraphNetNN :136-174; inverse support transform core/config.py:430-442,463-499; the driver's softmax / beta
// mcts_sampled.py:158-161), restructured around what bounded the first kernel at 2s3z / MMM2 / 27m batch sizes
// (profiles/r01_ncu_summary.md, profiles/r02_ncu_summary.md): one tile per CTA walks 25 dependent stages, and in every stage the tensor pipe waits for the
// epilogue warps and the epilogue warps for the tensor pipe (MMA + hand-offs were ~1/3 of a tile's time); and the attention
// over the agent axis was scalar code whose cost grew with the team size (27m: about half of the tile time).
//
//   * Ping-pong: a CTA owns tiles A and B.  The 16 epilogue warps alternate epi A(s), epi B(s), epi A(s+1), ...; the MMA warp
//     issues stage s+1 of a tile as soon as that tile's epilogue s has published its operands, i.e. WHILE the epilogue warps
//     work on the other tile.  tcgen05.mma execution, commit -> wait latency and the barrier hand-off of one tile hide behind
//     the other tile's epilogue.
//   * TMEM: 256 columns per tile (ACC0 | ACC1).  The fp32 residual stream of the first kernel (128 more columns per tile) is
//     gone: x lives only as the bf16 operand tile and `x + f(x)` is added in the epilogue from that tile.
//   * q|k|v is two stages of four heads each ([Q | K] in ACC0, V in ACC1): no stage needs more than 192 columns, and each has a
//     full attention epilogue behind it (a separate V stage had a 1 k-cycle epilogue that could not cover the next MMA group).
//   * Attention over the agents of a root on warp-level tensor-core MMAs (mma.sync.m16n8k16, bf16): a warp holds 32 token
//     rows (whole roots) and one head per stage; S = Q K^T (32 x 32 x 16) with a block-diagonal root mask, softmax on the accumulator
//     fragments, O = P V (32 x 16 x 32).  The tcgen05 operand layout is made of 8 x 16-byte core matrices, which is exactly
//     what ldmatrix reads: V fragments come straight from the operand tile (ldmatrix.trans).  16 MMAs per head and warp
//     whatever the team size (the scalar loop was ~110 instructions per key, head and row).
//   * The one-hot joint-action operand is gone: `W [h | onehot(a)]` = `W_h h + W_a[:, a]`, the column is added in the epilogue
//     from a bf16 [A][128] table (three fewer MMA groups, no one-hot tiles in shared memory).
//   * Weights stream through a 4 x 16 KB ring in K-halves (a 128 x 128 matrix is two pieces), ONCE per CTA: a stage's pieces
//     (at most 4) serve tile A and then tile B and are released by tcgen05.commit after tile B's MMAs.  Biases / LayerNorm
//     affines / heads are read from global memory (L1-resident): shared memory holds 4 operand tiles (128 KB) + 32 KB scratch
//     + the ring.
//   * Hand-off: the 512 epilogue threads publish a tile's operands by arriving on an mbarrier the MMA thread waits on; they
//     never wait for each other per stage.  Shared exchange areas are double-buffered by tile or quadrant-local behind
//     quadrant barriers; two CTA-wide barriers per pass fence the places where a warp-local area covers another quadrant's
//     buffer (DESIGN.md section 5d lists the hazards).
#pragma once
#include "infer_fused.cuh"

namespace maz {
namespace twin {

using namespace umma;
using fused::Desc;
using fused::GH;
using fused::GP;
using fused::H;
using fused::HD;
using fused::NEPI;
using fused::NTHREADS;
using fused::PARTS;
using fused::PH;
using fused::PP;
using fused::SUP;
using fused::Thr;
using fused::pack2;
using fused::store_cols;
using fused::sum_sq;

constexpr int NSLOT = 4;
constexpr uint32_t SLOT_BYTES = 128 * 64 * 2;      // one K-half of a 128-row weight matrix
constexpr uint32_t TILE_BYTES = 128 * 128 * 2;     // one bf16 operand tile
constexpr uint32_t SCRATCH_BYTES = 32768;          // attention Q/K blocks (16 warps x 2 KB) | graph-head partials 24 KB + row statistics 4 KB
constexpr uint32_t RED_OFF = 24576;
constexpr uint32_t TM_TILE = 256, TM_A0 = 0, TM_A1 = 128;
constexpr int NOPS = 32;                           // weight matrices = MMA groups per tile

__host__ __device__ inline size_t smem_bytes() { return 4 * (size_t)TILE_BYTES + SCRATCH_BYTES + NSLOT * (size_t)SLOT_BYTES + 1024; }

// One MMA group: D[tile ACC `dst`] (+)= A[tile `asrc`: 0 = sX, 1 = sT] * W[mat]^T; `last` closes a stage.
struct Op { unsigned char mat, asrc, dst, acc, last; };
#define MAZ_TW_LAYER(b) {b, 0, 0, 0, 0}, {b + 1, 0, 1, 0, 1}, {b + 2, 0, 0, 0, 0}, {b + 3, 0, 1, 0, 1}, {b + 4, 1, 0, 0, 1}, {b + 5, 0, 0, 0, 1}, {b + 6, 1, 0, 0, 1}
__constant__ Op kOps[NOPS] = {
    {0, 1, 0, 0, 1},                                       // in-proj on h
    MAZ_TW_LAYER(1), MAZ_TW_LAYER(8), MAZ_TW_LAYER(15),    // per layer: [Q|K heads 0-3, V heads 0-3] | [Q|K, V heads 4-7] | out-proj | linear1 | linear2
    {22, 1, 0, 0, 0}, {23, 0, 0, 1, 1},                    // fc_dynamic.0 on [h | . | attention output]
    {24, 1, 0, 0, 1}, {25, 0, 0, 0, 1},                    // fc_dynamic.3, fc_dynamic.6
    {26, 1, 0, 0, 1}, {27, 0, 0, 0, 1},                    // reward graph net layer 1 (on h'), layer 2
    {28, 1, 0, 0, 1}, {29, 0, 0, 0, 1},                    // value graph net
    {30, 1, 0, 0, 1}, {31, 0, 0, 0, 1},                    // fc_policy.0, fc_policy.3
};
#undef MAZ_TW_LAYER
__device__ __forceinline__ void mat_dims(int m, int NAP, uint32_t &n, uint32_t &k)
{
    n = 128; k = 128;
    if (m >= 1 && m <= 21 && ((m - 1) % 7 == 1 || (m - 1) % 7 == 3)) n = 64;      // V of four heads
    else if (m == 27 || m == 29) k = GH;
    else if (m == 30) n = PH;
    else if (m == 31) { n = (uint32_t)NAP; k = PH; }
}

// ---- small helpers ---------------------------------------------------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void add_gvec(float (&v)[NV], const float *__restrict__ p)
{
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p + i));
        v[i] += t.x; v[i + 1] += t.y; v[i + 2] += t.z; v[i + 3] += t.w;
    }
}
// 256-bit global accesses (sm_100): a thread that owns a row segment moves whole 32-byte sectors per instruction.  The LSU
// takes about one sector per clock and SM, and a row-per-thread access touches 32 different sectors per warp instruction:
// with 128-bit accesses every sector was requested twice (next_hidden, the gathers: ~12 k cycles per tile at 27m).
__device__ __forceinline__ void ldg256(const float *p, float (&v)[8])
{
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
__device__ __forceinline__ void stg256(float *p, const float (&v)[8])
{
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]),
                 "f"(v[6]), "f"(v[7]) : "memory");
}
// v += a per-row vector in global memory (one-hot weight column), 32-byte aligned
template <int NV>
__device__ __forceinline__ void add_grow(float (&v)[NV], const float *__restrict__ p)
{
#pragma unroll
    for (int i = 0; i < NV; i += 8) {
        float t[8];
        ldg256(p + i, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i + j] += t[j];
    }
}
// v += NV bf16 values stored as packed pairs in 32-bit words at p (one-hot weight tables: [A][64] words = [A][128] bf16)
template <int NV>
__device__ __forceinline__ void add_grow_bf16(float (&v)[NV], const float *__restrict__ p)
{
#pragma unroll
    for (int i = 0; i < NV; i += 16) {
        float t[8];
        ldg256(p + i / 2, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t w = __float_as_uint(t[j]);
            v[i + 2 * j] += __uint_as_float(w << 16);
            v[i + 2 * j + 1] += __uint_as_float(w & 0xffff0000u);
        }
    }
}
// v += the bf16 row segment [c, c + NV) of `row` in a K = 128 operand tile (the residual stream)
template <int NV>
__device__ __forceinline__ void add_xres(float (&v)[NV], uint32_t tile, int row, int c)
{
#pragma unroll
    for (int j = 0; j < NV / 8; ++j) {
        uint32_t w[4];
        lds4u(tile + operand_chunk_off(row, (c >> 3) + j, H, 128), w[0], w[1], w[2], w[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            v[8 * j + 2 * i] += __uint_as_float(w[i] << 16);
            v[8 * j + 2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
        }
    }
}
// v += b with Blackwell's packed fp32 adds
template <int NV>
__device__ __forceinline__ void add_regs(float (&v)[NV], const float (&b)[NV])
{
#pragma unroll
    for (int i = 0; i < NV; i += 2) {
        const float2 r = __fadd2_rn(make_float2(v[i], v[i + 1]), make_float2(b[i], b[i + 1]));
        v[i] = r.x; v[i + 1] = r.y;
    }
}
template <int NV>
__device__ __forceinline__ void load_gvec(float (&b)[NV], const float *__restrict__ p)
{
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(p + i));
        b[i] = t.x; b[i + 1] = t.y; b[i + 2] = t.z; b[i + 3] = t.w;
    }
}
// v = (v - mean) * rstd * g + b as a = rstd*g; v = v*a + (b - mean*a), packed
template <int NV>
__device__ __forceinline__ void ln_affine_p(float (&v)[NV], float mean, float rstd, const float *__restrict__ pg, const float *__restrict__ pb)
{
    const float2 r2 = make_float2(rstd, rstd), nm2 = make_float2(-mean, -mean);
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 g = __ldg(reinterpret_cast<const float4 *>(pg + i)), b = __ldg(reinterpret_cast<const float4 *>(pb + i));
        const float2 a0 = __fmul2_rn(r2, make_float2(g.x, g.y)), a1 = __fmul2_rn(r2, make_float2(g.z, g.w));
        const float2 c0 = __ffma2_rn(nm2, a0, make_float2(b.x, b.y)), c1 = __ffma2_rn(nm2, a1, make_float2(b.z, b.w));
        const float2 y0 = __ffma2_rn(make_float2(v[i], v[i + 1]), a0, c0), y1 = __ffma2_rn(make_float2(v[i + 2], v[i + 3]), a1, c1);
        v[i] = y0.x; v[i + 1] = y0.y; v[i + 2] = y1.x; v[i + 3] = y1.y;
    }
}
template <int NV>
__device__ __forceinline__ void ln_affine_g(float (&v)[NV], float mean, float rstd, const float *__restrict__ pg, const float *__restrict__ pb)
{
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 g = __ldg(reinterpret_cast<const float4 *>(pg + i)), b = __ldg(reinterpret_cast<const float4 *>(pb + i));
        v[i] = (v[i] - mean) * rstd * g.x + b.x; v[i + 1] = (v[i + 1] - mean) * rstd * g.y + b.y;
        v[i + 2] = (v[i + 2] - mean) * rstd * g.z + b.z; v[i + 3] = (v[i + 3] - mean) * rstd * g.w + b.w;
    }
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4])
{
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4])
{
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2f(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void sts32(uint32_t saddr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }

// combine (sum, sumsq) of the four column parts of a row.  Layout [part][row]: the 32 lanes of a warp write / read 256 contiguous
// bytes (the [row][part] layout of the first kernel is a 4-way bank conflict on every access).
__device__ __forceinline__ void row_stats_pr(const Thr &t, uint32_t aRed, float &sum, float &sq)
{
    sts2f(aRed + (uint32_t)(t.part * 128 + t.row) * 8u, sum, sq);
    named_bar_sync(1 + t.quad, 128);
    float S = 0.f, Q = 0.f;
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
        const float2 v = lds2f(aRed + (uint32_t)(p * 128 + t.row) * 8u);
        S += v.x; Q += v.y;
    }
    sum = S; sq = Q;
}

// ---- epilogues (NOT inlined: small code, see infer_fused.cuh) -----------------------------------------------------------------
// Thread layout as in infer_fused.cuh: 16 warps = 4 TMEM lane quadrants x 4 column parts; row = quad*32 + lane.
// `trow`: TMEM address of the tile's ACC0 at this warp's lanes; `oh`: this row's column of the one-hot weight block (or NULL).

// x0 = relu(acc + b_in + W_a[:, action]) + pos[agent] -> sX
static __device__ __noinline__ void epi_inproj(uint32_t trow, const float *__restrict__ pb, const float *__restrict__ oh, const float *__restrict__ pos,
                                        uint32_t aX)
{
    const Thr t;
    const int c = t.part * 32;
    float v[32];
    tmem_ld32(trow + TM_A0 + c, v);
    add_gvec(v, pb + c);
    if (oh) add_grow_bf16(v, oh + c / 2);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
    add_grow(v, pos + c);
    store_cols(aX, t.row, c, H, v);
}
// acc + b -> bf16 tile (V of the attention; relu != 0: relu(linear1))
static __device__ __noinline__ void epi_bias(uint32_t trow, const float *__restrict__ pb, int relu, uint32_t tile)
{
    const Thr t;
    const int c = t.part * 32;
    float v[32], b[32];
    load_gvec(b, pb + c);                      // (issued before the TMEM load: its wait covers the L1 latency)
    tmem_ld32(trow + TM_A0 + c, v);
    add_regs(v, b);
    if (relu) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
    }
    store_cols(tile, t.row, c, H, v);
}
// y = LN(acc + b [+ oh] [+ x from res_tile]) * g + be, optional ReLU -> dst tile (bf16)
static __device__ __noinline__ void epi_ln(uint32_t trow, const float *__restrict__ pb, const float *__restrict__ pg, const float *__restrict__ pbe,
                                    const float *__restrict__ oh, uint32_t res_tile, int relu_after, uint32_t dst_tile, uint32_t aRed, int dbg = 0)
{
    const Thr t;
    const int c = t.part * 32;
    float v[32], b[32];
    load_gvec(b, pb + c);                      // everything that does not depend on the accumulator first
    if (oh) add_grow_bf16(b, oh + c / 2);
    if (res_tile) add_xres(b, res_tile, t.row, c);
    if (dbg & 128) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0.f;
    } else
        tmem_ld32(trow + TM_A0 + c, v);
    add_regs(v, b);
    float sum, sq;
    sum_sq(v, sum, sq);
    if (!(dbg & 16)) row_stats_pr(t, aRed, sum, sq);
    const float mean = sum * (1.f / H);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / H) - mean * mean, 0.f) + 1e-5f);
    if (!(dbg & 32)) ln_affine_p(v, mean, rstd, pg + c, pbe + c);
    if (relu_after) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
    }
    if (!(dbg & 64)) store_cols(dst_tile, t.row, c, H, v);
}

// Scaled dot-product attention over the agents of a root (attention.py:36-43 -> nn.MultiheadAttention, 8 heads x 16).
// A layer's q|k|v projection is two stages of four heads each (`half`): ACC0 = [Q | K] of heads 4*half .. +3 (64 + 64 columns),
// ACC1 = V of the same heads (64 columns).  A warp (quad, part) owns token rows quad*32 .. +31 and head 4*half + part:
//   V (+ bias) of the 32 rows -> bf16 into the head's 16 columns of aT (the tile that receives the attention output);
//   Q (scaled by 1/sqrt(16), + bias) and K (+ bias) of the 32 rows -> two 32 x 16 bf16 blocks in the warp's scratch (core-matrix
//   layout), S[32 x 32] = Q K^T on 8 MMAs, keys of other roots masked, row softmax on the fragments (a row's 32 scores sit in
//   the 4 lanes of a quad), P as bf16 A fragments, O[32 x 16] = P V on 8 MMAs with V fragments by ldmatrix.trans from aT.
// Rows beyond the last whole root of the warp form a pseudo-root of their own (finite garbage, never stored anywhere).
static __device__ __noinline__ void epi_attention(uint32_t trow, uint32_t aT, const float *__restrict__ pqk, int N, uint32_t scratch, int half)
{
    const Thr t;
    const int l = t.lane, m = l >> 3;
    const uint32_t qb = scratch + (uint32_t)(t.part * 4 + t.quad) * 2048u, kb = qb + 1024u;
    const uint32_t mine = (uint32_t)(l >> 3) * 256u + (uint32_t)(l & 7) * 16u;    // my row in a 32 x 16 block (k8 = 1: + 128)
    int rs[2][2];                                                                    // first row of the root of my 4 fragment rows
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = mt * 16 + (l >> 2) + 8 * h;
            rs[mt][h] = (r / N) * N;
        }
    {
        const int hh = half * 4 + t.part;
        {
            float q[16], k[16];
            {
                float v[16];
                tmem_ld16(trow + TM_A1 + t.part * HD, v);
                add_gvec(v, pqk + 2 * H + hh * HD);
                uint4 a;
                a.x = pack2(v[0], v[1]); a.y = pack2(v[2], v[3]); a.z = pack2(v[4], v[5]); a.w = pack2(v[6], v[7]);
                sts4(aT + operand_chunk_off(t.row, hh * 2, H, 128), a);
                a.x = pack2(v[8], v[9]); a.y = pack2(v[10], v[11]); a.z = pack2(v[12], v[13]); a.w = pack2(v[14], v[15]);
                sts4(aT + operand_chunk_off(t.row, hh * 2 + 1, H, 128), a);
            }
            tmem_ld16(trow + TM_A0 + t.part * HD, q);
            tmem_ld16(trow + TM_A0 + 64 + t.part * HD, k);
            add_gvec(q, pqk + hh * HD);
            // (no K bias: q . (k + bk) = q . k + a per-query constant, which the softmax over the keys cancels)
#pragma unroll
            for (int i = 0; i < 16; ++i) q[i] *= 0.25f * 1.4426950408889634f;   // 1/sqrt(head_dim) * log2(e): scores in log2 units
            uint4 a;
            a.x = pack2(q[0], q[1]); a.y = pack2(q[2], q[3]); a.z = pack2(q[4], q[5]); a.w = pack2(q[6], q[7]);
            sts4(qb + mine, a);
            a.x = pack2(q[8], q[9]); a.y = pack2(q[10], q[11]); a.z = pack2(q[12], q[13]); a.w = pack2(q[14], q[15]);
            sts4(qb + mine + 128, a);
            a.x = pack2(k[0], k[1]); a.y = pack2(k[2], k[3]); a.z = pack2(k[4], k[5]); a.w = pack2(k[6], k[7]);
            sts4(kb + mine, a);
            a.x = pack2(k[8], k[9]); a.y = pack2(k[10], k[11]); a.z = pack2(k[12], k[13]); a.w = pack2(k[14], k[15]);
            sts4(kb + mine + 128, a);
        }
        __syncwarp();
        float S[2][4][4];
        {
            uint32_t kf[2][4];                                   // B fragments of K: [key pair of 8-blocks][b0, b1 of block 2j | b0, b1 of block 2j+1]
#pragma unroll
            for (int j = 0; j < 2; ++j) ldsm_x4(kb + (uint32_t)(2 * j + (m >> 1)) * 256u + (uint32_t)(m & 1) * 128u + (uint32_t)(l & 7) * 16u, kf[j]);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                uint32_t a[4];
                ldsm_x4(qb + (uint32_t)(2 * mt + (m & 1)) * 256u + (uint32_t)(m >> 1) * 128u + (uint32_t)(l & 7) * 16u, a);
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    S[mt][nt][0] = S[mt][nt][1] = S[mt][nt][2] = S[mt][nt][3] = 0.f;
                    mma16816(S[mt][nt], a, kf[nt >> 1][(nt & 1) * 2], kf[nt >> 1][(nt & 1) * 2 + 1]);
                }
            }
        }
        float inv[2][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float mx = -INFINITY;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int c = nt * 8 + 2 * (l & 3) + e;
                        const float s = ((unsigned)(c - rs[mt][h]) < (unsigned)N) ? S[mt][nt][2 * h + e] : -INFINITY;
                        S[mt][nt][2 * h + e] = s;
                        mx = fmaxf(mx, s);
                    }
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                float sum = 0.f;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float p = ex2f(S[mt][nt][2 * h + e] - mx);
                        S[mt][nt][2 * h + e] = p;
                        sum += p;
                    }
                sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                inv[mt][h] = 1.f / sum;
            }
        float O[2][2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2) O[mt][n2][0] = O[mt][n2][1] = O[mt][n2][2] = O[mt][n2][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            uint32_t vf[4];                                      // V^T fragments: [b0, b1 of dims 0..7 | b0, b1 of dims 8..15] of keys ks*16 .. +15
            ldsm_x4_t(aT + (uint32_t)(t.quad * 4 + ks * 2 + (m & 1)) * 2048u + (uint32_t)(hh * 2 + (m >> 1)) * 128u + (uint32_t)(l & 7) * 16u, vf);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                uint32_t pa[4];
                pa[0] = pack2(S[mt][2 * ks][0], S[mt][2 * ks][1]);
                pa[1] = pack2(S[mt][2 * ks][2], S[mt][2 * ks][3]);
                pa[2] = pack2(S[mt][2 * ks + 1][0], S[mt][2 * ks + 1][1]);
                pa[3] = pack2(S[mt][2 * ks + 1][2], S[mt][2 * ks + 1][3]);
                mma16816(O[mt][0], pa, vf[0], vf[1]);
                mma16816(O[mt][1], pa, vf[2], vf[3]);
            }
        }
        __syncwarp();                                            // every lane has its V fragments: the head's columns of aT may be overwritten
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int row = t.quad * 32 + mt * 16 + (l >> 2) + 8 * h;
                    sts32(aT + operand_chunk_off(row, hh * 2 + n2, H, 128) + (uint32_t)(l & 3) * 4u,
                          pack2(O[mt][n2][2 * h] * inv[mt][h], O[mt][n2][2 * h + 1] * inv[mt][h]));
                }
    }
}

// next_hidden = acc + b + hidden (fp32 residual straight from the pool); fp32 to global, bf16 to the tile
static __device__ __noinline__ void epi_next_hidden(uint32_t trow, const float *__restrict__ pb, const float *__restrict__ hrow, float *__restrict__ nh,
                                             int valid, uint32_t tile)
{
    const Thr t;
    const int c = t.part * 32;
    float v[32];
    tmem_ld32(trow + TM_A0 + c, v);
    add_gvec(v, pb + c);
    if (valid) {
        add_grow(v, hrow + c);
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = v[i + j];
            stg256(nh + c + i, o);
        }
    }
    store_cols(tile, t.row, c, H, v);
}
// fp32 pool row -> bf16 operand tile (K = 128), my 32 columns
static __device__ __noinline__ void gather_hidden(const float *__restrict__ hrow, int valid, uint32_t tile)
{
    const Thr t;
    const int c = t.part * 32;
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
    if (valid) add_grow(v, hrow + c);
    store_cols(tile, t.row, c, H, v);
}

// v[i] <- sum of v[i] over the lanes [lo, lo + N) of my root.  Small teams: N broadcasts per value; larger ones: a segmented
// inclusive scan (5 steps) + one broadcast from the root's last lane -- the shuffle crossbar moves one warp instruction per
// clock and SM, and 16 x N shuffles per thread were ~14 k cycles per graph-net stage at N = 27.
template <int NV>
__device__ __forceinline__ void root_sum(float (&v)[NV], int lane, int lo, int N)
{
    if (N <= 6) {
        float s[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) s[i] = 0.f;
#pragma unroll 1
        for (int j = 0; j < N; ++j) {
#pragma unroll
            for (int i = 0; i < NV; ++i) s[i] += __shfl_sync(0xffffffffu, v[i], lo + j);
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) v[i] = s[i];
        return;
    }
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) {
        const bool take = lane - dlt >= lo;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const float u = __shfl_up_sync(0xffffffffu, v[i], dlt);
            if (take) v[i] += u;
        }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = __shfl_sync(0xffffffffu, v[i], lo + N - 1);
}

// GraphNetNN layer (model.py:151-163) from one stacked GEMM: columns [0,64) = gc.lin(x), [64,128) = nn(x).
// y = LN(relu(sum_over_agents(gc + b_gc) + nn + b_nn)), no affine.  pb: [b_gc | b_nn | (head: V weights 11 x 64 | V bias)].
// head == 0: y (bf16) -> `tile` (K = 64 layout).
// head == 1: mean-pool over the agents, 64 -> 11 head, support transform.  The head is linear, so every thread first reduces ITS
//            16 features of ITS row to 11 partial logits; the four column parts of a row are combined through shared memory,
//            the rows of a root by the part-0 warp (root_sum over 11 values instead of 16 features x 4 parts).  The scalar is
//            returned by the part-0 thread of every row.
static __device__ __noinline__ float epi_gnn(uint32_t trow, const float *__restrict__ pb, const float *__restrict__ oh, int N, int root_lane0, int head,
                                      uint32_t tile, uint32_t aRed, uint32_t scratch, long long *clk = nullptr)
{
    const Thr t;
#define SUBTS(i) if (clk) clk[i] = clock64();
    SUBTS(0)
    const int c = t.part * GP;
    float y[GP], nn[GP];
    tmem_ld16(trow + TM_A0 + c, y);
    add_gvec(y, pb + c);
    if (oh) add_grow_bf16(y, oh + c / 2);
    SUBTS(1)
    root_sum(y, t.lane, root_lane0, N);
    SUBTS(2)
    tmem_ld16(trow + TM_A0 + GH + c, nn);
    add_gvec(nn, pb + GH + c);
    if (oh) add_grow_bf16(nn, oh + (GH + c) / 2);
    float sum = 0.f, sq = 0.f;
#pragma unroll
    for (int i = 0; i < GP; ++i) {
        y[i] = fmaxf(y[i] + nn[i], 0.f);
        sum += y[i];
        sq += y[i] * y[i];
    }
    SUBTS(3)
    row_stats_pr(t, aRed, sum, sq);
    SUBTS(4)
    const float mean = sum * (1.f / GH);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / GH) - mean * mean, 0.f) + 1e-5f);
#pragma unroll
    for (int i = 0; i < GP; ++i) y[i] = (y[i] - mean) * rstd;
    if (!head) {
        store_cols(tile, t.row, c, GH, y);
        return 0.f;
    }
    const float *pV = pb + 2 * GH, *pVb = pV + SUP * GH;
    // partial-logit exchange area [k = 0..11][part][row] (24 KB): every access of a warp is 128 contiguous bytes
#define PL(k, part, row) (scratch + (uint32_t)((((k) * PARTS + (part)) * 128 + (row)) * 4))
    SUBTS(5)
    named_bar_sync(1 + t.quad, 128);                 // the previous call's partials / results of this quadrant have been consumed
    SUBTS(6)
    // (1) partial logits of MY row over MY 16 features
#pragma unroll
    for (int k = 0; k < SUP; ++k) {
        float a = 0.f;
#pragma unroll
        for (int i = 0; i < GP; i += 4) {
            const float4 w = __ldg(reinterpret_cast<const float4 *>(pV + k * GH + c + i));
            a += w.x * y[i] + w.y * y[i + 1] + w.z * y[i + 2] + w.w * y[i + 3];
        }
        sts1f(PL(k, t.part, t.row), a);
    }
    sts1f(PL(11, t.part, t.row), 0.f);
    named_bar_sync(1 + t.quad, 128);
    SUBTS(7)
    // (2) column part p finishes logits 3p .. 3p+2: sum over the four parts of the row, then over the rows of the root; the root's
    //     first row keeps the result IN PLACE (slot (3p + j, part p, row) is read by nobody else)
    {
        float l3[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float a = 0.f;
#pragma unroll
            for (int q = 0; q < PARTS; ++q) a += lds1v(PL(t.part * 3 + j, q, t.row));
            l3[j] = a;
        }
        SUBTS(8)
        root_sum(l3, t.lane, root_lane0, N);
        if (t.lane == root_lane0) {
#pragma unroll
            for (int j = 0; j < 3; ++j) sts1f(PL(t.part * 3 + j, t.part, t.row), l3[j]);
        }
    }
    named_bar_sync(1 + t.quad, 128);
    SUBTS(9)
    // (3) mean, bias, softmax . support -> inv_h: the first row of every root, part 0
    float out = 0.f;
    if (t.part == 0 && t.lane == root_lane0) {
        const float invn = 1.f / (float)N;
        float l11[SUP];
#pragma unroll
        for (int k = 0; k < SUP; ++k) l11[k] = lds1v(PL(k, k / 3, t.row)) * invn + __ldg(pVb + k);
        out = fused::support_to_scalar(l11);
    }
    SUBTS(10)
#undef SUBTS
#undef PL
    return out;      // (valid on the first row of a root, part 0; no trailing barrier: the next writer of the partials synchronises first)
}

// policy hidden: p1 = relu(LN(acc + b) * g + be) over 32 columns -> operand tile (K = 32)
static __device__ __noinline__ void epi_policy_hidden(uint32_t trow, const float *__restrict__ pp, uint32_t tile, uint32_t aRed)
{
    const Thr t;
    const int c = t.part * PP;
    float p[PP];
    tmem_ld8(trow + TM_A0 + c, p);
    add_gvec(p, pp + c);
    float sum = 0.f, sq = 0.f;
#pragma unroll
    for (int i = 0; i < PP; ++i) { sum += p[i]; sq += p[i] * p[i]; }
    row_stats_pr(t, aRed, sum, sq);
    const float mean = sum * (1.f / PH);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / PH) - mean * mean, 0.f) + 1e-5f);
    ln_affine_g(p, mean, rstd, pp + PH + c, pp + 2 * PH + c);
#pragma unroll
    for (int i = 0; i < PP; ++i) p[i] = fmaxf(p[i], 0.f);
    store_cols(tile, t.row, c, PH, p);
}

// policy logits -> softmax -> probs, beta = probs^(1/tau) renormalised (mcts_sampled.py:158-161), greedy action.
// Column part p owns logits [NV p, NV p + NV) of its row, NV = 16 (narrow, NAP <= 64) or 32 (W: the wide variant, NAP <= 128; two
// 16-column TMEM blocks per part); parts beyond the padded action count idle.  Every part reduces its own columns (local maximum
// m_p, argmax, sum of exp(v - m_p), sum of exp((v - m_p)/tau)); ONE exchange through shared memory (ex: 8 KB) combines them:
// M = max m_p, s = sum s_p exp(m_p - M).  The parts are in column order, so the first part with the maximum holds the first
// maximum.  `stage`: the joint-mode staging area, 32 x 48 floats per quadrant from `stage` (narrow), 32 x 128 floats per quadrant in
// the two (free) sT operand tiles from `stage` = tile 0's sT (wide).
template <bool W>
static __device__ __noinline__ void epi_policy_out(const Desc &d, uint32_t trow, const float *__restrict__ pb2, int valid, int root, int agent,
                                            uint32_t ex, uint32_t stage, long long *clk = nullptr)
{
    const Thr t;
#define SUBTS(i) if (clk) clk[i] = clock64();
    SUBTS(0)
    constexpr int NV = W ? 32 : 16;
    const int A = d.A, cc = t.part * NV;
    const bool active = cc < d.NAP;                  // warp-uniform (tcgen05.ld is warp-collective)
    const bool unit_tau = (d.inv_tau == 1.0f);
    float v[NV];
    float m = -INFINITY, s = 0.f, sbeta = 0.f;
    int am = 0;
    if (active) {
#pragma unroll
        for (int b = 0; b < NV / 16; ++b) {
            float (&vb)[16] = *reinterpret_cast<float (*)[16]>(v + 16 * b);
            if (b == 0 || cc + 16 * b < d.NAP) {    // (warp-uniform)
                tmem_ld16(trow + TM_A0 + cc + 16 * b, vb);
                add_gvec(vb, pb2 + cc + 16 * b);
            }
        }
#pragma unroll
        for (int i = 0; i < NV; ++i)
            if (cc + i < A && v[i] > m) { m = v[i]; am = cc + i; }
        if (valid && d.logits_out) {
#pragma unroll
            for (int i = 0; i < NV; ++i)
                if (cc + i < A) d.logits_out[((size_t)root * d.N + agent) * A + cc + i] = v[i];
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const float e = (cc + i < A) ? __expf(v[i] - m) : 0.f;
            v[i] = e;
            s += e;
            sbeta += unit_tau ? e : ((cc + i < A) ? __powf(e, d.inv_tau) : 0.f);   // (e/s)^t = e^t / s^t
        }
    }
    SUBTS(1)
    sts4(ex + (uint32_t)(t.part * 128 + t.row) * 16u, make_uint4(__float_as_uint(m), (uint32_t)am, __float_as_uint(s), __float_as_uint(sbeta)));
    named_bar_sync(1 + t.quad, 128);
    SUBTS(2)
    float M = -INFINITY, mp[PARTS], sp[PARTS], bp[PARTS];
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {                // first maximum in column order, as torch.argmax
        uint32_t w0, w1, w2, w3;
        lds4u(ex + (uint32_t)(p * 128 + t.row) * 16u, w0, w1, w2, w3);
        mp[p] = __uint_as_float(w0); sp[p] = __uint_as_float(w2); bp[p] = __uint_as_float(w3);
        if (mp[p] > M) { M = mp[p]; am = (int)w1; }
    }
    s = 0.f; sbeta = 0.f;
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
        const float f = __expf(mp[p] - M);           // (idle parts: exp(-inf) = 0)
        s += sp[p] * f;
        sbeta += bp[p] * (unit_tau ? f : __powf(f, d.inv_tau));
    }
    const float mine = __expf(m - M);                // my columns were taken relative to my part's maximum
    if (t.part == 0 && valid && d.greedy) d.greedy[(size_t)root * d.N + agent] = am;
    const float invs = mine / s, invb = (unit_tau ? mine : __powf(mine, d.inv_tau)) / sbeta;
    SUBTS(3)
    if (d.cur < 0) {
        // joint mode: the rows of a quadrant are consecutive (root, agent) pairs, i.e. ONE contiguous block of probs / beta in
        // global memory: stage the quadrant's block in shared memory and copy it out with coalesced stores (a row-per-thread
        // store touches 32 sectors per instruction: ~13 k cycles per tile at 27m).  tau = 1: beta == probs, one pass.
        const uint32_t st = W ? stage + (uint32_t)(t.quad >> 1) * 2u * TILE_BYTES + (uint32_t)(t.quad & 1) * (32u * 128u * 4u)
                              : stage + (uint32_t)t.quad * (32u * 48u * 4u);
        const int rpw = 32 / d.N;
        const int q_root0 = __shfl_sync(0xffffffffu, root, 0);          // lane 0 holds the quadrant's first root
        const int nroots = max(0, min(rpw, d.B - q_root0));
        const int nflt = nroots * d.N * A;
        const size_t gbase = (size_t)q_root0 * d.N * A;
        const int idx = t.part * 32 + t.lane;
        const int npass = unit_tau ? 1 : 2;
#pragma unroll 1
        for (int pass = 0; pass < npass; ++pass) {
            if (pass) named_bar_sync(1 + t.quad, 128);                   // pass 0 has been copied out
            if (active) {
#pragma unroll
                for (int i = 0; i < NV; ++i)
                    if (cc + i < A) sts1f(st + (uint32_t)(t.lane * A + cc + i) * 4u, pass == 0 ? v[i] * invs : __powf(v[i], d.inv_tau) * invb);
            }
            SUBTS(4)
            named_bar_sync(1 + t.quad, 128);
            SUBTS(5)
            float *dst = (pass == 0 ? d.probs : d.beta) + gbase, *dst2 = d.beta + gbase;
            for (int k = idx; k < nflt; k += 128) {
                const float x = lds1v(st + (uint32_t)k * 4u);
                dst[k] = x;
                if (unit_tau) dst2[k] = x;
            }
        }
        SUBTS(6)
#undef SUBTS
        return;     // (the next writer of the staging area passes this function's first barrier again, after every warp's copy loop)
    }
    const int ta = (agent == d.cur ? 0 : -1);
    if (active && valid && ta >= 0) {
        float *po = d.probs + ((size_t)root * d.Nt + ta) * A, *bo = d.beta + ((size_t)root * d.Nt + ta) * A;
#pragma unroll
        for (int i = 0; i < NV; ++i)
            if (cc + i < A) {
                po[cc + i] = v[i] * invs;
                bo[cc + i] = (unit_tau ? v[i] * invs : __powf(v[i], d.inv_tau) * invb);
            }
    }
    named_bar_sync(1 + t.quad, 128);   // every warp of the quadrant has read `ex`: the next tile's call may overwrite it
}

// W: the wide variant (48 < NAP <= 128), which differs in the policy output epilogue only (epi_policy_out)
template <bool W>
__global__ void __launch_bounds__(NTHREADS, 1) k_recurrent_inference_twin(const __grid_constant__ Desc d)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_mma[2], bar_ready[2];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int N = d.N;
    uint8_t *s0 = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);
    const uint32_t aTile = smem_u32(s0);                         // tile tt: sX at aTile + tt*2*TILE_BYTES, sT right after it
    const uint32_t aScr = aTile + 4 * TILE_BYTES, aRed = aScr + RED_OFF;
    uint8_t *sW = s0 + 4 * TILE_BYTES + SCRATCH_BYTES;

    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        mbar_init(&bar_mma[0], 1);
        mbar_init(&bar_mma[1], 1);
        mbar_init(&bar_ready[0], NEPI);
        mbar_init(&bar_ready[1], NEPI);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (warp == NEPI / 32) {
        // ================================ weight producer: every piece once, in stage order (both tiles use it) ============
        if ((tid & 31) == 0) {
            int pc = 0;
#pragma unroll 1
            for (int o = 0; o < NOPS; ++o) {
                const int mat = kOps[o].mat;
                uint32_t n, k;
                mat_dims(mat, d.NAP, n, k);
                const uint8_t *src = reinterpret_cast<const uint8_t *>(d.wpk) + d.chunk_off[mat];
#pragma unroll 1
                for (uint32_t k0 = 0; k0 < k; k0 += 64, ++pc) {
                    const uint32_t kk = min(64u, k - k0), bytes = n * kk * 2u;
                    const int s = pc % NSLOT;
                    if (pc >= NSLOT) mbar_wait_backoff(&bar_empty[s], ((pc / NSLOT) - 1) & 1);
                    mbar_expect_tx(&bar_full[s], bytes);
                    bulk_g2s(sW + (size_t)s * SLOT_BYTES, src, bytes, &bar_full[s]);
                    src += bytes;
                }
            }
        }
    } else if (warp == NEPI / 32 + 1) {
        // ================================ MMA issuer ==========================================================================
        const bool issuer = (tid & 31) == 0;
        const uint32_t aW = smem_u32(sW);
        int pc = 0;
        uint32_t rph = 0;
#pragma unroll 1
        for (int i = 0; i < NOPS;) {
            int j = i;
            while (!kOps[j].last) ++j;
            const int pc0 = pc;      // a stage's pieces (<= NSLOT) stay resident for both tiles: tile 0 waits for them, tile 1 releases them
#pragma unroll 1
            for (int tt = 0; tt < 2; ++tt) {
                if (issuer) {
                    mbar_wait(&bar_ready[tt], (rph >> tt) & 1u);   // all 512 epilogue threads have published tile tt's operands
                    rph ^= 1u << tt;
                    tc_fence_after();
                    pc = pc0;
#pragma unroll 1
                    for (int o = i; o <= j; ++o) {
                        const Op op = kOps[o];
                        uint32_t n, k;
                        mat_dims(op.mat, d.NAP, n, k);
                        const uint32_t a_addr = aTile + (uint32_t)tt * 2u * TILE_BYTES + (op.asrc ? TILE_BYTES : 0u);
                        const uint32_t dst = tmem + (uint32_t)tt * TM_TILE + (op.dst ? TM_A1 : TM_A0);
#pragma unroll 1
                        for (uint32_t k0 = 0; k0 < k; k0 += 64, ++pc) {
                            const uint32_t kk = min(64u, k - k0);
                            const int s = pc % NSLOT;
                            if (tt == 0) {
                                mbar_wait(&bar_full[s], (pc / NSLOT) & 1);
                                tc_fence_after();
                            }
                            issue_gemm(dst, a_addr, k, k0, aW + (uint32_t)s * SLOT_BYTES, kk, 0, kk, n, op.acc != 0 || k0 != 0);
                            if (tt == 1) mma_commit(&bar_empty[s]);   // the slot is free once both tiles' MMAs have read it
                        }
                    }
                    mma_commit(&bar_mma[tt]);
                }
                __syncwarp();
            }
            i = j + 1;
        }
    } else {
        // ================================ epilogue warps ======================================================================
        const Thr t;
        const float *__restrict__ P = d.vec;
        const int rpw = 32 / N;
        const int rl = t.lane / N, agent = t.lane - rl * N;
        const int root_lane0 = (rl < rpw) ? rl * N : 0;
        const uint32_t trow0 = tmem + ((uint32_t)(t.quad * 32) << 16);
        uint32_t ph = 0;
        int ts_n = 0;
#define TS() \
    if (ts_on && ts_n < 256) d.dbg_clock[ts_n++] = clock64();
#define TILE_VARS                                                         \
    const uint32_t trow = trow0 + (uint32_t)tt * TM_TILE;                 \
    const uint32_t aX = aTile + (uint32_t)tt * 2u * TILE_BYTES, aT = aX + TILE_BYTES; \
    const int valid = tt ? valid1 : valid0;                               \
    const int root = root0 + tt * 4 * rpw;                                \
    const float *hrow = tt ? hrow1 : hrow0;                               \
    const int act = tt ? act1 : act0;                                     \
    const uint32_t aRedT = aRed + (uint32_t)tt * 4096u;                   \
    (void)trow, (void)aX, (void)aT, (void)valid, (void)root, (void)hrow, (void)act, (void)aRedT;
#define WAIT_MMA()                                 \
    mbar_wait(&bar_mma[tt], (ph >> tt) & 1u);      \
    ph ^= 1u << tt;                                \
    tc_fence_after();                              \
    TS();
#define PUBLISH()                      \
    TS();                              \
    fence_proxy_async();               \
    tc_fence_before();                 \
    mbar_arrive(&bar_ready[tt]);
#define STAGE(body)                            \
    _Pragma("unroll 1") for (int tt = 0; tt < 2; ++tt) { \
        TILE_VARS                              \
        WAIT_MMA();                            \
        body;                                  \
        PUBLISH();                             \
    }

        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        const int root0 = ((blockIdx.x * 2) * 4 + t.quad) * rpw + rl;          // tile tt: + tt * 4 * rpw
        const int valid0 = (rl < rpw) && (root0 < d.B), valid1 = (rl < rpw) && (root0 + 4 * rpw < d.B);
        const bool ts_on = d.dbg_clock != nullptr && blockIdx.x == 0 && tid == 0;
        // ---- per tile: the parent's hidden-state row and my agent's action ------------------------------------------------
        const float *hrow0 = d.pool, *hrow1 = d.pool;
        int act0 = -1, act1 = -1;
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) {
            const int valid = tt ? valid1 : valid0, root = root0 + tt * 4 * rpw;
            const float *hr = d.pool;
            int a = -1;
            if (valid) {
                const int ix = d.idx_x ? __ldcg(d.idx_x + root) : 0;
                hr = d.pool + ((size_t)ix * d.B + root) * (size_t)(N * H) + (size_t)agent * H;
                if (d.greedy_pool == nullptr || d.cur < 0)
                    a = __ldcg(d.actions + (size_t)root * N + agent);
                else if (agent == d.cur)                      // sequential-agent mode, joint action assembled here (mcts_sampled.py:116-147)
                    a = __ldcg(d.actions + root);
                else if (agent < d.cur)
                    a = d.factor ? __ldcg(d.factor + (size_t)root * N + agent) : 0;
                else
                    a = __ldcg(d.greedy_pool + ((size_t)ix * d.B + root) * N + agent);
                if (a < 0 || a >= d.A) a = -1;
            }
            if (tt) { hrow1 = hr; act1 = a; } else { hrow0 = hr; act0 = a; }
        }
        TS();
#pragma unroll 1
        for (int tt = 0; tt < 2; ++tt) {
            TILE_VARS
            gather_hidden(hrow, valid, aT);
            PUBLISH();
        }

        // ---- attention_stack[0..1]: x0 = relu(W_in [h | onehot] + b) + positional table ------------------------------------
        STAGE(epi_inproj(trow, P + d.o_bin, act >= 0 ? P + d.o_oh_in + act * (H / 2) : nullptr, P + d.o_pos + agent * H, aX));
        // ---- 3 x post-LN TransformerEncoderLayer over the agent axis (attention.py:36-43) ----------------------------------
#pragma unroll 1
        for (int l = 0; l < 3; ++l) {
            const float *lv = P + d.o_layer + l * 1280;   // bq bk bv bo g1 be1 b1 b2 g2 be2
            STAGE(epi_attention(trow, aT, lv, N, aScr, 0));                                           // heads 0-3: Q | K | V -> attention
            STAGE(epi_attention(trow, aT, lv, N, aScr, 1));                                           // heads 4-7
            named_bar_sync(5, NEPI);   // the warps' Q / K blocks cover the whole scratch area, row statistics included: nobody may
                                       // start the next LayerNorm while a slower warp is still in tile B's attention
            STAGE(epi_ln(trow, lv + 384, lv + 512, lv + 640, nullptr, aX, 0, aX, aRedT, d.dbg_flags));              // norm1(x + out_proj)
            STAGE(epi_bias(trow, lv + 768, 1, aT));                                                   // relu(linear1)
            STAGE(epi_ln(trow, lv + 896, lv + 1024, lv + 1152, nullptr, aX, 0, aX, aRedT, d.dbg_flags);             // norm2(x + linear2)
                  if (l == 2) gather_hidden(hrow, valid, aT));                                 // h (bf16) back for fc_dynamic
        }
        // ---- fc_dynamic: Linear-LN-ReLU, Linear-LN-ReLU, Linear; residual (model.py:262-268) --------------------------------
        const float *dv = P + d.o_dyn;
        STAGE(epi_ln(trow, dv, dv + 128, dv + 256, act >= 0 ? P + d.o_oh_dyn + act * (H / 2) : nullptr, 0, 1, aT, aRedT));
        STAGE(epi_ln(trow, dv + 384, dv + 512, dv + 640, nullptr, 0, 1, aX, aRedT));
        STAGE(epi_next_hidden(trow, dv + 768, hrow, d.next_hidden + (valid ? (size_t)root * (N * H) + (size_t)agent * H : 0), valid, aT));
        // ---- reward head: GraphNetNN on [next_hidden | onehot] (model.py:270-277) -------------------------------------------
        const float *rv = P + d.o_rg;
        STAGE(epi_gnn(trow, rv, act >= 0 ? P + d.o_oh_rg + act * (H / 2) : nullptr, N, root_lane0, 0, aX, aRedT, aScr));
        STAGE({
            const float r = epi_gnn(trow, rv + 128, nullptr, N, root_lane0, 1, 0, aRedT, aScr, ts_on ? d.dbg_clock + 128 + 16 * tt : nullptr);
            if (valid && agent == 0 && t.part == 0) d.reward[root] = r;
        });
        // ---- value head: GraphNetNN on next_hidden (model.py:359) -------------------------------------------------------------
        const float *vv = P + d.o_vg;
        STAGE(epi_gnn(trow, vv, nullptr, N, root_lane0, 0, aX, aRedT, aScr));
        STAGE({
            const float val = epi_gnn(trow, vv + 128, nullptr, N, root_lane0, 1, 0, aRedT, aScr);
            if (valid && agent == 0 && t.part == 0) d.value[root] = val;
        });
        // ---- policy head + the driver's softmax / beta ---------------------------------------------------------------------------
        const float *pv = P + d.o_pol;
        STAGE(epi_policy_hidden(trow, pv, aX, aRedT));
        named_bar_sync(5, NEPI);   // the policy exchange buffer covers both tiles' row-statistics buffers: every warp must have left
                                   // tile B's LayerNorm before the first one writes it
#pragma unroll 1
        for (int tt = 0; tt < 2; ++tt) {
            TILE_VARS
            WAIT_MMA();
            epi_policy_out<W>(d, trow, pv + 96, valid, root, agent, aRed, W ? aTile + TILE_BYTES : aScr,
                              ts_on ? d.dbg_clock + 160 + 16 * tt : nullptr);
            TS();
        }
#undef STAGE
#undef PUBLISH
#undef WAIT_MMA
#undef TILE_VARS
#undef TS
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace twin
}  // namespace maz
