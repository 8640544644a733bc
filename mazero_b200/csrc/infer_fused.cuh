// infer_fused.cuh -- ONE kernel for MAMuZeroNet.recurrent_inference inside the search (sm_100a).
//
// Reference computation: config/smac/model.py:562-574 (dynamics :251-282 with attention.py:27-43,
// prediction :335-373, GraphNetNN :136-174) + inverse support transform core/config.py:430-442,463-499
// + the driver's softmax / beta post-processing mcts_sampled.py:158-161.
//
// Tiling: a CTA of 128 threads owns a tile of 128 token rows (thread r == row r == TMEM lane r).  A token
// is one agent of one root; every warp holds floor(32/N) whole roots, so everything that mixes the
// agents of a root (attention over the agent axis, the all-ones-adjacency graph sums) stays inside a warp.
// The 32 weight chunks (<= 32 KB each, pre-packed on the host in the tcgen05 operand layout, in consumption
// order) stream from L2 through a 3-slot shared-memory ring (1-D bulk TMA + mbarriers); all biases /
// LayerNorm affines / heads arrive in shared memory with one more bulk copy.  Every GEMM is M=128 on the
// tensor cores with the fp32 accumulator in TMEM; the residual stream x lives in TMEM (columns 0..127) so
// `x + f(x)` is an accumulating MMA.  Per-row work (bias, ReLU, LayerNorm, softmax, support transform) is
// thread-local.  The epilogues are NON-inlined functions on purpose: the kernel is one long straight line,
// and v1 (everything inlined, ~600 KB of SASS executed once) spent most of its time in instruction-cache
// misses (profiles/r01_ncu_summary.md).
#pragma once
#include "../../include/maz_infer.h"
#include "umma.cuh"

namespace maz {
namespace fused {

using namespace umma;

constexpr int H = 128;        // hidden per agent            (config/smac/__init__.py:15)
constexpr int NHEAD = 8;      // attention.py:36
constexpr int HD = 16;
constexpr int GH = 64;        // GNN hidden                  (model.py:213,300 defaults)
constexpr int PH = 32;        // fc_policy_layers = [32]
constexpr int SUP = 11;       // DiscreteSupport(-5, 5)
constexpr int NLAYER = 3;     // AttentionEncoder(3, ...)    (model.py:221)
constexpr int NCHUNK = MAZ_INFER_NCHUNK;
constexpr int NSLOT = 3;
constexpr int NEPI_THREADS = 512;   // epilogue threads (16 warps)
constexpr uint32_t SLOT_BYTES = 128 * 128 * 2;

enum : uint32_t { TM_X = 0, TM_Q = 128, TM_K = 256, TM_V = 384, TM_ACC = 128 };

using Desc = ::maz_infer_desc;

__host__ __device__ inline size_t smem_bytes(int KA, int vec_floats)
{
    return 2 * operand_bytes(128, 128) + operand_bytes(128, KA) + NSLOT * (size_t)SLOT_BYTES + (size_t)vec_floats * 4 + 4096 + 1024;   // + row-statistics exchange
}

// ---- warp roles ---------------------------------------------------------------------------------------------
// warps 0..15 : epilogue (4 TMEM lane quadrants x 4 column parts)
// warp 16     : weight producer -- streams the 32 chunks through the 3-slot ring (bulk TMA), runs ahead freely
// warp 17     : MMA issuer -- waits for "operands ready" (bar_ready) and "chunk resident" (bar_full), issues the
//               tcgen05.mma's, releases ring slots (tcgen05.commit -> bar_empty) and signals bar_mma per stage
// Keeping the single-thread, long-latency async operations (mbarrier waits, bulk copies, MMA issue, commits) on
// their own warps takes them off the epilogue warps' critical path (v3 had thread 0 do all of it: ~2200 cycles
// per chunk between the barrier and the MMA completion).
struct Pipe {
    uint64_t *full, *empty, *mma, *ready;
    uint32_t slots;        // shared address of the ring
    uint32_t tmem;
    int c;                 // next chunk
    uint32_t ready_phase;
    int skip;              // profiling: do not issue the MMAs
};

// one weight chunk: D[dst] (+)= A[a_addr (row length a_K)] * W_c^T  (n_out columns).  MMA thread only; not inlined
// (called 32 times; small code = warm instruction cache).
static __device__ __noinline__ void mma_chunk(Pipe &p, uint32_t dst, uint32_t a_addr, uint32_t a_K, uint32_t n_out, uint32_t accum)
{
    const int c = p.c, s = c % NSLOT;
    mbar_wait(&p.full[s], (c / NSLOT) & 1);
    tc_fence_after();
    if (!(p.skip & 2)) issue_gemm(p.tmem + dst, a_addr, a_K, 0, p.slots + (uint32_t)s * SLOT_BYTES, a_K, 0, a_K, n_out, accum != 0);
    // (the ring slot is released by epilogue thread 0 after the stage's bar_mma completes: one tcgen05.commit per
    //  stage instead of one per chunk on this thread's serial path)
    p.c = c + 1;
}
// "operands ready" hand-off: the 512 epilogue threads and the 32 lanes of the MMA warp meet on hardware named
// barrier 5 (bar.sync, tens of cycles) -- one mbarrier hop less per stage than arrive + try_wait polling.
__device__ __forceinline__ void mma_stage_begin()
{
    named_bar_sync(5, NEPI_THREADS + 32);
    tc_fence_after();
}
__device__ __forceinline__ void mma_stage_end(Pipe &p)
{
    if (p.skip & 8) mbar_arrive(p.mma); else mma_commit(p.mma);   // (8: profiling, plain arrive instead of tcgen05.commit)
}

// ---- small per-thread helpers -----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack2(float a, float b)
{
    __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&p);
}
// write 16 consecutive columns [c, c+16) of row `row` into the bf16 operand tile at shared address `tile`
template <int NV>
__device__ __forceinline__ void store_cols(uint32_t tile, int row, int c, int K, const float (&v)[NV])
{
#pragma unroll
    for (int j = 0; j < NV; j += 8) {
        uint4 a;
        a.x = pack2(v[j], v[j + 1]); a.y = pack2(v[j + 2], v[j + 3]); a.z = pack2(v[j + 4], v[j + 5]); a.w = pack2(v[j + 6], v[j + 7]);
        sts4(tile + operand_chunk_off(row, (c + j) >> 3, K, 128), a);   // swizzled for K % 64 == 0
    }
}
// v += vec (shared memory), with Blackwell's packed fp32 adds (FADD2)
template <int NV>
__device__ __forceinline__ void add_svec(float (&v)[NV], uint32_t saddr)
{
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 t = lds4(saddr + 4 * i);
        const float2 a = __fadd2_rn(make_float2(v[i], v[i + 1]), make_float2(t.x, t.y));
        const float2 b = __fadd2_rn(make_float2(v[i + 2], v[i + 3]), make_float2(t.z, t.w));
        v[i] = a.x; v[i + 1] = a.y; v[i + 2] = b.x; v[i + 3] = b.y;
    }
}
// (sum, sumsq) of v with packed FADD2 / FFMA2
template <int NV>
__device__ __forceinline__ void sum_sq(const float (&v)[NV], float &sum, float &sq)
{
    float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < NV; i += 2) {
        const float2 x = make_float2(v[i], v[i + 1]);
        s2 = __fadd2_rn(s2, x);
        q2 = __ffma2_rn(x, x, q2);
    }
    sum = s2.x + s2.y;
    sq = q2.x + q2.y;
}
// v = (v - mean) * rstd * g + b  with g, b from shared memory: a = rstd*g; v = v*a + (b - mean*a)
template <int NV>
__device__ __forceinline__ void ln_affine(float (&v)[NV], float mean, float rstd, uint32_t sg, uint32_t sb)
{
    const float2 r2 = make_float2(rstd, rstd), nm2 = make_float2(-mean, -mean);
#pragma unroll
    for (int i = 0; i < NV; i += 4) {
        const float4 g = lds4(sg + 4 * i), b = lds4(sb + 4 * i);
        const float2 a0 = __fmul2_rn(r2, make_float2(g.x, g.y)), a1 = __fmul2_rn(r2, make_float2(g.z, g.w));
        const float2 c0 = __ffma2_rn(nm2, a0, make_float2(b.x, b.y)), c1 = __ffma2_rn(nm2, a1, make_float2(b.z, b.w));
        const float2 y0 = __ffma2_rn(make_float2(v[i], v[i + 1]), a0, c0);
        const float2 y1 = __ffma2_rn(make_float2(v[i + 2], v[i + 3]), a1, c1);
        v[i] = y0.x; v[i + 1] = y0.y; v[i + 2] = y1.x; v[i + 3] = y1.y;
    }
}

// inverse categorical transform of an 11-way support head (core/config.py:430-442, 463-499)
__device__ __forceinline__ float support_to_scalar(const float (&lg)[SUP])
{
    float m = lg[0];
#pragma unroll
    for (int t = 1; t < SUP; ++t) m = fmaxf(m, lg[t]);
    float s = 0.f, x = 0.f;
#pragma unroll
    for (int t = 0; t < SUP; ++t) {
        const float e = __expf(lg[t] - m);
        s += e;
        x += e * (float)(t - 5);
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

// ---- epilogues (one per stage kind; NOT inlined, see the header comment) ---------------------------------------
// Thread layout of a CTA: 16 warps = 4 TMEM lane quadrants x PARTS column parts.  warp = part*4 + quad;
// row = quad*32 + lane (a warp may only touch TMEM lanes 32*(warp%4)..+31); a thread owns the columns
// [part*W/PARTS, (part+1)*W/PARTS) of its row in a W-wide stage.  Row statistics (LayerNorm) are combined
// across the PARTS threads of a row through shared memory + a 128-thread named barrier per quadrant.
constexpr int PARTS = 4;
constexpr int NEPI = 128 * PARTS;          // epilogue threads
static_assert(NEPI == NEPI_THREADS, "epilogue thread count");
constexpr int NTHREADS = NEPI + 64;        // + producer warp + MMA warp
constexpr int CP = H / PARTS;        // 32
constexpr int GP = GH / PARTS;       // 16
constexpr int PP = PH / PARTS;       // 8
constexpr int HPP = NHEAD / PARTS;   // 2
constexpr uint32_t RED_BYTES = 128 * PARTS * 8;

struct Thr {            // who am I (recomputed from threadIdx in every epilogue: cheaper than passing it around)
    int lane, quad, part, row;
    __device__ __forceinline__ Thr()
    {
        const int tid = threadIdx.x, warp = tid >> 5;
        lane = tid & 31; quad = warp & 3; part = warp >> 2; row = quad * 32 + lane;
    }
};

// combine (sum, sumsq) of the PARTS threads that share a row
__device__ __forceinline__ void row_stats(const Thr &t, uint32_t aRed, float &sum, float &sq)
{
    sts2f(aRed + (uint32_t)(t.row * PARTS + t.part) * 8u, sum, sq);
    named_bar_sync(1 + t.quad, 128);
    float S = 0.f, Q = 0.f;
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
        const float2 v = lds2f(aRed + (uint32_t)(t.row * PARTS + p) * 8u);
        S += v.x; Q += v.y;
    }
    sum = S; sq = Q;
}

template <int NV>
__device__ __forceinline__ void tmem_store_cols(uint32_t taddr, const float (&v)[NV])
{
#pragma unroll
    for (int j = 0; j < NV; j += 16) {
        float w[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) w[i] = v[j + i];
        tmem_st16(taddr + j, w);
    }
}

// x0 = relu(acc + b_in) + pos[agent]  -> TMEM X (fp32) and operand tile (bf16)
static __device__ __noinline__ void epi_inproj(uint32_t trow, uint32_t sb, uint32_t spos, uint32_t tile)
{
    const Thr t;
    const int c = t.part * CP;
    float v[CP];
    tmem_ld32(trow + TM_ACC + c, v);
    add_svec(v, sb + 4 * c);
#pragma unroll
    for (int i = 0; i < CP; i += 4) {
        const float4 p = lds4(spos + 4 * (c + i));
        v[i] = fmaxf(v[i], 0.f) + p.x; v[i + 1] = fmaxf(v[i + 1], 0.f) + p.y;
        v[i + 2] = fmaxf(v[i + 2], 0.f) + p.z; v[i + 3] = fmaxf(v[i + 3], 0.f) + p.w;
    }
    tmem_store_cols(trow + TM_X + c, v);
    store_cols(tile, t.row, c, H, v);
    tmem_st_wait();
}

// f = relu(acc + b) -> operand tile
static __device__ __noinline__ void epi_bias_relu(uint32_t trow, uint32_t sb, uint32_t tile)
{
    const Thr t;
    const int c = t.part * CP;
    float v[CP];
    tmem_ld32(trow + TM_ACC + c, v);
    add_svec(v, sb + 4 * c);
#pragma unroll
    for (int i = 0; i < CP; ++i) v[i] = fmaxf(v[i], 0.f);
    store_cols(tile, t.row, c, H, v);
}

// y = LN(acc + bias) * g + be over the 128 TMEM columns at `tcol`; optional ReLU (mlp()); optional fp32 copy
// into the TMEM-resident residual stream X; always a bf16 copy into the operand tile.
static __device__ __noinline__ void epi_ln128(uint32_t trow, uint32_t tcol, uint32_t sb, uint32_t sg, uint32_t sbe, int relu_after,
                                       int store_x, uint32_t tile, uint32_t aRed)
{
    const Thr t;
    const int c = t.part * CP;
    float v[CP];
    tmem_ld32(trow + tcol + c, v);
    add_svec(v, sb + 4 * c);
    float sum, sq;
    sum_sq(v, sum, sq);
    row_stats(t, aRed, sum, sq);
    const float mean = sum * (1.f / H);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / H) - mean * mean, 0.f) + 1e-5f);
    ln_affine(v, mean, rstd, sg + 4 * c, sbe + 4 * c);
    if (relu_after) {
#pragma unroll
        for (int i = 0; i < CP; ++i) v[i] = fmaxf(v[i], 0.f);
    }
    if (store_x) tmem_store_cols(trow + TM_X + c, v);
    store_cols(tile, t.row, c, H, v);
    if (store_x) tmem_st_wait();
}

// scaled dot-product attention over the N agents of my root; each column part owns HPP heads.
// sb: shared address of [bq | bk | bv] (3 x 128 floats).  Output (bf16) into the operand tile.
// Small teams (N <= 4, e.g. 3m): two-phase softmax with everything unrolled -- all N score chains are independent
// (instruction-level parallelism; the online form below serialises max / exp / rescale per key) and the dot
// products use packed fp32 FMAs.  Larger N: one pass, online softmax.
template <int NN>
__device__ __forceinline__ void attention_head_small(uint32_t trow, uint32_t sb, int hh, int root_lane0, uint32_t tile, int row)
{
    float q[16], k[16], v[16];
    tmem_ld16(trow + TM_Q + hh * HD, q);
    tmem_ld16(trow + TM_K + hh * HD, k);
    tmem_ld16(trow + TM_V + hh * HD, v);
    add_svec(q, sb + 4 * (hh * HD));
    add_svec(k, sb + 4 * (H + hh * HD));
    add_svec(v, sb + 4 * (2 * H + hh * HD));
    float s[NN];
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
            const float2 kj = make_float2(__shfl_sync(0xffffffffu, k[i], root_lane0 + j), __shfl_sync(0xffffffffu, k[i + 1], root_lane0 + j));
            acc = __ffma2_rn(make_float2(q[i], q[i + 1]), kj, acc);
        }
        s[j] = (acc.x + acc.y) * 0.25f;   // 1/sqrt(head_dim)
    }
    float m = s[0];
#pragma unroll
    for (int j = 1; j < NN; ++j) m = fmaxf(m, s[j]);
    float l = 0.f;
#pragma unroll
    for (int j = 0; j < NN; ++j) { s[j] = __expf(s[j] - m); l += s[j]; }
    const float inv = 1.f / l;
    float2 o2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o2[i] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        const float pj = s[j] * inv;
        const float2 p2 = make_float2(pj, pj);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float2 vj = make_float2(__shfl_sync(0xffffffffu, v[2 * i], root_lane0 + j), __shfl_sync(0xffffffffu, v[2 * i + 1], root_lane0 + j));
            o2[i] = __ffma2_rn(p2, vj, o2[i]);
        }
    }
    float o[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[2 * i] = o2[i].x; o[2 * i + 1] = o2[i].y; }
    store_cols(tile, row, hh * HD, H, o);
}

static __device__ __noinline__ void epi_attention(uint32_t trow, uint32_t sb, int N, int root_lane0, uint32_t tile, uint32_t scratch)
{
    const Thr t;
    const uint32_t kv = scratch + (uint32_t)(t.part * 4 + t.quad) * 2048u;   // this warp's 32 x (K16 | V16) bf16 rows
#pragma unroll 1
    for (int hh = t.part * HPP; hh < (t.part + 1) * HPP; ++hh) {
        if (N <= 4) {   // warp-uniform
            switch (N) {
                case 1: attention_head_small<1>(trow, sb, hh, root_lane0, tile, t.row); break;
                case 2: attention_head_small<2>(trow, sb, hh, root_lane0, tile, t.row); break;
                case 3: attention_head_small<3>(trow, sb, hh, root_lane0, tile, t.row); break;
                default: attention_head_small<4>(trow, sb, hh, root_lane0, tile, t.row); break;
            }
            continue;
        }
        // Larger teams: K and V of the warp's 32 rows go through shared memory as bf16 (2 KB per warp, in the operand
        // tile that the QKV GEMM has just finished reading), so each key costs 4 broadcast LDS.128 instead of 32 warp
        // shuffles (the shuffle crossbar bounded this loop: 27 keys x 32 shuffles x 2 heads per warp and layer at N = 27).
        float q[16], o[16];
        {
            float k[16], v[16];
            tmem_ld16(trow + TM_Q + hh * HD, q);
            tmem_ld16(trow + TM_K + hh * HD, k);
            tmem_ld16(trow + TM_V + hh * HD, v);
            add_svec(q, sb + 4 * (hh * HD));
            add_svec(k, sb + 4 * (H + hh * HD));
            add_svec(v, sb + 4 * (2 * H + hh * HD));
            const uint32_t mine = kv + (uint32_t)t.lane * 64u;
            uint4 a, b2;
            a.x = pack2(k[0], k[1]); a.y = pack2(k[2], k[3]); a.z = pack2(k[4], k[5]); a.w = pack2(k[6], k[7]);
            b2.x = pack2(k[8], k[9]); b2.y = pack2(k[10], k[11]); b2.z = pack2(k[12], k[13]); b2.w = pack2(k[14], k[15]);
            sts4(mine, a);
            sts4(mine + 16, b2);
            a.x = pack2(v[0], v[1]); a.y = pack2(v[2], v[3]); a.z = pack2(v[4], v[5]); a.w = pack2(v[6], v[7]);
            b2.x = pack2(v[8], v[9]); b2.y = pack2(v[10], v[11]); b2.z = pack2(v[12], v[13]); b2.w = pack2(v[14], v[15]);
            sts4(mine + 32, a);
            sts4(mine + 48, b2);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 16; ++i) { q[i] *= 0.25f; o[i] = 0.f; }   // 1/sqrt(head_dim)
        float m = -INFINITY, lsum = 0.f;
#pragma unroll 1
        for (int j = 0; j < N; ++j) {
            const uint32_t rowp = kv + (uint32_t)(root_lane0 + j) * 64u;
            uint32_t w[16];
            lds4u(rowp, w[0], w[1], w[2], w[3]);
            lds4u(rowp + 16, w[4], w[5], w[6], w[7]);
            lds4u(rowp + 32, w[8], w[9], w[10], w[11]);
            lds4u(rowp + 48, w[12], w[13], w[14], w[15]);
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {   // bf16 pair -> two fp32: low half << 16, high half masked
                s += q[2 * i] * __uint_as_float(w[i] << 16) + q[2 * i + 1] * __uint_as_float(w[i] & 0xffff0000u);
            }
            const float mn = fmaxf(m, s);
            const float corr = __expf(m - mn), p = __expf(s - mn);
            lsum = lsum * corr + p;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                o[2 * i] = o[2 * i] * corr + p * __uint_as_float(w[8 + i] << 16);
                o[2 * i + 1] = o[2 * i + 1] * corr + p * __uint_as_float(w[8 + i] & 0xffff0000u);
            }
            m = mn;
        }
        const float inv = 1.f / lsum;
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] *= inv;
        store_cols(tile, t.row, hh * HD, H, o);
        __syncwarp();   // every lane is done with this head's K / V before the next head overwrites them
    }
}

// next_hidden = acc + b + hidden (fp32 residual straight from the pool); fp32 to global, bf16 to the tile
static __device__ __noinline__ void epi_next_hidden(uint32_t trow, uint32_t sb, const float *__restrict__ hrow, float *__restrict__ nh,
                                             int valid, uint32_t tile)
{
    const Thr t;
    const int c = t.part * CP;
    float v[CP];
    tmem_ld32(trow + TM_ACC + c, v);
    add_svec(v, sb + 4 * c);
    if (valid) {
#pragma unroll
        for (int i = 0; i < CP; i += 4) {
            const float4 h = __ldcg(reinterpret_cast<const float4 *>(hrow + c + i));
            v[i] += h.x; v[i + 1] += h.y; v[i + 2] += h.z; v[i + 3] += h.w;
            *reinterpret_cast<float4 *>(nh + c + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
    }
    store_cols(tile, t.row, c, H, v);
}

// GraphNetNN layer (model.py:151-163) from one stacked GEMM: columns [0,64) = gc.lin(x), [64,128) = nn(x).
// y = LN(relu(sum_over_agents(gc + b_gc) + nn + b_nn)), no affine.  sb: [b_gc | b_nn] (2 x 64 floats).
// head == 0: y (bf16) -> operand tile (K = 64) for the second layer.
// head == 1: mean-pool over the agents, 64 -> 11 head (V weights at sb + 128 floats, bias after), support
//            transform; partial logits of the column parts are combined through `scratch` (shared, 24 KB);
//            the scalar is returned by the part-0 thread of every row (0 elsewhere).
static __device__ __noinline__ float epi_gnn(uint32_t trow, uint32_t sb, int N, int root_lane0, int head, uint32_t tile, uint32_t aRed,
                                      uint32_t scratch)
{
    const Thr t;
    const int c = t.part * GP;
    float y[GP], nn[GP];
    {
        float g[GP];
        tmem_ld16(trow + TM_ACC + c, g);
        add_svec(g, sb + 4 * c);
#pragma unroll
        for (int i = 0; i < GP; ++i) y[i] = 0.f;
#pragma unroll 1
        for (int j = 0; j < N; ++j) {
#pragma unroll
            for (int i = 0; i < GP; ++i) y[i] += __shfl_sync(0xffffffffu, g[i], root_lane0 + j);
        }
    }
    tmem_ld16(trow + TM_ACC + GH + c, nn);
    add_svec(nn, sb + 4 * (GH + c));
    float sum = 0.f, sq = 0.f;
#pragma unroll
    for (int i = 0; i < GP; ++i) {
        y[i] = fmaxf(y[i] + nn[i], 0.f);
        sum += y[i];
        sq += y[i] * y[i];
    }
    row_stats(t, aRed, sum, sq);
    const float mean = sum * (1.f / GH);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / GH) - mean * mean, 0.f) + 1e-5f);
#pragma unroll
    for (int i = 0; i < GP; ++i) y[i] = (y[i] - mean) * rstd;
    if (!head) {
        store_cols(tile, t.row, c, GH, y);
        return 0.f;
    }
    const float invn = 1.f / (float)N;
#pragma unroll
    for (int i = 0; i < GP; ++i) {
        float s = 0.f;
        const float mine = y[i];
#pragma unroll 1
        for (int j = 0; j < N; ++j) s += __shfl_sync(0xffffffffu, mine, root_lane0 + j);
        y[i] = s * invn;
    }
    const uint32_t sV = sb + 4 * (2 * GH), sVb = sV + 4 * (SUP * GH);
    const uint32_t mine_out = scratch + (uint32_t)((t.row * PARTS + t.part) * 12) * 4u;
#pragma unroll 1
    for (int k = 0; k < SUP; ++k) {   // partial logits over my GP columns (rolled: executed twice per kernel)
        float a = 0.f;
#pragma unroll
        for (int i = 0; i < GP; i += 4) {
            const float4 w = lds4(sV + 4 * (k * GH + c + i));
            a += w.x * y[i] + w.y * y[i + 1] + w.z * y[i + 2] + w.w * y[i + 3];
        }
        sts1f(mine_out + 4 * k, a);
    }
    named_bar_sync(1 + t.quad, 128);
    if (t.part != 0) return 0.f;
    // softmax . support -> inv_h (core/config.py:430-442, 463-499), two rolled passes over the 11 logits
    const uint32_t rowp = scratch + (uint32_t)(t.row * PARTS * 12) * 4u;
    float m = -INFINITY;
#pragma unroll 1
    for (int k = 0; k < SUP; ++k) {
        float a = lds1v(sVb + 4 * k);
#pragma unroll
        for (int p = 0; p < PARTS; ++p) a += lds1v(rowp + (uint32_t)(p * 12 + k) * 4u);
        sts1f(rowp + 4 * k, a);          // total logit k overwrites part 0's slot
        m = fmaxf(m, a);
    }
    float ssum = 0.f, x = 0.f;
#pragma unroll 1
    for (int k = 0; k < SUP; ++k) {
        const float e = __expf(lds1v(rowp + 4 * k) - m);
        ssum += e;
        x += e * (float)(k - 5);
    }
    x /= ssum;
    const float eps = 0.001f;
    const float r = (sqrtf(1.f + 4.f * eps * (fabsf(x) + 1.f + eps)) - 1.f) / (2.f * eps);
    float out = r * r - 1.f;
    out = (x < 0.f) ? -out : out;
    if (!(out == out)) out = 0.f;
    if (fabsf(out) < eps) out = 0.f;
    return out;
}

// policy hidden: p1 = relu(LN(acc + b) * g + be) over 32 columns -> operand tile (K = 32)
static __device__ __noinline__ void epi_policy_hidden(uint32_t trow, uint32_t sp, uint32_t tile, uint32_t aRed)
{
    const Thr t;
    const int c = t.part * PP;
    float p[PP];
    tmem_ld8(trow + TM_ACC + c, p);
    add_svec(p, sp + 4 * c);
    float sum = 0.f, sq = 0.f;
#pragma unroll
    for (int i = 0; i < PP; ++i) { sum += p[i]; sq += p[i] * p[i]; }
    row_stats(t, aRed, sum, sq);
    const float mean = sum * (1.f / PH);
    const float rstd = rsqrtf(fmaxf(sq * (1.f / PH) - mean * mean, 0.f) + 1e-5f);
#pragma unroll
    for (int i = 0; i < PP; i += 4) {
        const float4 g = lds4(sp + 4 * (PH + c + i)), b = lds4(sp + 4 * (2 * PH + c + i));
        p[i] = fmaxf((p[i] - mean) * rstd * g.x + b.x, 0.f); p[i + 1] = fmaxf((p[i + 1] - mean) * rstd * g.y + b.y, 0.f);
        p[i + 2] = fmaxf((p[i + 2] - mean) * rstd * g.z + b.z, 0.f); p[i + 3] = fmaxf((p[i + 3] - mean) * rstd * g.w + b.w, 0.f);
    }
    store_cols(tile, t.row, c, PH, p);
}

// policy logits -> softmax -> probs, beta = probs^(1/tau) renormalised (mcts_sampled.py:158-161), greedy action.
// Executed by the part-0 warps only (A <= 48 columns), as three rolled passes over 16-column TMEM chunks
// (small code: this runs once per kernel, see issue_chunk's note on instruction fetch).
static __device__ __noinline__ void epi_policy_out(const Desc &d, uint32_t trow, uint32_t sb2, int valid, int root, int agent)
{
    const int A = d.A, NAP = d.NAP;
    float m = -INFINITY;
    int am = 0;
#pragma unroll 1
    for (int cc = 0; cc < NAP; cc += 16) {
        float v[16];
        tmem_ld16(trow + TM_ACC + cc, v);
        add_svec(v, sb2 + 4 * cc);
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (cc + i < A && v[i] > m) { m = v[i]; am = cc + i; }
        if (valid && d.logits_out) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (cc + i < A) d.logits_out[((size_t)root * d.N + agent) * A + cc + i] = v[i];
        }
    }
    const int ta = (d.cur < 0) ? agent : (agent == d.cur ? 0 : -1);
    const bool unit_tau = (d.inv_tau == 1.0f);
    float s = 0.f, sbeta = 0.f;
#pragma unroll 1
    for (int cc = 0; cc < NAP; cc += 16) {
        float v[16];
        tmem_ld16(trow + TM_ACC + cc, v);
        add_svec(v, sb2 + 4 * cc);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float e = (cc + i < A) ? __expf(v[i] - m) : 0.f;
            s += e;
            sbeta += unit_tau ? e : ((cc + i < A) ? __powf(e, d.inv_tau) : 0.f);   // (e/s)^t = e^t / s^t
        }
    }
    if (valid && d.greedy) d.greedy[(size_t)root * d.N + agent] = am;
    // NOTE: no early return before the last tcgen05.ld: it is warp-collective (.sync.aligned), every lane of the
    // warp must execute it; only the stores are predicated.
    const bool writer = valid && ta >= 0;
    const float invs = 1.f / s, invb = 1.f / sbeta;
    float *po = d.probs + (writer ? ((size_t)root * d.Nt + ta) * A : 0);
    float *bo = d.beta + (writer ? ((size_t)root * d.Nt + ta) * A : 0);
#pragma unroll 1
    for (int cc = 0; cc < NAP; cc += 16) {
        float v[16];
        tmem_ld16(trow + TM_ACC + cc, v);
        add_svec(v, sb2 + 4 * cc);
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (writer && cc + i < A) {
                const float e = __expf(v[i] - m);
                po[cc + i] = e * invs;
                bo[cc + i] = (unit_tau ? e : __powf(e, d.inv_tau)) * invb;
            }
    }
}

// fp32 pool row -> bf16 operand tile (K = 128), my 32 columns
static __device__ __noinline__ void gather_hidden(const float *__restrict__ hrow, int valid, uint32_t tile)
{
    const Thr t;
    const int c = t.part * CP;
    float v[CP];
#pragma unroll
    for (int i = 0; i < CP; i += 4) {
        const float4 h = valid ? __ldcg(reinterpret_cast<const float4 *>(hrow + c + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[i] = h.x; v[i + 1] = h.y; v[i + 2] = h.z; v[i + 3] = h.w;
    }
    store_cols(tile, t.row, c, H, v);
}

#ifndef MAZ_FUSED_NO_KERNEL   // (translation units that only need the device functions define it)
__global__ void __launch_bounds__(NTHREADS, 1) k_recurrent_inference(const __grid_constant__ Desc d)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_mma, bar_ready, bar_vec;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int N = d.N, KA = d.KA;
    uint8_t *sX = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);   // 128 x 128 bf16, 1 KB aligned (swizzle atoms)
    uint8_t *sT = sX + operand_bytes(128, 128);       // 128 x 128 bf16
    uint8_t *sOne = sT + operand_bytes(128, 128);     // 128 x KA  bf16 (one-hot joint action)
    uint8_t *sW = sOne + operand_bytes(128, KA);      // weight ring, NSLOT x 32 KB
    uint8_t *sR = sW + NSLOT * (size_t)SLOT_BYTES;    // row-statistics exchange, 4 KB
    uint8_t *sP = sR + RED_BYTES;                     // fp32 parameters (d.vec)

    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        mbar_init(&bar_mma, 1);
        mbar_init(&bar_ready, 1);
        mbar_init(&bar_vec, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const uint32_t aX = smem_u32(sX), aT = smem_u32(sT), aOne = smem_u32(sOne), aP = smem_u32(sP), aRed = smem_u32(sR);

    if (warp == NEPI / 32) {
        // ================================ weight producer =====================================================
        if ((tid & 31) == 0) {
            mbar_expect_tx(&bar_vec, (uint32_t)d.vec_floats * 4u);
            bulk_g2s(sP, d.vec, (uint32_t)d.vec_floats * 4u, &bar_vec);
#pragma unroll 1
            for (int c = 0; c < NCHUNK; ++c) {
                const int s = c % NSLOT;
                if (c >= NSLOT) mbar_wait_backoff(&bar_empty[s], ((c / NSLOT) - 1) & 1);
                const uint32_t nbytes = (d.dbg_flags & 4) ? 16u : d.chunk_bytes[c];   // profiling: tiny copies
                mbar_expect_tx(&bar_full[s], nbytes);
                bulk_g2s(sW + (size_t)s * SLOT_BYTES, reinterpret_cast<const uint8_t *>(d.wpk) + d.chunk_off[c], nbytes, &bar_full[s]);
            }
        }
    } else if (warp == NEPI / 32 + 1) {
        // ================================ MMA issuer ==========================================================
        {
            const bool issuer = (tid & 31) == 0;   // all 32 lanes take part in the named barrier, lane 0 issues
            Pipe p{bar_full, bar_empty, &bar_mma, &bar_ready, smem_u32(sW), tmem, 0, 0, (d.dbg_flags & (2 | 8))};
            const uint32_t uKA = (uint32_t)KA;
            mma_stage_begin();                                   // in-proj: W_in [h | onehot]
            if (issuer) mma_chunk(p, TM_ACC, aT, H, 128, 0);
            if (issuer) mma_chunk(p, TM_ACC, aOne, uKA, 128, 1);
            if (issuer) mma_stage_end(p);
            __syncwarp();
#pragma unroll 1
            for (int l = 0; l < NLAYER; ++l) {
                mma_stage_begin();                               // q, k, v projections
                if (issuer) mma_chunk(p, TM_Q, aX, H, 128, 0);
                if (issuer) mma_chunk(p, TM_K, aX, H, 128, 0);
                if (issuer) mma_chunk(p, TM_V, aX, H, 128, 0);
                if (issuer) mma_stage_end(p);
                __syncwarp();
                mma_stage_begin();                               // x += sa Wo^T (residual = accumulate into X)
                if (issuer) mma_chunk(p, TM_X, aT, H, 128, 1);
                if (issuer) mma_stage_end(p);
                __syncwarp();
                mma_stage_begin();                               // linear1
                if (issuer) mma_chunk(p, TM_ACC, aX, H, 128, 0);
                if (issuer) mma_stage_end(p);
                __syncwarp();
                mma_stage_begin();                               // x += f W2^T
                if (issuer) mma_chunk(p, TM_X, aT, H, 128, 1);
                if (issuer) mma_stage_end(p);
                __syncwarp();
            }
            mma_stage_begin();                                   // fc_dynamic.0 on [h | onehot | attn]
            if (issuer) mma_chunk(p, TM_ACC, aT, H, 128, 0);
            if (issuer) mma_chunk(p, TM_ACC, aOne, uKA, 128, 1);
            if (issuer) mma_chunk(p, TM_ACC, aX, H, 128, 1);
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aT, H, 128, 0);                  // fc_dynamic.3
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aX, H, 128, 0);                  // fc_dynamic.6
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();                                   // reward GNN layer 1 on [h' | onehot]
            if (issuer) mma_chunk(p, TM_ACC, aT, H, 128, 0);
            if (issuer) mma_chunk(p, TM_ACC, aOne, uKA, 128, 1);
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aX, GH, 128, 0);                 // reward GNN layer 2
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aT, H, 128, 0);                  // value GNN layer 1
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aX, GH, 128, 0);                 // value GNN layer 2
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aT, H, PH, 0);                   // fc_policy.0
            if (issuer) mma_stage_end(p);
            __syncwarp();
            mma_stage_begin();
            if (issuer) mma_chunk(p, TM_ACC, aX, PH, (uint32_t)d.NAP, 0);     // fc_policy.3
            if (issuer) mma_stage_end(p);
            __syncwarp();
        }
    } else {
        // ================================ epilogue warps ======================================================
        const Thr t;
        const uint32_t trow = tmem + ((uint32_t)(t.quad * 32) << 16);   // this warp's 32 TMEM lanes
        // token <-> (root, agent): every quadrant-warp holds floor(32/N) whole roots
        const int rpw = 32 / N;
        const int rl = t.lane / N, agent = t.lane - rl * N;
        const int root = (blockIdx.x * 4 + t.quad) * rpw + rl;
        const int valid = (rl < rpw) && (root < d.B);
        const int root_lane0 = (rl < rpw) ? rl * N : 0;   // first lane of my root inside the warp
        uint32_t mma_phase = 0;
        int c_ep = 0;   // chunks consumed so far (ring-slot release bookkeeping)
        const bool do_epi = !(d.dbg_flags & 1);
        int ts_n = 0;
        const bool ts_on = d.dbg_clock != nullptr && blockIdx.x == 0 && tid == 0;
#define TS() \
    if (ts_on && ts_n < 256) d.dbg_clock[ts_n++] = clock64();
// publish my operand writes to the async proxy, tell the MMA warp, wait for the stage's accumulator
#define HANDOFF(nchunks)            \
    TS();                           \
    fence_proxy_async();            \
    tc_fence_before();              \
    named_bar_sync(5, NEPI + 32);   \
    mbar_wait(&bar_mma, mma_phase); \
    mma_phase ^= 1;                 \
    tc_fence_after();               \
    if (tid == 0) {                 \
        for (int i__ = 0; i__ < (nchunks); ++i__) mbar_arrive(&bar_empty[(c_ep + i__) % NSLOT]); \
    }                               \
    c_ep += (nchunks);              \
    TS();

        // PDL: everything up to here (and the producer warp's weight streaming) may overlap the tail of the tree kernel
        // that produces idx_x / actions; wait for it before touching its outputs or the pool.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        // Only NOW may the next tree kernel start: its pre-wait section prefetches tree state, which the tree kernel
        // we just waited for was still writing.  (The tree kernel itself triggers at its start: this kernel's
        // pre-wait section touches nothing but constants.)
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        // ---- gather the parent's hidden state and build the one-hot action operand ------------------------
        const float *hrow = d.pool;
        int my_action = -1;
        if (valid) {
            const int ix = d.idx_x ? __ldcg(d.idx_x + root) : 0;   // .cg: produced by the kernel we may have overlapped (PDL)
            hrow = d.pool + ((size_t)ix * d.B + root) * (size_t)(N * H) + (size_t)agent * H;
            if (d.greedy_pool == nullptr || d.cur < 0)
                my_action = __ldcg(d.actions + (size_t)root * N + agent);
            else if (agent == d.cur)                  // sequential-agent mode, joint action assembled here (mcts_sampled.py:116-147)
                my_action = __ldcg(d.actions + root);
            else if (agent < d.cur)
                my_action = d.factor ? __ldcg(d.factor + (size_t)root * N + agent) : 0;
            else
                my_action = __ldcg(d.greedy_pool + ((size_t)ix * d.B + root) * N + agent);
        }
        gather_hidden(hrow, valid, aT);
        if (t.part * 16 < KA) {
            const int c0 = t.part * 16;
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = ((c0 + i) == my_action) ? 1.f : 0.f;
            store_cols(aOne, t.row, c0, KA, v);
        }
        mbar_wait(&bar_vec, 0);   // parameters resident
        // ---- attention_stack[0..1]: x0 = relu(W_in [h | onehot] + b) + positional table --------------------
        HANDOFF(2);
        if (do_epi) epi_inproj(trow, aP + 4 * d.o_bin, aP + 4 * (d.o_pos + agent * H), aX);
        // ---- 3 x post-LN TransformerEncoderLayer over the agent axis (attention.py:36-43) ---------------------
#pragma unroll 1
        for (int l = 0; l < NLAYER; ++l) {
            const uint32_t lv = aP + 4 * (d.o_layer + l * 1280);   // bq bk bv bo g1 be1 b1 b2 g2 be2
            HANDOFF(3);
            if (do_epi) epi_attention(trow, lv, N, root_lane0, aT, aX);   // sX is free: the QKV GEMM is done with it
            HANDOFF(1);
            if (do_epi) epi_ln128(trow, TM_X, lv + 4 * 384, lv + 4 * 512, lv + 4 * 640, 0, 1, aX, aRed);     // norm1
            HANDOFF(1);
            if (do_epi) epi_bias_relu(trow, lv + 4 * 768, aT);                                                 // relu(linear1)
            HANDOFF(1);
            if (do_epi) epi_ln128(trow, TM_X, lv + 4 * 896, lv + 4 * 1024, lv + 4 * 1152, 0, 1, aX, aRed);   // norm2
        }
        // ---- fc_dynamic: Linear-LN-ReLU, Linear-LN-ReLU, Linear; residual (model.py:262-268) ------------------
        const uint32_t dv = aP + 4 * d.o_dyn;
        gather_hidden(hrow, valid, aT);   // h (bf16) back into sT; sX holds the attention output
        HANDOFF(3);
        if (do_epi) epi_ln128(trow, TM_ACC, dv, dv + 4 * 128, dv + 4 * 256, 1, 0, aT, aRed);
        HANDOFF(1);
        if (do_epi) epi_ln128(trow, TM_ACC, dv + 4 * 384, dv + 4 * 512, dv + 4 * 640, 1, 0, aX, aRed);
        HANDOFF(1);
        {
            float *nh = d.next_hidden + (valid ? (size_t)root * (N * H) + (size_t)agent * H : 0);
            if (do_epi) epi_next_hidden(trow, dv + 4 * 768, hrow, nh, valid, aT);
        }
        // ---- reward head: GraphNetNN on [next_hidden | onehot] (model.py:270-277) -----------------------------
        const uint32_t rv = aP + 4 * d.o_rg;
        HANDOFF(2);
        if (do_epi) epi_gnn(trow, rv, N, root_lane0, 0, aX, aRed, 0);
        HANDOFF(1);
        {
            const float r = !do_epi ? 0.f : epi_gnn(trow, rv + 4 * 128, N, root_lane0, 1, 0, aRed, aX);   // sX is free: scratch
            if (valid && agent == 0 && t.part == 0) d.reward[root] = r;
        }
        // ---- value head: GraphNetNN on next_hidden (model.py:359) ----------------------------------------------
        const uint32_t vv = aP + 4 * d.o_vg;
        HANDOFF(1);
        if (do_epi) epi_gnn(trow, vv, N, root_lane0, 0, aX, aRed, 0);
        HANDOFF(1);
        {
            const float val = !do_epi ? 0.f : epi_gnn(trow, vv + 4 * 128, N, root_lane0, 1, 0, aRed, aX);
            if (valid && agent == 0 && t.part == 0) d.value[root] = val;
        }
        // ---- policy head + the driver's softmax / beta ------------------------------------------------------------
        const uint32_t pv = aP + 4 * d.o_pol;
        HANDOFF(1);
        if (do_epi) epi_policy_hidden(trow, pv, aX, aRed);
        HANDOFF(1);
        if (do_epi && t.part == 0) epi_policy_out(d, trow, pv + 4 * 96, valid, root, agent);
        TS();
#undef HANDOFF
#undef TS
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}
#endif  // MAZ_FUSED_NO_KERNEL

}  // namespace fused
}  // namespace maz
