// infer_initial.cuh -- MAMuZeroNet.initial_inference (config/smac/model.py:542-559) as one small-batch kernel (sm_100a).
//
// The tile of infer_hmma.cuh (32 token rows = floor(32 / N) whole roots, 2*NQ compute warps on bf16 mma.sync with fp32
// accumulate, one producer warp streaming the weights through the 3-slot ring) fed from observations instead of a dynamics step:
//   1. feature_norm: LayerNorm over obs_dim with affine, fp32 (two passes over the row in global memory: mean, then the
//      variance of the deviations, so that observations with large offsets keep their precision), rounded to bf16;
//   2. mlp([obs_dim, 128, 128, 128]) (config/smac/model.py:176-195): Linear -> LN -> ReLU -> Linear -> LN -> ReLU -> Linear.
//      The first Linear runs over column blocks of <= 128 features: each block of the normalised observation is written to
//      tile HH and multiplied with its own weight chunk, K padded to 16 with zero weight columns.  The last output is the root
//      hidden state: fp32 to global (B, N*128), bf16 to tile T, the operand of the heads;
//   3. the prediction heads through the root variant (R = true) of stage_heads1 / stage_heads2: value graph net -> inverse
//      value transform -> value (B,); policy MLP 128 -> 32 -> A -> logits (B, N, A), no softmax / beta (root preparation,
//      maz_root_prepare_dev, does that with the noise and the legal mask).  The reward of initial_inference is zero.
// Ring chunks, in order: the nb = ceil(K16 / 128) column blocks of mlp.0, mlp.3, mlp.6, then chunks 27, 28, 30, 31 of the
// small-batch packing (value graph net layer 1, fc_policy.0, value graph net layer 2, fc_policy.3).
#pragma once
#include "infer_hmma.cuh"

namespace maz {
namespace hmma {

constexpr int OBS_MAX = 640;                                   // = MAZ_MLP_MAXWIDTH of the row-wise kernel
constexpr int INIT_MAXCHUNK = (OBS_MAX + 127) / 128 + 2 + 4;

struct InitialArgs {
    Desc d;                    // the heads' view: B, N, A, KA, NAP, roots_per_tile 0, o_rg = o_vg / o_pol (rebased), vec, vec_floats
    const float *obs;          // (B*N, obs_dim) fp32
    float *hidden, *value, *logits;
    const float *rep_vec;      // feature_norm w | b (kp each), mlp.0 b, mlp.1 w | b, mlp.3 b, mlp.4 w | b, mlp.6 b (128 each)
    int rep_floats;            // 2 * kp + 7 * 128
    int obs_dim, kp;           // kp = obs_dim rounded up to 16
    int nchunk;
    const uint8_t *chunk_src[INIT_MAXCHUNK];
    uint32_t chunk_bytes[INIT_MAXCHUNK];
};

__host__ __device__ inline size_t initial_smem_bytes(int vec_floats, int rep_floats)
{
    return smem_bytes(vec_floats) + (size_t)rep_floats * 4;
}

// producer (one thread): the heads' parameters and the representation's parameters behind them, then the chunk list once
__device__ __forceinline__ void produce_initial(const InitialArgs &a, uint64_t *bar_full, uint64_t *bar_empty, uint64_t *bar_vec)
{
    HSM_DECL;
    const uint32_t vb = (uint32_t)a.d.vec_floats * 4u, rb = (uint32_t)a.rep_floats * 4u;
    mbar_expect_tx(bar_vec, vb + rb);
    bulk_g2s(hsm + OFF_P, a.d.vec, vb, bar_vec);
    bulk_g2s(hsm + OFF_P + vb, a.rep_vec, rb, bar_vec);
#pragma unroll 1
    for (int c = 0; c < a.nchunk; ++c) {
        const int s = c % NSLOT;
        if (c >= NSLOT) mbar_wait_backoff(&bar_empty[s], ((c / NSLOT) - 1) & 1);
        const uint32_t nbytes = a.chunk_bytes[c];
        uint8_t *dst = hsm + OFF_W + (size_t)s * SLOT_BYTES;
        mbar_expect_tx(&bar_full[s], nbytes);
        for (uint32_t o = 0; o < nbytes; o += PIECE) {
            const uint32_t n = (nbytes - o < PIECE) ? (nbytes - o) : PIECE;
            bulk_g2s(dst + o, a.chunk_src[c] + o, n, &bar_full[s]);
        }
    }
}

// acc = bias + LayerNorm(128) + ReLU epilogue of a 128-wide representation layer, bf16 -> tile `dst`
__device__ __forceinline__ void rep_ln_relu(float (&acc)[NT][4], const Thr &th, uint32_t dst, uint32_t p, int n0)
{
    add_bias<NT>(acc, th, p, n0);
    layer_norm128(acc, th, p + 4u * H, p + 8u * H, n0, true);
    store_tile<NT>(dst, LDA, th, n0, acc);
    cta_sync();
}

// observation rows -> feature_norm -> mlp -> root hidden state (global fp32, tile T bf16)
static __device__ __noinline__ void stage_representation(const InitialArgs &a, Ring &ring)
{
    HSM_DECL;
    const Thr th;
    const uint32_t sb = sbase();
    const int n0 = CW * th.nq, tid = threadIdx.x, r = (tid >> 3) & (TM - 1), part = tid & 7;
    const int K = a.obs_dim, KP = a.kp;
    const uint32_t fw = sb + OFF_P + 4u * a.d.vec_floats, fb = fw + 4u * KP, pb = fb + 4u * KP;   // feature_norm w, b; mlp params
    const RowInfo ri = row_info(r);
    const bool mine = tid < TM * 8 && ri.valid;      // 8 threads per row (warp-uniform: tid < TM * 8)
    const float *x = a.obs + (size_t)(mine ? ri.root * a.d.N + ri.agent : 0) * K;
    // feature_norm statistics over the row, fp32, two passes (every lane runs the shuffles)
    const int kk = mine ? K : 0;
    float s = 0.f;
    for (int c = part; c < kk; c += 8) s += __ldg(x + c);
#pragma unroll
    for (int o = 1; o <= 4; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)K;
    float q = 0.f;
    for (int c = part; c < kk; c += 8) {
        const float dv = __ldg(x + c) - mean;
        q += dv * dv;
    }
#pragma unroll
    for (int o = 1; o <= 4; o <<= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q / (float)K + 1e-5f);
    // mlp.0 over column blocks of <= 128 features of the normalised observation (tile HH)
    float acc[NT][4];
    zero<NT>(acc);
#pragma unroll 1
    for (int k0 = 0; k0 < KP; k0 += 128) {
        const int kc = KP - k0 < 128 ? KP - k0 : 128;
        if (tid < TM * 8) {
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = k0 + part * 16 + 2 * i;
                float v0 = 0.f, v1 = 0.f;
                if (mine && c < K) v0 = (__ldg(x + c) - mean) * rstd * lds1(fw + 4u * c) + lds1(fb + 4u * c);
                if (mine && c + 1 < K) v1 = (__ldg(x + c + 1) - mean) * rstd * lds1(fw + 4u * (c + 1)) + lds1(fb + 4u * (c + 1));
                w[i] = pack2(v0, v1);
            }
            uint4 *dst = reinterpret_cast<uint4 *>(hsm + OFF_HH + (size_t)r * LDA + part * 32);
            dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
            dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
        cta_sync();
        const uint32_t wc = ring.acquire();
        if (kc == 128) gemm_fixed<NT, 8>(acc, th, sb + OFF_HH, LDA, wc, LDA, n0);
        else gemm_rt<NT>(acc, th, sb + OFF_HH, LDA, wc, (kc + PAD) * 2, n0, kc);
        ring.release(th.lane);
        cta_sync();                                  // tile HH takes the next block
    }
    rep_ln_relu(acc, th, sb + OFF_X, pb, n0);                                    // mlp.0 bias, mlp.1 LN, ReLU -> X
    zero<NT>(acc);
    uint32_t wc = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_X, LDA, wc, LDA, n0);
    ring.release(th.lane);
    rep_ln_relu(acc, th, sb + OFF_HH, pb + 4u * (3 * H), n0);                    // mlp.3 bias, mlp.4 LN, ReLU -> HH
    zero<NT>(acc);
    wc = ring.acquire();
    gemm_fixed<NT, 8>(acc, th, sb + OFF_HH, LDA, wc, LDA, n0);
    ring.release(th.lane);
    add_bias<NT>(acc, th, pb + 4u * (6 * H), n0);                                // mlp.6 bias: the root hidden state
    const RowInfo ra = row_info(th.rA), rb = row_info(th.rB);
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
        const RowInfo &rr = hf ? rb : ra;
        if (!rr.valid) continue;
        float *hp = a.hidden + (size_t)rr.root * (a.d.N * H) + (size_t)rr.agent * H;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
            *reinterpret_cast<float2 *>(hp + n0 + 8 * nt + 2 * th.t) = make_float2(acc[nt][2 * hf], acc[nt][2 * hf + 1]);
    }
    store_tile<NT>(sb + OFF_T, LDA, th, n0, acc);
    cta_sync();
}

template <bool W>
__global__ void __launch_bounds__(NTHREADS, 1) k_initial_inference_small(const __grid_constant__ InitialArgs a)
{
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_vec;
    const int tid = threadIdx.x, warp = tid >> 5;
    const Desc &d = a.d;
    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], NCONS / 32); }
        mbar_init(&bar_vec, 1);
        mbar_fence_init();
    }
    setup_rows(d);
    __syncthreads();
    if (warp == NCONS / 32) {
        if ((tid & 31) == 0) produce_initial(a, bar_full, bar_empty, &bar_vec);
        return;
    }
    Ring ring{bar_full, bar_empty, 0};
    const SimIo io{nullptr, nullptr, nullptr, a.value, nullptr, nullptr, 0, a.hidden, nullptr, a.logits};
    mbar_wait(&bar_vec, 0);          // parameters resident
    setup_head_copies(d);            // (o_rg = o_vg: both padded copies hold the value head; phase E reads the value one)
    stage_representation(a, ring);
    stage_heads1<W, true>(d, ring);
    stage_heads2<W, true>(d, ring, io, nullptr);
}

}  // namespace hmma
}  // namespace maz
