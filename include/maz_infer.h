/*
 * maz_infer.h -- C ABI of the fused network forward used inside the search (libmaz_b200.so).
 *
 * Replaces, for the search only, the reference's per-simulation model calls
 *   model.recurrent_inference(hidden, action)   config/smac/model.py:562-574
 *   model.prediction(hidden)                    config/smac/model.py:494-501
 * (called from core/mcts/tree_search/mcts_sampled.py:137,151) with one sm_100a kernel whose GEMMs run on
 * the tcgen05 tensor cores in bf16 with fp32 accumulation in TMEM.  Device pointers only; asynchronous on
 * the given stream.  Same error convention as maz_tree.h (maz_last_error()).
 */
#ifndef MAZ_INFER_H
#define MAZ_INFER_H

#ifdef __cplusplus
extern "C" {
#endif

/* Self-test of the tensor-core GEMM stage: out[128 x n] (fp32) = bf16(a[128 x k]) * w_packed[n x k]^T.
 * `w_packed` is bf16 in the kernels' shared-memory operand layout (see mazero_b200/csrc/umma.cuh):
 * W.view(n/8, 8, k/8, 8).permute(0, 2, 1, 3).  n, k multiples of 16, n <= 256, k <= 512. */
int maz_dbg_umma_gemm(const float *a, const void *w_packed, float *out, int n, int k, void *cuda_stream);

/* Everything one launch of the fused recurrent_inference kernel needs.  All pointers are DEVICE pointers.
 * Fixed architecture (config/smac/__init__.py:15-27): hidden 128 per agent, 3 encoder layers x 8 heads,
 * dim_feedforward 128, fc_dynamic [128,128], GNN hidden 64, fc_policy [32], support 11; agents N <= 32,
 * actions A <= 128 (KA > 48 launches the wide instances of the small-batch and the two-tiles-in-flight kernels; the first-generation
 * kernel, tc_layout 0, takes A <= 48 and returns MAZ_ERR_UNSUPPORTED above).  Weight packing: see mazero_b200/fused.py (pack_weights). */
#define MAZ_INFER_NCHUNK 32
typedef struct maz_infer_desc {
    int B, N, A, KA, NAP;        /* roots, agents, actions, A rounded up to 16 (twice) */
    int Nt, cur;                 /* agents in the tree (N joint / 1 sequential), sequential agent index or -1 */
    float inv_tau;               /* 1 / sampled_tau (mcts_sampled.py:160) */
    const float *pool;           /* hidden-state pool: row (idx*B + b), N*128 floats */
    const int *idx_x;            /* (B,) pool index of the parent of each root's leaf, or NULL (= 0) */
    const int *actions;          /* (B,N) joint action */
    float *next_hidden;          /* (B, N*128) */
    float *reward, *value;       /* (B,) scalars after the inverse support transform */
    float *probs, *beta;         /* (B,Nt,A) softmax of the policy logits and probs^(1/tau) renormalised */
    int *greedy;                 /* (B,N) argmax_a of the policy logits, or NULL */
    float *logits_out;           /* (B,N,A) raw policy logits, or NULL */
    const void *wpk;             /* bf16 weight chunks in tcgen05 operand layout */
    const float *vec;            /* fp32 biases / LayerNorm affine / positional table / heads */
    int vec_floats;              /* length of vec, multiple of 4 (copied to shared memory in one bulk copy) */
    unsigned int chunk_off[MAZ_INFER_NCHUNK];
    unsigned int chunk_bytes[MAZ_INFER_NCHUNK];
    int o_bin, o_pos, o_layer, o_dyn, o_rg, o_vg, o_pol;   /* float offsets into vec */
    long long *dbg_clock;        /* optional (NULL): SM-cycle timestamps of CTA 0's stages, 256 entries (profiling) */
    int dbg_flags;               /* profiling only: 1 = skip the epilogue math, 2 = skip the MMAs (results are garbage) */
    int roots_per_tile;          /* small-batch kernel only: whole roots per 32-row tile, 0 = floor(32 / N) */
    /* Sequential-agent mode with the joint action assembled IN the kernel (mcts_sampled.py:116-147), when greedy_pool is
     * non-NULL and cur >= 0: `actions` is then the TREE's action (B,1) of agent `cur`; agents k < cur take factor[b][k]
     * (zeros when factor is NULL), agents k > cur take greedy_pool[idx_x[b]][b][k] = argmax_a prediction(parent).policy. */
    const int *factor;           /* (B,N) or NULL */
    const int *greedy_pool;      /* (S+1,B,N): row (idx*B + b), or NULL (`actions` is the full (B,N) joint action) */
    /* maz_infer_recurrent only: which large-batch kernel `wpk` / `vec` / the chunk table are packed for.
     * 0: one tile per CTA (csrc/infer_fused.cuh; 32 chunks, `vec` copied to shared memory).
     * 1: two tiles in flight per CTA (csrc/infer_twin.cuh; 32 matrices stored as K-halves in the order of its stage table,
     *    `vec` read from global memory and followed by the three one-hot weight blocks W_a^T as bf16 [A][128] tables,
     *    i.e. [A][64] 32-bit words). */
    int tc_layout;
    int o_oh_in, o_oh_dyn, o_oh_rg;   /* tc_layout 1: float offsets into vec of the one-hot blocks of attention_stack.0 /
                                         fc_dynamic.0 / reward_predictor layer 1 (gc | nn stacked) */
} maz_infer_desc;

/* replaces model.recurrent_inference + the driver's softmax/beta (mcts_sampled.py:150-161): one kernel launch */
int maz_infer_recurrent(const maz_infer_desc *desc, void *cuda_stream);

/* The same computation for SMALL batches (mazero_b200/csrc/infer_hmma.cuh): 32-row tiles on warp-level bf16 MMAs, so
 * that 1024 roots x 3 agents fill 103 SMs instead of 26 and the per-simulation latency chain is short.  `wpk` and the
 * chunk tables are in the row-major padded layout of mazero_b200/fused.py::HmmaParams (chunk = [out][K + 8] bf16);
 * `vec` and all other fields as above. */
int maz_infer_recurrent_small(const maz_infer_desc *desc, void *cuda_stream);
/* number of column groups the small-batch kernel was compiled for (4 or 8): the stacked graph-net weights are
 * interleaved in groups of 64 / nq features (gc rows, then nn rows) by the host-side packer. */
int maz_infer_small_nq(void);
/* opt both kernels into their dynamic shared-memory sizes ahead of time (called by maz_search_create, so that the launches
 * captured into a CUDA graph do not have to); vec_floats / ka as in the descriptor */
int maz_infer_configure(int vec_floats, int ka);

/* ---- MLP-family network (the reference's matrix-game MAMuZeroNet) --------------------------------------------
 * Replaces, for the search only, config/matrix/model.py:358-368 `recurrent_inference` (= `dynamics` :334-343 /
 * DynamicsNetwork.forward :118-126 + PredictionNetwork.forward :163-166) and the driver's softmax / beta
 * (mcts_sampled.py:158-161).  fp32 SIMT kernel, one CTA per root; device pointers; asynchronous on the stream.
 * A layer computes y = W x + b followed by nothing (MAZ_MLP_LINEAR), ReLU then LayerNorm (MAZ_MLP_RELU_LN, the
 * matrix mlp() order, config/matrix/model.py:44-46) or LayerNorm then ReLU (MAZ_MLP_LN_RELU, the SMAC order).
 * `wt` is the weight TRANSPOSED to [in][out] (row-major). */
#define MAZ_MLP_MAXLAYERS 6
#define MAZ_MLP_MAXWIDTH 640
enum { MAZ_MLP_LINEAR = 0, MAZ_MLP_RELU_LN = 1, MAZ_MLP_LN_RELU = 2, MAZ_MLP_LN_ONLY = 3 /* maz_mlp_forward only: LayerNorm of the input, no Linear */ };
typedef struct maz_mlp_layer {
    const float *wt, *b, *ln_w, *ln_b;   /* ln_* NULL for MAZ_MLP_LINEAR */
    int in, out, kind;
} maz_mlp_layer;
typedef struct maz_mlp_net {
    int n;
    maz_mlp_layer l[MAZ_MLP_MAXLAYERS];
} maz_mlp_net;
typedef struct maz_mlp_desc {
    int B, N, A, H;              /* roots, agents, actions per agent, hidden size per agent */
    int Nt, cur;                 /* agents in the tree (N joint / 1 sequential), sequential agent index or -1 */
    float inv_tau;               /* 1 / sampled_tau */
    const float *pool;           /* hidden-state pool: row (idx*B + b), N*H floats */
    const int *idx_x;            /* (B,) or NULL (= 0) */
    const int *actions;          /* (B,N) joint action */
    float *next_hidden;          /* (B, N*H) */
    float *reward, *value;       /* (B,) scalars after the inverse support transform */
    float *probs, *beta;         /* (B,Nt,A) */
    int *greedy;                 /* (B,N) argmax_a of the policy logits, or NULL */
    float *logits_out;           /* (B,N,A) raw policy logits, or NULL */
    maz_mlp_net dyn, rew, val, pol;   /* fc_dynamic (N*H+N*A -> N*H), fc_reward (N*H+N*A -> support),
                                         fc_value (N*H -> support), fc_policy (H -> A, applied per agent) */
    int reward_support_min, reward_support_size;   /* size 1: scalar head, no transform (use_vectorization=False) */
    int value_support_min, value_support_size;
    const int *factor;           /* in-kernel joint-action assembly of the sequential-agent mode: see maz_infer_desc */
    const int *greedy_pool;
} maz_mlp_desc;

int maz_mlp_recurrent(const maz_mlp_desc *desc, void *cuda_stream);

/* Row-wise MLP, y[r] = net(x[r]) for `rows` independent rows: the representation network of `initial_inference`
 * (config/smac/model.py:176-195 with its feature LayerNorm as a MAZ_MLP_LN_ONLY first layer, :470-489; config/matrix/model.py:54-83),
 * one row per agent observation.  x (rows, net->l[0].in), y (rows, out of the last layer); fp32; device pointers. */
int maz_mlp_forward(const maz_mlp_net *net, const float *x, int rows, float *y, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* MAZ_INFER_H */
