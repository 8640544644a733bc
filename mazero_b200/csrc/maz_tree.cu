// maz_tree.cu -- host side of libmaz_b200.so: arena management, kernel launches, the C ABI of
// include/maz_tree.h.  No CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/maz_tree.h"
#include "tree_host.h"
#include "tree_kernels.cuh"

using namespace maz;

static thread_local std::string g_last_error;

static int set_err(int code, const std::string &msg)
{
    g_last_error = msg;
    return code;
}
namespace maz {
int set_last_error(int code, const std::string &msg) { return set_err(code, msg); }  // shared with maz_infer.cu
// Programmatic dependent launch between the two kernels of the on-device loop: MAZ_PDL bit 0 = inference kernel,
// bit 1 = tree kernel.  OFF by default: measured on B200 inside the CUDA graph it buys nothing (5.668 ms vs 5.664 ms
// per 1024 x 50 search), and it needs care: an early-resident dependent grid can hit STALE L1 lines of buffers that
// the predecessor is still writing (the per-simulation reward / value / probs / beta buffers are re-used every
// simulation) -- data produced by the predecessor is therefore read with ld.global.cg (L2) in both kernels.
int pdl_mask()
{
    static const int m = [] { const char *e = getenv("MAZ_PDL"); return e ? atoi(e) : 0; }();
    return m;
}
bool pdl_enabled() { return pdl_mask() != 0; }
}

#define CU_TRY(expr)                                                                                          \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return set_err(MAZ_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));                \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static const char *dev_err_msg(int code)
{
    switch (code) {
        case kErrValueSetInvariant: return "SubTreeValueSet::update: cur_size+1!=size_lim.";
        case kErrPoolExhausted: return "node pool exhausted (more expansions than simulation_num allows)";
        case kErrLogOverflow: return "value log overflow (more simulations than simulation_num)";
        case kErrPathOverflow: return "search path longer than simulation_num + 1";
        default: return "unknown device-side failure";
    }
}

namespace maz { const char *device_error_message(int code) { return dev_err_msg(code); } }

static unsigned align_up(unsigned long long x, unsigned a) { return (unsigned)((x + a - 1) / a * a); }

static int build_layout(TreeLayout &L, int B, int N, int A, int K, int S, float delta_lb, float rho, float lam)
{
    if (B <= 0 || N <= 0 || A <= 0 || K <= 0 || S < 0) return set_err(MAZ_ERR_INVALID, "maz_tree_create: dimensions must be positive");
    if (K > kMaxSampledTimes) return set_err(MAZ_ERR_UNSUPPORTED, "sampled_times > 32 is not supported by the warp-per-tree kernels");
    if (A > 255) return set_err(MAZ_ERR_UNSUPPORTED, "action_space_size > 255 is not supported (actions are stored as bytes)");
    const long long P = (long long)K * (S + 2);
    if (P > 65535 || S > 32000) return set_err(MAZ_ERR_UNSUPPORTED, "sampled_times*(simulation_num+2) > 65535 is not supported (16-bit node slots)");
    L.B = B; L.N = N; L.A = A; L.K = K; L.S = S;
    L.P = (int)P;
    L.L = 1 + S * (S + 3) / 2 + 8;
    L.delta_lb = delta_lb;
    L.one_minus_rho = 1 - rho;  // float, as in utils.cpp:31
    L.lam = lam;
    const unsigned Pp = align_up(P, 32);
    unsigned long long o = sizeof(TreeHdr);
    auto take = [&](unsigned long long bytes) { o = align_up(o, 128); unsigned at = (unsigned)o; o += bytes; return at; };
    L.off_mt = take(4ull * kMtN);
    L.off_rec = take(sizeof(NodeRec) * Pp);
    L.off_pred_prob = take(4ull * Pp);
    L.off_beta = take(4ull * Pp);
    L.off_beta_hat = take(4ull * Pp);
    L.off_qdelta = take(4ull * Pp);
    L.off_actions = take(1ull * Pp * N);
    L.off_expslot = take(2ull * (S + 4));
    L.off_path = take(2ull * (S + 4));
    L.off_vskey = take(4ull * L.L);
    L.off_vsval = take(4ull * L.L);
    L.off_depth = take(2ull * (S + 4));      // depth of the e-th expanded node (its distance from the root)
    {   // wide selection: worth it once the sequential descent (~2 k cycles per level) costs more than one pass over all expanded
        // nodes (~4 k cycles per 32 of them).  MAZ_SELECT_WIDE=0 never, 1 always: identical results
        // (the fused-step cases of tests/test_tree_gpu.py and tests/test_deep_trees_gpu.py run all three settings).
        const char *e = getenv("MAZ_SELECT_WIDE");
        const int chunks = (S + 1 + 31) / 32;
        L.wide_min_len = e ? (atoi(e) ? 0 : 1 << 30) : 3 + 2 * chunks;
    }
    L.slab_bytes = align_up(o, 256);
    if (o > 0xfffffff0ull) return set_err(MAZ_ERR_UNSUPPORTED, "per-tree slab exceeds 4 GiB");
    return MAZ_OK;
}

static int upload_lam_pow(maz_tree *t)
{
    std::vector<float> lp(t->L.S + 2);
    for (int d = 0; d < (int)lp.size(); ++d) lp[d] = (d == 0) ? 1.0f : lp[d - 1] * t->L.lam;
    CU_TRY(cudaMemcpyAsync(t->d_lam_pow, lp.data(), lp.size() * sizeof(float), cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaStreamSynchronize(t->stream));
    return MAZ_OK;
}

extern "C" {

int maz_abi_version(void) { return MAZ_ABI_VERSION; }
const char *maz_last_error(void) { return g_last_error.c_str(); }

int maz_tree_create(maz_tree **out, int B, int N, int A, int K, int S, float delta_lb, unsigned int seed, float rho, float lam)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_err(MAZ_ERR_CUDA, "no CUDA device available (libmaz_b200 has no CPU fallback)");
    return maz_tree_create_ex(out, B, N, A, K, S, delta_lb, seed, rho, lam, dev, 0u);
}

int maz_tree_create_ex(maz_tree **out, int B, int N, int A, int K, int S, float delta_lb, unsigned int seed, float rho,
                       float lam, int device, unsigned int root_index_offset)
{
    if (!out) return set_err(MAZ_ERR_INVALID, "maz_tree_create: out is NULL");
    *out = nullptr;
    TreeLayout L{};
    int rc = build_layout(L, B, N, A, K, S, delta_lb, rho, lam);
    if (rc) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return set_err(MAZ_ERR_CUDA, "no CUDA device available (libmaz_b200 has no CPU fallback)");
    if (device < 0 || device >= ndev) return set_err(MAZ_ERR_INVALID, "maz_tree_create: bad device index");
    DeviceGuard g(device);
    if (!g.ok) return set_err(MAZ_ERR_CUDA, "cudaSetDevice failed");

    maz_tree *t = new maz_tree();
    t->L = L;
    t->device = device;
    t->seed = seed;
    t->root_offset = root_index_offset;
    t->arena_bytes = (size_t)L.slab_bytes * (size_t)B;
    t->table_len = S + 2;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    // one warp per tree; keep at least ~8 blocks per SM in flight before packing more trees per block
    t->wpb = (B <= sms * 8) ? 1 : (B <= sms * 16) ? 2 : 4;
    t->scratch_per_warp = tree_scratch_bytes(N, A, K, S);

    auto fail = [&](int code, const std::string &m) { maz_tree_destroy(t); return set_err(code, m); };
    cudaError_t e;
    if ((e = cudaMalloc(&t->arena, t->arena_bytes)) != cudaSuccess)
        return fail(MAZ_ERR_CUDA, std::string("cudaMalloc(arena): ") + cudaGetErrorString(e));
    if ((e = cudaMalloc(&t->d_lam_pow, sizeof(float) * t->table_len)) != cudaSuccess ||
        (e = cudaMalloc(&t->d_logterm, sizeof(float) * t->table_len)) != cudaSuccess ||
        (e = cudaMalloc(&t->d_sqrtn, sizeof(double) * t->table_len)) != cudaSuccess ||
        (e = cudaMalloc(&t->d_err, sizeof(int))) != cudaSuccess ||
        (e = cudaMalloc(&t->d_sums, 2 * sizeof(unsigned long long))) != cudaSuccess)
        return fail(MAZ_ERR_CUDA, std::string("cudaMalloc(tables): ") + cudaGetErrorString(e));
    if ((e = cudaMemset(t->d_err, 0, sizeof(int))) != cudaSuccess) return fail(MAZ_ERR_CUDA, cudaGetErrorString(e));
    // the expansion kernels use dynamic shared memory: wpb * scratch_per_warp
    const size_t dyn = t->scratch_per_warp * t->wpb;
    if (dyn > 227 * 1024) return fail(MAZ_ERR_UNSUPPORTED, "agent_num*action_space_size too large for the shared-memory staging");
    if (dyn > 48 * 1024) {
        if ((e = cudaFuncSetAttribute(k_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn)) != cudaSuccess ||
            (e = cudaFuncSetAttribute(k_expand_backup, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn)) != cudaSuccess ||
            (e = cudaFuncSetAttribute(k_expand_backup_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn)) != cudaSuccess ||
            (e = cudaFuncSetAttribute(k_expand_backup_select2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn)) != cudaSuccess)
            return fail(MAZ_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    }
    if ((rc = upload_lam_pow(t)) != MAZ_OK) { std::string m = g_last_error; return fail(rc, m); }
    *out = t;
    return MAZ_OK;
}

void maz_tree_destroy(maz_tree *t)
{
    if (!t) return;
    DeviceGuard g(t->device);
    cudaFree(t->arena);
    cudaFree(t->d_lam_pow);
    cudaFree(t->d_logterm);
    cudaFree(t->d_sqrtn);
    cudaFree(t->d_pbc);
    cudaFree(t->d_err);
    cudaFree(t->d_sums);
    cudaFree(t->s_rewards);
    cudaFree(t->s_values);
    cudaFree(t->s_probs);
    cudaFree(t->s_beta);
    cudaFree(t->s_noises);
    cudaFree(t->s_idx);
    cudaFree(t->s_readout);
    delete t;
}

int maz_tree_reset(maz_tree *t, unsigned int seed, float delta_lb, float rho, float lam, unsigned int root_index_offset)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    DeviceGuard g(t->device);
    t->seed = seed;
    t->root_offset = root_index_offset;
    t->L.delta_lb = delta_lb;
    t->L.one_minus_rho = 1 - rho;
    t->prepared = false;
    if (lam != t->L.lam) {
        t->L.lam = lam;
        return upload_lam_pow(t);
    }
    return MAZ_OK;
}

int maz_tree_set_stream(maz_tree *t, void *stream)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    t->stream = static_cast<cudaStream_t>(stream);
    return MAZ_OK;
}

int maz_tree_check(maz_tree *t)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    DeviceGuard g(t->device);
    int code = 0;
    CU_TRY(cudaMemcpyAsync(&code, t->d_err, sizeof(int), cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaStreamSynchronize(t->stream));
    if (code) return set_err(MAZ_ERR_DEVICE, dev_err_msg(code));
    return MAZ_OK;
}

int maz_tree_set_puct(maz_tree *t, float c_base, float c_init)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (t->puct_set && t->c_base == c_base && t->c_init == c_init) return MAZ_OK;
    DeviceGuard g(t->device);
    std::vector<float> lt(t->table_len);
    std::vector<double> sq(t->table_len);
    for (int n = 0; n < t->table_len; ++n) {
        // cnode.cpp:313: pb_c = log((n + pb_c_base + 1) / pb_c_base) + pb_c_init, with the overloads the
        // reference's toolchain resolves: float quotient, double log (glibc), double sum, stored to float.
        float ratio = ((float)n + c_base + 1) / c_base;
        lt[n] = (float)(std::log((double)ratio) + (double)c_init);
        sq[n] = std::sqrt((double)n);  // cnode.cpp:314: sqrt(int) -> double
    }
    CU_TRY(cudaMemcpyAsync(t->d_logterm, lt.data(), lt.size() * sizeof(float), cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->d_sqrtn, sq.data(), sq.size() * sizeof(double), cudaMemcpyHostToDevice, t->stream));
    // the whole prior coefficient as a 2-D table: fp64 divide + multiply cost ~600 cycles per tree level on the device
    // (few fp64 units), the table is one L1/L2-resident float load.  Same IEEE double operations, evaluated here.
    const size_t T = (size_t)t->table_len;
    if (T * T <= (size_t)4 << 20) {
        std::vector<float> pbc(T * T);
        for (size_t n = 0; n < T; ++n)
            for (size_t v = 0; v < T; ++v) pbc[n * T + v] = (float)((double)lt[n] * (sq[n] / (double)(v + 1)));
        if (!t->d_pbc) CU_TRY(cudaMalloc(&t->d_pbc, sizeof(float) * T * T));
        CU_TRY(cudaMemcpyAsync(t->d_pbc, pbc.data(), pbc.size() * sizeof(float), cudaMemcpyHostToDevice, t->stream));
        CU_TRY(cudaStreamSynchronize(t->stream));
        t->L.pbc_table = t->d_pbc;
        t->L.pbc_dim = (int)T;
    } else {
        t->L.pbc_table = nullptr;
        t->L.pbc_dim = 0;
    }
    CU_TRY(cudaStreamSynchronize(t->stream));
    t->c_base = c_base;
    t->c_init = c_init;
    t->puct_set = true;
    return MAZ_OK;
}

static inline dim3 tree_grid(const maz_tree *t) { return dim3((unsigned)((t->L.B + t->wpb - 1) / t->wpb)); }
static inline dim3 tree_block(const maz_tree *t) { return dim3(32u * t->wpb); }

int maz_tree_prepare_dev(maz_tree *t, const float *rewards, const float *values, const float *probs, const float *beta,
                         int K, float eps, const float *noises)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (K < 1 || K > t->L.K) return set_err(MAZ_ERR_INVALID, "prepare: sampled_times must be in [1, constructor's sampled_times]");
    if (!rewards || !values || !probs || !beta || (eps > 0 && !noises)) return set_err(MAZ_ERR_INVALID, "prepare: NULL input");
    DeviceGuard g(t->device);
    const unsigned seed_base = t->seed * 2333u + t->root_offset;  // cnode.cpp:574
    k_seed<<<(t->L.B + 127) / 128, 128, 0, t->stream>>>(t->L, t->arena, seed_base);   // 4 warps x 32 trees per block
    k_prepare<<<tree_grid(t), tree_block(t), t->scratch_per_warp * t->wpb, t->stream>>>(
        t->L, t->arena, t->d_lam_pow, rewards, values, probs, beta, K, eps, noises, t->d_err);
    CU_TRY(cudaGetLastError());
    t->prepared = true;
    return MAZ_OK;
}

int maz_tree_batch_selection_dev(maz_tree *t, float c_base, float c_init, float discount, int *idx_x, int *idx_y, int *act)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!t->prepared) return set_err(MAZ_ERR_INVALID, "batch_selection before prepare");
    if (!idx_x || !idx_y || !act) return set_err(MAZ_ERR_INVALID, "batch_selection: NULL output");
    int rc = maz_tree_set_puct(t, c_base, c_init);
    if (rc) return rc;
    DeviceGuard g(t->device);
    k_select<<<tree_grid(t), tree_block(t), 0, t->stream>>>(t->L, t->arena, t->d_logterm, t->d_sqrtn, t->table_len,
                                                             discount, idx_x, idx_y, act, t->d_err);
    CU_TRY(cudaGetLastError());
    return MAZ_OK;
}

int maz_tree_batch_expansion_and_backup_dev(maz_tree *t, int hidx, float discount, int K, const float *rewards,
                                            const float *values, const float *probs, const float *beta)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!t->prepared) return set_err(MAZ_ERR_INVALID, "batch_expansion_and_backup before prepare");
    if (K < 1 || K > t->L.K) return set_err(MAZ_ERR_INVALID, "expansion: sampled_times must be in [1, constructor's sampled_times]");
    if (hidx < 0 || hidx > 32767) return set_err(MAZ_ERR_INVALID, "expansion: hidden_state_index_x out of range");
    if (!rewards || !values || !probs || !beta) return set_err(MAZ_ERR_INVALID, "expansion: NULL input");
    DeviceGuard g(t->device);
    k_expand_backup<<<tree_grid(t), tree_block(t), t->scratch_per_warp * t->wpb, t->stream>>>(
        t->L, t->arena, t->d_lam_pow, hidx, discount, K, rewards, values, probs, beta, t->d_err);
    CU_TRY(cudaGetLastError());
    return MAZ_OK;
}

int maz_tree_expansion_backup_selection_dev(maz_tree *t, int hidx, float discount, int K, const float *rewards,
                                            const float *values, const float *probs, const float *beta, float c_base,
                                            float c_init, int *idx_x, int *idx_y, int *act)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!t->prepared) return set_err(MAZ_ERR_INVALID, "expansion before prepare");
    if (K < 1 || K > t->L.K) return set_err(MAZ_ERR_INVALID, "expansion: sampled_times must be in [1, constructor's sampled_times]");
    if (hidx < 0 || hidx > 32767) return set_err(MAZ_ERR_INVALID, "expansion: hidden_state_index_x out of range");
    if (!rewards || !values || !probs || !beta || !idx_x || !idx_y || !act) return set_err(MAZ_ERR_INVALID, "NULL argument");
    int rc = maz_tree_set_puct(t, c_base, c_init);
    if (rc) return rc;
    DeviceGuard g(t->device);
    // launched as a programmatic dependent of the inference kernel: the tree-state prefetch overlaps its tail
    cudaLaunchConfig_t cfg = {};
    // two warps per tree (expansion || backup): wpb trees per block -> 64 * wpb threads
    cfg.gridDim = tree_grid(t);
    cfg.blockDim = dim3(64u * t->wpb);
    cfg.dynamicSmemBytes = t->scratch_per_warp * t->wpb;
    cfg.stream = t->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (maz::pdl_mask() & 2) ? 1 : 0;
    const float *lam = t->d_lam_pow, *lt = t->d_logterm;
    const double *sq = t->d_sqrtn;
    CU_TRY(cudaLaunchKernelEx(&cfg, k_expand_backup_select2, t->L, t->arena, lam, hidx, discount, K, rewards, values, probs, beta,
                              lt, sq, t->table_len, idx_x, idx_y, act, t->d_err));
    return MAZ_OK;
}

// ---- host-pointer entry points: stage through device buffers owned by the handle ---------------------
static int ensure_staging(maz_tree *t)
{
    if (t->s_rewards) return MAZ_OK;
    const size_t B = t->L.B, NA = (size_t)t->L.N * t->L.A;
    CU_TRY(cudaMalloc(&t->s_rewards, 4 * B));
    CU_TRY(cudaMalloc(&t->s_values, 4 * B));
    CU_TRY(cudaMalloc(&t->s_probs, 4 * B * NA));
    CU_TRY(cudaMalloc(&t->s_beta, 4 * B * NA));
    CU_TRY(cudaMalloc(&t->s_noises, 4 * B * NA));
    CU_TRY(cudaMalloc(&t->s_idx, 4 * B * (2 + t->L.N)));
    return MAZ_OK;
}

static int sync_and_check(maz_tree *t, int code_from_copy)
{
    CU_TRY(cudaStreamSynchronize(t->stream));
    if (code_from_copy) return set_err(MAZ_ERR_DEVICE, dev_err_msg(code_from_copy));
    return MAZ_OK;
}

int maz_tree_prepare(maz_tree *t, const float *rewards, const float *values, const float *probs, const float *beta, int K,
                     float eps, const float *noises)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!rewards || !values || !probs || !beta || (eps > 0 && !noises)) return set_err(MAZ_ERR_INVALID, "prepare: NULL input");
    DeviceGuard g(t->device);
    int rc = ensure_staging(t);
    if (rc) return rc;
    const size_t B = t->L.B, NA = (size_t)t->L.N * t->L.A;
    CU_TRY(cudaMemcpyAsync(t->s_rewards, rewards, 4 * B, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_values, values, 4 * B, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_probs, probs, 4 * B * NA, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_beta, beta, 4 * B * NA, cudaMemcpyHostToDevice, t->stream));
    if (noises) CU_TRY(cudaMemcpyAsync(t->s_noises, noises, 4 * B * NA, cudaMemcpyHostToDevice, t->stream));
    rc = maz_tree_prepare_dev(t, t->s_rewards, t->s_values, t->s_probs, t->s_beta, K, eps, t->s_noises);
    if (rc) return rc;
    return maz_tree_check(t);
}

int maz_tree_batch_selection(maz_tree *t, float c_base, float c_init, float discount, int *idx_x, int *idx_y, int *act)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!idx_x || !idx_y || !act) return set_err(MAZ_ERR_INVALID, "batch_selection: NULL output");
    DeviceGuard g(t->device);
    int rc = ensure_staging(t);
    if (rc) return rc;
    const size_t B = t->L.B;
    int *dx = t->s_idx, *dy = t->s_idx + B, *da = t->s_idx + 2 * B;
    rc = maz_tree_batch_selection_dev(t, c_base, c_init, discount, dx, dy, da);
    if (rc) return rc;
    int code = 0;
    CU_TRY(cudaMemcpyAsync(idx_x, dx, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaMemcpyAsync(idx_y, dy, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaMemcpyAsync(act, da, 4 * B * t->L.N, cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaMemcpyAsync(&code, t->d_err, sizeof(int), cudaMemcpyDeviceToHost, t->stream));
    return sync_and_check(t, code);
}

int maz_tree_batch_expansion_and_backup(maz_tree *t, int hidx, float discount, int K, const float *rewards,
                                        const float *values, const float *probs, const float *beta)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!rewards || !values || !probs || !beta) return set_err(MAZ_ERR_INVALID, "expansion: NULL input");
    DeviceGuard g(t->device);
    int rc = ensure_staging(t);
    if (rc) return rc;
    const size_t B = t->L.B, NA = (size_t)t->L.N * t->L.A;
    CU_TRY(cudaMemcpyAsync(t->s_rewards, rewards, 4 * B, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_values, values, 4 * B, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_probs, probs, 4 * B * NA, cudaMemcpyHostToDevice, t->stream));
    CU_TRY(cudaMemcpyAsync(t->s_beta, beta, 4 * B * NA, cudaMemcpyHostToDevice, t->stream));
    rc = maz_tree_batch_expansion_and_backup_dev(t, hidx, discount, K, t->s_rewards, t->s_values, t->s_probs, t->s_beta);
    if (rc) return rc;
    // like the reference (`except +` on this method, ctree.pxd:20) failures surface from this call
    return maz_tree_check(t);
}

// ---- readouts ----------------------------------------------------------------------------------------------
int maz_tree_readout_dev(maz_tree *t, float discount, float *values, int *mv, float *mp, int *nc, int *actions, int *visits,
                         float *pred_probs, float *beta, float *beta_hat, float *priors, float *imp_ratio,
                         float *pred_values, float *mcts_values, float *rewards, float *qvalues)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!t->prepared) return set_err(MAZ_ERR_INVALID, "readout before prepare");
    DeviceGuard g(t->device);
    ReadoutPtrs o{values, mv, mp, nc, actions, visits, pred_probs, beta, beta_hat, priors, imp_ratio,
                  pred_values, mcts_values, rewards, qvalues};
    k_readout<<<tree_grid(t), tree_block(t), 0, t->stream>>>(t->L, t->arena, discount, o);
    CU_TRY(cudaGetLastError());
    return MAZ_OK;
}

int maz_tree_readout(maz_tree *t, float discount, float *values, int *mv, float *mp, int *nc, int *actions, int *visits,
                     float *pred_probs, float *beta, float *beta_hat, float *priors, float *imp_ratio, float *pred_values,
                     float *mcts_values, float *rewards, float *qvalues)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    DeviceGuard g(t->device);
    const size_t B = t->L.B, NA = (size_t)t->L.N * t->L.A, K = t->L.K, N = t->L.N;
    // device mirror: values B | mv B*NA | mp B*NA | nc B | actions B*K*N | visits B*K | 9 x B*K floats
    const size_t words = B + 2 * B * NA + B + B * K * N + B * K + 9 * B * K;
    if (!t->s_readout) CU_TRY(cudaMalloc(&t->s_readout, 4 * words));
    int *w = reinterpret_cast<int *>(t->s_readout);
    size_t o = 0;
    auto take = [&](size_t n) { int *p = w + o; o += n; return p; };
    float *d_values = (float *)take(B);
    int *d_mv = take(B * NA);
    float *d_mp = (float *)take(B * NA);
    int *d_nc = take(B);
    int *d_act = take(B * K * N);
    int *d_vis = take(B * K);
    float *d_f[9];
    for (int i = 0; i < 9; ++i) d_f[i] = (float *)take(B * K);
    float *h_f[9] = {pred_probs, beta, beta_hat, priors, imp_ratio, pred_values, mcts_values, rewards, qvalues};
    int rc = maz_tree_readout_dev(t, discount, values ? d_values : nullptr, mv ? d_mv : nullptr, mp ? d_mp : nullptr,
                                  nc ? d_nc : nullptr, actions ? d_act : nullptr, visits ? d_vis : nullptr,
                                  h_f[0] ? d_f[0] : nullptr, h_f[1] ? d_f[1] : nullptr, h_f[2] ? d_f[2] : nullptr,
                                  h_f[3] ? d_f[3] : nullptr, h_f[4] ? d_f[4] : nullptr, h_f[5] ? d_f[5] : nullptr,
                                  h_f[6] ? d_f[6] : nullptr, h_f[7] ? d_f[7] : nullptr, h_f[8] ? d_f[8] : nullptr);
    if (rc) return rc;
    if (values) CU_TRY(cudaMemcpyAsync(values, d_values, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    if (mv) CU_TRY(cudaMemcpyAsync(mv, d_mv, 4 * B * NA, cudaMemcpyDeviceToHost, t->stream));
    if (mp) CU_TRY(cudaMemcpyAsync(mp, d_mp, 4 * B * NA, cudaMemcpyDeviceToHost, t->stream));
    if (nc) CU_TRY(cudaMemcpyAsync(nc, d_nc, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    if (actions) CU_TRY(cudaMemcpyAsync(actions, d_act, 4 * B * K * N, cudaMemcpyDeviceToHost, t->stream));
    if (visits) CU_TRY(cudaMemcpyAsync(visits, d_vis, 4 * B * K, cudaMemcpyDeviceToHost, t->stream));
    for (int i = 0; i < 9; ++i)
        if (h_f[i]) CU_TRY(cudaMemcpyAsync(h_f[i], d_f[i], 4 * B * K, cudaMemcpyDeviceToHost, t->stream));
    return maz_tree_check(t);
}

int maz_tree_get_roots_values(maz_tree *t, float *out)
{
    return maz_tree_readout(t, 0.0f, out, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            nullptr, nullptr, nullptr, nullptr, nullptr);
}
int maz_tree_get_roots_marginal_visit_count(maz_tree *t, int *out)
{
    return maz_tree_readout(t, 0.0f, nullptr, out, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            nullptr, nullptr, nullptr, nullptr, nullptr);
}
int maz_tree_get_roots_marginal_priors(maz_tree *t, float *out)
{
    return maz_tree_readout(t, 0.0f, nullptr, nullptr, out, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            nullptr, nullptr, nullptr, nullptr, nullptr);
}
int maz_tree_get_roots_num_children(maz_tree *t, int *out)
{
    return maz_tree_readout(t, 0.0f, nullptr, nullptr, nullptr, out, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            nullptr, nullptr, nullptr, nullptr, nullptr);
}

int maz_tree_stats(maz_tree *t, int *tot_nodes, int *last_len, long long *sum_len, long long *sum_expanded)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    if (!t->prepared) return set_err(MAZ_ERR_INVALID, "stats before prepare");
    DeviceGuard g(t->device);
    int rc = ensure_staging(t);
    if (rc) return rc;
    const size_t B = t->L.B;
    int *d_tot = t->s_idx, *d_len = t->s_idx + B;
    CU_TRY(cudaMemsetAsync(t->d_sums, 0, 2 * sizeof(unsigned long long), t->stream));
    k_stats<<<(unsigned)((B + 127) / 128), 128, 0, t->stream>>>(t->L, t->arena, d_tot, d_len, t->d_sums);
    CU_TRY(cudaGetLastError());
    unsigned long long sums[2] = {0, 0};
    if (tot_nodes) CU_TRY(cudaMemcpyAsync(tot_nodes, d_tot, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    if (last_len) CU_TRY(cudaMemcpyAsync(last_len, d_len, 4 * B, cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaMemcpyAsync(sums, t->d_sums, sizeof(sums), cudaMemcpyDeviceToHost, t->stream));
    CU_TRY(cudaStreamSynchronize(t->stream));
    if (sum_len) *sum_len = (long long)sums[0];
    if (sum_expanded) *sum_expanded = (long long)sums[1];
    return MAZ_OK;
}

int maz_tree_set_debug_clock(maz_tree *t, long long *p)
{
    if (!t) return set_err(MAZ_ERR_INVALID, "null handle");
    t->L.dbg_clock = p;
    return MAZ_OK;
}

size_t maz_tree_arena_bytes(const maz_tree *t) { return t ? t->arena_bytes : 0; }

}  // extern "C"
