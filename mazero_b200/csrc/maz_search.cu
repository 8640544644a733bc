// maz_search.cu -- the whole search behind the C ABI (include/maz_search.h): root preparation, tree construction, the
// simulation loop (persistent kernel or a CUDA graph built here with the runtime API) and the readouts.
// Replaces the body of SampledMCTS.batch_search (core/mcts/tree_search/mcts_sampled.py:51-200).
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/maz_search.h"
#include "../../include/maz_turn.h"
#define MAZ_HMMA_NO_KERNEL   // the one-step kernel of infer_hmma.cuh lives in maz_infer.cu
#include "search_persist.cuh"
#include "tree_host.h"

using namespace maz;

#define CU_TRY(expr)                                                                                          \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return set_last_error(MAZ_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));         \
    } while (0)
#define MAZ_TRY(expr)          \
    do {                       \
        int rc__ = (expr);     \
        if (rc__) return rc__; \
    } while (0)

namespace {

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DevGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

struct GraphKey {
    int cur;
    float inv_tau, c_base, c_init, discount, delta_lb, rho, lam;
    bool operator==(const GraphKey &o) const { return std::memcmp(this, &o, sizeof(GraphKey)) == 0; }
};
struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec;
    unsigned long long used;
};
constexpr size_t kMaxGraphs = 40;   // one per (agent turn, constants); least recently used is dropped

}  // namespace

struct maz_search {
    maz_search_config cfg{};
    maz_infer_desc tc{}, sm{};
    maz_mlp_desc mlp{};
    int Nt = 1, D = 0, rpt = 1, strategy = MAZ_SEARCH_GRAPH;
    bool use_small = false;         // graph strategy, SMAC: which one-step kernel
    cudaStream_t stream = nullptr, cap_stream = nullptr;
    maz_tree *tree = nullptr;
    bool own_pool = false;
    float *pool = nullptr;
    int *greedy = nullptr;          // (S+1, B, N)
    int *idx_x = nullptr, *idx_y = nullptr, *act = nullptr, *factor = nullptr;
    float *sim_r = nullptr, *sim_v = nullptr, *sim_p = nullptr, *sim_b = nullptr;
    float *root_p = nullptr, *root_b = nullptr, *root_n = nullptr;
    size_t bytes = 0;
    // record (parity replay)
    float *rec_r = nullptr, *rec_v = nullptr, *rec_p = nullptr, *rec_b = nullptr;
    int *rec_ix = nullptr, *rec_act = nullptr;
    long long *dbg_clock = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // timing of the simulation loop (maz_search_set_timing)
    bool timing = false, timed = false;
    std::vector<GraphEntry> graphs;
    unsigned long long tick = 0;
    // host-pointer entry point: one pinned block + device mirror per direction
    char *h_in = nullptr, *d_in = nullptr, *h_out = nullptr, *d_out = nullptr;
    size_t in_bytes = 0, out_bytes = 0;
};

static int dmalloc(maz_search *s, void **p, size_t bytes)
{
    CU_TRY(cudaMalloc(p, bytes));
    s->bytes += bytes;
    return MAZ_OK;
}

static int env_strategy()
{
    const char *e = getenv("MAZ_SEARCH_STRATEGY");
    if (!e) return MAZ_SEARCH_AUTO;
    if (!strcmp(e, "persistent")) return MAZ_SEARCH_PERSISTENT;
    if (!strcmp(e, "graph")) return MAZ_SEARCH_GRAPH;
    return MAZ_SEARCH_AUTO;
}
static int env_int(const char *name, int dflt)
{
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}

extern "C" {

int maz_search_create(maz_search **out, const maz_search_config *cfg)
{
    if (!out || !cfg) return set_last_error(MAZ_ERR_INVALID, "maz_search_create: NULL argument");
    *out = nullptr;
    if (cfg->B <= 0 || cfg->N <= 0 || cfg->A <= 0 || cfg->K <= 0 || cfg->S <= 0 || cfg->hidden <= 0)
        return set_last_error(MAZ_ERR_INVALID, "maz_search_create: dimensions must be positive");
    if (cfg->net_kind == MAZ_NET_SMAC && (!cfg->smac_tc || !cfg->smac_small || cfg->hidden != hmma::H))
        return set_last_error(MAZ_ERR_INVALID, "maz_search_create: MAZ_NET_SMAC needs both weight packings and hidden 128");
    if (cfg->net_kind == MAZ_NET_SMAC && cfg->A > hmma::KA_WIDE)
        return set_last_error(MAZ_ERR_UNSUPPORTED, "maz_search_create: the fused SMAC inference supports at most 128 actions per agent");
    if (cfg->net_kind == MAZ_NET_MLP && !cfg->mlp) return set_last_error(MAZ_ERR_INVALID, "maz_search_create: MAZ_NET_MLP needs the MLP descriptor");
    if (cfg->net_kind != MAZ_NET_SMAC && cfg->net_kind != MAZ_NET_MLP) return set_last_error(MAZ_ERR_INVALID, "maz_search_create: bad net_kind");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return set_last_error(MAZ_ERR_CUDA, "no CUDA device available (libmaz_b200 has no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return set_last_error(MAZ_ERR_INVALID, "maz_search_create: bad device index");
    DevGuard g(cfg->device);

    maz_search *s = new maz_search();
    s->cfg = *cfg;
    if (cfg->net_kind == MAZ_NET_SMAC) { s->tc = *cfg->smac_tc; s->sm = *cfg->smac_small; }
    else s->mlp = *cfg->mlp;
    s->cfg.smac_tc = s->cfg.smac_small = nullptr;
    s->cfg.mlp = nullptr;
    const int B = cfg->B, N = cfg->N, A = cfg->A, K = cfg->K, S = cfg->S;
    s->Nt = cfg->joint ? N : 1;
    s->D = N * cfg->hidden;
    auto fail = [&](int rc) { std::string m = maz_last_error(); maz_search_destroy(s); set_last_error(rc, m); return rc; };

    int rc = maz_tree_create_ex(&s->tree, B, s->Nt, A, K, S, 0.01f, 0u, 0.75f, 0.8f, cfg->device, 0u);
    if (rc) return fail(rc);
    s->bytes += maz_tree_arena_bytes(s->tree);

    // ---- strategy ------------------------------------------------------------------------------------------------
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
    int strat = cfg->strategy != MAZ_SEARCH_AUTO ? cfg->strategy : env_strategy();
    const int rpt_fit = hmma::TM / N;                               // whole roots per 32-row tile
    int rpt = rpt_fit < 8 ? rpt_fit : 8;                            // one warp per tree, 8 compute warps
    const int rpt_env = env_int("MAZ_SEARCH_RPT", 0);
    if (rpt_env > 0 && rpt_env < rpt) rpt = rpt_env;
    // the persistent kernel's shared memory: the inference map + the trees' hot state and the exchange arrays
    int optin = 227 * 1024;
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
    // (the wide instance, KA > 48, places the tree-step scratch that the PH..Q alias cannot hold elsewhere: search_persist.cuh)
    const bool wide = cfg->net_kind == MAZ_NET_SMAC && s->sm.KA > hmma::KA_NARROW;
    bool persist_ok = cfg->net_kind == MAZ_NET_SMAC && N <= hmma::TM && rpt >= 1 &&
                      (wide ? persist::persist_smem_bytes_wide(s->sm.vec_floats, rpt, s->Nt, A, K, S) + 256 <= (size_t)optin
                            : (size_t)rpt * tree_scratch_bytes(s->Nt, A, K, S) <= persist::TREE_SCRATCH_BYTES &&
                                  persist::persist_smem_bytes(s->sm.vec_floats, rpt, s->Nt, A, S) + 256 <= (size_t)optin);
    if (strat == MAZ_SEARCH_PERSISTENT && !persist_ok) {
        set_last_error(MAZ_ERR_UNSUPPORTED, "maz_search_create: the persistent kernel does not support this network / shape");
        return fail(MAZ_ERR_UNSUPPORTED);
    }
    {
        const char *k = getenv("MAZ_INFER_KERNEL");      // "tcgen05" pins the 128-row kernel's arithmetic: graph strategy
        if (strat == MAZ_SEARCH_AUTO && k && !strcmp(k, "tcgen05")) strat = MAZ_SEARCH_GRAPH;
    }
    if (strat == MAZ_SEARCH_AUTO) {
        // one CTA per SM in ONE wave: each CTA runs its roots' whole search; above that the CUDA-graph loop with the
        // 128-row tcgen05 tiles re-reads the weights 4x less often (measured cross-over: DESIGN.md)
        const int waves_max = env_int("MAZ_SEARCH_PERSIST_MAX_CTAS", sms);
        strat = (persist_ok && (B + rpt - 1) / rpt <= waves_max) ? MAZ_SEARCH_PERSISTENT : MAZ_SEARCH_GRAPH;
    }
    s->strategy = strat;
    s->rpt = rpt;
    if (cfg->net_kind == MAZ_NET_SMAC) {
        const char *k = getenv("MAZ_INFER_KERNEL");
        const int small_max = env_int("MAZ_INFER_SMALL_MAX_TILES", 222);
        s->use_small = k && !strcmp(k, "small") ? true : k && !strcmp(k, "tcgen05") ? false : (B + rpt_fit - 1) / rpt_fit <= small_max;
    }

    // ---- buffers -----------------------------------------------------------------------------------------------------
    const size_t NA = (size_t)s->Nt * A;
    if (cfg->pool) s->pool = cfg->pool;
    else {
        if ((rc = dmalloc(s, (void **)&s->pool, sizeof(float) * (size_t)(S + 1) * B * s->D))) return fail(rc);
        s->own_pool = true;
    }
    if ((rc = dmalloc(s, (void **)&s->greedy, sizeof(int) * (size_t)(S + 1) * B * N)) ||
        (rc = dmalloc(s, (void **)&s->idx_x, sizeof(int) * B)) || (rc = dmalloc(s, (void **)&s->idx_y, sizeof(int) * B)) ||
        (rc = dmalloc(s, (void **)&s->act, sizeof(int) * B * s->Nt)) || (rc = dmalloc(s, (void **)&s->factor, sizeof(int) * B * N)) ||
        (rc = dmalloc(s, (void **)&s->sim_r, sizeof(float) * B)) || (rc = dmalloc(s, (void **)&s->sim_v, sizeof(float) * B)) ||
        (rc = dmalloc(s, (void **)&s->sim_p, sizeof(float) * B * NA)) || (rc = dmalloc(s, (void **)&s->sim_b, sizeof(float) * B * NA)) ||
        (rc = dmalloc(s, (void **)&s->root_p, sizeof(float) * B * NA)) || (rc = dmalloc(s, (void **)&s->root_b, sizeof(float) * B * NA)) ||
        (rc = dmalloc(s, (void **)&s->root_n, sizeof(float) * B * NA)))
        return fail(rc);
    if (cudaMemset(s->greedy, 0, sizeof(int) * (size_t)(S + 1) * B * N) != cudaSuccess ||
        cudaMemset(s->factor, 0, sizeof(int) * B * N) != cudaSuccess) {
        set_last_error(MAZ_ERR_CUDA, "cudaMemset failed");
        return fail(MAZ_ERR_CUDA);
    }
    if (s->strategy == MAZ_SEARCH_PERSISTENT) {
        const void *kfn = wide ? (const void *)persist::k_search_persistent<false, true> : (const void *)persist::k_search_persistent<false, false>;
        const void *kprof = wide ? (const void *)persist::k_search_persistent<true, true> : (const void *)persist::k_search_persistent<true, false>;
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kfn);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kprof, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
        if (e != cudaSuccess) {
            set_last_error(MAZ_ERR_CUDA, std::string("cudaFuncSetAttribute(k_search_persistent): ") + cudaGetErrorString(e));
            return fail(MAZ_ERR_CUDA);
        }
        int nb = 0;
        const size_t dyn = wide ? persist::persist_smem_bytes_wide(s->sm.vec_floats, rpt, s->Nt, A, K, S)
                                : persist::persist_smem_bytes(s->sm.vec_floats, rpt, s->Nt, A, S);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, persist::PERSIST_THREADS, dyn);
        if (e != cudaSuccess || nb < 1) {
            set_last_error(MAZ_ERR_CUDA, "k_search_persistent does not fit on an SM: " + std::to_string(fa.numRegs) + " registers x " +
                                             std::to_string(persist::PERSIST_THREADS) + " threads, " + std::to_string(dyn) + " + " +
                                             std::to_string(fa.sharedSizeBytes) + " bytes of shared memory (opt-in limit " + std::to_string(optin) + ")");
            return fail(MAZ_ERR_CUDA);
        }
    } else {
        if (cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
            set_last_error(MAZ_ERR_CUDA, "cudaStreamCreate failed");
            return fail(MAZ_ERR_CUDA);
        }
        if (cfg->net_kind == MAZ_NET_SMAC && (rc = maz_infer_configure(s->sm.vec_floats, s->sm.KA))) return fail(rc);
    }
    *out = s;
    return MAZ_OK;
}

void maz_search_destroy(maz_search *s)
{
    if (!s) return;
    DevGuard g(s->cfg.device);
    for (auto &e : s->graphs) cudaGraphExecDestroy(e.exec);
    if (s->cap_stream) cudaStreamDestroy(s->cap_stream);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    maz_tree_destroy(s->tree);
    if (s->own_pool) cudaFree(s->pool);
    void *ptrs[] = {s->greedy, s->idx_x, s->idx_y, s->act, s->factor, s->sim_r, s->sim_v, s->sim_p, s->sim_b,
                    s->root_p, s->root_b, s->root_n, s->d_in, s->d_out};
    for (void *p : ptrs) cudaFree(p);
    if (s->h_in) cudaFreeHost(s->h_in);
    if (s->h_out) cudaFreeHost(s->h_out);
    delete s;
}

int maz_search_set_stream(maz_search *s, void *stream)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    s->stream = static_cast<cudaStream_t>(stream);
    return maz_tree_set_stream(s->tree, stream);
}
int maz_search_strategy(const maz_search *s) { return s ? s->strategy : 0; }
size_t maz_search_device_bytes(const maz_search *s) { return s ? s->bytes : 0; }
float *maz_search_pool(maz_search *s) { return s ? s->pool : nullptr; }
maz_tree *maz_search_tree(maz_search *s) { return s ? s->tree : nullptr; }
int maz_search_root_arrays(maz_search *s, const float **probs, const float **beta, const float **noises)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    if (probs) *probs = s->root_p;
    if (beta) *beta = s->root_b;
    if (noises) *noises = s->root_n;
    return MAZ_OK;
}
int maz_search_check(maz_search *s)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    return maz_tree_check(s->tree);
}
int maz_search_set_record(maz_search *s, float *rewards, float *values, float *probs, float *beta, int *idx_x, int *actions)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    if (rewards && (!values || !probs || !beta || !idx_x || !actions))
        return set_last_error(MAZ_ERR_INVALID, "maz_search_set_record: all six arrays or none");
    s->rec_r = rewards; s->rec_v = values; s->rec_p = probs; s->rec_b = beta; s->rec_ix = idx_x; s->rec_act = actions;
    return MAZ_OK;
}
int maz_search_set_debug_clock(maz_search *s, long long *p)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    s->dbg_clock = p;
    return MAZ_OK;
}

int maz_search_set_timing(maz_search *s, int on)
{
    if (!s) return set_last_error(MAZ_ERR_INVALID, "null handle");
    DevGuard g(s->cfg.device);
    if (on && !s->ev0) {
        CU_TRY(cudaEventCreate(&s->ev0));
        CU_TRY(cudaEventCreate(&s->ev1));
    }
    s->timing = on != 0;
    s->timed = false;
    return MAZ_OK;
}
int maz_search_loop_ms(maz_search *s, float *ms)
{
    if (!s || !ms) return set_last_error(MAZ_ERR_INVALID, "maz_search_loop_ms: NULL argument");
    if (!s->timed) return set_last_error(MAZ_ERR_INVALID, "maz_search_loop_ms: no timed search yet (maz_search_set_timing)");
    DevGuard g(s->cfg.device);
    CU_TRY(cudaEventSynchronize(s->ev1));
    CU_TRY(cudaEventElapsedTime(ms, s->ev0, s->ev1));
    return MAZ_OK;
}
int maz_search_roots_per_cta(const maz_search *s) { return s && s->strategy == MAZ_SEARCH_PERSISTENT ? s->rpt : 0; }

}  // extern "C"

// ---- one simulation's network forward (graph strategy / eager record loop) ------------------------------------------------
static int launch_inference(maz_search *s, const maz_search_call *c, int sim, const int *idx_x, const int *act, float *r, float *v,
                            float *p, float *b, cudaStream_t stream)
{
    const int B = s->cfg.B, N = s->cfg.N;
    const bool seq = !s->cfg.joint;
    float *next_hidden = s->pool + (size_t)(sim + 1) * B * s->D;
    int *greedy = seq ? s->greedy + (size_t)(sim + 1) * B * N : nullptr;
    if (s->cfg.net_kind == MAZ_NET_SMAC) {
        maz_infer_desc d = s->use_small ? s->sm : s->tc;
        d.B = B; d.Nt = s->Nt; d.cur = seq ? c->cur : -1; d.inv_tau = 1.0f / c->tau;
        d.pool = s->pool; d.idx_x = idx_x; d.actions = act; d.next_hidden = next_hidden;
        d.reward = r; d.value = v; d.probs = p; d.beta = b; d.greedy = greedy; d.logits_out = nullptr;
        d.dbg_clock = nullptr; d.roots_per_tile = 0;
        d.factor = seq ? s->factor : nullptr;
        d.greedy_pool = seq ? s->greedy : nullptr;
        return s->use_small ? maz_infer_recurrent_small(&d, stream) : maz_infer_recurrent(&d, stream);
    }
    maz_mlp_desc d = s->mlp;
    d.B = B; d.Nt = s->Nt; d.cur = seq ? c->cur : -1; d.inv_tau = 1.0f / c->tau;
    d.pool = s->pool; d.idx_x = idx_x; d.actions = act; d.next_hidden = next_hidden;
    d.reward = r; d.value = v; d.probs = p; d.beta = b; d.greedy = greedy; d.logits_out = nullptr;
    d.factor = seq ? s->factor : nullptr;
    d.greedy_pool = seq ? s->greedy : nullptr;
    return maz_mlp_recurrent(&d, stream);
}

// S simulations as 1 + 2 S launches on `stream` (captured into a graph, or eager with per-simulation record slices)
static int enqueue_loop(maz_search *s, const maz_search_call *c, cudaStream_t stream, bool record)
{
    const int B = s->cfg.B, S = s->cfg.S, K = s->cfg.K;
    const size_t NA = (size_t)s->Nt * s->cfg.A;
    maz_tree *t = s->tree;
    cudaStream_t keep = t->stream;
    t->stream = stream;
    auto slice = [&](int sim, int *&ix, int *&act, float *&r, float *&v, float *&p, float *&b) {
        const size_t o = record ? (size_t)sim : 0;
        ix = (record ? s->rec_ix : s->idx_x) + o * B;
        act = (record ? s->rec_act : s->act) + o * B * s->Nt;
        r = (record ? s->rec_r : s->sim_r) + o * B;
        v = (record ? s->rec_v : s->sim_v) + o * B;
        p = (record ? s->rec_p : s->sim_p) + o * B * NA;
        b = (record ? s->rec_b : s->sim_b) + o * B * NA;
    };
    int *ix, *act, *ixn, *actn;
    float *r, *v, *p, *b, *rn, *vn, *pn, *bn;
    slice(0, ix, act, r, v, p, b);
    int rc = maz_tree_batch_selection_dev(t, c->pb_c_base, c->pb_c_init, c->discount, ix, s->idx_y, act);
    for (int sim = 0; sim < S && !rc; ++sim) {
        rc = launch_inference(s, c, sim, ix, act, r, v, p, b, stream);
        if (rc) break;
        if (sim + 1 < S) {
            slice(sim + 1, ixn, actn, rn, vn, pn, bn);
            rc = maz_tree_expansion_backup_selection_dev(t, sim + 1, c->discount, K, r, v, p, b, c->pb_c_base, c->pb_c_init, ixn,
                                                         s->idx_y, actn);
            ix = ixn; act = actn; r = rn; v = vn; p = pn; b = bn;
        } else {
            rc = maz_tree_batch_expansion_and_backup_dev(t, sim + 1, c->discount, K, r, v, p, b);
        }
    }
    t->stream = keep;
    return rc;
}

static int graph_for(maz_search *s, const maz_search_call *c, cudaGraphExec_t *out)
{
    GraphKey key;
    std::memset(&key, 0, sizeof(key));
    key.cur = s->cfg.joint ? -1 : c->cur;
    key.inv_tau = 1.0f / c->tau; key.c_base = c->pb_c_base; key.c_init = c->pb_c_init; key.discount = c->discount;
    key.delta_lb = c->delta_lb; key.rho = c->rho; key.lam = c->lam;
    for (auto &e : s->graphs)
        if (e.key == key) {
            e.used = ++s->tick;
            *out = e.exec;
            return MAZ_OK;
        }
    // kernel parameters (tree layout with delta_lb / rho, discount, tau, agent index) are frozen into the graph nodes: one
    // graph per distinct set, least recently used dropped
    cudaGraph_t graph = nullptr;
    CU_TRY(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue_loop(s, c, s->cap_stream, false);
    cudaError_t e = cudaStreamEndCapture(s->cap_stream, &graph);
    if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    if (e != cudaSuccess) return set_last_error(MAZ_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return set_last_error(MAZ_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
    if (s->graphs.size() >= kMaxGraphs) {
        size_t lru = 0;
        for (size_t i = 1; i < s->graphs.size(); ++i)
            if (s->graphs[i].used < s->graphs[lru].used) lru = i;
        cudaGraphExecDestroy(s->graphs[lru].exec);
        s->graphs.erase(s->graphs.begin() + lru);
    }
    s->graphs.push_back(GraphEntry{key, exec, ++s->tick});
    *out = exec;
    return MAZ_OK;
}

static int launch_persistent(maz_search *s, const maz_search_call *c, bool record)
{
    const int B = s->cfg.B;
    const bool seq = !s->cfg.joint;
    maz_tree *t = s->tree;
    persist::SearchParams P;
    std::memset(&P, 0, sizeof(P));
    P.d = s->sm;
    maz_infer_desc &d = P.d;
    d.B = B; d.Nt = s->Nt; d.cur = seq ? c->cur : -1; d.inv_tau = 1.0f / c->tau;
    d.pool = s->pool; d.next_hidden = s->pool + (size_t)B * s->D;
    d.idx_x = nullptr; d.actions = nullptr;              // (the exchange arrays live in the kernel's shared memory)
    d.reward = d.value = d.probs = d.beta = nullptr;
    d.greedy = nullptr; d.logits_out = nullptr; d.dbg_clock = nullptr;
    d.roots_per_tile = s->rpt;
    d.factor = seq ? s->factor : nullptr;
    d.greedy_pool = seq ? s->greedy : nullptr;
    P.L = t->L;
    P.arena = t->arena;
    P.lam_pow = t->d_lam_pow; P.logterm = t->d_logterm; P.sqrtn = t->d_sqrtn; P.table_len = t->table_len;
    P.discount = c->discount; P.K = s->cfg.K; P.S = s->cfg.S;
    P.g_err = t->d_err;
    P.idx_y = s->idx_y;
    P.greedy_w = seq ? s->greedy : nullptr;
    if (record) { P.rec_r = s->rec_r; P.rec_v = s->rec_v; P.rec_p = s->rec_p; P.rec_b = s->rec_b; P.rec_ix = s->rec_ix; P.rec_act = s->rec_act; }
    P.tree_clock = s->dbg_clock;
    const unsigned grid = (unsigned)((B + s->rpt - 1) / s->rpt);
    const bool wide = d.KA > hmma::KA_NARROW;
    const size_t dyn = wide ? persist::persist_smem_bytes_wide(s->sm.vec_floats, s->rpt, s->Nt, s->cfg.A, s->cfg.K, s->cfg.S)
                            : persist::persist_smem_bytes(s->sm.vec_floats, s->rpt, s->Nt, s->cfg.A, s->cfg.S);
    if (P.tree_clock != nullptr) {
        if (wide) persist::k_search_persistent<true, true><<<grid, persist::PERSIST_THREADS, dyn, s->stream>>>(P);
        else persist::k_search_persistent<true, false><<<grid, persist::PERSIST_THREADS, dyn, s->stream>>>(P);
    } else {
        if (wide) persist::k_search_persistent<false, true><<<grid, persist::PERSIST_THREADS, dyn, s->stream>>>(P);
        else persist::k_search_persistent<false, false><<<grid, persist::PERSIST_THREADS, dyn, s->stream>>>(P);
    }
    CU_TRY(cudaGetLastError());
    return MAZ_OK;
}

extern "C" int maz_search_run_dev(maz_search *s, const maz_search_call *c)
{
    if (!s || !c) return set_last_error(MAZ_ERR_INVALID, "maz_search_run_dev: NULL argument");
    const int B = s->cfg.B, N = s->cfg.N, A = s->cfg.A, K = s->cfg.K;
    const bool seq = !s->cfg.joint;
    if (seq ? (c->cur < 0 || c->cur >= N) : (c->cur >= 0))
        return set_last_error(MAZ_ERR_INVALID, "maz_search_run_dev: current agent index does not match the handle's mode");
    if (!c->rewards || !c->values || !c->logits || !c->noise) return set_last_error(MAZ_ERR_INVALID, "maz_search_run_dev: NULL input");
    if (!(c->tau > 0.f)) return set_last_error(MAZ_ERR_INVALID, "maz_search_run_dev: sampled_tau must be positive");
    DevGuard g(s->cfg.device);
    cudaStream_t st = s->stream;
    if (c->root_hidden && c->root_hidden != s->pool)
        CU_TRY(cudaMemcpyAsync(s->pool, c->root_hidden, sizeof(float) * (size_t)B * s->D, cudaMemcpyDeviceToDevice, st));
    // root preparation (mcts_sampled.py:57-106) + greedy actions of the roots (pool slot 0)
    MAZ_TRY(maz_root_prepare_dev(c->logits, c->legal, c->noise, B, N, A, seq ? c->cur : -1, c->noise_eps, 1.0f / c->tau, s->root_p,
                                 s->root_b, s->root_n, s->greedy, st));
    if (seq && c->cur > 0) {
        if (c->factor) {
            if (c->factor != s->factor) CU_TRY(cudaMemcpyAsync(s->factor, c->factor, sizeof(int) * (size_t)B * N, cudaMemcpyDeviceToDevice, st));
        } else {
            CU_TRY(cudaMemsetAsync(s->factor, 0, sizeof(int) * (size_t)B * N, st));      // mcts_sampled.py:116-120
        }
    }
    // Tree_batch(...) + prepare (mcts_sampled.py:89,106): the arena is re-armed, not re-allocated
    MAZ_TRY(maz_tree_set_stream(s->tree, st));
    MAZ_TRY(maz_tree_reset(s->tree, c->seed, c->delta_lb, c->rho, c->lam, c->root_index_offset));
    MAZ_TRY(maz_tree_set_puct(s->tree, c->pb_c_base, c->pb_c_init));
    MAZ_TRY(maz_tree_prepare_dev(s->tree, c->rewards, c->values, s->root_p, s->root_b, K, c->noise_eps, s->root_n));
    const bool record = s->rec_r != nullptr;
    if (s->timing) CU_TRY(cudaEventRecord(s->ev0, st));
    if (s->strategy == MAZ_SEARCH_PERSISTENT) {
        MAZ_TRY(launch_persistent(s, c, record));
    } else if (record) {
        MAZ_TRY(enqueue_loop(s, c, st, true));
    } else {
        cudaGraphExec_t exec = nullptr;
        MAZ_TRY(graph_for(s, c, &exec));
        CU_TRY(cudaGraphLaunch(exec, st));
    }
    if (s->timing) {
        CU_TRY(cudaEventRecord(s->ev1, st));
        s->timed = true;
    }
    const maz_search_readout &o = c->out;
    return maz_tree_readout_dev(s->tree, c->discount, o.values, o.marginal_visit_count, o.marginal_priors, o.num_children, o.actions,
                                o.visit_count, o.pred_probs, o.beta, o.beta_hat, o.priors, o.imp_ratio, o.pred_values, o.mcts_values,
                                o.rewards, o.qvalues);
}

// ---- host pointers: one pinned block in, one out ---------------------------------------------------------------------------
extern "C" int maz_search_run(maz_search *s, const maz_search_call *c)
{
    if (!s || !c) return set_last_error(MAZ_ERR_INVALID, "maz_search_run: NULL argument");
    if (!c->root_hidden || !c->rewards || !c->values || !c->logits || !c->noise)
        return set_last_error(MAZ_ERR_INVALID, "maz_search_run: NULL input");
    DevGuard g(s->cfg.device);
    const size_t B = s->cfg.B, N = s->cfg.N, A = s->cfg.A, K = s->cfg.K, Nt = s->Nt, D = s->D;
    const size_t n_hidden = B * D, n_b = B, n_bna = B * N * A, n_noise = B * Nt * A, n_fac = B * N;
    const size_t in_words = n_hidden + 2 * n_b + 2 * n_bna + n_noise + n_fac;
    const size_t n_mv = B * Nt * A, n_act = B * K * Nt, n_k = B * K;
    const size_t out_words = n_b + 2 * n_mv + n_b + n_act + n_k + 9 * n_k;
    if (!s->h_in) {
        CU_TRY(cudaMallocHost((void **)&s->h_in, 4 * in_words));
        CU_TRY(cudaMallocHost((void **)&s->h_out, 4 * out_words));
        MAZ_TRY(dmalloc(s, (void **)&s->d_in, 4 * in_words));
        MAZ_TRY(dmalloc(s, (void **)&s->d_out, 4 * out_words));
        s->in_bytes = 4 * in_words;
        s->out_bytes = 4 * out_words;
    }
    size_t o = 0;
    auto put = [&](const void *src, size_t words) {
        const size_t at = o;
        if (src) std::memcpy(s->h_in + 4 * at, src, 4 * words);
        o += words;
        return at;
    };
    const size_t o_hid = put(c->root_hidden, n_hidden), o_r = put(c->rewards, n_b), o_v = put(c->values, n_b),
                 o_log = put(c->logits, n_bna), o_leg = put(c->legal, n_bna), o_noi = put(c->noise, n_noise), o_fac = put(c->factor, n_fac);
    CU_TRY(cudaMemcpyAsync(s->d_in, s->h_in, 4 * in_words, cudaMemcpyHostToDevice, s->stream));
    maz_search_call dc = *c;
    auto din = [&](size_t at) { return s->d_in + 4 * at; };
    dc.root_hidden = (const float *)din(o_hid);
    dc.rewards = (const float *)din(o_r);
    dc.values = (const float *)din(o_v);
    dc.logits = (const float *)din(o_log);
    dc.legal = c->legal ? (const float *)din(o_leg) : nullptr;
    dc.noise = (const float *)din(o_noi);
    dc.factor = c->factor ? (const int *)din(o_fac) : nullptr;
    size_t q = 0;
    auto take = [&](size_t words) { char *p = s->d_out + 4 * q; q += words; return p; };
    maz_search_readout &r = dc.out;
    r.values = (float *)take(n_b);
    r.marginal_visit_count = (int *)take(n_mv);
    r.marginal_priors = (float *)take(n_mv);
    r.num_children = (int *)take(n_b);
    r.actions = (int *)take(n_act);
    r.visit_count = (int *)take(n_k);
    float **f9[9] = {&r.pred_probs, &r.beta, &r.beta_hat, &r.priors, &r.imp_ratio, &r.pred_values, &r.mcts_values, &r.rewards, &r.qvalues};
    for (auto pf : f9) *pf = (float *)take(n_k);
    MAZ_TRY(maz_search_run_dev(s, &dc));
    CU_TRY(cudaMemcpyAsync(s->h_out, s->d_out, 4 * out_words, cudaMemcpyDeviceToHost, s->stream));
    MAZ_TRY(maz_search_check(s));
    // scatter to the caller's arrays (any may be NULL)
    const maz_search_readout &u = c->out;
    q = 0;
    auto give = [&](void *dst, size_t words) {
        if (dst) std::memcpy(dst, s->h_out + 4 * q, 4 * words);
        q += words;
    };
    give(u.values, n_b); give(u.marginal_visit_count, n_mv); give(u.marginal_priors, n_mv); give(u.num_children, n_b);
    give(u.actions, n_act); give(u.visit_count, n_k);
    float *uf[9] = {u.pred_probs, u.beta, u.beta_hat, u.priors, u.imp_ratio, u.pred_values, u.mcts_values, u.rewards, u.qvalues};
    for (float *p : uf) give(p, n_k);
    return MAZ_OK;
}
