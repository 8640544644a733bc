// search_persist.cuh -- ONE kernel per search: a CTA owns a group of roots for all S simulations (sm_100a).
//
// Replaces the per-simulation loop of SampledMCTS.batch_search (core/mcts/tree_search/mcts_sampled.py:114-172):
//     selection -> gather parent hidden -> recurrent_inference (+ prediction) -> softmax / beta -> expansion + backup
// The two-kernel loop (fused inference + tree step, 2 launches per simulation inside a CUDA graph) ends every simulation with
// the slowest of ALL trees and pays two kernel boundaries; here the trees of a CTA only wait for each other:
//   * the CTA's 8 compute warps run the fused recurrent_inference of its tile on the tensor cores (the stages of
//     infer_hmma.cuh, unchanged arithmetic), then each of the first `rpt` warps steps ONE tree (expansion, backup, the next
//     selection: tree_step.cuh, the same bit-exact code as the stand-alone tree kernels) and gathers that root's parent hidden
//     state + joint action into the activation tiles of the next inference;
//   * no grid-wide barrier, no host, no launch between simulations: CTAs drift apart freely;
//   * everything the tree step exchanges with the network -- selection results in, reward / value / probs / beta out -- and the
//     tree's header, path, q-delta entries and expansion tables live in SHARED memory for the whole search (each of these was an
//     L2 round trip on the per-simulation critical path); node records, the value log and the generator state stay in the HBM
//     arena (L2-resident);
//   * the producer warp keeps streaming the weight chunks through the shared-memory ring across simulations, so the first
//     chunks of simulation s+1 arrive during the tree step of simulation s;
//   * the expansion scratch of the tree warps aliases activation tiles that are idle during the tree step.
// Trees are independent (cnode.cpp:571-576), so the grouping changes nothing in the results: every readout is bit-identical
// to the two-kernel loop (tests/test_search_native_gpu.py).
#pragma once
#include "infer_hmma.cuh"
#include "tree_step.cuh"

namespace maz {
namespace persist {

using namespace hmma;

struct SearchParams {
    Desc d;                    // network parameters + buffers.  d.pool: hidden-state pool (S+1, B, N*H); d.next_hidden: pool slot 1
    TreeLayout L;              // tree arena layout (L.N = agents in the tree = d.Nt)
    char *arena;
    const float *lam_pow, *logterm;
    const double *sqrtn;
    int table_len;
    float discount;
    int K, S;
    int *g_err;
    int *idx_y;                // (B,) the reference's second selection output (= arange)
    int *greedy_w;             // (S+1, B, N) greedy actions of every expanded node (sequential-agent mode), or NULL
    // parity replay (NULL = off): simulation s stores what the reference's loop passes between its steps
    float *rec_r, *rec_v, *rec_p, *rec_b;     // (S,B), (S,B), (S,B,Nt,A), (S,B,Nt,A)
    int *rec_ix, *rec_act;                    // (S,B), (S,B,Nt)
    long long *tree_clock;     // profiling (NULL): [2 s + {0,1}] = CTA 0's inference / tree-step cycles of simulation s; then per CTA c at
                               // [2 S + 4 c + ...]: total SM cycles, total nanoseconds (%globaltimer), sum of inference cycles, sum of tree
                               // cycles; then 64 stage timestamps of CTA 0's middle simulation; then per tree 4 counters
};

__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// tree-step scratch: the policy-hidden tile and the q|k|v region are idle during the tree step (the X / T / HH / one-hot tiles
// are not: the tree warps write the next simulation's HH / one-hot rows there)
constexpr uint32_t TREE_SCRATCH_OFF = OFF_PH;
constexpr uint32_t TREE_SCRATCH_BYTES = OFF_STAT - OFF_PH;
// The wide instance (W, 48 < KA <= 128) has larger tree-step scratch (it grows with N*A and S): 2c_vs_64zg (N = 2, A = 70, 8 trees per
// CTA) needs 8 x 4608 bytes at S = 50 and 8 x 6112 at S = 100, more than the alias above holds.  Its trees beyond that take slots in
// the X + T tiles, idle during the tree step too (the inference's last reads of them precede the barrier that ends it; the next
// inference writes them after the barrier that ends the tree step), and then behind the extra map below.
constexpr uint32_t TREE_SCRATCH_XT_BYTES = OFF_HH - OFF_X;
__host__ __device__ inline size_t tree_scratch_tail_bytes(int rpt, size_t ts)
{
    const int n = rpt - (int)(TREE_SCRATCH_BYTES / ts) - (int)(TREE_SCRATCH_XT_BYTES / ts);
    return n > 0 ? (size_t)n * ts : 0;
}

// ---- the CTA's extra shared memory, after the inference kernel's map --------------------------------------------------------
struct ExtraMap {
    uint32_t hot_stride;       // bytes per tree: header | qd | path | expslot | depth
    uint32_t o_qd, o_path, o_exp, o_dep;
    uint32_t o_xr, o_xv, o_xp, o_xb, o_xi, o_xa;    // exchange arrays (offsets from the extra base): reward, value, probs, beta, idx_x, actions
    uint32_t bytes;
};
__host__ __device__ inline uint32_t al16(uint32_t x) { return (x + 15u) & ~15u; }
__host__ __device__ inline ExtraMap extra_map(int rpt, int Nt, int A, int S)
{
    ExtraMap m;
    const uint32_t lv = (uint32_t)S + 2;
    m.o_qd = 64;
    m.o_path = m.o_qd + al16(4 * lv);
    m.o_exp = m.o_path + al16(2 * lv);
    m.o_dep = m.o_exp + al16(2 * lv);
    m.hot_stride = m.o_dep + al16(2 * lv);
    uint32_t o = m.hot_stride * (uint32_t)rpt;
    const uint32_t NA = (uint32_t)Nt * A;
    m.o_xr = o; o += al16(4 * rpt);
    m.o_xv = o; o += al16(4 * rpt);
    m.o_xp = o; o += al16(4 * rpt * NA);
    m.o_xb = o; o += al16(4 * rpt * NA);
    m.o_xi = o; o += al16(4 * rpt);
    m.o_xa = o; o += al16(4 * rpt * Nt);
    m.bytes = o;
    return m;
}
__host__ __device__ inline size_t persist_smem_bytes(int vec_floats, int rpt, int Nt, int A, int S)
{
    return ((smem_bytes(vec_floats) + 15) & ~(size_t)15) + extra_map(rpt, Nt, A, S).bytes;
}
// ... of the wide instance: + the tree-step scratch slots behind the extra map
__host__ __device__ inline size_t persist_smem_bytes_wide(int vec_floats, int rpt, int Nt, int A, int K, int S)
{
    return persist_smem_bytes(vec_floats, rpt, Nt, A, S) + tree_scratch_tail_bytes(rpt, tree_scratch_bytes(Nt, A, K, S));
}

// The parent hidden state and the joint action of ONE root -> its rows of the HH / one-hot tiles (what stage_gather does for the
// whole tile in the one-step kernel), by the warp that has just selected that root's leaf.  mcts_sampled.py:116-147.
// W (wide variant): the one-hot tile region holds the row's action instead of its one-hot row.
template <bool W>
__device__ __forceinline__ void gather_root(const Desc &d, int root, int rl, int ix, const int *tree_act, int lane)
{
    HSM_DECL;
    const int N = d.N;
#pragma unroll 1
    for (int j0 = 0; j0 < N; j0 += 4) {
        float4 v[4];
        int act[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            if (j < N) {
                v[u] = __ldcg(reinterpret_cast<const float4 *>(d.pool + ((size_t)ix * d.B + root) * (size_t)(N * H) + (size_t)j * H) + lane);
                if (d.greedy_pool == nullptr || d.cur < 0) act[u] = tree_act[j];
                else if (j == d.cur) act[u] = tree_act[0];
                else if (j < d.cur) act[u] = d.factor ? __ldcg(d.factor + (size_t)root * N + j) : 0;
                else act[u] = __ldcg(d.greedy_pool + ((size_t)ix * d.B + root) * N + j);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            if (j < N) {
                const int r = rl * N + j;
                *reinterpret_cast<uint2 *>(hsm + OFF_HH + (size_t)r * LDA + lane * 8) = make_uint2(pack2(v[u].x, v[u].y), pack2(v[u].z, v[u].w));
                if (W) {
                    if (lane == 0) *reinterpret_cast<int *>(hsm + OFF_ONE + (size_t)r * 4) = act[u];
                } else if (2 * lane < d.KA)
                    *reinterpret_cast<uint32_t *>(hsm + OFF_ONE + (size_t)r * LDO + lane * 4) =
                        pack2((2 * lane == act[u]) ? 1.f : 0.f, (2 * lane + 1 == act[u]) ? 1.f : 0.f);
            }
        }
    }
}

// 8 compute / tree warps (two warpgroups) + a third warpgroup whose first warp streams the weights.  Registers are allocated to
// warps in groups of four, so a 9-warp CTA is charged for 12: every thread would be capped at 168 registers, and the tree step
// inlined next to the inference stages spills at that.  The warpgroups re-balance at kernel start (setmaxnreg): the producer
// group keeps 40 registers per thread, the two compute groups take 232.
constexpr int PERSIST_THREADS = NCONS + 128;
constexpr int REGS_COMPUTE = 232, REGS_PRODUCER = 40;

// kProf: the instance with the in-kernel cycle counters (P.tree_clock); the production instance carries none of their registers.
// W: the wide variant of the inference stages (48 < KA <= 128, infer_hmma.cuh).
template <bool kProf, bool W>
__global__ void __launch_bounds__(PERSIST_THREADS, 1) k_search_persistent(const __grid_constant__ SearchParams P)
{
    HSM_DECL;
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_vec;
    const Desc &d = P.d;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], NCONS / 32); }
        mbar_init(&bar_vec, 1);
        mbar_fence_init();
    }
    setup_rows(d);
    // the HH / one-hot tiles: rows of roots this CTA does not have stay zero (wide variant: action -1) for the whole search
    for (uint32_t o = tid * 16u; o < TM * (uint32_t)LDA + TM * (uint32_t)LDO; o += PERSIST_THREADS * 16u) {
        const uint32_t f = (W && o >= TM * (uint32_t)LDA) ? 0xffffffffu : 0u;
        *reinterpret_cast<uint4 *>(hsm + OFF_HH + o) = make_uint4(f, f, f, f);
    }
    __syncthreads();
    if (warp >= NCONS / 32) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_PRODUCER));
        if (warp == NCONS / 32 && lane == 0) produce_weights(d, bar_full, bar_empty, &bar_vec, P.S);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_COMPUTE));
    // ==================================== compute warps =========================================================
    Ring ring{bar_full, bar_empty, 0};
    // (profiling instance: phase timestamps of tree 0's step, MAZ_TS, go after the per-tree counters)
    TreeLayout Lprof = P.L;
    if (kProf && P.tree_clock != nullptr)
        Lprof.dbg_clock = P.tree_clock + 2 * P.S + 4 * (long long)gridDim.x + 64 + 4 * (long long)P.d.B;
    const TreeLayout &L = kProf ? Lprof : P.L;
    const int rpt = tile_rpt(d);
    const int root0 = blockIdx.x * rpt;
    const int tree = root0 + warp;
    const bool has_tree = warp < rpt && tree < d.B;
    char *tb = P.arena + (size_t)(has_tree ? tree : 0) * L.slab_bytes;
    const size_t B = (size_t)d.B, NA = (size_t)L.N * L.A;
    const size_t ts = tree_scratch_bytes(L.N, L.A, L.K, L.S);
    char *const base = reinterpret_cast<char *>(hsm);
    // (wide instance: slots in the PH..Q alias, then in the X + T tiles, then behind the extra map)
    const int n0 = W ? (int)(TREE_SCRATCH_BYTES / ts) : rpt, n1 = W ? n0 + (int)(TREE_SCRATCH_XT_BYTES / ts) : rpt;
    const size_t tail0 = ((smem_bytes(d.vec_floats) + 15) & ~(size_t)15) + (W ? extra_map(rpt, L.N, L.A, L.S).bytes : 0);
    const StepScratch scr = carve_step_scratch(!W || warp < n0 ? base + TREE_SCRATCH_OFF + (size_t)warp * ts
                                               : warp < n1     ? base + OFF_X + (size_t)(warp - n0) * ts
                                                               : base + tail0 + (size_t)(warp - n1) * ts,
                                               L.N, L.A, L.K, L.S);
    // ---- shared-memory residents: this warp's tree (header + hot arrays) and the CTA's exchange arrays ------------------------
    const ExtraMap xm = extra_map(rpt, L.N, L.A, L.S);
    char *xbase = reinterpret_cast<char *>(hsm) + ((smem_bytes(d.vec_floats) + 15) & ~(size_t)15);
    char *hb = xbase + (size_t)(warp < rpt ? warp : 0) * xm.hot_stride;
    TreeHdr *hdr = reinterpret_cast<TreeHdr *>(hb);
    const TreeHot hot{reinterpret_cast<uint16_t *>(hb + xm.o_path), reinterpret_cast<float *>(hb + xm.o_qd),
                      reinterpret_cast<uint16_t *>(hb + xm.o_exp), reinterpret_cast<uint16_t *>(hb + xm.o_dep)};
    float *x_r = reinterpret_cast<float *>(xbase + xm.o_xr), *x_v = reinterpret_cast<float *>(xbase + xm.o_xv);
    float *x_p = reinterpret_cast<float *>(xbase + xm.o_xp), *x_b = reinterpret_cast<float *>(xbase + xm.o_xb);
    int *x_i = reinterpret_cast<int *>(xbase + xm.o_xi), *x_a = reinterpret_cast<int *>(xbase + xm.o_xa);
    if (has_tree) {
        const TreeHot g = hot_from_slab(L, tb);                  // as k_prepare left it
        if (lane < 16) reinterpret_cast<int *>(hdr)[lane] = reinterpret_cast<const int *>(f_hdr(tb))[lane];
        for (int i = lane; i < L.S + 2; i += 32) {
            hot.path[i] = g.path[i]; hot.qd[i] = g.qd[i]; hot.expslot[i] = g.expslot[i]; hot.depth[i] = g.depth[i];
        }
    }
    __syncwarp();

    long long *clk = (kProf && P.tree_clock != nullptr && blockIdx.x == 0 && tid == 0) ? P.tree_clock : nullptr;
    long long *cta_clk = (kProf && P.tree_clock != nullptr && tid == 0) ? P.tree_clock + 2 * P.S + 4 * blockIdx.x : nullptr;
    const long long k0 = cta_clk ? clock64() : 0;
    const unsigned long long g0 = cta_clk ? globaltimer_ns() : 0;
    long long sum_inf = 0, sum_tree = 0;
    // per tree (after the 64 stage timestamps): cycles in expansion + backup, cycles in selection (+ gather), sum of path lengths, max
    long long *tree_clk = (kProf && P.tree_clock != nullptr && has_tree && lane == 0)
                              ? P.tree_clock + 2 * P.S + 4 * (long long)gridDim.x + 64 + 4 * (long long)tree : nullptr;
    long long tc_eb = 0, tc_sel = 0, tc_len = 0, tc_max = 0;

    mbar_wait(&bar_vec, 0);          // parameters resident
    setup_head_copies(d);
    cta_sync();

    // the network's view of the exchange arrays (shared memory, indexed by root - root0)
    SimIo io;
    io.idx_x = x_i; io.actions = x_a; io.reward = x_r; io.value = x_v; io.probs = x_p; io.beta = x_b; io.root0 = root0;
    io.logits_out = nullptr;

    // Iteration s: [tree warps] expansion + backup of simulation s-1 (its network outputs are in the exchange arrays), then the
    // selection of simulation s and the gather of its parent hidden state;  [all compute warps] recurrent_inference of
    // simulation s.  One call site per tree function: a single inlined copy of each.
#pragma unroll 1
    for (int s = 0; s <= P.S; ++s) {
        const long long t1 = cta_clk ? clock64() : 0;
        if (has_tree) {
            const long long q0 = tree_clk ? clock64() : 0;
            if (s > 0) {
                if (P.rec_r != nullptr) {       // parity replay: what batch_expansion_and_backup(s, ...) receives
                    const size_t o = (size_t)(s - 1) * B + tree;
                    if (lane == 0) { P.rec_r[o] = x_r[warp]; P.rec_v[o] = x_v[warp]; }
                    for (int t = lane; t < (int)NA; t += 32) {
                        P.rec_p[o * NA + t] = x_p[(size_t)warp * NA + t];
                        P.rec_b[o * NA + t] = x_b[(size_t)warp * NA + t];
                    }
                }
                expand_backup_device<false>(L, tb, hdr, hot, P.lam_pow, s, P.discount, P.K, x_r + warp, x_v + warp, x_p + (size_t)warp * NA,
                                            x_b + (size_t)warp * NA, scr, lane, P.g_err, kProf ? tree : -1);
            }
            __syncwarp();
            if (kProf && s > 0 && L.dbg_clock != nullptr && tree == 0 && lane == 0) {     // accumulate tree 0's phase times (slots 16..31)
                const int order[11] = {0, 1, 2, 11, 12, 13, 14, 15, 3, 4, 5};
                for (int i = 1; i < 11; ++i) L.dbg_clock[16 + i] += L.dbg_clock[order[i]] - L.dbg_clock[order[i - 1]];
            }
            const long long q1 = tree_clk ? clock64() : 0;
            if (s < P.S) {
                // (idx / act are indexed by tree - root0 = warp: the selection writes x_i[warp], x_a[warp * Nt ...])
                select_next_device(L, tb, hdr, hot, P.logterm, P.sqrtn, P.table_len, P.discount, warp, lane, &scr, x_i, nullptr, x_a,
                                   P.g_err);
                __syncwarp();
                const int ix = x_i[warp];
                if (P.rec_ix != nullptr) {      // parity replay: what batch_selection returns
                    const size_t o = (size_t)s * B + tree;
                    if (lane == 0) P.rec_ix[o] = ix;
                    for (int j = lane; j < L.N; j += 32) P.rec_act[o * L.N + j] = x_a[warp * L.N + j];
                }
                gather_root<W>(d, tree, warp, ix, x_a + warp * L.N, lane);
            }
            if (tree_clk) {
                const long long q2 = clock64();
                const int pl = hdr->path_len;
                tc_eb += q1 - q0; tc_sel += q2 - q1; tc_len += pl; tc_max = pl > tc_max ? pl : tc_max;
            }
        }
        cta_sync();                  // the HH / one-hot rows and idx of simulation s are in place; the tree scratch is free
        const long long t2 = cta_clk ? clock64() : 0;
        if (cta_clk) {
            sum_tree += t2 - t1;
            if (clk && s > 0) clk[2 * (s - 1) + 1] = t2 - t1;
        }
        if (s == P.S) break;
        io.next_hidden = d.next_hidden + (size_t)s * B * (size_t)(d.N * H);
        io.greedy = P.greedy_w ? P.greedy_w + (size_t)(s + 1) * B * d.N : nullptr;
        // profiling: stage timestamps of CTA 0 in the middle simulation, after the per-CTA counters (64 entries)
        long long *sclk = (clk && s == P.S / 2) ? P.tree_clock + 2 * P.S + 4 * (long long)gridDim.x : nullptr;
        if (sclk) { sclk[0] = t2; sclk[1] = t2; }
        infer_stages<W>(d, io, ring, sclk);
        cta_sync();                  // the tile's network outputs are visible to the tree warps; the scratch tiles are free
        if (cta_clk) {
            const long long t3 = clock64();
            sum_inf += t3 - t2;
            if (clk) clk[2 * s] = t3 - t2;
        }
    }
    // the header back to the arena (statistics / later calls read it there)
    if (has_tree && lane < 16) reinterpret_cast<int *>(f_hdr(tb))[lane] = reinterpret_cast<const int *>(hdr)[lane];
    if (tree_clk) { tree_clk[0] = tc_eb; tree_clk[1] = tc_sel; tree_clk[2] = tc_len; tree_clk[3] = tc_max; }
    if (cta_clk) {
        cta_clk[0] = clock64() - k0;
        cta_clk[1] = (long long)(globaltimer_ns() - g0);
        cta_clk[2] = sum_inf;
        cta_clk[3] = sum_tree;
    }
}

}  // namespace persist
}  // namespace maz
