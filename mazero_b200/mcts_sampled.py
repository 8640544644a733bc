"""`SampledMCTS.batch_search` / `SearchOutput`: the search driver, API-compatible with the reference's
core/mcts/tree_search/mcts_sampled.py:12-200, so core/selfplay_worker.py:201-211 and
core/reanalyze_worker.py:121-129,284-294,540-550 can call it unchanged.

Two execution paths, same results contract:

* device path  -- the model is a SMAC `MAMuZeroNet`-shaped network (or a `SmacInference`): the whole
  select -> gather hidden -> recurrent_inference -> softmax/beta -> expand+backup loop runs on the GPU
  as one CUDA graph; the host touches nothing between `prepare` and the readout.
* step path    -- any other `BaseNet` (e.g. the reference's mock models): the reference's simulation loop
  verbatim, with `cytree.Tree_batch` (CUDA) in place of the Cython tree.  Still no CPU tree.

Extension over the fork's signature: `current_agent_idx=None` selects JOINT mode (tree agent_num =
true_num_agents, the upstream MAZero behaviour the BASELINE configs describe); an int selects the fork's
sequential-agent mode (tree agent_num = 1, mcts_sampled.py:53,89).
"""
from collections.abc import Sequence
from typing import List, NamedTuple, Optional, Tuple

import numpy as np
import torch

import ctypes as C
import weakref

import os
from collections import OrderedDict

from . import cytree, hostrng
from ._lib import check, lib
from .search_native import NativeSearch
from .inference import SmacInference
from .inference_mlp import MlpInference
from . import inference_mlp


class SearchOutput(NamedTuple):  # mcts_sampled.py:12-26
    value: np.ndarray
    marginal_visit_count: np.ndarray
    marginal_priors: np.ndarray
    sampled_actions: List[np.ndarray]
    sampled_visit_count: List[np.ndarray]
    sampled_pred_probs: List[np.ndarray]
    sampled_beta: List[np.ndarray]
    sampled_beta_hat: List[np.ndarray]
    sampled_priors: List[np.ndarray]
    sampled_imp_ratio: List[np.ndarray]
    sampled_pred_values: List[np.ndarray]
    sampled_mcts_values: List[np.ndarray]
    sampled_rewards: List[np.ndarray]
    sampled_qvalues: List[np.ndarray]


class AgentTurnsOutput(NamedTuple):
    """Result of `SampledMCTS.search_agents`: what the workers' per-agent loops build on the host."""
    actions: np.ndarray        # (B,N) int32   temp_agent_actions / current_actions
    policy_dist: np.ndarray    # (B,N,A) f64   marginal_visits / sum   (reanalyze_worker.py:319-320)
    prob: np.ndarray           # (B,) f64      product over agents of policy_dist[agent, action]   (:334-345)
    entropy: np.ndarray        # (B,N) f64     base-2 visit entropy of select_action (sample turns)
    search_outputs: list       # N x SearchOutput


class Ragged(Sequence):
    """Lazy list-of-arrays view over a padded (B,K,...) array + per-root lengths: element b is
    padded[b, :n[b]].  The reference materialises 11*B tiny numpy arrays per search
    (cytree.pyx:111-241); callers only index `[b]`, iterate, and use `.size` / `[pos, 0]` / np.sum."""

    __slots__ = ("_pad", "_n")

    def __init__(self, padded, n):
        self._pad, self._n = padded, n

    def __len__(self):
        return len(self._n)

    def __getitem__(self, b):
        if isinstance(b, slice):
            return [self[i] for i in range(*b.indices(len(self)))]
        if b < 0:
            b += len(self)
        return self._pad[b, : self._n[b]]

    def __eq__(self, other):
        return len(self) == len(other) and all(np.array_equal(a, b) for a, b in zip(self, other))


def _softmax_np(logits):
    p = np.exp(logits - np.max(logits, axis=-1, keepdims=True))
    return p / np.sum(p, axis=-1, keepdims=True)


def _output_from_readout(r):
    n = r["num_children"]
    rg = lambda k: Ragged(r[k], n)
    return SearchOutput(r["value"], r["marginal_visit_count"], r["marginal_priors"], rg("actions"), rg("visit_count"),
                        rg("pred_probs"), rg("beta"), rg("beta_hat"), rg("priors"), rg("imp_ratio"), rg("pred_values"),
                        rg("mcts_values"), rg("rewards"), rg("qvalues"))


def _local_agent_turns(plan, count):
    """The first `count` roots of a sequential-agent plan's step results (one D2H copy, one sync): a rank's own slice."""
    outs, actions, dist, prob, entropy = plan.finish_turns()
    return AgentTurnsOutput(actions[:count], dist[:count], prob[:count], entropy[:count],
                            [_output_from_readout({k: v[:count] for k, v in r.items()}) for r in outs])


class _DevicePlan:
    """Static buffers + the captured CUDA graphs of S simulations for one problem shape.  The sequential-agent turns
    (current_agent_idx = 0..N-1) share ONE plan -- tree arena, hidden-state pool and staging buffers are by far the
    largest allocations -- and differ only in their captured graph (`graphs[cur]`)."""

    def __init__(self, inf: SmacInference, B, K, S, cur, cfg, tau, use_graph=True, strategy="auto"):
        self.inf, self.B, self.K, self.S, self.cur, self.tau = inf, B, K, S, cur, float(tau)
        self.N, self.A, self.H = inf.N, inf.A, inf.H
        self.joint = cur is None
        self.Nt = self.N if cur is None else 1  # agents in the tree
        dev = inf.device
        self.dev = dev
        self.c_base, self.c_init, self.discount = float(cfg.pb_c_base), float(cfg.pb_c_init), float(cfg.discount)
        f32, i32 = torch.float32, torch.int32
        D = self.N * self.H
        self.pool = torch.zeros(S + 1, B, D, dtype=f32, device=dev)          # hidden_states_pool (mcts_sampled.py:86)
        z = lambda *s: torch.zeros(*s, dtype=f32, device=dev)
        self.graphs = {}   # legacy path: current_agent_idx (or None) -> captured CUDA graph
        self.use_graph = use_graph
        self.record = None  # when a list: per-simulation injected arrays are appended (parity replay tests)
        self._rec_pending = []
        # The product path: the whole search behind the C ABI (include/maz_search.h) -- tree arena, loop buffers, the
        # persistent kernel / the CUDA graph all live in the library.  Only the fp32 parity mode (plain torch ops for the
        # network, no fused kernel) keeps the loop below.
        self.native = None
        if getattr(inf, "fused", None) is not None and strategy != "legacy":
            self.native = NativeSearch(inf, B, K, S, self.joint, pool=self.pool, strategy=strategy)
            self.tree = self.native.tree
            self.root_p, self.root_b, self.root_n = self.native.root_arrays()
        else:
            self.tree = cytree.Tree_batch(B, self.Nt, self.A, K, S, float(cfg.tree_value_stat_delta_lb), 0,
                                          float(cfg.mcts_rho), float(cfg.mcts_lambda), device=dev.index or 0)
            self.tree.set_puct(self.c_base, self.c_init)
            self.greedy = torch.zeros(S + 1, B, self.N, dtype=i32, device=dev)   # argmax_a prediction(node).policy (A.11)
            self.idx_x = torch.zeros(B, dtype=i32, device=dev)
            self.idx_y = torch.zeros(B, dtype=i32, device=dev)
            self.act = torch.zeros(B, self.Nt, dtype=i32, device=dev)
            self.rows = torch.arange(B, dtype=torch.int64, device=dev)
            self.root_p, self.root_b, self.root_n = z(B, self.Nt, self.A), z(B, self.Nt, self.A), z(B, self.Nt, self.A)
            # per-simulation network outputs (fused path writes them in place)
            self.sim_r, self.sim_v = z(B), z(B)
            self.sim_p, self.sim_b = z(B, self.Nt, self.A), z(B, self.Nt, self.A)
        self.factor = torch.zeros(B, max(self.N, 1), dtype=i32, device=dev)
        f64 = torch.float64
        # ---- host -> device staging: every small root input lives in ONE pinned buffer (one H2D copy per search) ----
        T = 1 if cur is None else self.N            # turns served by this plan (sequential-agent mode: one per agent)
        self.T = T
        in_spec = [("rewards", f32, (B,)), ("values", f32, (B,)), ("logits", f32, (B, self.N, self.A)),
                   ("legal", f32, (B, self.N, self.A)), ("factor_in", i32, (B, self.N))]
        for t in range(T):    # per-turn block (depends on the host RNG): contiguous, so one H2D copy per turn
            in_spec += [(f"uniforms{t}", f64, (B,)), (f"noise_raw{t}", f32, (B, self.Nt, self.A)), (f"eps_u{t}", f32, (B,)),
                        (f"rand_act{t}", i32, (B,))]
        self.inp, self.inp_np, self.in_flat, self.in_host, off = self._flat(in_spec, dev)
        self.in_common = (0, off["uniforms0"][0])
        self.in_turn = [(off[f"uniforms{t}"][0], off[f"rand_act{t}"][1]) for t in range(T)]
        self.root_r, self.root_v = self.inp["rewards"], self.inp["values"]
        self.has_legal = False
        self._dev_fields = []
        # ---- device -> host: all readouts of all turns + the turn results in ONE buffer / ONE D2H copy -------------
        spec = [("value", f32, (B,)), ("marginal_visit_count", i32, (B, self.Nt, self.A)),
                ("marginal_priors", f32, (B, self.Nt, self.A)), ("num_children", i32, (B,)),
                ("actions", i32, (B, K, self.Nt)), ("visit_count", i32, (B, K))]
        spec += [(f, f32, (B, K)) for f in cytree._FLOAT_FIELDS]
        self.readout_spec = [(n, np.float32 if dt is f32 else np.int32, shp) for n, dt, shp in spec]
        words = sum(int(np.prod(shp)) for _, _, shp in spec)
        words += words & 1
        out_spec = [(f"t{t}", i32, (words,)) for t in range(T)]
        out_spec += [("turn_actions", i32, (B, self.N)), ("prob_prod", f64, (B,)),
                     ("policy_dist", f64, (B, self.N, self.A)), ("entropy", f64, (B, self.N))]
        self.res, self.res_np, self.res_flat, self.res_host, self.res_off = self._flat(out_spec, dev)
        self.words = words
        self.turn_out, self.turn_out_np = [], []
        for t in range(T):
            o, d, dn = 0, {}, {}
            for name, dt, shp in spec:
                n = int(np.prod(shp))
                d[name] = self.res[f"t{t}"][o:o + n].view(dt).view(*shp)
                dn[name] = self.res_np[f"t{t}"][o:o + n].view(np.float32 if dt is f32 else np.int32).reshape(shp)
                o += n
            self.turn_out.append(d)
            self.turn_out_np.append(dn)
        # single-search view (turn 0): what `run` / bench.py / the sharded all-gather use
        self.out, self.out_np = self.turn_out[0], self.turn_out_np[0]
        self.out_flat, self.out_host = self.res["t0"], self.res_host[: words]
        if cur is not None:
            # the agents' chosen actions (= `factor` of the later turns) live in the result buffer: written by
            # k_agent_turn on the device, or copied from the caller's host `factor`
            self.factor = self.res["turn_actions"]

    def gather_buffers(self, world):
        """(device, pinned host) int32 buffers for the all-gather of `world` packed readout blocks."""
        g = getattr(self, "_gather", None)
        if g is None or g[0].numel() != world * self.out_flat.numel():
            dev = torch.empty(world * self.out_flat.numel(), dtype=torch.int32, device=self.dev)
            g = (dev, torch.empty(dev.numel(), dtype=torch.int32).pin_memory())
            self._gather = g
        return g

    def turn_gather_buffers(self, world):
        """(device, pinned host) int32 buffers for the all-gather of `world` whole step buffers (`res_flat`: every agent's
        readouts + the turn results)."""
        g = getattr(self, "_turn_gather", None)
        if g is None or g[0].numel() != world * self.res_flat.numel():
            dev = torch.empty(world * self.res_flat.numel(), dtype=torch.int32, device=self.dev)
            g = (dev, torch.empty(dev.numel(), dtype=torch.int32).pin_memory())
            self._turn_gather = g
        return g

    def turn_layout(self):
        """Where everything lives in `res_flat` (int32 words): (readout_spec, word offset of each turn's readout block,
        [(name, numpy dtype, shape, word offset)] of the turn fields) -- what `sharding.split_turn_block` reads."""
        npdt = {torch.float32: np.float32, torch.int32: np.int32, torch.float64: np.float64}
        fields = [(n, npdt[self.res[n].dtype], tuple(self.res[n].shape), self.res_off[n][0])
                  for n in ("turn_actions", "prob_prod", "policy_dist", "entropy")]
        return self.readout_spec, [self.res_off[f"t{t}"][0] for t in range(self.T)], fields

    def device_bytes(self):
        """HBM held by this plan (pool + arena + loop buffers + staging mirrors)."""
        n = self.pool.numel() * 4 + self.in_flat.numel() * 4 + self.res_flat.numel() * 4
        if self.native is not None:
            return n + self.native.device_bytes()
        return n + self.tree.arena_bytes() + self.greedy.numel() * 4

    def close(self):
        """Free the native objects now (cache eviction); the torch buffers go with the last reference."""
        self.graphs.clear()
        if self.native is not None:
            self.native.close()
            self.native = None
        self.tree = None

    @staticmethod
    def _flat(spec, dev):
        """One device buffer + one pinned host mirror holding all arrays of `spec` (4-byte words; float64 entries are
        placed at even word offsets).  Returns (device views, host numpy views, device flat, host flat, offsets)."""
        f64 = torch.float64
        npdt = {torch.float32: np.float32, torch.int32: np.int32, torch.float64: np.float64}
        off, o = {}, 0
        for name, dt, shp in spec:
            n = int(np.prod(shp)) * (2 if dt is f64 else 1)
            if dt is f64 and o % 2:
                o += 1
            off[name] = (o, o + n)
            o += n
        o += o & 1
        flat = torch.zeros(o, dtype=torch.int32, device=dev)
        host = torch.zeros(o, dtype=torch.int32).pin_memory()
        host_np = host.numpy()
        dv, hv = {}, {}
        for name, dt, shp in spec:
            a, b = off[name]
            dv[name] = flat[a:b].view(dt).view(*shp)
            hv[name] = host_np[a:b].view(npdt[dt]).reshape(shp)
        return dv, hv, flat, host, off

    def _simulate(self, s, select_first=True, select_next=False):
        """One simulation.  select_first: run the selection kernel at the start (else the previous simulation's
        fused expand+backup+select launch already did); select_next: fuse the NEXT simulation's selection into
        this simulation's expansion+backup launch."""
        t, B = self.tree, self.B
        if select_first:
            t.batch_selection_device(self.c_base, self.c_init, self.discount, self.idx_x, self.idx_y, self.act)
        flat = None
        if self.cur is None:
            joint = self.act
        else:                                                                 # mcts_sampled.py:116-147
            flat = self.idx_x.long() * B + self.rows                          # row of the parent in the pool
            g = self.greedy.view(-1, self.N).index_select(0, flat)
            joint = torch.cat([self.factor[:, : self.cur], self.act, g[:, self.cur + 1:]], dim=1).contiguous()
        if self.inf.fused is not None:
            # ONE kernel: gather parent hidden, recurrent_inference on the tensor cores, inverse support
            # transforms, softmax / beta of the tree agents, greedy actions of every agent
            self.inf.recurrent_fused(B, self.pool, self.idx_x, joint, self.pool[s + 1], self.sim_r, self.sim_v, self.sim_p,
                                     self.sim_b, self.greedy[s + 1] if self.cur is not None else None, None, self.Nt,
                                     -1 if self.cur is None else self.cur, 1.0 / self.tau)
            if self.record is not None:
                self.record.append((self.sim_r.clone(), self.sim_v.clone(), self.sim_p.clone(), self.sim_b.clone(),
                                    self.idx_x.clone(), self.act.clone()))
            if select_next:
                t.expansion_backup_selection_device(s + 1, self.discount, self.K, self.sim_r, self.sim_v, self.sim_p,
                                                    self.sim_b, self.c_base, self.c_init, self.idx_x, self.idx_y, self.act)
            else:
                t.batch_expansion_and_backup(s + 1, self.discount, self.K, self.sim_r, self.sim_v, self.sim_p, self.sim_b)
            return
        if flat is None:
            flat = self.idx_x.long() * B + self.rows
        h = self.pool.view(-1, self.N * self.H).index_select(0, flat)
        _, rew, val, logits = self.inf.recurrent(h, joint, out_hidden=self.pool[s + 1])
        if self.cur is not None:
            self.greedy[s + 1].copy_(logits.argmax(dim=-1))
            logits = logits[:, self.cur: self.cur + 1]
        p = torch.softmax(logits, dim=-1)                                     # mcts_sampled.py:158-161
        b = p if self.tau == 1.0 else p ** (1.0 / self.tau)
        b = b / b.sum(dim=-1, keepdim=True)
        p, b = p.contiguous(), b.contiguous()
        if self.record is not None:
            self.record.append((rew.clone(), val.clone(), p.clone(), b.clone(), self.idx_x.clone(), self.act.clone()))
        if select_next:
            t.expansion_backup_selection_device(s + 1, self.discount, self.K, rew, val, p, b, self.c_base, self.c_init,
                                                self.idx_x, self.idx_y, self.act)
        else:
            t.batch_expansion_and_backup(s + 1, self.discount, self.K, rew, val, p, b)

    def _loop(self):
        # two launches per simulation: [inference] -> [expand + backup + next selection]
        fuse = self.record is None
        for s in range(self.S):
            self._simulate(s, select_first=(s == 0 or not fuse), select_next=(fuse and s + 1 < self.S))

    @property
    def graph(self):
        return self.graphs.get(self.cur)

    # ---- host -> device staging ------------------------------------------------------------------------------
    def _stream(self):
        stream = torch.cuda.current_stream(self.dev)
        if self.native is not None:
            self.native.set_stream(stream.cuda_stream)
        else:
            self.tree.set_stream(stream.cuda_stream)
        return stream

    def stage_roots(self, root_hidden, rewards, values, logits, legal, factor=None, cur=None):
        """Everything that does not depend on the host RNG: the root hidden state goes straight into the pool
        (asynchronously when pinned), the small arrays into the pinned staging block (copied by `_h2d`)."""
        B, h = self.B, self.inp_np
        src = root_hidden if torch.is_tensor(root_hidden) else torch.from_numpy(np.ascontiguousarray(root_hidden))
        self.pool[0].copy_(src.reshape(B, -1), non_blocking=True)
        self._dev_fields = []      # inputs that already live on the device: copied over the staging block after its H2D

        def put(name, x, shape):
            if torch.is_tensor(x) and x.is_cuda:
                self._dev_fields.append((name, x.detach().reshape(shape)))
            else:
                h[name][:] = (x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)).reshape(shape)

        put("rewards", rewards, (B,))
        put("values", values, (B,))
        put("logits", logits, (B, self.N, self.A))
        self.has_legal = legal is not None
        if legal is not None:
            put("legal", legal, (B, self.N, self.A))
        if cur:
            if factor is None:                       # the reference leaves zeros for the earlier agents (mcts_sampled.py:116-120)
                h["factor_in"][:, :cur] = 0
            else:
                f = factor.detach().cpu().numpy() if torch.is_tensor(factor) else np.asarray(factor)
                assert f.shape[0] == B and f.shape[1] >= cur, "factor must hold the actions of agents 0..current_agent_idx-1"
                h["factor_in"][:, :cur] = f[:, :cur]

    def _apply_dev_fields(self):
        for name, t in self._dev_fields:
            self.inp[name].copy_(t, non_blocking=True)

    def _h2d(self, a, b):
        self.in_flat[a:b].copy_(self.in_host[a:b], non_blocking=True)

    # ---- one search, fully asynchronous -------------------------------------------------------------------------
    def _enqueue_search(self, slot, cur, seed, cfg, noise_eps, root_index_offset):
        """root preparation -> reset -> prepare -> S simulations -> readout into result slot `slot`."""
        self.cur = cur
        stream = self._stream()
        if self.native is not None:      # ONE library call: root preparation, tree construction, S simulations, readout
            if self.record is not None or self._rec_on:
                self._arm_record()
            self.native.run_dev(cur, seed, cfg, noise_eps, self.tau, self.root_r, self.root_v, self.inp["logits"],
                                self.inp["legal"] if self.has_legal else None, self.inp[f"noise_raw{slot}"],
                                self.factor if cur else None, self.turn_out[slot], root_index_offset=root_index_offset,
                                cache_key=(slot, bool(cur), self.has_legal))
            return
        ptr = lambda t: C.c_void_p(t.data_ptr())
        check(lib.maz_root_prepare_dev(                                         # mcts_sampled.py:57-106 on the device
            ptr(self.inp["logits"]), ptr(self.inp["legal"]) if self.has_legal else None, ptr(self.inp[f"noise_raw{slot}"]),
            self.B, self.N, self.A, -1 if cur is None else int(cur), float(noise_eps), 1.0 / self.tau,
            ptr(self.root_p), ptr(self.root_b), ptr(self.root_n), ptr(self.greedy[0]), C.c_void_p(stream.cuda_stream)))

        def prepare():
            self.tree.reset(seed, float(cfg.tree_value_stat_delta_lb), float(cfg.mcts_rho), float(cfg.mcts_lambda), root_index_offset)
            self.tree.prepare(self.root_r, self.root_v, self.root_p, self.root_b, self.K, float(noise_eps), self.root_n)

        if self.use_graph and self.record is None:
            if self.cur not in self.graphs:
                prepare()          # the capture warm-up runs one real simulation: it needs valid roots
                self._capture()
            prepare()
            self.graphs[self.cur].replay()
        else:
            prepare()
            self._loop()
        self.tree.readout_device(self.discount, self.turn_out[slot])

    _rec_on = False

    def _arm_record(self):
        """Parity instrumentation of the native search: per-simulation selections + injected network outputs."""
        if self.record is None:
            self.native.set_record(None)
            self._rec_on = False
            return
        S, B, Nt, A, dev = self.S, self.B, self.Nt, self.A, self.dev
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        i = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
        rec = {"rewards": f(S, B), "values": f(S, B), "probs": f(S, B, Nt, A), "beta": f(S, B, Nt, A), "idx_x": i(S, B),
               "actions": i(S, B, Nt)}
        self.native.set_record(rec)
        self._rec_on = True
        self._rec_pending.append(rec)

    def _flush_record(self):
        for rec in self._rec_pending:
            for s in range(self.S):
                self.record.append((rec["rewards"][s], rec["values"][s], rec["probs"][s], rec["beta"][s], rec["idx_x"][s],
                                    rec["actions"][s]))
        self._rec_pending = []

    def run(self, seed, cfg, noise_eps, noise_raw, root_index_offset=0, cur=None):
        """One search after `stage_roots`: `noise_raw` (B,Nt,A) are the raw Dirichlet draws (host).  Returns the
        padded readout dict (host numpy)."""
        assert (cur is None) == self.joint, "a plan is either joint or sequential"
        self._stream()
        self.inp_np["noise_raw0"][:] = noise_raw
        self._h2d(0, self.in_turn[0][1])
        self._apply_dev_fields()
        if cur:
            self.factor[:, :cur].copy_(self.inp["factor_in"][:, :cur], non_blocking=True)
        self._enqueue_search(0, cur, seed, cfg, noise_eps, root_index_offset)
        self.out_host.copy_(self.out_flat, non_blocking=True)
        self.tree.check()          # synchronises the stream and surfaces device-side invariant failures
        if self._rec_pending:
            self._flush_record()
        return {k: v.copy() for k, v in self.out_np.items()}

    def enqueue(self, seed, cfg, noise_eps, noise_raw, root_index_offset=0, cur=None):
        """`run` without the device -> host copy and without synchronising: the readouts stay in `out_flat` (device)."""
        assert (cur is None) == self.joint, "a plan is either joint or sequential"
        self._stream()
        self.inp_np["noise_raw0"][:] = noise_raw
        self._h2d(0, self.in_turn[0][1])
        self._apply_dev_fields()
        if cur:
            self.factor[:, :cur].copy_(self.inp["factor_in"][:, :cur], non_blocking=True)
        self._enqueue_search(0, cur, seed, cfg, noise_eps, root_index_offset)

    # ---- the N sequential-agent turns of one environment step, back to back on the device -------------------------
    def begin_turns(self):
        self._stream()
        self._h2d(*self.in_common)
        self._apply_dev_fields()

    def enqueue_turn(self, k, mode, seed, cfg, noise_eps, noise_raw, inv_temperature=1.0, uniforms=None, greedy_epsilon=0.0,
                     eps_u=None, rand_act=None, root_index_offset=0):
        """Turn of agent k: its search (factor = the actions chosen on the device in the earlier turns), then the
        worker's action choice (maz_agent_turn_dev).  Nothing synchronises."""
        h = self.inp_np
        h[f"noise_raw{k}"][:] = noise_raw
        if uniforms is not None:
            h[f"uniforms{k}"][:] = uniforms
        inject = eps_u is not None and rand_act is not None
        if inject:
            h[f"eps_u{k}"][:] = eps_u
            h[f"rand_act{k}"][:] = rand_act
        self._h2d(*self.in_turn[k])
        self._enqueue_search(k, k, seed, cfg, noise_eps, root_index_offset)
        o, ptr = self.turn_out[k], (lambda t: C.c_void_p(t.data_ptr()))
        stream = torch.cuda.current_stream(self.dev)
        check(lib.maz_agent_turn_dev(
            int(mode), self.B, self.N, self.A, self.K, int(k), ptr(o["num_children"]), ptr(o["actions"]), ptr(o["visit_count"]),
            ptr(o["marginal_visit_count"]), ptr(self.inp["legal"]) if self.has_legal else None, float(inv_temperature),
            ptr(self.inp[f"uniforms{k}"]), float(greedy_epsilon), ptr(self.inp[f"eps_u{k}"]) if inject else None,
            ptr(self.inp[f"rand_act{k}"]) if inject else None, ptr(self.res["turn_actions"]), ptr(self.res["policy_dist"]),
            ptr(self.res["prob_prod"]), ptr(self.res["entropy"]), C.c_void_p(stream.cuda_stream)))

    def finish_turns(self):
        self.res_host.copy_(self.res_flat, non_blocking=True)      # ONE D2H copy for all turns
        self.tree.check()
        if self._rec_pending:
            self._flush_record()
        r = self.res_np
        outs = [{k: v.copy() for k, v in d.items()} for d in self.turn_out_np]
        return (outs, r["turn_actions"].copy(), r["policy_dist"].copy(), r["prob_prod"].copy(), r["entropy"].copy())

    def _capture(self):
        cur = torch.cuda.current_stream(self.dev)
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):   # warm-up outside capture (cuBLAS handles, workspaces, allocator)
            self.tree.set_stream(side.cuda_stream)
            self._simulate(0)
            self.tree.check()
        cur.wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.tree.set_stream(torch.cuda.current_stream(self.dev).cuda_stream)
            self._loop()
        self.tree.set_stream(cur.cuda_stream)
        self.graphs[self.cur] = g


# The workers build a NEW `SampledMCTS(config, np_random)` for every environment step / every agent
# (selfplay_worker.py:191, reanalyze_worker.py:284), so the expensive device objects -- packed weights, tree arena,
# hidden-state pool, CUDA graphs -- are cached per PROCESS, not per instance: keyed by the model object and the problem
# shape / search constants.  Both caches are bounded: plans by a byte budget with least-recently-used eviction (a reanalyze
# worker whose batch size varies would otherwise keep one arena + pool per size), inference objects by the life of their
# model (weak reference + finalizer).
_INFERENCE_CACHE = {}          # (id(model), device, mode) -> (weakref to the model, SmacInference | MlpInference)
_PLAN_CACHE = OrderedDict()    # plan key -> _DevicePlan, least recently used first
PLAN_CACHE_BYTES = int(float(os.environ.get("MAZ_PLAN_CACHE_GB", "32")) * (1 << 30))


def _plan_cache_bytes():
    return sum(p.device_bytes() for p in _PLAN_CACHE.values())


def _plan_cache_put(key, plan):
    _PLAN_CACHE[key] = plan
    _PLAN_CACHE.move_to_end(key)
    # evict least recently used plans until the budget holds; the plan just inserted always stays
    while len(_PLAN_CACHE) > 1 and _plan_cache_bytes() > PLAN_CACHE_BYTES:
        _, old = _PLAN_CACHE.popitem(last=False)
        old.close()            # frees the arena / loop buffers now, not when the last Python reference dies


def _drop_inference(key):
    hit = _INFERENCE_CACHE.pop(key, None)
    if hit is None:
        return
    inf = hit[1]
    for k in [k for k, p in _PLAN_CACHE.items() if p.inf is inf]:
        _PLAN_CACHE.pop(k).close()


def clear_caches():
    """Drop every cached device object (arenas, pools, graphs) of this process."""
    for p in _PLAN_CACHE.values():
        p.close()
    _INFERENCE_CACHE.clear()
    _PLAN_CACHE.clear()


def _weights_signature(tensors):
    """Cheap change detector of a module's parameters: in-place updates bump `_version`, re-assigned storages
    (`param.data = ...`, load_state_dict(assign=True)) change `data_ptr`."""
    v = 0
    for t in tensors:
        v = (v * 1000003 + int(t._version) * 8191 + t.data_ptr()) & 0xFFFFFFFFFFFFFFFF
    return v


class SampledMCTS(object):
    def __init__(self, config, np_random: np.random.RandomState = None, use_cuda_graph: bool = True,
                 inference_mode: str = "auto", speculate_noise: bool = True, search_strategy: str = "auto"):
        """inference_mode: "bf16" = fused tensor-core kernel, "fp32" = parity mode (plain fp32 torch ops on the
        device), "auto" = bf16 when the network has the reference SMAC architecture, else fp32.
        speculate_noise: draw the NEXT search's exploration noise on a background thread while the GPU runs the current
        search; it is used only if `np_random` is still in exactly the state it was left in (mazero_b200/hostrng.py)."""
        self.config = config
        self.speculate_noise = speculate_noise
        self.np_random = np.random if np_random is None else np_random
        self.use_cuda_graph = use_cuda_graph
        self.inference_mode = inference_mode
        # "auto" | "persistent" | "graph": how the library runs the loop (include/maz_search.h); "legacy": the round-1 Python /
        # torch.cuda.CUDAGraph loop over the per-step C ABI (kept as a cross-check of the native search)
        self.search_strategy = search_strategy
        self._inference = {}
        self._plans = {}

    # ---- model adaptation ---------------------------------------------------------------------------------
    def _device_inference(self, model, device) -> Optional[SmacInference]:
        if isinstance(model, (SmacInference, MlpInference)):
            return model
        if not isinstance(model, torch.nn.Module):
            return None
        # fast path: this model object was adapted before -- no state_dict() walk, only the change signature of its tensors
        probe = getattr(model, "_maz_inference", None)
        if probe is not None:
            dev_s = str(torch.device(device)) if device is not None else probe.get("default_dev")
            key = (id(model), dev_s, self.inference_mode)
            hit = _INFERENCE_CACHE.get(key)
            if hit is not None and hit[0]() is model:
                inf = hit[1]
                sig = _weights_signature(inf._src_tensors)
                if sig != inf._src_signature:                 # weights were updated (set_weights / load_state_dict)
                    inf.refresh(model.state_dict())
                    inf._src_signature = sig
                self._inference[key] = inf
                return inf
        try:
            sd = model.state_dict()
        except Exception:
            return None
        smac = "dynamics_network.attention_stack.0.weight" in sd and "prediction_network.fc_policy.0.weight" in sd
        mlp = not smac and inference_mlp.supported(sd)     # the matrix-game family (config/matrix/model.py)
        if not smac and not mlp:
            return None
        dev = torch.device(device) if device is not None else sd["prediction_network.fc_policy.0.weight"].device
        if dev.type != "cuda":
            return None
        key = (id(model), str(dev), self.inference_mode)      # "fp32" parity mode must never be served a cached bf16 object
        hit = _INFERENCE_CACHE.get(key)
        inf = hit[1] if hit is not None and hit[0]() is model else None      # (ids are reused after garbage collection)
        if inf is None and hit is not None:
            _drop_inference(key)
        if inf is None and mlp:
            inf = MlpInference.from_model(model, device=dev, mode="torch" if self.inference_mode in ("torch", "fp32torch") else "fp32")
        elif inf is None:
            mode = self.inference_mode
            if mode == "auto":
                from . import fused

                h = int(getattr(model, "hidden_state_size_per_agent", getattr(model, "hidden", 128)))
                mode = "bf16" if fused.supported(sd, int(model.num_agents), int(model.action_space_size), h) else "fp32"
                if mode == "fp32":      # not silent: the fused kernels cover the reference SMAC architecture only (fused.supported)
                    import warnings

                    warnings.warn("mazero_b200: this network is not the reference SMAC architecture (hidden 128, 3 x 8-head encoder "
                                  "layers, support 11, <= 30 agents, <= 128 actions): the search runs its forward as plain fp32 torch "
                                  "ops on the device (parity mode), not through the fused tensor-core kernels", RuntimeWarning,
                                  stacklevel=3)
            inf = SmacInference.from_model(model, device=dev, mode=mode)
        else:
            inf.refresh(sd)
        inf._src_tensors = list(model.parameters()) + list(model.buffers())
        inf._src_signature = _weights_signature(inf._src_tensors)
        if hit is None or hit[1] is not inf:
            _INFERENCE_CACHE[key] = (weakref.ref(model), inf)
            weakref.finalize(model, _drop_inference, key)     # a dead model releases its packed weights and its plans
        try:
            marks = getattr(model, "_maz_inference", None) or {}
            marks["default_dev"] = str(dev) if device is None else marks.get("default_dev")
            model._maz_inference = marks
        except Exception:
            pass
        self._inference[key] = inf
        return inf

    # ---- the entry point (mcts_sampled.py:34-46) -----------------------------------------------------------
    def batch_search(
        self,
        model,
        network_output,
        current_agent_idx: Optional[int],
        factor: np.ndarray,
        true_num_agents: int,
        legal_actions_lst: np.ndarray = None,
        device: torch.device = None,
        add_noise: bool = False,
        sampled_tau: float = 1.0,
        sampled_actions_res: Tuple[np.ndarray, np.ndarray] = None,
        root_index_offset: int = 0,
    ) -> SearchOutput:
        cfg = self.config
        noise_alpha, noise_epsilon = cfg.root_dirichlet_alpha, cfg.root_exploration_fraction
        A, K = cfg.action_space_size, cfg.sampled_action_times
        joint = current_agent_idx is None
        Nt = true_num_agents if joint else 1
        B = network_output.hidden_state.shape[0]

        def host(x):
            return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)

        if not add_noise:
            noise_epsilon = 0.0

        inf = self._device_inference(model, device)
        plan = None
        if inf is not None:
            plan = self._plan(inf, B, current_agent_idx, sampled_tau)
            # the copies that do not depend on the host RNG are in flight while the noise is drawn; reward / value / logits may
            # be numpy (the reference's eval-mode NetworkOutput) or CUDA tensors (`inf.initial_inference`: nothing leaves the GPU)
            plan.stage_roots(network_output.hidden_state, network_output.reward, network_output.value, network_output.policy_logits,
                             legal_actions_lst, factor, current_agent_idx)
        else:
            batch_rewards, batch_values = host(network_output.reward), host(network_output.value)
            all_logits = host(network_output.policy_logits)
            assert batch_values.shape == (B, 1) and all_logits.size == B * true_num_agents * A

        # exploration noise (:68-70): drawn even when add_noise is False, one Dirichlet per (root, tree agent)
        # (hostrng: the same values and the same final generator state as np_random.dirichlet, on all host cores)
        noises = hostrng.dirichlet_f32(self.np_random, noise_alpha, A, B * Nt if joint else B).reshape(B, Nt, A)
        seed = self.np_random.choice(256)                                            # :89 (after the Dirichlet)
        if sampled_actions_res is not None:
            raise NotImplementedError                                                # :108-109
        if plan is not None:
            if self.speculate_noise:   # the next search's noise draw overlaps this search (used only if np_random is untouched)
                hostrng.speculate(self.np_random, noise_alpha, A, B * Nt if joint else B)
            # root preparation (:57-106) runs on the device (maz_root_prepare_dev)
            r = plan.run(int(seed), cfg, noise_epsilon, noises, root_index_offset, cur=current_agent_idx)
            return _output_from_readout(r)

        if joint:
            logits = all_logits.reshape(B, Nt, A)
        else:
            logits = all_logits[:, current_agent_idx, :].reshape(B, 1, A)           # mcts_sampled.py:60-61
        probs = _softmax_np(logits)                                                  # :64-65
        legal = None
        if legal_actions_lst is not None:                                            # :73-83
            legal = (legal_actions_lst.reshape(B, Nt, A) if joint
                     else legal_actions_lst[:, current_agent_idx, :].reshape(B, 1, A))
            probs *= legal
            probs += legal * 1e-4
            assert ~(np.sum(probs, axis=-1) == 0).sum()
            probs = probs / np.sum(probs, axis=-1, keepdims=True)
            noises *= legal
            noises += legal * 1e-4
            noises = noises / np.sum(noises, axis=-1, keepdims=True)
        beta = probs * (1 - noise_epsilon) + noises * noise_epsilon                  # :93-100
        beta = beta ** (1 / sampled_tau)
        if legal is not None:
            beta *= legal
            assert ~(np.sum(beta, axis=-1) == 0).sum()
        beta = beta / np.sum(beta, axis=-1, keepdims=True)
        batch_rewards = batch_rewards.reshape(B).astype(np.float32)
        batch_values = batch_values.reshape(B).astype(np.float32)
        probs, beta, noises = probs.astype(np.float32), beta.astype(np.float32), noises.astype(np.float32)
        return self._search_step_path(model, network_output, current_agent_idx, factor, true_num_agents, device, sampled_tau,
                                      seed, noise_epsilon, batch_rewards, batch_values, probs, beta, noises, root_index_offset)

    # ---- SURVEY 8(e): roots sharded over the ranks of a process group, ONE exchange per search ------------------------------
    def batch_search_sharded(self, model, network_output, current_agent_idx, factor, true_num_agents, total_roots: int,
                             legal_actions_lst=None, device=None, add_noise: bool = False, sampled_tau: float = 1.0, group=None,
                             gather: bool = True) -> SearchOutput:
        """`batch_search` for a batch of `total_roots` roots split over the ranks of `group` (torch.distributed, NCCL): this rank
        passes ITS contiguous slice `sharding.shard_range(total_roots, rank, world)` of every per-root argument, searches it with
        the trees seeded by their GLOBAL root index (results do not depend on the number of ranks, cnode.cpp:574), and ONE
        all-gather of the packed readouts (device tensors, NCCL over NVLink) gives every rank the SearchOutput of all roots.
        Every rank must hold `np_random` in the same state (the noise of ALL roots and the tree seed are drawn on every rank, as
        the single-process reference would, and sliced).  gather=False returns the local slice only (no collective)."""
        import torch.distributed as dist

        from . import sharding

        cfg = self.config
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        start, count = sharding.shard_range(total_roots, rank, world)
        Bp = sharding.shard_range(total_roots, 0, world)[1]               # the largest shard: every rank searches Bp roots
        joint = current_agent_idx is None
        A, Nt = cfg.action_space_size, (true_num_agents if joint else 1)
        if network_output.hidden_state.shape[0] != count:
            raise ValueError(f"rank {rank}: expected {count} local roots, got {network_output.hidden_state.shape[0]}")
        inf = self._device_inference(model, device)
        if inf is None:
            raise RuntimeError("batch_search_sharded needs a network with a device path (SMAC / matrix MAMuZeroNet on a CUDA device)")
        pad = lambda x: None if x is None else sharding.pad_rows(x, Bp)
        plan = self._plan(inf, Bp, current_agent_idx, sampled_tau)
        plan.stage_roots(pad(network_output.hidden_state), pad(network_output.reward), pad(network_output.value),
                         pad(network_output.policy_logits), pad(legal_actions_lst), pad(factor), current_agent_idx)
        noises = hostrng.dirichlet_f32(self.np_random, cfg.root_dirichlet_alpha, A, total_roots * Nt).reshape(total_roots, Nt, A)
        seed = self.np_random.choice(256)
        plan.enqueue(int(seed), cfg, cfg.root_exploration_fraction if add_noise else 0.0, pad(noises[start:start + count]),
                     root_index_offset=start, cur=current_agent_idx)
        if not gather or world == 1:
            plan.out_host.copy_(plan.out_flat, non_blocking=True)
            plan.tree.check()
            r = {k: v[:count].copy() for k, v in plan.out_np.items()}
            return _output_from_readout(r)
        gbuf, ghost = plan.gather_buffers(world)
        dist.all_gather_into_tensor(gbuf, plan.out_flat, group=group)                # the one collective of the search
        ghost.copy_(gbuf, non_blocking=True)
        plan.tree.check()
        blocks = ghost.numpy().reshape(world, -1)
        return _output_from_readout(sharding.merge_shards(blocks, plan.readout_spec, total_roots, world))

    def _plan(self, inf, B, current_agent_idx, sampled_tau) -> _DevicePlan:
        cfg = self.config
        # The native search takes every search constant per call (its CUDA graphs are keyed by them inside the library), so a
        # plan depends on the shape only; the legacy loop freezes the constants into its captured graphs: they are in its key.
        key = (id(inf), B, cfg.sampled_action_times, cfg.num_simulations, current_agent_idx is None, float(sampled_tau),
               self.search_strategy)
        if self.search_strategy == "legacy" or getattr(inf, "fused", None) is None:
            key += (float(cfg.pb_c_base), float(cfg.pb_c_init), float(cfg.discount), float(cfg.tree_value_stat_delta_lb),
                    float(cfg.mcts_rho), float(cfg.mcts_lambda), bool(self.use_cuda_graph))
        plan = _PLAN_CACHE.get(key)                                                  # all sequential turns share a plan
        if plan is not None and (plan.inf is not inf or plan.tree is None):
            plan = None
        if plan is None:
            plan = _DevicePlan(inf, B, cfg.sampled_action_times, cfg.num_simulations, current_agent_idx, cfg, sampled_tau,
                               self.use_cuda_graph, strategy=self.search_strategy)
        plan.c_base, plan.c_init, plan.discount = float(cfg.pb_c_base), float(cfg.pb_c_init), float(cfg.discount)
        _plan_cache_put(key, plan)
        self._plans[key] = plan
        return plan

    # ---- SURVEY 8(f): the workers' per-agent loop as ONE device-resident call ------------------------------------------
    def search_agents(self, model, network_output, true_num_agents: int, legal_actions_lst: np.ndarray = None,
                      device: torch.device = None, add_noise: bool = True, sampled_tau: float = 1.0, turn: str = "greedy",
                      temperature: float = 1.0, greedy_epsilon: float = 0.0, eps_randoms=None,
                      root_index_offset: int = 0) -> "AgentTurnsOutput":
        """The N sequential per-agent searches of one environment step (selfplay_worker.py:196-257,
        reanalyze_worker.py:278-327) without returning to the host in between: agent k's search takes `factor` =
        the actions agents 0..k-1 chose ON THE DEVICE, and the host synchronises once, after the last agent.

        turn="greedy"  reanalyze: action = argmax(marginal_visits * legal)                     (reanalyze_worker.py:298-317)
        turn="sample"  self-play: select_action(sampled_visit_count, temperature) with np_random, then eps_greedy_action
                       (selfplay_worker.py:230-257).  `eps_randoms` = (eps_u (N,B) float32, random_action (N,B) int32) are the
                       draws `torch.rand_like` / `Categorical(legal).sample()` of core/utils.py:328-330, which depend only
                       on the legal mask; None = no epsilon-greedy override.

        `self.np_random` is consumed in exactly the reference's order -- per agent: dirichlet, choice(256), then (sample
        mode) one random_sample per root for np_random.choice inside select_action -- and the host draws agent k+1's
        numbers while the GPU searches for agent k."""
        cfg = self.config
        N, A = int(true_num_agents), cfg.action_space_size
        inf = self._device_inference(model, device)
        if inf is None:
            raise RuntimeError("search_agents needs a network with a device path (SMAC / matrix MAMuZeroNet on a CUDA device)")
        if turn not in ("greedy", "sample"):
            raise ValueError(turn)
        B = network_output.hidden_state.shape[0]
        host = lambda x: x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
        noise_epsilon = cfg.root_exploration_fraction if add_noise else 0.0
        plan = self._plan(inf, B, 0, sampled_tau)
        plan.stage_roots(network_output.hidden_state, network_output.reward, network_output.value,
                         network_output.policy_logits, legal_actions_lst)
        plan.begin_turns()
        eps_u, rand_act = (None, None) if eps_randoms is None else eps_randoms
        for k in range(N):
            noises = hostrng.dirichlet_f32(self.np_random, cfg.root_dirichlet_alpha, A, B).reshape(B, 1, A)
            seed = self.np_random.choice(256)
            u = self.np_random.random_sample(B) if turn == "sample" else None        # B x np_random.choice(n, p=...)
            plan.enqueue_turn(k, 1 if turn == "sample" else 0, int(seed), cfg, noise_epsilon, noises, 1.0 / temperature, u,
                              greedy_epsilon, None if eps_u is None else eps_u[k], None if rand_act is None else rand_act[k],
                              root_index_offset)
        outs, actions, dist, prob, entropy = plan.finish_turns()
        return AgentTurnsOutput(actions, dist, prob, entropy, [_output_from_readout(r) for r in outs])

    # ---- SURVEY 8(e) + 8(f): the per-agent loop of one environment step with the roots sharded over the ranks, ONE exchange ------
    def search_agents_sharded(self, model, network_output, true_num_agents: int, total_roots: int, legal_actions_lst=None,
                              device=None, add_noise: bool = True, sampled_tau: float = 1.0, turn: str = "greedy",
                              temperature: float = 1.0, greedy_epsilon: float = 0.0, eps_randoms=None, group=None,
                              gather: bool = True) -> AgentTurnsOutput:
        """`search_agents` for a batch of `total_roots` roots split over the ranks of `group` (torch.distributed, NCCL).  This rank
        passes ITS contiguous slice `sharding.shard_range(total_roots, rank, world)` of every per-root argument (`network_output`,
        `legal_actions_lst`, and each (N, count) array of `eps_randoms`) and runs all N turns on it with no exchange: agent k+1's
        `factor` for a root depends only on that root's own trees.  After the last turn ONE all-gather of the whole step buffer
        (every agent's readouts + the turn results) gives every rank the AgentTurnsOutput of all roots in global order.
        Every rank must hold `np_random` in the same state: each draws what single-process `search_agents` over `total_roots`
        roots would draw and keeps its slice, so the result and the final generator state do not depend on the number of ranks.
        gather=False returns the local slice only (no collective)."""
        import torch.distributed as dist

        from . import sharding

        world, rank = dist.get_world_size(group), dist.get_rank(group)
        plan, count = self._search_agents_rank(model, network_output, true_num_agents, total_roots, rank, world, legal_actions_lst,
                                               device, add_noise, sampled_tau, turn, temperature, greedy_epsilon, eps_randoms)
        if not gather or world == 1:
            return _local_agent_turns(plan, count)
        gbuf, ghost = plan.turn_gather_buffers(world)
        dist.all_gather_into_tensor(gbuf, plan.res_flat, group=group)              # the one collective of the environment step
        ghost.copy_(gbuf, non_blocking=True)
        plan.tree.check()
        outs, t = sharding.merge_turn_shards(ghost.numpy().reshape(world, -1), plan.turn_layout(), total_roots, world)
        return AgentTurnsOutput(t["turn_actions"], t["policy_dist"], t["prob_prod"], t["entropy"], [_output_from_readout(r) for r in outs])

    def _search_agents_rank(self, model, network_output, true_num_agents, total_roots, rank, world, legal_actions_lst=None,
                            device=None, add_noise=True, sampled_tau=1.0, turn="greedy", temperature=1.0, greedy_epsilon=0.0,
                            eps_randoms=None):
        """The body of `search_agents_sharded` on rank `rank` of `world`, with no collective and no host sync: the N turns of
        this rank's slice, padded to the largest shard, are enqueued on the plan's stream.  Returns (plan, local root count);
        the step's results land in `plan.res_flat`."""
        from . import sharding

        cfg = self.config
        N, A = int(true_num_agents), cfg.action_space_size
        inf = self._device_inference(model, device)
        if inf is None:
            raise RuntimeError("search_agents_sharded needs a network with a device path (SMAC / matrix MAMuZeroNet on a CUDA device)")
        if turn not in ("greedy", "sample"):
            raise ValueError(turn)
        start, count = sharding.shard_range(total_roots, rank, world)
        Bp = sharding.shard_range(total_roots, 0, world)[1]               # the largest shard: every rank searches Bp roots
        if count == 0:
            raise ValueError(f"{total_roots} roots cannot be split over {world} ranks")
        eps_u, rand_act = (None, None) if eps_randoms is None else eps_randoms
        for x in (network_output.hidden_state, legal_actions_lst):
            if x is not None and x.shape[0] != count:
                raise ValueError(f"rank {rank}: expected {count} local roots, got {x.shape[0]}")
        for x in (eps_u, rand_act):
            if x is not None and tuple(np.shape(x)) != (N, count):
                raise ValueError(f"rank {rank}: expected {count} local roots, got eps_randoms of shape {tuple(np.shape(x))}")
        pad = lambda x: None if x is None else sharding.pad_rows(x, Bp)
        noise_epsilon = cfg.root_exploration_fraction if add_noise else 0.0
        plan = self._plan(inf, Bp, 0, sampled_tau)
        plan.stage_roots(pad(network_output.hidden_state), pad(network_output.reward), pad(network_output.value),
                         pad(network_output.policy_logits), pad(legal_actions_lst))
        plan.begin_turns()
        mine = slice(start, start + count)
        for k in range(N):       # np_random is consumed as single-process search_agents over total_roots roots consumes it
            noises = hostrng.dirichlet_f32(self.np_random, cfg.root_dirichlet_alpha, A, total_roots).reshape(total_roots, 1, A)
            seed = self.np_random.choice(256)
            u = self.np_random.random_sample(total_roots)[mine] if turn == "sample" else None
            if self.speculate_noise:   # the next agent's noise draw overlaps this turn's enqueue (used only if np_random is untouched)
                hostrng.speculate(self.np_random, cfg.root_dirichlet_alpha, A, total_roots)
            plan.enqueue_turn(k, 1 if turn == "sample" else 0, int(seed), cfg, noise_epsilon, pad(noises[mine]), 1.0 / temperature,
                              pad(u), greedy_epsilon, None if eps_u is None else pad(np.asarray(eps_u[k])),
                              None if rand_act is None else pad(np.asarray(rand_act[k])), root_index_offset=start)
        return plan, count

    # ---- reference simulation loop with the CUDA tree (any BaseNet) --------------------------------------------
    def _search_step_path(self, model, network_output, cur, factor, true_num_agents, device, sampled_tau, seed,
                          noise_epsilon, batch_rewards, batch_values, probs, beta, noises, root_index_offset):
        cfg = self.config
        A, K = cfg.action_space_size, cfg.sampled_action_times
        joint = cur is None
        Nt = true_num_agents if joint else 1
        B = network_output.hidden_state.shape[0]
        hidden_states_pool = [network_output.hidden_state]
        dev_index = None
        if device is not None and torch.device(device).type == "cuda":
            dev_index = torch.device(device).index or 0
        trees = cytree.Tree_batch(B, Nt, A, K, cfg.num_simulations, cfg.tree_value_stat_delta_lb, seed, cfg.mcts_rho,
                                  cfg.mcts_lambda, device=dev_index, root_index_offset=root_index_offset)
        trees.prepare(batch_rewards, batch_values, probs, beta, K, noise_epsilon, noises)
        with torch.no_grad():
            if hasattr(model, "eval"):
                model.eval()
            for index_simulation in range(cfg.num_simulations):
                ix, iy, batch_actions = trees.batch_selection(cfg.pb_c_base, cfg.pb_c_init, cfg.discount)
                hs = torch.vstack([hidden_states_pool[x][y] for x, y in zip(ix, iy)])
                if joint:
                    joint_action = batch_actions.astype(np.int32)
                else:
                    joint_action = np.zeros((B, true_num_agents), dtype=np.int32)
                    if factor is not None:
                        for k in range(cur):
                            joint_action[:, k] = factor[:, k]
                    joint_action[:, cur] = batch_actions.squeeze()
                    if cur + 1 < true_num_agents:
                        prior_logits, _ = model.prediction(hs)
                        if isinstance(prior_logits, torch.Tensor):
                            prior_logits = prior_logits.cpu().numpy()
                        for k in range(cur + 1, true_num_agents):
                            joint_action[:, k] = np.argmax(prior_logits[:, k, :], axis=-1)
                out = model.recurrent_inference(hs, torch.from_numpy(joint_action).to(device))
                hidden_states_pool.append(out.hidden_state)
                host = lambda x: x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
                pl = host(out.policy_logits)
                pl = pl.reshape(B, Nt, A) if joint else pl[:, cur, :].reshape(B, 1, A)
                p = _softmax_np(pl)
                b = p ** (1 / sampled_tau)
                b = b / np.sum(b, axis=-1, keepdims=True)
                trees.batch_expansion_and_backup(index_simulation + 1, cfg.discount, K,
                                                 host(out.reward).reshape(B).astype(np.float32),
                                                 host(out.value).reshape(B).astype(np.float32),
                                                 p.astype(np.float32), b.astype(np.float32))
        return _output_from_readout(trees.readout(cfg.discount))
