#!/usr/bin/env python
"""bench.py -- MCTS simulations/second of the batched sampled-MCTS hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 3m] [--mode joint|seq] [--impl ours|reference]
                    [--total-roots T] [--legal-frac 0.7] [--no-extras] [--dump-outputs DIR]

A "step" is ONE whole search of the workload: B roots x S simulations (root preparation -> tree construction -> S x [select ->
gather hidden -> recurrent_inference -> softmax/beta -> expand+backup] -> 13 readouts).  Default workload is BASELINE.json
configs[1]: SMAC 3m-shaped, 3 agents x 9 actions, 1024 roots x 50 sims, K = 10 sampled joint actions, synthetic root hidden
states and random-init weights of the reference architecture.

`value`   device-resident throughput: every input already in HBM (root hidden states, reward / value / logits, noise), the
          readouts left in HBM; the step is the library's whole search (`maz_search_run_dev`: root-preparation kernel, seeding,
          prepare, the simulation loop, readout kernel); CUDA events on the launching stream.
`e2e`     the same metric through the public API a worker calls (`SampledMCTS.batch_search`) with HOST buffers: host noise draw,
          H2D of the root tensors from pinned memory, the search, D2H of all readouts; wall clock after a device sync.
`roofline`       the dominant kernel (the persistent search kernel `k_search_persistent`, one launch per search; or the fused
                 inference kernel of the graph strategy) against the measured sustained bf16 peak, timed with CUDA events
                 inside the library around that launch alone.
`roofline_tree`  the tree step against the measured HBM copy peak.
`cpu_baseline`, `cpu_baseline_ctree_only`, `reference_native`: the three baselines of BASELINE.md section 3 on this box.
`--impl reference` times the reference's CPU path alone (the reference arm).
N > 1: roots sharded by rank (weak scaling by default, `--total-roots` = strong scaling), ONE all-gather of the packed readouts per
search (`SampledMCTS.batch_search_sharded` is the product entry; the device-resident step issues the same collective).
`--dump-outputs DIR` writes the readouts of the last timed device-resident search (rank 0's roots) as DIR/<name>.npy: the inputs
depend only on the arguments, so two builds can be compared output for output.

libmaz_b200.so is rebuilt only when it is missing or older than its sources, and the CPU checker (oracle/) is loaded as built,
compiled only when missing: on a tree that `__graft_entry__.build()` has built, the benchmark compiles and writes nothing, so
that tree may be read-only.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_JSON_FD = None     # set when fd 1 has been redirected (multi-rank runs)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


METRIC = "mcts_sims_per_sec"
UNIT = "root-sims/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="3m")
    ap.add_argument("--mode", default="joint", choices=["joint", "seq"])
    ap.add_argument("--roots", type=int, default=0, help="override roots per GPU")
    ap.add_argument("--total-roots", type=int, default=0, help="strong scaling: total roots, split over the ranks")
    ap.add_argument("--sims", type=int, default=0, help="override simulations")
    ap.add_argument("--legal-frac", type=float, default=0.0, help="random legal-action mask with this fraction legal (0 = all legal)")
    ap.add_argument("--strategy", default="auto", choices=["auto", "persistent", "graph", "legacy"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sequential-mode / legal-mask / other-config legs")
    ap.add_argument("--inference", default="bf16", choices=["bf16", "fp32"], help="bf16 = fused kernels, fp32 = parity mode")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the readouts of the last timed search as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


DUMP_LIMIT = 64 << 20


def dump_outputs(path, out, limit=DUMP_LIMIT):
    """Write the readouts of one search (`out`: name -> device tensor with the roots along dim 0) as path/<name>.npy in float32
    (the integer readouts -- counts, actions -- are exact in float32).  When all roots would take more than `limit` bytes, a fixed
    sample of roots (seed 0, in root order) is written, and its root indices as root_index.npy (float64)."""
    arrs = {k: v.cpu().numpy().astype(np.float32) for k, v in out.items()}
    B = len(arrs["value"])
    hdr = 128 * (len(arrs) + 1)                                    # one .npy header per file
    per_root = sum(a[0].nbytes for a in arrs.values())
    if B * per_root + hdr > limit:
        keep = np.sort(np.random.RandomState(0).choice(B, (limit - hdr) // (per_root + 8), replace=False))
        arrs = {k: a[keep] for k, a in arrs.items()}
        arrs["root_index"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(path, k + ".npy"), a)


def workload(args, world=1):
    from mazero_b200.synthetic import WORKLOADS

    N, A, B, S, K = WORKLOADS[args.workload]
    if args.roots:
        B = args.roots
    if args.total_roots:
        assert args.total_roots % world == 0, "--total-roots must be a multiple of the number of ranks"
        B = args.total_roots // world
    if args.sims:
        S = args.sims
    return N, A, B, S, K


def config_dict(args, N, A, B, S, K):
    """The workload description shared by BOTH arms (the driver compares the two lines' `config`)."""
    return {"workload": f"{args.workload}-shaped: {N} agents x {A} actions, {B} roots per step and GPU x {S} sims, K={K}, {args.mode} mode",
            "roots_per_gpu": B, "sims": S, "sampled_times": K, "mode": args.mode}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops_sustained)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


# algorithmic FLOPs of one recurrent_inference per root (SURVEY.md 8d / BASELINE.md section 4)
FLOP_PER_ROOT = {"3m": 2.61e6, "2s3z": 4.36e6, "mmm2": 8.81e6, "27m": 24.41e6}


def tree_bytes_per_root_sim(Nt, A, dbar, cbar):
    """algorithmic bytes of one tree step (SURVEY.md 8d):
    expansion + backup: 8 + 8*N*A  reward, value, probs, beta in;  16 + C*(4N + 36)  leaf header + per-child fields;
                        40*(d+1)   visit, wsum/wtot r/w, value-log append, min-max entry r/w
    selection:          d*(16 + 20*C) parent header + per-child prior, visit, reward, wsum, wtot;  4*(2+N) idx, idy, act"""
    return 8 + 8 * Nt * A + 16 + cbar * (4 * Nt + 36) + 40 * (dbar + 1) + dbar * (16 + 20 * cbar) + 4 * (2 + Nt)


class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                       "-lms", "20", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                out["sm_max_mhz"] = float(r[1])
                for n, v in zip(names, r[2:6]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------ CPU / reference baselines
def _reference_model(N, A, sd, device="cpu"):
    from oracle.model_oracle import OracleMAMuZeroNet

    return OracleMAMuZeroNet(N, A).load_reference_state_dict(sd).eval().to(device)


def cpu_reference_search(args, N, A, B, S, K, sd, hidden, steps, warmup, device="cpu"):
    """The reference's path restated (oracle/search_oracle.py = mcts_sampled.py:34-200 line by line, pinned to the reference's own
    driver by tests/test_reference_driver_cpu.py) over the reference's OWN C++ tree compiled into oracle/_ref (else the C port),
    with the same weights.  device="cpu": everything on the host (BASELINE.md 3-ii).  device="cuda": the reference's native
    deployment (3-iii): CPU tree, network on the GPU under autocast, per-simulation host<->device round trips
    (mcts_sampled.py:130-156)."""
    import torch
    from mazero_b200.synthetic import SearchConfig
    from oracle import pyoracle
    from oracle.model_oracle import inverse_support_transform
    from oracle.search_oracle import NetworkOutput, reference_batch_search

    kind = "reference" if pyoracle.available("reference") else "port"
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = _reference_model(N, A, sd, device)
    cfg = SearchConfig(A, S, K)
    hidden = hidden.float().to(device)
    with torch.no_grad():
        pol, vlog = model.prediction(hidden)
        value = inverse_support_transform(vlog, -5, 5)
    out0 = NetworkOutput(hidden, np.zeros((B, 1), np.float32), value.cpu().numpy(), pol.cpu().numpy())
    cur = None if args.mode == "joint" else 0
    rs = np.random.RandomState(1)
    times = []
    for i in range(warmup + steps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        if device != "cpu":
            with torch.autocast("cuda", dtype=torch.float16):          # the reference's `with autocast():` (:136,150)
                reference_batch_search(cfg, rs, model, out0, cur, None, N, None, device, add_noise=True, tree_kind=kind)
            torch.cuda.synchronize()
        else:
            reference_batch_search(cfg, rs, model, out0, cur, None, N, None, "cpu", add_noise=True, tree_kind=kind)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return float(np.mean(times)), kind, cores


def cpu_ctree_only(N, A, B, S, K, joint, steps=2, warmup=1):
    """BASELINE.md 3-i: the compiled reference tree alone (prepare + S x [selection, expansion+backup] + readouts) with
    pre-generated network outputs, single-threaded by construction (cnode.cpp:563)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _harness import MCTS, Inputs, drive
    from oracle import pyoracle

    kind = "reference" if pyoracle.available("reference") else "port"
    Nt = N if joint else 1
    inp = Inputs(B, Nt, A, S, seed=0, mode="random")
    times = []
    for i in range(warmup + steps):
        t = pyoracle.OracleTreeBatch(B, Nt, A, K, S, MCTS["delta_lb"], 11 + i, MCTS["rho"], MCTS["lam"], kind=kind)
        t0 = time.perf_counter()
        drive(t, inp, K, record_steps=False)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return float(np.mean(times)), kind


def run_reference_arm(args):
    import torch
    from mazero_b200.synthetic import random_state_dict, root_hidden

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    N, A, B, S, K = workload(args, world)
    # bounded sample of the workload: at most 1024 roots per step (the full 3m configuration)
    Bs = min(B, 1024)
    sd = random_state_dict(N, A, seed=0)
    hidden = root_hidden(Bs, N, seed=0)
    sec, kind, cores = cpu_reference_search(args, N, A, Bs, S, K, sd, hidden, args.steps, args.warmup)
    val = Bs * S / sec
    sample = (f"{Bs} roots x {S} sims per step, {args.steps} steps; the reference's own C++ tree ({kind}: oracle/_ref, single-threaded by "
              f"construction) + its Python loop and network restated (oracle/search_oracle.py, model_oracle.py) on torch CPU, {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong" if args.total_roots else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, N, A, B, S, K),
        "details": {"sample_roots": Bs},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
class Problem:
    """One workload on this rank: weights, plan (native search handle + staging), NSETS synthetic input batches resident in HBM
    and mirrored on the host."""

    def __init__(self, args, name, N, A, B, S, K, dev, rank, cur, legal_frac=0.0, nsets=5, strategy="auto", inference="bf16"):
        import torch
        from mazero_b200.inference import SmacInference
        from mazero_b200.mcts_sampled import SampledMCTS
        from mazero_b200.synthetic import NetworkOutput, SearchConfig, random_state_dict, root_hidden

        self.name, self.N, self.A, self.B, self.S, self.K, self.dev, self.rank, self.cur = name, N, A, B, S, K, dev, rank, cur
        self.Nt = N if cur is None else 1
        self.cfg = SearchConfig(A, S, K)
        self.sd = random_state_dict(N, A, seed=0)
        self.inf = SmacInference(self.sd, N, A, device=dev, mode=inference)
        self.mcts = SampledMCTS(self.cfg, np.random.RandomState(1), search_strategy=strategy)
        self.nsets = nsets
        base_seed = int(os.environ.get("MAZ_BENCH_SEED", "0"))
        self.root_off = rank * B                        # global index of this rank's first root (tree RNG seeding, cnode.cpp:574)
        self.legal = None
        if legal_frac > 0:
            rng = np.random.RandomState(17 + rank)
            self.legal = (rng.rand(B, N, A) < legal_frac).astype(np.float32)
            self.legal[..., 1] = 1.0                    # action 1 always legal (SURVEY 8d)
        self.host, self.devs = [], []
        for k in range(nsets):
            self.host.append(self.make_inputs(base_seed + k + rank * nsets, pinned=True))
            h = self.host[-1]
            noise = np.random.RandomState(1000 + k + 31 * rank).dirichlet([0.3] * A, B * self.Nt).astype(np.float32).reshape(B, self.Nt, A)
            to = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
            self.devs.append(dict(hidden=h.hidden_state.to(dev), rewards=to(h.reward.reshape(B)), values=to(h.value.reshape(B)),
                                  logits=to(h.policy_logits), noise=to(noise)))
        # builds the plan (library handle, staging buffers) through the public entry point
        first = self.api(0)
        assert int(first.marginal_visit_count[0, 0].sum()) == S
        self.plan = next(iter(self.mcts._plans.values()))
        if self.legal is not None:
            self.plan.inp["legal"].copy_(torch.from_numpy(self.legal).to(dev))
        self.NetworkOutput = NetworkOutput

    def make_inputs(self, seed, pinned=False, B=None):
        import torch
        from mazero_b200.synthetic import NetworkOutput, root_hidden

        B = self.B if B is None else B
        hidden_host = root_hidden(B, self.N, seed=seed, pinned=pinned)
        pol, vlog = self.inf.prediction(hidden_host.to(self.dev))
        value = self.inf._inv_transform(vlog, self.inf.vsup)
        return NetworkOutput(hidden_host, np.zeros((B, 1), np.float32), value.cpu().numpy().reshape(B, 1), pol.cpu().numpy())

    def api(self, i, cur="default"):
        """One search through the worker-facing entry point with HOST buffers."""
        cur = self.cur if cur == "default" else cur
        return self.mcts.batch_search(self.inf, self.host[i % self.nsets], cur, None, self.N, self.legal, self.dev, add_noise=True,
                                      root_index_offset=self.root_off)

    def dev_step(self, i, seed=None):
        """One search with every input already in HBM: stage the i-th input set device-to-device, run the library's search."""
        p, d = self.plan, self.devs[i % self.nsets]
        p.pool[0].copy_(d["hidden"], non_blocking=True)
        p.inp["rewards"].copy_(d["rewards"], non_blocking=True)
        p.inp["values"].copy_(d["values"], non_blocking=True)
        p.inp["logits"].copy_(d["logits"], non_blocking=True)
        p.inp["noise_raw0"].copy_(d["noise"], non_blocking=True)
        p.has_legal = self.legal is not None
        p._enqueue_search(0, self.cur, 100 + i if seed is None else seed, self.cfg, self.cfg.root_exploration_fraction, self.root_off)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from mazero_b200 import build
    build.build()
    from mazero_b200.mcts_sampled import clear_caches
    from mazero_b200.synthetic import WORKLOADS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- mazero_b200 has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL printf()s its version banner to fd 1 at communicator creation, so fd 1 is
        # pointed at stderr for the whole run and the JSON line goes to a saved copy of the original stdout
        sys.stdout.flush()
        global _JSON_FD
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)

    N, A, B, S, K = workload(args, world)
    cur = None if args.mode == "joint" else 0
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    steps, warm = args.steps, max(args.warmup, 3)

    def timed(fn, n, w, wall=False):
        """n timed calls after w warm-up calls, barrier + synchronize on both sides, L2 flushed before every call; CUDA events on
        the launching stream (wall=False) or wall clock around calls that synchronise themselves (wall=True); max over ranks."""
        for i in range(w):
            fn(i)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        evs, walls = [], []
        for i in range(n):
            flush.zero_()
            if wall:
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                fn(w + i)
                torch.cuda.synchronize(dev)
                walls.append((time.perf_counter() - t0) * 1e3)
            else:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                fn(w + i)
                b.record(stream)
                evs.append((a, b))
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = float(np.mean(walls)) if wall else float(np.mean([a.elapsed_time(b) for a, b in evs]))
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    prob = Problem(args, args.workload, N, A, B, S, K, dev, rank, cur, legal_frac=args.legal_frac, strategy=args.strategy,
                   inference=args.inference)
    plan, cfg, inf = prob.plan, prob.cfg, prob.inf
    native = plan.native
    strategy = native.strategy if native is not None else "legacy"

    # ---- the exchange of the multi-GPU path: ONE all-gather of the packed readouts per search, on its own stream so that the
    # collective of search i overlaps search i+1 (it needs every rank to arrive: run synchronously it would add the rank skew
    # of every search to the step).  Each timed step contains the wait for the previous step's exchange.
    class Exchange:
        def __init__(self, on):
            self.on = on and world > 1
            if self.on:
                self.gather, _ = plan.gather_buffers(world)
                self.comm = torch.cuda.Stream(dev)
                self.ready, self.done = torch.cuda.Event(), torch.cuda.Event()
                self.done.record(stream)

        def before_readout(self):
            if self.on:
                stream.wait_event(self.done)               # the previous search's readouts have been sent

        def after_search(self):
            if self.on:
                self.ready.record(stream)
                with torch.cuda.stream(self.comm):
                    self.comm.wait_event(self.ready)
                    dist.all_gather_into_tensor(self.gather, plan.out_flat)
                    self.done.record(self.comm)

    def make_dev_step(ex):
        def step(i):
            ex.before_readout()
            prob.dev_step(i)
            ex.after_search()
        return step

    sampler = ClockSampler(local) if rank == 0 else None
    ex = Exchange(True)
    ms_dev = timed(make_dev_step(ex), steps, warm)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, plan.out)        # before any further search overwrites the readouts
    # a default run times 10 short searches: shorter than nvidia-smi's start-up.  Keep the GPU under the same load (untimed
    # steps, the same number on every rank) until ~0.4 s have passed, so that the clocks are sampled under load.
    extra = int(max(0.0, 0.4 - steps * ms_dev * 1e-3) / (ms_dev * 1e-3)) + 1
    for i in range(extra):
        make_dev_step(ex)(1000 + i)
    torch.cuda.synchronize(dev)
    clocks = sampler.stop() if sampler else None
    plan.tree.check()
    ms_nogather = None
    if world > 1:                                          # A/B: the same steps without the exchange (what limits scaling?)
        ms_nogather = timed(make_dev_step(Exchange(False)), steps, warm)

    # ---- gather check: rank 0 recomputes ANOTHER rank's shard alone (same inputs, same global root offset) and compares it bit
    # for bit with what the all-gather delivered
    gather_check = None
    if world > 1:
        torch.cuda.synchronize(dev)
        dist.barrier()
        ex2 = Exchange(True)
        step = make_dev_step(ex2)
        step(7)                                            # every rank: input set 7 % nsets, tree seed 107
        torch.cuda.synchronize(dev)
        dist.barrier()
        if rank == 0:
            peer = world - 1
            got = ex2.gather.view(world, -1)[peer].clone()
            saved_off, saved_devs = prob.root_off, prob.devs
            other = Problem(args, args.workload, N, A, B, S, K, dev, peer, cur, legal_frac=args.legal_frac, strategy=args.strategy,
                            inference=args.inference)     # regenerates rank `peer`'s synthetic inputs (seeded by rank)
            other.dev_step(7)
            torch.cuda.synchronize(dev)
            gather_check = "ok" if torch.equal(other.plan.out_flat, got) else "MISMATCH"
            del other
        dist.barrier()

    # ---- end to end through the public API with host buffers (pinned hidden state, numpy everything else); wall clock
    ms_e2e = timed(lambda i: prob.api(i), steps, warm, wall=True)
    h2d = prob.host[0].hidden_state.numel() * 4 + 4 * plan.in_turn[0][1]      # root hidden state + the pinned staging block
    d2h = plan.out_flat.numel() * 4

    # ---- roofline of the dominant kernel: CUDA events INSIDE the library around the simulation loop only
    hbm_peak, bf16_peak, peak_src = peaks()
    roofline = tree_roof = None
    tot_nodes, last_len, sum_len, sum_exp = plan.tree.stats()
    dbar = sum_len / float(B * S)
    cbar = float((tot_nodes.sum() - B)) / float(sum_exp)
    bytes_tree = B * tree_bytes_per_root_sim(prob.Nt, A, dbar, cbar)          # per simulation, all trees of this GPU
    if native is not None:
        native.set_timing(True)
        clk = torch.zeros(2 * S + 4 * (B + 8) + 64 + 4 * B, dtype=torch.int64, device=dev)
        native.set_debug_clock(clk if strategy == "persistent" else None)
        loop_ms = []
        for i in range(5):
            flush.zero_()
            prob.dev_step(50 + i)
            loop_ms.append(native.loop_ms())
        native.set_timing(False)
        native.set_debug_clock(None)
        loop = float(np.mean(loop_ms[1:]))
        flop = B * S * FLOP_PER_ROOT.get(args.workload, 0.0)
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp))
        if strategy == "persistent":
            rpc = native.roots_per_cta()
            ncta = (B + rpc - 1) // rpc
            c = clk.cpu().numpy()
            per = c[2 * S:2 * S + 4 * ncta].reshape(ncta, 4).astype(np.float64)
            share_tree = float(per[:, 3].sum() / max(per[:, 0].sum(), 1.0))      # tree-step share of the CTAs' cycles
            roofline = {"bound": "tensor", "kernel": "k_search_persistent", "achieved": flop / (loop * 1e-3) / 1e12, "peak": bf16_peak,
                        "unit": "TFLOP/s", "frac": flop / (loop * 1e-3) / 1e12 / bf16_peak,
                        "traffic": traffic.get(f"k_search_persistent:{args.workload}:{args.mode}"),
                        "peak_source": peak_src, "algorithmic_flop_per_launch": flop, "launch_ms": loop, "launches_per_search": 1,
                        "ctas": ncta, "roots_per_cta": rpc,
                        "cta_cycles": {"mean": float(per[:, 0].mean()), "max": float(per[:, 0].max()),
                                       "inference_per_sim": float(per[:, 2].mean() / S), "tree_per_sim": float(per[:, 3].mean() / S)},
                        "note": "ONE launch = the whole search (S x [fused recurrent_inference on warp-level bf16 MMAs + tree step]); "
                                "the kernel is a dependent chain per CTA (latency-bound), not tensor-throughput-bound: DESIGN.md section 5"}
            tree_ms = loop * share_tree
            tree_roof = {"bound": "hbm", "kernel": "k_search_persistent (tree-step phases)", "achieved": bytes_tree * S / (tree_ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": bytes_tree * S / (tree_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_tree * S, "launch_ms": tree_ms,
                         "note": "share of the persistent kernel's CTA cycles spent in the tree step (in-kernel cycle counters) x its duration"}
        else:
            # graph strategy: 2 S launches; time the inference kernel and the tree kernel alone (eager, behind a GPU sleep)
            ms_inf, ms_tree = time_graph_kernels(prob, dev, stream)
            fl = B * FLOP_PER_ROOT.get(args.workload, 0.0)
            from mazero_b200 import fused as _fused
            small = _fused.use_small(B, N)
            kname = "k_recurrent_inference_small" if small else ("k_recurrent_inference_twin" if _fused.use_twin(B, N) else "k_recurrent_inference")
            roofline = {"bound": "tensor", "kernel": kname, "achieved": fl / (ms_inf * 1e-3) / 1e12, "peak": bf16_peak, "unit": "TFLOP/s",
                        "frac": fl / (ms_inf * 1e-3) / 1e12 / bf16_peak, "traffic": traffic.get(f"{kname}:{args.workload}:{args.mode}"),
                        "peak_source": peak_src, "algorithmic_flop_per_launch": fl, "launch_ms": ms_inf, "launches_per_search": S,
                        "loop_ms": loop}
            tree_roof = {"bound": "hbm", "kernel": "k_expand_backup_select2", "achieved": bytes_tree / (ms_tree * 1e-3) / 1e9, "peak": hbm_peak,
                         "unit": "GB/s", "frac": bytes_tree / (ms_tree * 1e-3) / 1e9 / hbm_peak,
                         "traffic": traffic.get(f"k_expand_backup_select2:{args.workload}:{args.mode}"), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_tree, "launch_ms": ms_tree}

    extras = {}
    if not args.no_extras:
        # ---- the fork's sequential-agent mode (what the workers call): one environment step = N per-agent searches
        # (selfplay_worker.py:196-257, reanalyze_worker.py:278-327).  (a) the workers' loop over N batch_search calls with the
        # host choosing each agent's action in between; (b) SampledMCTS.search_agents: the same N searches back to back on
        # the device, one sync.
        seq = prob if cur is not None else Problem(args, args.workload, N, A, B, S, K, dev, rank, 0, strategy=args.strategy,
                                                   inference=args.inference)
        ms_seq = timed(lambda i: seq.dev_step(i), max(3, steps // 2), 3)

        def loop_step(i):
            acts = np.zeros((B, N), dtype=np.int32)
            for k in range(N):
                o = seq.mcts.batch_search(seq.inf, seq.host[i % seq.nsets], k, acts[:, :k].copy() if k else None, N, None, dev,
                                          add_noise=True, root_index_offset=seq.root_off)
                acts[:, k] = np.argmax(o.marginal_visit_count[:, 0, :], axis=-1)      # reanalyze_worker.py:309

        def fused_step(i):
            seq.mcts.search_agents(seq.inf, seq.host[i % seq.nsets], N, None, dev, add_noise=True, turn="greedy",
                                   root_index_offset=seq.root_off)

        fused_step(0)
        ms_loop = timed(loop_step, max(3, steps // 2), 3, wall=True)
        ms_fused = timed(fused_step, max(3, steps // 2), 3, wall=True)
        extras["sequential_mode"] = {
            "unit": UNIT, "agents": N, "value": world * B * S / (ms_seq * 1e-3), "ms_per_search": ms_seq,
            "what": "one search of agent 0 in the fork's sequential-agent mode (tree agent_num = 1, later agents greedy), device-resident"}
        extras["e2e_agent_turns"] = {
            "unit": UNIT, "agents": N, "host_loop": world * B * S * N / (ms_loop * 1e-3), "host_loop_ms": ms_loop,
            "search_agents": world * B * S * N / (ms_fused * 1e-3), "search_agents_ms": ms_fused,
            "what": "one environment step = N per-agent searches, host buffers; host_loop = N x batch_search with the action choice on "
                    "the host, search_agents = one device-resident call (one host sync)"}
        if seq is not prob:
            del seq
        # ---- the 70 %-legal-mask run of SURVEY 8d (the timed configuration has every action legal)
        if args.legal_frac == 0:
            lm = Problem(args, args.workload, N, A, B, S, K, dev, rank, cur, legal_frac=0.7, strategy=args.strategy, inference=args.inference)
            ms_lm = timed(lambda i: lm.dev_step(i), max(3, steps // 2), 3)
            ms_lm_e2e = timed(lambda i: lm.api(i), max(3, steps // 2), 3, wall=True)
            extras["legal_mask_70"] = {"unit": UNIT, "value": world * B * S / (ms_lm * 1e-3), "ms_per_step": ms_lm,
                                       "e2e": world * B * S / (ms_lm_e2e * 1e-3), "legal_fraction": float(lm.legal.mean())}
            del lm
        # ---- the other BASELINE configurations on the SAME number of GPUs (compact): roots sharded over the ranks
        if args.workload == "3m" and not args.roots and not args.total_roots and not args.sims and os.environ.get("MAZ_BENCH_OTHER", "1") != "0":
            del prob, plan
            clear_caches()
            torch.cuda.empty_cache()
            others = {}
            for name in ("2s3z", "mmm2", "27m"):
                n2, a2, b2, s2, k2 = WORKLOADS[name]
                if b2 % world:
                    continue
                bl = b2 // world
                o = Problem(args, name, n2, a2, bl, s2, k2, dev, rank, None, nsets=2, strategy=args.strategy, inference=args.inference)
                gbuf, _ = o.plan.gather_buffers(world) if world > 1 else (None, None)

                def ostep(i, o=o, gbuf=gbuf):
                    o.dev_step(i)
                    if gbuf is not None:
                        dist.all_gather_into_tensor(gbuf, o.plan.out_flat)

                ms_o = timed(ostep, 2, 3)
                ms_oe = timed(lambda i, o=o: o.api(i), 2, 3, wall=True)
                nat = o.plan.native
                nat.set_timing(True)
                ostep(9)
                loop_o = nat.loop_ms()
                nat.set_timing(False)
                others[name] = {"roots_total": b2, "roots_per_gpu": bl, "sims": s2, "ranks": world, "value": b2 * s2 / (ms_o * 1e-3),
                                "ms_per_step": ms_o, "e2e": b2 * s2 / (ms_oe * 1e-3), "strategy": nat.strategy,
                                "tensor_frac": bl * s2 * FLOP_PER_ROOT[name] / (loop_o * 1e-3) / 1e12 / bf16_peak,
                                "scaling": "strong (BASELINE total roots split over the ranks)" if world > 1 else "single GPU"}
                del o
                clear_caches()
                torch.cuda.empty_cache()
            extras["other_configs"] = others

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_sims = world * B * S
    launches_per_search = 5 if strategy == "persistent" else 4 + (2 if inf.fused is not None else 1) * S
    line = {
        "metric": METRIC, "value": total_sims / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong" if args.total_roots else "weak",
        "vs_baseline": None, "dtype": "bf16" if inf.fused is not None else "f32", "data": "synthetic",
        "config": config_dict(args, N, A, B, S, K),
        "details": {"tree_agents": N if cur is None else 1, "inference": inf.mode, "search_strategy": strategy,
                    "l2": "flushed (256 MiB memset) between timed steps",
                    "inputs": "5 synthetic batches of root hidden states rotated per step (rank offset)",
                    "legal_mask": args.legal_frac or "all legal", "mean_search_depth": dbar, "mean_children": cbar,
                    "parallelism": f"roots sharded x{world}",
                    **({"exchange": "one all_gather of the packed readouts per search (NCCL), overlapped with the next search",
                        "ms_per_step_without_exchange": ms_nogather, "gather_check": gather_check} if world > 1 else {})},
        "e2e": {"value": total_sims / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e, "api": "SampledMCTS.batch_search (host numpy + pinned hidden state); wall clock"},
        # our kernels per search: k_root_prepare, k_seed, k_prepare, the persistent search kernel (or k_select + per simulation the
        # fused inference kernel and the tree kernel), k_readout
        "gpu_launches": int(steps * launches_per_search),
        "clocks": clocks,
        "roofline": roofline,
        "roofline_tree": tree_roof,
    }
    if world > 1:
        line["gather_check"] = gather_check
    line.update(extras)
    if not args.no_cpu_baseline and world == 1:
        from mazero_b200.synthetic import random_state_dict, root_hidden
        sd = random_state_dict(N, A, seed=0)
        Bs = min(B, 1024)
        # (ii) the reference's full CPU path; (i) its compiled tree alone; (iii) its native deployment: CPU tree + network on this GPU
        sec, kind, cores = cpu_reference_search(args, N, A, Bs, S, K, sd, root_hidden(Bs, N, seed=0), 2, 1)
        line["cpu_baseline"] = {"value": Bs * S / sec, "unit": UNIT, "cores": cores, "kind": kind,
                                "sample": f"{Bs} roots x {S} sims, 2 timed searches after 1 warm-up; reference C++ tree ({kind}) single-threaded "
                                          f"+ restated Python loop / network on torch CPU, {cores} threads"}
        sec_t, kind_t = cpu_ctree_only(N, A, Bs, S, K, cur is None)
        line["cpu_baseline_ctree_only"] = {"value": Bs * S / sec_t, "unit": UNIT, "cores": 1, "kind": kind_t,
                                           "sample": f"{Bs} roots x {S} sims, tree only with pre-generated network outputs, 2 timed searches"}
        sec_n, kind_n, _ = cpu_reference_search(args, N, A, Bs, S, K, sd, root_hidden(Bs, N, seed=0), 2, 1, device=str(dev))
        line["reference_native"] = {"value": Bs * S / sec_n, "unit": UNIT, "kind": kind_n,
                                    "sample": f"{Bs} roots x {S} sims: reference tree on the CPU + the same network on this GPU under fp16 "
                                              "autocast, per-simulation H2D / D2H as mcts_sampled.py:130-156; 2 timed searches"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def time_graph_kernels(prob, dev, stream):
    """Graph strategy: average duration of the fused inference kernel and of the tree kernel (expand + backup + next selection),
    launched eagerly one by one through the per-step C ABI behind a GPU sleep (CUDA events around each launch)."""
    import torch
    from mazero_b200 import cytree

    cfg, inf, B, N, A, S, K, Nt = prob.cfg, prob.inf, prob.B, prob.N, prob.A, prob.S, prob.K, prob.Nt
    plan = prob.plan
    f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
    tree = cytree.Tree_batch(B, Nt, A, K, S, cfg.tree_value_stat_delta_lb, 7, cfg.mcts_rho, cfg.mcts_lambda, device=dev.index or 0)
    tree.set_puct(cfg.pb_c_base, cfg.pb_c_init)
    tree.set_stream(stream.cuda_stream)
    idx_x, idx_y, act = i32(B), i32(B), i32(B, Nt)
    r, v, p, b = f(B), f(B), f(B, Nt, A), f(B, Nt, A)
    tree.prepare(plan.inp["rewards"], plan.inp["values"], plan.root_p, plan.root_b, K, cfg.root_exploration_fraction, plan.root_n)
    tree_ev, inf_ev = [], []
    torch.cuda._sleep(int(2.0e8))
    tree.batch_selection_device(cfg.pb_c_base, cfg.pb_c_init, cfg.discount, idx_x, idx_y, act)
    n = min(S, 20)
    for s in range(n):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(stream)
        inf.recurrent_fused(B, plan.pool, idx_x, act, plan.pool[s + 1], r, v, p, b, None, None, Nt, -1, 1.0)
        e[1].record(stream)
        e[2].record(stream)
        tree.expansion_backup_selection_device(s + 1, cfg.discount, K, r, v, p, b, cfg.pb_c_base, cfg.pb_c_init, idx_x, idx_y, act)
        e[3].record(stream)
        inf_ev.append((e[0], e[1]))
        tree_ev.append((e[2], e[3]))
    torch.cuda.synchronize(dev)
    return float(np.mean([a.elapsed_time(b) for a, b in inf_ev])), float(np.mean([a.elapsed_time(b) for a, b in tree_ev]))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)
