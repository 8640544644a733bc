#!/usr/bin/env python
"""One environment step of the fork's sequential-agent mode (N per-agent searches) with the roots sharded over the GPUs:
`SampledMCTS.search_agents_sharded`, one all-gather of the whole step buffer per step.

    torchrun --nproc_per_node W profiles/prof_agents_sharded.py [--steps 3] [--warmup 1] [--turn greedy|sample]
                                                                [--configs 3m-weak,3m-strong,mmm2,27m] [--out FILE]
    python profiles/prof_agents_sharded.py ...          (one GPU: a one-rank gloo group, no exchange)

Rank 0 prints one JSON line per configuration (and appends it to FILE):
  step_ms        environment step, wall clock from a barrier to the end of the call (the call synchronises; a device sync
                 follows), mean over the timed steps, max over ranks;
  root_sims_per_s  total_roots * S * N / step time;
  loop_ms_per_rank the rank body alone (`_search_agents_rank`: the N turns of the rank's slice, no collective) to a device
                 sync, mean over the timed steps, one entry per rank;
  exchange_ms    step_ms minus the slowest rank body: the all-gather, the D2H copy of the gathered buffers and the merge;
  gather_check   rank 0 recomputes the last rank's shard alone from the same generator state and input batch, with the same
                 global root offset, and compares its step buffer word for word with the gathered block; the generator must
                 end in the same state.
Input batches (root hidden states and the prediction heads' logits / values of the random-init reference network) are
rotated per step (DESIGN section 7: search time depends on the inputs); they are generated for ALL roots from a seed and
sliced, so every rank count searches the same problem.  No legal mask (every action legal).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CONFIGS = {       # name -> (workload, roots: per GPU for weak scaling, total for strong)
    "3m-weak": ("3m", "weak"),
    "3m-strong": ("3m", "strong"),
    "mmm2": ("mmm2", "strong"),
    "27m": ("27m", "strong"),
}
NSETS = 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--turn", default="greedy", choices=["greedy", "sample"])
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch.distributed as dist

    from mazero_b200 import build
    build.build()
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.sharding import shard_range
    from mazero_b200.synthetic import WORKLOADS, NetworkOutput, SearchConfig, random_state_dict, root_hidden

    if not torch.cuda.is_available():
        raise SystemExit("prof_agents_sharded.py: no CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    else:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29500 + os.getpid() % 1000))
        dist.init_process_group("gloo", rank=0, world_size=1)       # the public entry resolves rank / world from a group
    gpu = card() if rank == 0 else None

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world == 1:
            return [x]
        out = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.tolist()

    for name in args.configs.split(","):
        wl, scaling = CONFIGS[name]
        N, A, B, S, K = WORKLOADS[wl]
        total = B * world if scaling == "weak" else B
        cfg = SearchConfig(A, S, K)
        inf = SmacInference(random_state_dict(N, A, seed=0), N, A, device=dev, mode="bf16")
        peer = world - 1

        def inputs(s, r):
            """input batch s, the slice of rank r (device tensors, as `inf.initial_inference` would leave them)"""
            start, count = shard_range(total, r, world)
            h = root_hidden(total, N, seed=s)[start:start + count].to(dev)
            pol, vlog = inf.prediction(h)
            value = inf._inv_transform(vlog, inf.vsup).reshape(count, 1)
            return NetworkOutput(h, torch.zeros(count, 1, device=dev), value, pol)

        sets = [inputs(s, rank) for s in range(NSETS)]
        mcts = SampledMCTS(cfg, np.random.RandomState(1))
        call = lambda i: mcts.search_agents_sharded(inf, sets[i % NSETS], N, total, None, dev, add_noise=True, turn=args.turn)
        for i in range(max(args.warmup, 1)):
            call(i)
        step_ms = []
        for i in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            call(args.warmup + i)
            torch.cuda.synchronize(dev)
            step_ms.append((time.perf_counter() - t0) * 1e3)
        loop_ms = []
        for i in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            mcts._search_agents_rank(inf, sets[i % NSETS], N, total, rank, world, None, dev, add_noise=True, turn=args.turn)
            torch.cuda.synchronize(dev)
            loop_ms.append((time.perf_counter() - t0) * 1e3)

        # ---- gather check: the last rank's shard recomputed alone on rank 0, compared with the gathered block
        barrier()
        state = mcts.np_random.get_state()
        out = call(7)
        plan = next(iter(mcts._plans.values()))          # the one sequential-agent plan of this shard size
        torch.cuda.synchronize(dev)
        got = plan.turn_gather_buffers(world)[0].view(world, -1)[peer].clone() if world > 1 else plan.res_flat.clone()
        check = None
        if rank == 0:
            rs = np.random.RandomState()
            rs.set_state(state)
            again = SampledMCTS(cfg, rs)
            p2, _ = again._search_agents_rank(inf, inputs(7 % NSETS, peer), N, total, peer, world, None, dev, add_noise=True,
                                              turn=args.turn)
            torch.cuda.synchronize(dev)
            same_rng = all(np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
                           for a, b in zip(rs.get_state(), mcts.np_random.get_state()))
            check = "ok" if torch.equal(p2.res_flat, got) and same_rng and out.actions.shape == (total, N) else "MISMATCH"
        barrier()

        step = max_over_ranks(float(np.mean(step_ms)))
        loops = gather_floats(float(np.mean(loop_ms)))
        if rank == 0:
            line = {"config": name, "workload": f"{wl}-shaped: {N} agents x {A} actions, K={K}, sequential-agent mode",
                    "scaling": scaling, "n_gpus": world, "total_roots": total, "roots_per_gpu": shard_range(total, 0, world)[1],
                    "sims": S, "agents": N, "turn": args.turn, "steps": args.steps, "warmup": max(args.warmup, 1),
                    "step_ms": step, "root_sims_per_s": total * S * N / (step * 1e-3),
                    "loop_ms_per_rank": loops, "exchange_ms": step - max(loops),
                    "step_ms_samples_rank0": step_ms, "gather_check": check,
                    "strategy": plan.native.strategy if plan.native is not None else "legacy",
                    "gather_bytes_per_rank": plan.res_flat.numel() * 4,
                    "inputs": f"{NSETS} batches rotated per step, generated for all roots and sliced; every action legal",
                    "gpu": gpu}
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
        del sets, mcts, plan, inf, call
        clear_caches()
        torch.cuda.empty_cache()
    barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
