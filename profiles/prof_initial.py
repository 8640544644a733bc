#!/usr/bin/env python
"""Root inference (`MAMuZeroNet.initial_inference`, config/smac/model.py:542-559): the fp32 path (`SmacInference(mode="fp32")
.initial_inference(obs)`: the row-wise representation kernel + ~25 torch ops for the heads) against the bf16 root-inference
kernel (`SmacInference(mode="bf16").initial_inference(obs, fused=True)`, csrc/infer_initial.cuh), per call.

    python profiles/prof_initial.py [--shapes 3m,2s3z,mmm2,27m,2c_vs_64zg] [--batches 8,64,1536] [--reps 5] [--out FILE]

One JSON line per (shape, B), also appended to FILE:
  fp32_us / fused_us   median over `reps` timed windows of the mean time per call (CUDA events around `iters` back-to-back
                       calls on one stream, after a warm-up of every shape); both include the output allocation the call makes;
  *_spread_us          max - min over the windows (the two paths alternate window by window);
  speedup              fp32_us / fused_us;
  err_*                max |fused - fp32| / max(1, max |fp32|) per output on the timed inputs (bf16 against fp32).
B = 8 and 64 are self-play sizes (one call per environment step), 1536 the reanalyze batch (B * (U + 1) roots).  obs_dim is
the per-agent observation size of the SMAC map.  Inputs are a few MB: they stay in L2 between calls, as in the workers.
Weights: the reference initialisation (oracle/model_oracle.py::init_like_reference)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OBS_DIM = {"3m": 30, "2s3z": 80, "mmm2": 176, "27m": 285, "2c_vs_64zg": 332}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def window(fn, iters):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1000.0 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=",".join(OBS_DIM))
    ap.add_argument("--batches", default="8,64,1536")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_initial.py needs a CUDA device")
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import WORKLOADS
    from oracle.model_oracle import OracleMAMuZeroNet

    dev = "cuda:0"
    gpu = card()
    for shape in args.shapes.split(","):
        N, A = WORKLOADS[shape][:2]
        obs = OBS_DIM[shape]
        sd = OracleMAMuZeroNet(N, A, obs_size=obs).init_like_reference(0).state_dict()
        f32 = SmacInference(sd, N, A, device=dev, mode="fp32")
        b16 = SmacInference(sd, N, A, device=dev, mode="bf16")
        for B in (int(b) for b in args.batches.split(",")):
            g = torch.Generator().manual_seed(B)
            x = (torch.randn(B, N, obs, generator=g) * 3 + 1).to(dev)
            run32 = lambda: f32.initial_inference(x)
            run16 = lambda: b16.initial_inference(x, fused=True)
            for _ in range(20):                       # warm-up: module loads, allocator, torch kernels of this shape
                run32(), run16()
            torch.cuda.synchronize()
            t = window(run16, 10)
            iters = max(20, min(2000, int(200000 / max(t, 1.0))))     # >= ~0.2 s per window of the fused path
            t32, t16 = [], []
            for _ in range(args.reps):
                t32.append(window(run32, iters))
                t16.append(window(run16, iters))
            a, b = run32(), run16()
            torch.cuda.synchronize()
            err = {n: ((getattr(b, n) - getattr(a, n)).abs().max() / max(1.0, getattr(a, n).abs().max().item())).item()
                   for n in ("hidden_state", "policy_logits", "value")}
            med = lambda v: sorted(v)[len(v) // 2]
            line = dict(shape=shape, N=N, A=A, obs_dim=obs, B=B, iters=iters, reps=args.reps,
                        fp32_us=round(med(t32), 2), fp32_spread_us=round(max(t32) - min(t32), 2),
                        fused_us=round(med(t16), 2), fused_spread_us=round(max(t16) - min(t16), 2),
                        speedup=round(med(t32) / med(t16), 2), **{f"err_{k}": float(f"{v:.3g}") for k, v in err.items()},
                        gpu=gpu)
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as fh:
                    fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
