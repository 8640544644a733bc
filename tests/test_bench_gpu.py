"""GPU: bench.py --dump-outputs writes the readouts of the last timed search: they equal a separate host-buffer search
(maz_search_run) of that step's input batch and tree seed, two runs with the same arguments write the same arrays, and
--steps (which decides the last timed step) changes them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, S, WARMUP = 64, 8, 3


def bench(d, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--roots", str(B), "--sims", str(S), "--steps", str(steps),
                          "--warmup", str(WARMUP), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def last_step_host_search(steps):
    """The search of timed step `steps - 1` (after WARMUP warm-up steps) through maz_search_run with host buffers."""
    import torch

    import bench as bench_mod
    from mazero_b200.mcts_sampled import clear_caches
    from mazero_b200.synthetic import WORKLOADS

    N, A, _, _, K = WORKLOADS["3m"]
    prob = bench_mod.Problem(None, "3m", N, A, B, S, K, torch.device("cuda", 0), 0, None)   # regenerates bench.py's inputs
    i = WARMUP + steps - 1                                # bench.py's step index: input set i % nsets, tree seed 100 + i
    d = {k: v.cpu().numpy() for k, v in prob.devs[i % prob.nsets].items()}
    r = prob.plan.native.run_host(None, 100 + i, prob.cfg, prob.cfg.root_exploration_fraction, prob.plan.tau, d["hidden"],
                                  d["rewards"], d["values"], d["logits"], None, d["noise"], None, root_index_offset=prob.root_off)
    del prob
    clear_caches()
    return r


def test_dump_outputs_are_the_last_timed_search_and_reproducible(built_lib, tmp_path):
    a, b, c = bench(tmp_path / "a", 3), bench(tmp_path / "b", 3), bench(tmp_path / "c", 2)
    want = last_step_host_search(3)
    assert set(a) == set(want) == set(b) == set(c)
    for k in a:
        assert a[k].dtype == np.float32 and a[k].shape == want[k].shape, k
        assert np.array_equal(a[k], want[k].astype(np.float32)), k
        assert np.array_equal(a[k], b[k]), k
    assert (a["marginal_visit_count"].sum(axis=2) == S).all()
    assert not np.array_equal(a["value"], c["value"])      # another last step: another input batch and tree seed
