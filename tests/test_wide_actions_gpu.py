"""GPU: the wide instances of the fused kernels (49 to 128 actions per agent; 2c_vs_64zg has 70).

1. the small-batch and the twin kernel against the fp32 restatement of the network (`SmacInference(mode="fp32")`, pinned to the
   real reference network by tests/test_model128_cpu.py and tests/test_infer128_gpu.py; it has no branch on the action count),
   two chained steps, the tolerances of test_infer128_gpu.py; the first-generation kernel is refused above 48 actions;
2. the persistent kernel fits the 2c_vs_64zg shape, and the persistent, graph and legacy loops agree bit for bit at (2, 70);
   the device path replays bit for bit through the CPU oracle tree;
3. the device-resident environment step (`search_agents`) equals the workers' host loop at (2, 70);
4. a bf16 search against an fp32 search at 2c_vs_64zg 1024 roots x 50 simulations;
5. exact ties of two policy rows: every kernel takes the first of the tied columns (np.argmax), joint and sequential mode;
6. every placement of the persistent wide kernel's tree-step scratch (the PH..Q alias, the X + T tiles, behind the extra map;
   tests/test_wide_actions_cpu.py: PERSIST_CASES) against the legacy loop, bit for bit; above the shared-memory limit the
   persistent strategy is refused and "auto" takes the graph loop."""
import os

import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_infer128_gpu import TOL_BF16, _relerr
from test_search_gpu import device_path_replay, root_output, smac_model
from test_search_native_gpu import _equal, _problem
from test_wide_actions_cpu import OPTIN_B200, PERSIST_CASES, persist_layout

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHAPES = [(2, 49), (2, 70), (8, 100), (2, 128)]


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ("MAZ_INFER_TC", "MAZ_INFER_KERNEL", "MAZ_SEARCH"):
        monkeypatch.delenv(k, raising=False)


def _hidden(B, N, seed):
    rng = np.random.RandomState(seed)
    return torch.from_numpy((rng.randint(-32768, 32768, size=(B, N * 128)) / 16384.0).astype(np.float32)).to(DEV)


@pytest.mark.parametrize("kernel", ["twin", "small"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"N{n}A{a}" for n, a in SHAPES])
def test_wide_kernels_match_fp32(built_lib, shape, kernel):
    """Two chained recurrent_inference steps; 301 roots leave the last tile of every kernel ragged."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import exact_state_dict

    N, A = shape
    B = 301
    sd = exact_state_dict(N, A, seed=N + A)
    ref = SmacInference(sd, N, A, device=DEV, mode="fp32")
    inf = SmacInference(sd, N, A, device=DEV, mode="bf16")
    rng = np.random.RandomState(A)
    acts = [torch.from_numpy(rng.randint(0, A, size=(B, N)).astype(np.int32)).to(DEV) for _ in range(2)]
    nan = lambda *s: torch.full(s, float("nan"), device=DEV)
    pool = torch.zeros(3, B, N * 128, device=DEV)
    pool[0] = _hidden(B, N, seed=A)
    idx = torch.zeros(B, dtype=torch.int32, device=DEV)
    ref_h = pool[0].clone()
    for step, act in enumerate(acts):
        ref_h, ref_r, ref_v, ref_logits = ref.recurrent(ref_h, act)
        rew, val, probs, beta, logits = nan(B), nan(B), nan(B, N, A), nan(B, N, A), nan(B, N, A)
        greedy = torch.full((B, N), -1, dtype=torch.int32, device=DEV)
        idx.fill_(step)
        inf.recurrent_fused(B, pool, idx, act, pool[step + 1], rew, val, probs, beta, greedy, logits, kernel=kernel)
        torch.cuda.synchronize()
        scale = 1.0 + step * 0.5          # the second step starts from the kernel's own (bf16-path) hidden state
        for name, got, want in (("hidden", pool[step + 1], ref_h), ("policy_logits", logits, ref_logits), ("reward", rew, ref_r),
                                ("value", val, ref_v), ("probs", probs, torch.softmax(ref_logits, -1))):
            assert torch.isfinite(got).all(), name
            e = _relerr(got, want.reshape(got.shape).cpu().numpy())
            print(f"{kernel} N={N} A={A} step {step} {name}: {e:.3g} (tol {TOL_BF16[name] * scale:.3g})")
            assert e <= TOL_BF16[name] * scale, f"{name}: {e}"
        assert torch.equal(beta, probs)                              # inv_tau = 1
        top2 = ref_logits.topk(2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > 2 * TOL_BF16["policy_logits"] * max(1.0, ref_logits.abs().max().item())
        assert torch.equal(greedy.long()[clear], ref_logits.argmax(-1)[clear])
        assert clear.float().mean().item() > 0.5
        # the greedy action is the first maximum of the kernel's own logits (torch.argmax)
        assert torch.equal(greedy.long(), logits.argmax(-1))


def test_first_generation_kernel_refused_above_48_actions(built_lib, monkeypatch):
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import exact_state_dict

    N, A, B = 2, 70, 4096
    inf = SmacInference(exact_state_dict(N, A, seed=1), N, A, device=DEV, mode="bf16")
    z = lambda *s: torch.zeros(s, device=DEV)
    pool, idx, act = z(2, B, N * 128), torch.zeros(B, dtype=torch.int32, device=DEV), torch.zeros(B, N, dtype=torch.int32, device=DEV)
    args = (B, pool, idx, act, pool[1], z(B), z(B), z(B, N, A), z(B, N, A))
    with pytest.raises(ValueError, match="at most 48 actions"):
        inf.recurrent_fused(*args, kernel="tcgen05")
    monkeypatch.setenv("MAZ_INFER_TC", "v1")
    monkeypatch.setenv("MAZ_INFER_KERNEL", "tcgen05")
    with pytest.raises(ValueError, match="MAZ_INFER_TC=v1"):
        inf.recurrent_fused(*args)


@pytest.mark.parametrize("S", [50, 100])
@pytest.mark.parametrize("joint", [True, False], ids=["joint", "seq"])
def test_persistent_kernel_fits_2c_vs_64zg(built_lib, joint, S):
    from mazero_b200.inference import SmacInference
    from mazero_b200.search_native import NativeSearch
    from mazero_b200.synthetic import WORKLOADS, exact_state_dict

    N, A, B, _, K = WORKLOADS["2c_vs_64zg"]
    inf = SmacInference(exact_state_dict(N, A, seed=0), N, A, device=DEV, mode="bf16")
    ns = NativeSearch(inf, B, K, S, joint, strategy="persistent")      # maz_search_create refuses when persist_ok fails
    assert ns.strategy == "persistent"
    smem, *where = persist_layout(inf.fused.vec.numel(), 8, N if joint else 1, A, S)
    print(f"2c_vs_64zg {'joint' if joint else 'seq'} S={S}: persistent kernel shared memory {smem} bytes ({smem / 1024:.1f} KB), "
          f"tree scratch alias / X + T / tail {where}")
    del ns


@pytest.mark.parametrize("cur", [None, 0, 1])
def test_loops_agree_bit_for_bit_at_70_actions(built_lib, cur):
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    N, A, B, K, S = 2, 70, 48, 10, 25
    inf, out0, factor, legal = _problem(N, A, B)
    cfg = MockConfig(N, A, S, K)
    outs = {}
    for strat in ("persistent", "graph", "legacy"):
        mcts = SampledMCTS(cfg, np.random.RandomState(1), search_strategy=strat)
        outs[strat] = mcts.batch_search(inf, out0, cur, factor, N, legal, DEV, add_noise=True, sampled_tau=1.0 if cur != 1 else 0.7)
        plan = next(iter(mcts._plans.values()))
        if strat != "legacy":
            assert plan.native is not None and plan.native.strategy == strat
        else:
            assert plan.native is None
    clear_caches()
    Nt = N if cur is None else 1
    print(f"(2, 70) cur={cur}: persistent kernel shared memory, tree scratch alias / X + T / tail "
          f"{persist_layout(inf.fused.vec.numel(), 8, Nt, A, S)}")
    _equal(outs["persistent"], outs["legacy"], "persistent vs legacy: ")
    _equal(outs["graph"], outs["legacy"], "graph vs legacy: ")
    assert int(outs["persistent"].marginal_visit_count[0, 0].sum()) == S


# P2 (joint, S = 100): two trees per CTA behind the extra map, the last CTA with only the first of them
@pytest.mark.parametrize("cur,B,S", [pytest.param(None, 48, 25, id="None"), pytest.param(1, 48, 25, id="1"),
                                     pytest.param(None, PERSIST_CASES["P2"][5], PERSIST_CASES["P2"][3], id="None-P2")])
def test_device_path_replays_through_oracle_tree_at_70_actions(built_lib, oracle_built, cur, B, S):
    from mazero_b200.inference import SmacInference

    N, A, K = 2, 70, 10
    model = smac_model(N, A)
    inf = SmacInference.from_model(model, device=DEV, mode="bf16")
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    device_path_replay(inf, out0, N, A, B, K, S, cur, oracle_built)


@pytest.mark.parametrize("turn", ["greedy", "sample"])
def test_search_agents_equals_the_workers_host_loop_at_70_actions(built_lib, turn):
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS
    from oracle import turn_oracle

    N, A, B, K, S = 2, 70, 40, 10, 20
    cfg = MockConfig(N, A, S, K)
    model = smac_model(N, A)
    inf = SmacInference.from_model(model, device=DEV, mode="bf16")
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1
    rng = np.random.RandomState(9)
    eps_u = rng.rand(N, B).astype(np.float32)
    rand_act = np.stack([[rng.choice(np.where(legal[b, k] > 0)[0]) for b in range(B)] for k in range(N)]).astype(np.int32)
    temperature, eps = 0.5, 0.3

    fused = SampledMCTS(cfg, np.random.RandomState(21))
    got = fused.search_agents(inf, out0, N, legal, DEV, add_noise=True, sampled_tau=1.0, turn=turn, temperature=temperature,
                              greedy_epsilon=eps, eps_randoms=(eps_u, rand_act) if turn == "sample" else None)

    host_rs = np.random.RandomState(21)
    looped = SampledMCTS(cfg, host_rs)
    search_fn = lambda k, factor: looped.batch_search(inf, out0, k, factor, N, legal, DEV, add_noise=True, sampled_tau=1.0)
    if turn == "greedy":
        actions, dist, prob, outs = turn_oracle.reanalyze_turns(search_fn, B, N, A, legal)
        assert np.array_equal(got.prob, prob)
    else:
        actions, ent, outs = turn_oracle.selfplay_turns(search_fn, host_rs, B, N, A, legal, temperature, eps, eps_u, rand_act)
        np.testing.assert_allclose(got.entropy, ent, rtol=1e-12, atol=1e-14)
        dist = np.stack([np.stack([turn_oracle.visit_policy(outs[k].marginal_visit_count[b, 0], legal[b, k], A) for k in range(N)])
                         for b in range(B)])
    assert np.array_equal(got.actions, actions)
    assert np.array_equal(got.policy_dist, dist)
    for k in range(N):
        _equal(got.search_outputs[k], outs[k], f"agent {k}: ")
    assert np.array_equal(fused.np_random.get_state()[1], host_rs.get_state()[1])


def test_bf16_vs_fp32_search_report_2c_vs_64zg(built_lib):
    """2c_vs_64zg, 1024 roots x 50 simulations, joint mode: bf16 kernels vs fp32 parity mode, the bounds of
    test_infer128_gpu.py::test_bf16_vs_fp32_search_report."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.synthetic import WORKLOADS, NetworkOutput, SearchConfig, exact_state_dict

    N, A, B, S, K = WORKLOADS["2c_vs_64zg"]
    sd = exact_state_dict(N, A, seed=103)
    cfg = SearchConfig(A, S, K)
    hidden = _hidden(B, N, seed=5)
    outs = {}
    for mode in ("fp32", "bf16"):
        inf = SmacInference(sd, N, A, device=DEV, mode=mode)
        pol, vlog = SmacInference(sd, N, A, device=DEV, mode="fp32").prediction(hidden)
        value = inf._inv_transform(vlog, inf.vsup).reshape(B, 1)
        root = NetworkOutput(hidden, np.zeros((B, 1), np.float32), value.cpu().numpy(), pol.cpu().numpy())
        mcts = SampledMCTS(cfg, np.random.RandomState(9), inference_mode=mode)
        outs[mode] = mcts.batch_search(inf, root, None, None, N, None, DEV, add_noise=True)
        clear_caches()
    f, h = outs["fp32"], outs["bf16"]
    dv = np.abs(f.value - h.value)
    vf = f.marginal_visit_count.astype(np.float64) / S
    vh = h.marginal_visit_count.astype(np.float64) / S
    tv = 0.5 * np.abs(vf - vh).sum(-1)
    flip = (vf.argmax(-1) != vh.argmax(-1)).mean()
    same_sets = np.mean([np.array_equal(f.sampled_actions[b], h.sampled_actions[b]) for b in range(B)])
    print(f"bf16 vs fp32 search (2c_vs_64zg 1024x50): root value |diff| mean {dv.mean():.4g} max {dv.max():.4g} "
          f"(value range {np.abs(f.value).max():.3g}); visit-distribution TV mean {tv.mean():.4g}; "
          f"visit-argmax differs for {100 * flip:.2f}% of (root, agent); identical root sampled sets {100 * same_sets:.2f}%")
    assert same_sets == 1.0
    assert dv.mean() < 0.02 * max(1.0, np.abs(f.value).max())
    assert tv.mean() < 0.15


TIES = ([(40, k, p) for k in ("twin", "tcgen05", "small") for p in ((3, 11), (15, 16), (7, 39))] +
        [(A, k, p) for A in (70, 128) for k in ("twin", "small") for p in ((5, 21), (31, 32), (2, 67), (1, A - 1))])


@pytest.mark.parametrize("A,kernel,pair", TIES, ids=[f"A{a}-{k}-{p[0]}-{p[1]}" for a, k, p in TIES])
def test_exact_ties_take_the_first_maximum(built_lib, A, kernel, pair):
    """fc_policy.3 rows and biases j1 < j2 made equal, + 20 on both biases: the two columns tie as the maximum of every row.
    The kernels reduce across 16-column blocks, 32-column parts (twin) and 8 lanes per row (small-batch); each must keep the
    first maximum, j1, as np.argmax does (mcts_sampled.py:145), and give both columns the same probability and beta."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import exact_state_dict

    N, B = 2, 301
    j1, j2 = pair
    sd = {k: v.clone() for k, v in exact_state_dict(N, A, seed=A).items()}
    w, b = sd["prediction_network.fc_policy.3.weight"], sd["prediction_network.fc_policy.3.bias"]
    w[j2], b[j2] = w[j1], b[j1]
    b[[j1, j2]] += 20.0
    inf = SmacInference(sd, N, A, device=DEV, mode="bf16")
    pool = torch.stack([_hidden(B, N, seed=A), torch.zeros(B, N * 128, device=DEV)])
    idx = torch.zeros(B, dtype=torch.int32, device=DEV)
    act = torch.from_numpy(np.random.RandomState(A).randint(0, A, size=(B, N)).astype(np.int32)).to(DEV)
    for cur in (None, N - 1):
        Nt = N if cur is None else 1
        probs, beta, logits = (torch.full((B, n, A), float("nan"), device=DEV) for n in (Nt, Nt, N))
        greedy = torch.full((B, N), -1, dtype=torch.int32, device=DEV)
        mode = dict(tree_agents=1, cur=cur, inv_tau=0.5) if cur is not None else {}
        inf.recurrent_fused(B, pool, idx, act, pool[1], torch.zeros(B, device=DEV), torch.zeros(B, device=DEV), probs, beta, greedy,
                            logits, kernel=kernel, **mode)
        torch.cuda.synchronize()
        what = f"{kernel} A={A} ({j1}, {j2}) {'joint' if cur is None else f'cur={cur}'}"
        # premise: the tied columns are bit-identical maxima of every row
        assert torch.equal(logits[..., j1], logits[..., j2]), f"{what}: tied logits differ"
        assert torch.equal(logits[..., j1], logits.max(-1).values), f"{what}: the tie is not the maximum"
        assert (greedy == j1).all(), f"{what}: greedy {greedy[greedy != j1][:8].tolist()}"
        assert torch.equal(probs[..., j1], probs[..., j2]) and torch.equal(beta[..., j1], beta[..., j2]), what


@pytest.mark.parametrize("name", sorted(PERSIST_CASES))
def test_persistent_kernel_every_tree_scratch_placement(built_lib, monkeypatch, name):
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.search_native import NativeSearch

    N, A, cur, S, rpt, B, counts, nbytes = PERSIST_CASES[name]
    K = 10
    if rpt < min(8, 32 // N):
        monkeypatch.setenv("MAZ_SEARCH_RPT", str(rpt))
    assert min(8, 32 // N, int(os.environ.get("MAZ_SEARCH_RPT", "8"))) == rpt    # the roots per CTA of maz_search_create
    inf, out0, factor, legal = _problem(N, A, B or 16)
    layout = persist_layout(inf.fused.vec.numel(), rpt, N if cur is None else 1, A, S)
    print(f"{name}: (N, A) = ({N}, {A}) {'joint' if cur is None else f'cur={cur}'} S={S} rpt={rpt} B={B}: {layout[0]} bytes, "
          f"tree scratch alias / X + T / tail {layout[1:]}")
    assert layout == (nbytes, *counts)
    if B is None:
        assert nbytes + 256 > OPTIN_B200
        with pytest.raises(RuntimeError, match="persistent kernel does not support"):
            NativeSearch(inf, 16, K, S, cur is None, strategy="persistent")
        assert NativeSearch(inf, 16, K, S, cur is None).strategy == "graph"
        return
    ns = NativeSearch(inf, B, K, S, cur is None)
    assert ns.strategy == "persistent"                              # "auto": within the limit, one wave of CTAs
    del ns
    cfg = MockConfig(N, A, S, K)
    outs = {}
    for strat in ("persistent", "legacy"):
        mcts = SampledMCTS(cfg, np.random.RandomState(1), search_strategy=strat)
        outs[strat] = mcts.batch_search(inf, out0, cur, factor, N, legal, DEV, add_noise=True)
        plan = next(iter(mcts._plans.values()))
        assert (plan.native.strategy if plan.native is not None else "legacy") == strat
    clear_caches()
    _equal(outs["persistent"], outs["legacy"], f"{name}: persistent vs legacy: ")
    assert int(outs["persistent"].marginal_visit_count[0, 0].sum()) == S

