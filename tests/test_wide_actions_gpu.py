"""GPU: the wide instances of the fused kernels (49 to 128 actions per agent; 2c_vs_64zg has 70).

1. the small-batch and the twin kernel against the fp32 restatement of the network (`SmacInference(mode="fp32")`, pinned to the
   real reference network by tests/test_model128_cpu.py and tests/test_infer128_gpu.py; it has no branch on the action count),
   two chained steps, the tolerances of test_infer128_gpu.py; the first-generation kernel is refused above 48 actions;
2. the persistent kernel fits the 2c_vs_64zg shape, and the persistent, graph and legacy loops agree bit for bit at (2, 70);
   the device path replays bit for bit through the CPU oracle tree;
3. the device-resident environment step (`search_agents`) equals the workers' host loop at (2, 70);
4. a bf16 search against an fp32 search at 2c_vs_64zg 1024 roots x 50 simulations."""
import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_infer128_gpu import TOL_BF16, _relerr
from test_search_gpu import device_path_replay, root_output, smac_model
from test_search_native_gpu import _equal, _problem

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


def _persist_smem_bytes(vec_floats, rpt, Nt, A, S, K=10):
    """persist::persist_smem_bytes_wide (csrc/search_persist.cuh) restated, for the report."""
    al16 = lambda x: (x + 15) // 16 * 16
    lv, na = S + 2, Nt * A
    ts = al16(al16(16 * na + 256 + 4 * 128 + K * Nt) + 24 * lv + 4 * lv + al16(2 * lv))   # tree_scratch_bytes
    tail = max(0, rpt - 27648 // ts - 17408 // ts) * ts
    TM, LDA, LDO, LDP, LDQ, NQ, SUP, LDV = 32, 272, 112, 80, 784, 4, 11, 68
    off_row = TM * LDA * 3 + TM * LDO + TM * LDP + TM * LDQ + 3 * TM * NQ * 8 + 2 * SUP * LDV * 4
    off_p = (off_row + TM * 16 + 127) // 128 * 128 + 3 * 128 * 136 * 2
    lv = S + 2
    hot = 64 + al16(4 * lv) + 3 * al16(2 * lv)
    extra = hot * rpt + 3 * al16(4 * rpt) + 2 * al16(4 * rpt * Nt * A) + al16(4 * rpt * Nt)
    return al16(off_p + vec_floats * 4 + 128) + extra + tail


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
    smem = _persist_smem_bytes(inf.fused.vec.numel(), 8, N if joint else 1, A, S)
    print(f"2c_vs_64zg {'joint' if joint else 'seq'} S={S}: persistent kernel shared memory {smem} bytes ({smem / 1024:.1f} KB)")
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
    print(f"(2, 70) cur={cur}: persistent kernel shared memory {_persist_smem_bytes(inf.fused.vec.numel(), 8, Nt, A, S)} bytes")
    _equal(outs["persistent"], outs["legacy"], "persistent vs legacy: ")
    _equal(outs["graph"], outs["legacy"], "graph vs legacy: ")
    assert int(outs["persistent"].marginal_visit_count[0, 0].sum()) == S


@pytest.mark.parametrize("cur", [None, 1])
def test_device_path_replays_through_oracle_tree_at_70_actions(built_lib, oracle_built, cur):
    from mazero_b200.inference import SmacInference

    N, A, B, K, S = 2, 70, 48, 10, 25
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
