"""GPU: the whole search behind the C ABI (include/maz_search.h, mazero_b200/search_native.py).

* the three ways to run the loop -- persistent kernel, CUDA graph built in the library, and the round-1 Python loop over the
  per-step C ABI ("legacy") -- give bit-identical SearchOutputs (joint and every sequential turn, legal mask + noise);
* `maz_search_run` driven through ctypes with HOST numpy buffers only (what a non-Python host would bind) equals
  `SampledMCTS.batch_search` bit for bit;
* search constants (rho, delta_lb, lambda, discount, c_init) changed between searches on the SAME cached handle take effect
  (the library keys its CUDA graphs by them; round 1 replayed stale graphs);
* the process-wide plan cache respects its byte budget."""
import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_search_gpu import root_output, smac_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _equal(a, b, what=""):
    for f in a._fields:
        x, y = getattr(a, f), getattr(b, f)
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y), f"{what}{f}"
        else:
            assert x == y, f"{what}{f}"


def _problem(N=3, A=9, B=48, seed=0):
    from mazero_b200.inference import SmacInference

    model = smac_model(N, A, seed=seed)
    inf = SmacInference.from_model(model, device=DEV, mode="bf16")
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    factor = np.random.RandomState(5).randint(0, A, size=(B, N)).astype(np.int32)
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1
    return inf, out0, factor, legal


@pytest.mark.parametrize("cur", [None, 0, 1, 2])
def test_persistent_graph_and_legacy_loops_agree_bit_for_bit(built_lib, cur):
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    N, A, B, K, S = 3, 9, 48, 10, 25
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
    _equal(outs["persistent"], outs["legacy"], "persistent vs legacy: ")
    _equal(outs["graph"], outs["legacy"], "graph vs legacy: ")
    assert int(outs["persistent"].marginal_visit_count[0, 0].sum()) == S


@pytest.mark.parametrize("shape", [(5, 11, 20), (10, 18, 7), (27, 36, 3), (1, 5, 33), (2, 40, 17)])
def test_persistent_kernel_other_team_shapes(built_lib, shape):
    """roots per CTA = min(8, floor(32 / N)): 6, 3, 1, 8, 8 -- ragged last CTA included."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.synthetic import NetworkOutput, exact_state_dict

    N, A, B = shape
    K, S = 6, 12
    inf = SmacInference(exact_state_dict(N, A, seed=N), N, A, device=DEV, mode="bf16")
    g = torch.Generator().manual_seed(3)
    hidden = torch.randn(B, N * 128, generator=g).to(DEV)
    pol, vlog = inf.prediction(hidden)
    value = inf._inv_transform(vlog, inf.vsup).reshape(B, 1).cpu().numpy()
    root = NetworkOutput(hidden, np.zeros((B, 1), np.float32), value, pol.cpu().numpy())
    cfg = MockConfig(N, A, S, K)
    outs = {}
    for strat in ("persistent", "graph"):
        mcts = SampledMCTS(cfg, np.random.RandomState(2), search_strategy=strat)
        outs[strat] = [mcts.batch_search(inf, root, None, None, N, None, DEV, add_noise=True)]
        if N > 1:   # a sequential turn of the last agent (factor given) and of the first one (later agents greedy)
            fac = np.random.RandomState(4).randint(0, A, size=(B, N)).astype(np.int32)
            outs[strat].append(mcts.batch_search(inf, root, N - 1, fac, N, None, DEV, add_noise=True))
            outs[strat].append(mcts.batch_search(inf, root, 0, None, N, None, DEV, add_noise=False))
    clear_caches()
    for a, b in zip(outs["persistent"], outs["graph"]):
        _equal(a, b)


def test_ctypes_host_call_equals_batch_search(built_lib):
    """maz_search_create / maz_search_run / maz_search_destroy with host buffers only."""
    from mazero_b200 import hostrng
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.search_native import NativeSearch

    N, A, B, K, S = 3, 9, 40, 10, 20
    inf, out0, factor, legal = _problem(N, A, B)
    cfg = MockConfig(N, A, S, K)
    for cur in (None, 1):
        ref = SampledMCTS(cfg, np.random.RandomState(7)).batch_search(inf, out0, cur, factor, N, legal, DEV, add_noise=True)
        rng = np.random.RandomState(7)                                   # the two host draws of mcts_sampled.py:68,89
        Nt = N if cur is None else 1
        noise = hostrng.dirichlet_f32(rng, cfg.root_dirichlet_alpha, A, B * Nt).reshape(B, Nt, A)
        seed = rng.choice(256)
        ns = NativeSearch(inf, B, K, S, joint=cur is None)
        r = ns.run_host(cur, seed, cfg, cfg.root_exploration_fraction, 1.0, out0.hidden_state.cpu().numpy(), out0.reward,
                        out0.value, out0.policy_logits, legal, noise, factor)
        ns.close()
        assert np.array_equal(r["value"], ref.value)
        assert np.array_equal(r["marginal_visit_count"], ref.marginal_visit_count)
        assert np.array_equal(r["marginal_priors"], ref.marginal_priors)
        for b in range(B):
            n = r["num_children"][b]
            assert np.array_equal(r["actions"][b, :n], ref.sampled_actions[b])
            assert np.array_equal(r["visit_count"][b, :n], ref.sampled_visit_count[b])
            assert np.array_equal(r["qvalues"][b, :n], ref.sampled_qvalues[b])
            assert np.array_equal(r["imp_ratio"][b, :n], ref.sampled_imp_ratio[b])
    clear_caches()


@pytest.mark.parametrize("strategy", ["persistent", "graph"])
def test_search_constants_changed_on_a_cached_handle_take_effect(built_lib, strategy):
    """ADVICE r1: a captured graph froze delta_lb / rho / lambda; a second SampledMCTS with other values replayed it."""
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    N, A, B, K, S = 3, 9, 32, 10, 20
    inf, out0, factor, legal = _problem(N, A, B)
    variants = [dict(), dict(mcts_rho=0.25), dict(tree_value_stat_delta_lb=0.5), dict(mcts_lambda=0.5), dict(discount=0.9),
                dict(pb_c_init=2.5), dict()]
    got, want = [], []
    for kw in variants:
        cfg = MockConfig(N, A, S, K)
        for k, v in kw.items():
            setattr(cfg, k, v)
        got.append(SampledMCTS(cfg, np.random.RandomState(3), search_strategy=strategy)
                   .batch_search(inf, out0, None, None, N, legal, DEV, add_noise=True))     # same cached handle every time
    from mazero_b200.mcts_sampled import _PLAN_CACHE
    assert len(_PLAN_CACHE) == 1
    clear_caches()
    for kw in variants:
        cfg = MockConfig(N, A, S, K)
        for k, v in kw.items():
            setattr(cfg, k, v)
        want.append(SampledMCTS(cfg, np.random.RandomState(3), search_strategy="legacy", use_cuda_graph=False)
                    .batch_search(inf, out0, None, None, N, legal, DEV, add_noise=True))
        clear_caches()                                                                       # fresh objects every time
    for i, (a, b) in enumerate(zip(got, want)):
        _equal(a, b, f"variant {i}: ")
    assert not np.array_equal(got[0].value, got[1].value) and not np.array_equal(got[0].value, got[3].value)
    _equal(got[0], got[-1])


def test_inference_mode_is_part_of_the_cache_key(built_lib):
    """ADVICE r1: SampledMCTS(inference_mode='fp32') must not be served the cached bf16 object of an earlier instance."""
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    N, A, B, K, S = 3, 9, 16, 10, 8
    model = smac_model(N, A).to(DEV)
    out0 = root_output(smac_model(N, A), B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    cfg = MockConfig(N, A, S, K)
    a = SampledMCTS(cfg, np.random.RandomState(1), inference_mode="bf16")
    a.batch_search(model, out0, None, None, N, None, DEV)
    b = SampledMCTS(cfg, np.random.RandomState(1), inference_mode="fp32")
    b.batch_search(model, out0, None, None, N, None, DEV)
    ia, ib = next(iter(a._inference.values())), next(iter(b._inference.values()))
    assert ia is not ib and ia.fused is not None and ib.fused is None
    clear_caches()


def test_plan_cache_respects_its_byte_budget(built_lib):
    from mazero_b200 import mcts_sampled as ms

    N, A, K, S = 3, 9, 10, 10
    inf, out0, _, _ = _problem(N, A, 64)
    cfg = MockConfig(N, A, S, K)
    ms.clear_caches()
    torch.cuda.synchronize()
    old = ms.PLAN_CACHE_BYTES
    try:
        probe = ms.SampledMCTS(cfg, np.random.RandomState(0))
        probe.batch_search(inf, out0._replace(hidden_state=out0.hidden_state[:64]), None, None, N, None, DEV)
        one = ms._plan_cache_bytes()
        ms.clear_caches()
        ms.PLAN_CACHE_BYTES = 3 * one
        free0 = torch.cuda.mem_get_info()[0]
        low = free0
        for B in range(64, 44, -1):          # 20 different batch sizes, as a self-play worker whose episodes end one by one
            o = out0._replace(hidden_state=out0.hidden_state[:B], reward=out0.reward[:B], value=out0.value[:B],
                              policy_logits=out0.policy_logits[:B])
            ms.SampledMCTS(cfg, np.random.RandomState(0)).batch_search(inf, o, None, None, N, None, DEV)
            assert ms._plan_cache_bytes() <= ms.PLAN_CACHE_BYTES
            assert len(ms._PLAN_CACHE) <= 4          # (smaller batches make slightly smaller plans)
            low = min(low, torch.cuda.mem_get_info()[0])
        # device memory held: a handful of plans, not twenty (torch may cache freed blocks: allow 8 plans' worth + 64 MiB)
        assert free0 - low <= 8 * one + (64 << 20), (free0 - low, one)
    finally:
        ms.PLAN_CACHE_BYTES = old
        ms.clear_caches()


@pytest.mark.parametrize("N,A,gen,cur", [pytest.param(3, 9, g, c, id=f"{c}-{g}") for c in (None, 0, 2) for g in ("twin", "v1")] +
                         [pytest.param(2, 70, "twin", c, id=f"{c}-twin-A70") for c in (None, 0, 1)])
def test_graph_loop_on_the_tcgen05_kernels_equals_the_legacy_loop(built_lib, monkeypatch, N, A, gen, cur):
    """The library-built graph with the 128-row tcgen05 kernels (both generations; forced: at this batch size the small-batch
    kernel would be picked) against the round-1 Python loop on the same kernel: in the sequential-agent mode the former assembles
    the joint action INSIDE the inference kernel (factor | tree action | greedy of the parent, mcts_sampled.py:116-147), the latter
    in Python -- bit-identical SearchOutputs prove the in-kernel assembly of either generation, and of the wide twin instance
    (70 actions: only the twin kernel has one)."""
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    monkeypatch.setenv("MAZ_INFER_KERNEL", "tcgen05")
    monkeypatch.setenv("MAZ_INFER_TC", gen)
    B, K, S = 100, 10, 20
    inf, out0, factor, legal = _problem(N, A, B, seed=3)
    cfg = MockConfig(N, A, S, K)
    outs = {}
    for strat in ("graph", "legacy"):
        mcts = SampledMCTS(cfg, np.random.RandomState(1), search_strategy=strat)
        outs[strat] = mcts.batch_search(inf, out0, cur, factor, N, legal, DEV, add_noise=True)
    clear_caches()
    _equal(outs["graph"], outs["legacy"], f"graph vs legacy ({gen}): ")
