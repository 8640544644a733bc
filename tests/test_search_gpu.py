"""GPU: the search driver `SampledMCTS.batch_search` (drop-in for mcts_sampled.py:34-200).

* step path  (any model, CUDA tree): reproduces the real reference's known answers exactly;
* device path (SMAC network, whole loop on the GPU, CUDA graph): every simulation's network outputs are
  recorded and REPLAYED through the CPU oracle tree -- selections, sampled sets and visit counts must be
  bit-exact, values/Q bit-exact too (same injected fp32 arrays);  graph replay == eager loop."""
import numpy as np
import pytest
import torch

from _mock import MockConfig, MockModel, sequential_search
from test_search_oracle import check_kat, kat_legal

pytestmark = pytest.mark.gpu


def smac_model(n, a, h=128, seed=0):
    from oracle.model_oracle import OracleMAMuZeroNet

    m = OracleMAMuZeroNet(n, a, hidden_state_size=h, fc_dynamic_layers=(h, h)).init_like_reference(seed).eval()
    # the reference init leaves the heads at ~0 (uniform policy, value 0): perturb for a non-degenerate search
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(torch.randn(p.shape, generator=g) * 0.03)
    return m


def root_output(model, B, seed=0):
    from oracle.search_oracle import NetworkOutput

    g = torch.Generator().manual_seed(seed)
    hidden = torch.randn(B, model.num_agents * model.hidden, generator=g)
    with torch.no_grad():
        pol, vlog = model.prediction(hidden)
        from oracle.model_oracle import inverse_support_transform
        value = inverse_support_transform(vlog, -5, 5)
    return NetworkOutput(hidden, np.zeros((B, 1), np.float32), value.numpy(), pol.numpy())


def test_step_path_reproduces_reference_known_answers(built_lib):
    from mazero_b200.mcts_sampled import SampledMCTS

    cfg, model = MockConfig(), MockModel(2, 3)
    mcts = SampledMCTS(cfg, np.random.RandomState(123))
    fn = lambda m, o, k, f, n, l: mcts.batch_search(m, o, k, f, n, l, torch.device("cpu"), add_noise=True)
    check_kat(*sequential_search(fn, cfg, model, legal=kat_legal()))


def device_path_replay(inf, out0, N, A, B, K, S, cur, oracle_built, strategy="auto"):
    """Run the on-device search eagerly with every simulation's network outputs recorded, replay them through the CPU
    oracle tree (bit-exact selections, sampled sets, visit counts, values, Q), then require graph replay == eager.
    Returns the search output and the oracle's path length of every simulation and tree, (S, B)."""
    from mazero_b200.mcts_sampled import SampledMCTS

    cfg = MockConfig(N, A, S, K)
    factor = np.random.RandomState(5).randint(0, A, size=(B, N)).astype(np.int32)
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1

    def run(graph, record):
        mcts = SampledMCTS(cfg, np.random.RandomState(1), use_cuda_graph=graph, search_strategy=strategy)
        if record is not None:
            mcts.batch_search(inf, out0, cur, factor, N, legal, "cuda:0", add_noise=True)  # builds the plan
            plan = next(iter(mcts._plans.values()))
            plan.record = record
            mcts.np_random = np.random.RandomState(1)
        return mcts.batch_search(inf, out0, cur, factor, N, legal, "cuda:0", add_noise=True), mcts

    rec = []
    eager, mcts = run(False, rec)
    assert len(rec) == S
    # replay the recorded network outputs through the CPU oracle tree with the same seed / root arrays
    plan = next(iter(mcts._plans.values()))
    Nt = N if cur is None else 1
    seed = np.random.RandomState(1)
    seed.dirichlet([cfg.root_dirichlet_alpha] * A, B * Nt if cur is None else B)
    tree_seed = seed.choice(256)
    orc = oracle_built.OracleTreeBatch(B, Nt, A, K, S, cfg.tree_value_stat_delta_lb, tree_seed, cfg.mcts_rho, cfg.mcts_lambda)
    orc.prepare(plan.root_r.cpu().numpy(), plan.root_v.cpu().numpy(), plan.root_p.cpu().numpy(), plan.root_b.cpu().numpy(),
                K, cfg.root_exploration_fraction, plan.root_n.cpu().numpy())
    lens = []
    for s, (rew, val, p, b, ix, act) in enumerate(rec):
        oix, _, oact = orc.batch_selection(cfg.pb_c_base, cfg.pb_c_init, cfg.discount)
        lens.append(orc.stats()[1])
        assert np.array_equal(np.asarray(oix, np.int32), ix.cpu().numpy()), f"sim {s}: hidden_state_index_x"
        assert np.array_equal(oact, act.cpu().numpy()), f"sim {s}: selected actions"
        orc.batch_expansion_and_backup(s + 1, cfg.discount, K, rew.cpu().numpy(), val.cpu().numpy(), p.cpu().numpy(), b.cpu().numpy())
    ro = orc.readout(cfg.discount)
    assert np.array_equal(eager.marginal_visit_count, orc.get_roots_marginal_visit_count())
    assert np.array_equal(eager.value, orc.get_roots_values())
    for b in range(B):
        n = ro["num_children"][b]
        assert np.array_equal(eager.sampled_actions[b], ro["actions"][b, :n])
        assert np.array_equal(eager.sampled_visit_count[b], ro["visit_count"][b, :n])
        assert np.array_equal(eager.sampled_qvalues[b], ro["qvalues"][b, :n])
    assert int(eager.marginal_visit_count[0, 0].sum()) == S

    graphed, _ = run(True, None)
    for f in eager._fields:
        x, y = getattr(eager, f), getattr(graphed, f)
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y), f
        else:
            assert x == y, f
    return eager, np.stack(lens)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("cur", [None, 0, 1, 2])
def test_device_path_replays_bit_exact_through_oracle_tree(built_lib, oracle_built, cur, mode):
    from mazero_b200.inference import SmacInference

    N, A, B, K, S = 3, 9, 48, 10, 25
    model = smac_model(N, A)
    inf = SmacInference.from_model(model, device="cuda:0", mode=mode)
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    device_path_replay(inf, out0, N, A, B, K, S, cur, oracle_built)


def test_device_path_accepts_reference_style_module(built_lib):
    """A torch module with the reference's parameter names on the GPU is adapted automatically."""
    from mazero_b200.mcts_sampled import SampledMCTS

    N, A, B, K, S = 3, 9, 16, 5, 10
    cfg = MockConfig(N, A, S, K)
    model = smac_model(N, A).cuda()
    model.hidden_state_size_per_agent = model.hidden
    out0 = root_output(smac_model(N, A), B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    mcts = SampledMCTS(cfg, np.random.RandomState(3))
    o = mcts.batch_search(model, out0, 0, None, N, None, torch.device("cuda:0"), add_noise=False)
    assert len(mcts._plans) == 1
    assert o.value.shape == (B,) and o.marginal_visit_count.shape == (B, 1, A)
    assert (o.marginal_visit_count.sum(axis=(1, 2)) == S).all()
    assert all(o.sampled_actions[b].shape[1] == 1 for b in range(B))
    with pytest.raises(NotImplementedError):
        mcts.batch_search(model, out0, 0, None, N, None, torch.device("cuda:0"), sampled_actions_res=(None, None))


class _RefStyleModel:
    """Reference-style interface (numpy reward / value / logits, torch hidden) around the CPU fp32 network."""

    def __init__(self, net):
        self.net = net

    def eval(self):
        return self

    def prediction(self, hidden):
        pol, vlog = self.net.prediction(hidden)
        return pol.detach().numpy(), vlog.detach().numpy()

    def recurrent_inference(self, hidden, action):
        from oracle.search_oracle import NetworkOutput

        nxt, r, v, pl = self.net.recurrent_inference(hidden, action)
        return NetworkOutput(nxt, r.numpy(), v.numpy(), pl.numpy())


@pytest.mark.parametrize("cur", [None, 0, 2])
def test_step_path_equals_restated_reference_driver(built_lib, oracle_built, cur):
    """Whole `batch_search` of the product (CUDA tree, reference loop, real fp32 network on the CPU) against the restated
    reference driver over the CPU oracle tree: identical network outputs by construction, so EVERY field of SearchOutput
    must be bit-identical (root preparation, RNG consumption order, legal mask, noise, sequential-agent joint actions)."""
    from mazero_b200.mcts_sampled import SampledMCTS
    from oracle.search_oracle import reference_batch_search

    N, A, B, K, S = 3, 9, 20, 10, 15
    cfg = MockConfig(N, A, S, K)
    net = smac_model(N, A, h=32)
    model = _RefStyleModel(net)
    out0 = root_output(net, B)
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1
    factor = np.random.RandomState(5).randint(0, A, size=(B, N)).astype(np.int32)
    ours = SampledMCTS(cfg, np.random.RandomState(11)).batch_search(model, out0, cur, factor, N, legal.copy(), torch.device("cpu"),
                                                                     add_noise=True, sampled_tau=1.0)
    ref = reference_batch_search(cfg, np.random.RandomState(11), model, out0, cur, factor, N, legal.copy(), torch.device("cpu"),
                                 add_noise=True, sampled_tau=1.0, tree_kind="port")
    for f in ours._fields:
        x, y = getattr(ours, f), getattr(ref, f)
        if isinstance(y, np.ndarray):
            assert np.array_equal(x, y), f
        else:
            assert len(x) == len(y) and all(np.array_equal(a, b) for a, b in zip(x, y)), f


def test_sequential_turns_share_one_plan_without_leaking_state(built_lib):
    """The per-agent loop of the workers (selfplay_worker.py:196-211) calls batch_search N times on one SampledMCTS:
    one device plan (arena, pool) serves all turns, one captured graph per turn, and a turn's result does not depend
    on the turns run before it."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS

    N, A, B, K, S = 3, 9, 24, 10, 12
    cfg = MockConfig(N, A, S, K)
    model = smac_model(N, A)
    inf = SmacInference.from_model(model, device="cuda:0", mode="bf16")
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    factor = np.random.RandomState(5).randint(0, A, size=(B, N)).astype(np.int32)
    shared = SampledMCTS(cfg, np.random.RandomState(0))
    looped = []
    for cur in (0, 1, 2, 1):
        shared.np_random = np.random.RandomState(100 + cur)
        looped.append(shared.batch_search(inf, out0, cur, factor, N, None, "cuda:0", add_noise=True))
    assert len(shared._plans) == 1
    plan = next(iter(shared._plans.values()))
    assert plan.native is not None or sorted(plan.graphs) == [0, 1, 2]     # (the native search keeps its graphs in the library)
    fresh = SampledMCTS(cfg, np.random.RandomState(101)).batch_search(inf, out0, 1, factor, N, None, "cuda:0", add_noise=True)
    for o in (looped[1], looped[3]):
        assert np.array_equal(o.value, fresh.value)
        assert np.array_equal(o.marginal_visit_count, fresh.marginal_visit_count)
        assert o.sampled_qvalues == fresh.sampled_qvalues


def test_new_instances_reuse_the_cached_device_objects(built_lib):
    """The workers build a new SampledMCTS per environment step / per agent (selfplay_worker.py:191, reanalyze_worker.py:284):
    packed weights, tree arena, hidden-state pool and captured graphs are cached per process, keyed by the model object and
    the problem shape, and a search through a new instance gives the same bits as through the first one."""
    from mazero_b200 import mcts_sampled
    from mazero_b200.mcts_sampled import SampledMCTS

    N, A, B, K, S = 3, 9, 16, 5, 10
    cfg = MockConfig(N, A, S, K)
    model = smac_model(N, A).cuda()
    model.hidden_state_size_per_agent = model.hidden
    out0 = root_output(smac_model(N, A), B)
    out0 = out0._replace(hidden_state=out0.hidden_state.cuda())
    first = SampledMCTS(cfg, np.random.RandomState(3))
    r1 = first.batch_search(model, out0, 1, None, N, None, torch.device("cuda:0"), add_noise=True)
    second = SampledMCTS(cfg, np.random.RandomState(3))
    r2 = second.batch_search(model, out0, 1, None, N, None, torch.device("cuda:0"), add_noise=True)
    assert next(iter(first._plans.values())) is next(iter(second._plans.values()))
    assert next(iter(first._inference.values())) is next(iter(second._inference.values()))
    assert np.array_equal(r1.value, r2.value) and np.array_equal(r1.marginal_visit_count, r2.marginal_visit_count)
    assert r1.sampled_qvalues == r2.sampled_qvalues
    # another configuration of the search constants: the native search takes them per call (its graphs are keyed by them inside
    # the library), so the plan IS shared and the new constants take effect (tests/test_search_native_gpu.py)
    cfg2 = MockConfig(N, A, S, K)
    cfg2.discount = 0.9
    third = SampledMCTS(cfg2, np.random.RandomState(3))
    r3 = third.batch_search(model, out0, 1, None, N, None, torch.device("cuda:0"), add_noise=True)
    assert next(iter(third._plans.values())) is next(iter(first._plans.values()))
    assert not all(np.array_equal(a, b) for a, b in zip(r3.sampled_qvalues, r1.sampled_qvalues))
    # another batch size does not
    out1 = out0._replace(hidden_state=out0.hidden_state[:B - 1], reward=out0.reward[:B - 1], value=out0.value[:B - 1],
                         policy_logits=out0.policy_logits[:B - 1])
    fourth = SampledMCTS(cfg, np.random.RandomState(3))
    fourth.batch_search(model, out1, 1, None, N, None, torch.device("cuda:0"), add_noise=True)
    assert next(iter(fourth._plans.values())) is not next(iter(first._plans.values()))
    n = len(mcts_sampled._PLAN_CACHE)
    mcts_sampled.clear_caches()
    assert n >= 2 and not mcts_sampled._PLAN_CACHE
