"""GPU: the SURVEY 8(f) rows -- device root preparation (mcts_sampled.py:57-106), the per-agent turn logic of the
workers (selfplay_worker.py:196-257, reanalyze_worker.py:278-345) and the device-resident N-agent pipeline
`SampledMCTS.search_agents` -- against the restated reference logic (oracle/turn_oracle.py, pinned to the reference's
own functions by tests/test_turn_oracle.py)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_search_gpu import root_output, smac_model

pytestmark = pytest.mark.gpu
KAT = os.path.join(os.path.dirname(__file__), "golden", "turns_kat.npz")
DEV = "cuda:0"


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("cur", [None, 0, 2])
@pytest.mark.parametrize("with_legal,tau", [(True, 1.0), (False, 1.0), (True, 2.0)])
@pytest.mark.parametrize("A", [9, 36, 200])
def test_root_prepare_kernel_matches_numpy_block(built_lib, cur, with_legal, tau, A):
    """fp32 on both sides, different exp / summation order: 2e-6 relative (the tree parity tests then use the DEVICE's
    arrays as the injected inputs of the oracle tree)."""
    from mazero_b200._lib import check, lib
    from oracle.turn_oracle import root_prepare

    B, N = 37, 3
    rng = np.random.RandomState(A + (0 if cur is None else cur + 1))
    logits = (rng.randn(B, N, A) * 2).astype(np.float32)
    legal = (rng.rand(B, N, A) < 0.6).astype(np.float32)
    legal[..., 1] = 1
    Nt = N if cur is None else 1
    noises = rng.dirichlet([0.3] * A, B * Nt).astype(np.float32).reshape(B, Nt, A)
    if A == 200:   # every row's maximum twice, the copy before or after it: the greedy action is the first one (np.argmax)
        rows = logits.reshape(B * N, A)
        first = rows.argmax(-1)
        other = (first + rng.randint(1, A, size=B * N)) % A
        rows[np.arange(B * N), other] = rows[np.arange(B * N), first]
        assert np.array_equal(rows.argmax(-1), np.minimum(first, other)) and (other < first).any() and (other > first).any()
    p_ref, b_ref, n_ref = root_prepare(logits, cur, legal.astype(np.float64) if with_legal else None, noises, 0.25, tau)
    d = lambda x: torch.from_numpy(x).to(DEV)
    dl, dm, dn = d(logits), d(legal), d(noises)
    p, b, n = (torch.full((B, Nt, A), float("nan"), device=DEV) for _ in range(3))
    g = torch.full((B, N), -1, dtype=torch.int32, device=DEV)
    check(lib.maz_root_prepare_dev(_ptr(dl), _ptr(dm) if with_legal else None, _ptr(dn), B, N, A, -1 if cur is None else cur,
                                   0.25, 1.0 / tau, _ptr(p), _ptr(b), _ptr(n), _ptr(g), _stream()))
    torch.cuda.synchronize()
    tol = dict(rtol=2e-6, atol=1e-9) if tau == 1.0 else dict(rtol=2e-5, atol=1e-9)    # powf on both sides for tau != 1
    np.testing.assert_allclose(p.cpu().numpy(), p_ref, **tol)
    np.testing.assert_allclose(n.cpu().numpy(), n_ref, **tol)
    np.testing.assert_allclose(b.cpu().numpy(), b_ref, **tol)
    assert np.array_equal(g.cpu().numpy(), logits.argmax(-1))
    if with_legal:   # illegal actions get exactly zero probability, legal ones strictly positive
        m = legal if cur is None else legal[:, cur:cur + 1]
        assert ((p.cpu().numpy() > 0) == (m > 0)).all() and ((b.cpu().numpy() > 0) == (m > 0)).all()


def _agent_turn(mode, B, N, A, K, agent, nchild, sact, svis, mvis, legal, inv_t, uniforms, eps, eps_u, rand_act, actions, dist, prob, ent):
    from mazero_b200._lib import check, lib

    check(lib.maz_agent_turn_dev(mode, B, N, A, K, agent, _ptr(nchild), _ptr(sact), _ptr(svis), _ptr(mvis), _ptr(legal),
                                 float(inv_t), _ptr(uniforms), float(eps), _ptr(eps_u), _ptr(rand_act), _ptr(actions), _ptr(dist),
                                 _ptr(prob), _ptr(ent), _stream()))


def test_agent_turn_sample_reproduces_reference_known_answers(built_lib):
    """select_action + np_random.choice of the reference (tests/golden/turns_kat.npz): positions bit-exact with the
    injected uniform, visit entropy to 1e-12 (device log vs glibc log)."""
    z = np.load(KAT)
    counts, lens, temps = z["counts"], z["lens"], z["temps"]
    M, K = counts.shape
    A = K
    for T in np.unique(temps):
        sel = np.where(temps == T)[0]
        B = len(sel)
        d = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x)).to(dt).to(DEV)
        sact = torch.arange(K, dtype=torch.int32, device=DEV).repeat(B, 1).contiguous()       # action == position
        mvis = d(counts[sel], torch.int32)                                                   # A == K: marginal == counts
        actions = torch.full((B, 1), -1, dtype=torch.int32, device=DEV)
        dist = torch.zeros(B, 1, A, dtype=torch.float64, device=DEV)
        prob = torch.zeros(B, dtype=torch.float64, device=DEV)
        ent = torch.zeros(B, 1, dtype=torch.float64, device=DEV)
        _agent_turn(1, B, 1, A, K, 0, d(lens[sel], torch.int32), sact, d(counts[sel], torch.int32), mvis, None, 1.0 / float(T),
                    d(z["uniforms"][sel], torch.float64), 0.0, None, None, actions, dist, prob, ent)
        torch.cuda.synchronize()
        assert np.array_equal(actions.cpu().numpy()[:, 0], z["pos"][sel]), T
        np.testing.assert_allclose(ent.cpu().numpy()[:, 0], z["entropy"][sel], rtol=1e-12, atol=1e-14)
        ref_dist = counts[sel] / counts[sel].sum(-1, keepdims=True)
        assert np.array_equal(dist.cpu().numpy()[:, 0], ref_dist)                            # float64 quotient: bit-exact
        assert np.array_equal(prob.cpu().numpy(), ref_dist[np.arange(B), z["pos"][sel]])


def test_agent_turn_eps_greedy_and_greedy_modes(built_lib):
    from oracle.turn_oracle import eps_greedy_action

    z = np.load(KAT)
    E, A = z["masks"].shape
    K = 4
    d = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x)).to(dt).to(DEV)
    # SAMPLE with one child whose action is the "greedy" action of the fixture, then the injected epsilon-greedy draws
    nchild = torch.ones(E, dtype=torch.int32, device=DEV)
    sact = torch.zeros(E, K, dtype=torch.int32, device=DEV)
    sact[:, 0] = d(z["greedy"], torch.int32)
    svis = torch.zeros(E, K, dtype=torch.int32, device=DEV)
    svis[:, 0] = 5
    mv = np.zeros((E, A), np.int32)
    mv[np.arange(E), z["greedy"]] = 5
    actions = torch.full((E, 2), -1, dtype=torch.int32, device=DEV)
    dist = torch.zeros(E, 2, A, dtype=torch.float64, device=DEV)
    prob = torch.zeros(E, dtype=torch.float64, device=DEV)
    ent = torch.zeros(E, 2, dtype=torch.float64, device=DEV)
    legal = torch.ones(E, 2, A, device=DEV)
    legal[:, 1] = d(z["masks"], torch.float32)
    _agent_turn(1, E, 2, A, K, 1, nchild, sact, svis, d(mv, torch.int32), legal, 1.0, torch.full((E,), 0.5, dtype=torch.float64, device=DEV),
                float(z["eps"]), d(z["eps_u"], torch.float32), d(z["rand_act"], torch.int32), actions, dist, prob, ent)
    torch.cuda.synchronize()
    got = actions.cpu().numpy()
    assert np.array_equal(got[:, 1], z["eps_result"]) and (got[:, 0] == -1).all()
    assert all(eps_greedy_action(z["greedy"][i], float(z["eps"]), z["eps_u"][i], z["rand_act"][i]) == got[i, 1] for i in range(E))
    # GREEDY: argmax(marginal_visits * legal), first maximum
    rng = np.random.RandomState(0)
    mv = rng.randint(0, 6, size=(E, A)).astype(np.int32)
    mv[:, 0] += 1
    _agent_turn(0, E, 2, A, K, 1, nchild, sact, svis, d(mv, torch.int32), legal, 1.0, None, 0.0, None, None, actions, dist, prob, ent)
    torch.cuda.synchronize()
    assert np.array_equal(actions.cpu().numpy()[:, 1], np.argmax(mv * z["masks"], axis=-1))
    assert np.array_equal(dist.cpu().numpy()[:, 1], mv / mv.sum(-1, keepdims=True))


def test_device_dirichlet_has_the_reference_distribution(built_lib):
    """Opt-in device noise: same distribution as np_random.dirichlet([alpha]*A) (mcts_sampled.py:68), not the same stream."""
    from mazero_b200._lib import check, lib

    rows, A, alpha = 40000, 9, 0.3
    out = torch.full((rows, A), float("nan"), device=DEV)
    check(lib.maz_dirichlet_dev(_ptr(out), rows, A, alpha, 12345, _stream()))
    torch.cuda.synchronize()
    x = out.double().cpu().numpy()
    assert np.isfinite(x).all() and (x >= 0).all()
    np.testing.assert_allclose(x.sum(-1), 1, rtol=1e-5)
    a0 = alpha * A
    mean, var = 1.0 / A, (1.0 / A) * (1 - 1.0 / A) / (a0 + 1)
    assert abs(x.mean(0) - mean).max() < 4 * np.sqrt(var / rows)
    assert abs(x.var(0) - var).max() < 0.05 * var
    ref = np.random.RandomState(0).dirichlet([alpha] * A, rows)
    for q in (0.1, 0.5, 0.9, 0.99):        # marginal Beta(alpha, alpha*(A-1)) quantiles
        assert abs(np.quantile(x[:, 0], q) - np.quantile(ref[:, 0], q)) < 0.02 + 0.05 * np.quantile(ref[:, 0], q)
    out2 = torch.empty_like(out)
    check(lib.maz_dirichlet_dev(_ptr(out2), rows, A, alpha, 12345, _stream()))
    torch.cuda.synchronize()
    assert torch.equal(out, out2)                 # counter-based: reproducible from (seed, row)


@pytest.mark.parametrize("turn", ["greedy", "sample"])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_search_agents_equals_the_workers_host_loop(built_lib, turn, mode):
    """ONE device-resident call for the N per-agent searches == the workers' loop (restated) over N separate
    `batch_search` calls with the host doing the action choice in between: same np_random consumption order, same
    actions, same visit distributions, same SearchOutput of every agent -- bit for bit."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS
    from oracle import turn_oracle

    N, A, B, K, S = 3, 9, 40, 10, 20
    cfg = MockConfig(N, A, S, K)
    model = smac_model(N, A)
    inf = SmacInference.from_model(model, device=DEV, mode=mode)
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
        for f in outs[k]._fields:
            x, y = getattr(got.search_outputs[k], f), getattr(outs[k], f)
            if isinstance(y, np.ndarray):
                assert np.array_equal(x, y), (k, f)
            else:
                assert x == y, (k, f)
    # both host RNG streams are at the same position afterwards
    assert fused.np_random.random_sample() == host_rs.random_sample()
