"""GPU: the matrix-game configuration (BASELINE configs[0]: 2 agents x 3 actions, 16 roots x 50 sims, K=5).

* the fp32 MLP kernel (csrc/maz_mlp.cu) against outputs of the REAL reference network
  (tests/golden/model_matrix_*.npz, config/matrix/model.py imported in the build container);
* the whole on-device search of that network: every simulation's network outputs recorded and replayed
  through the CPU oracle tree (bit-exact), graph replay == eager, joint and both sequential-agent turns."""
import numpy as np
import pytest
import torch

from test_model_oracle import MODEL_GOLDEN, load_model_golden  # noqa: E402
from test_search_gpu import device_path_replay

pytestmark = pytest.mark.gpu
MATRIX_GOLDEN = [p for p in MODEL_GOLDEN if "matrix" in p]


def _inference(z, sd, n, a, h, mode="fp32"):
    from mazero_b200.inference_mlp import MlpInference

    r0, r1, v0, v1 = [int(x) for x in z["supports"]]
    tsd = {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}
    return MlpInference(tsd, n, a, h, reward_support=(r0, r1), value_support=(v0, v1), device="cuda:0", mode=mode)


@pytest.mark.parametrize("path", MATRIX_GOLDEN, ids=[p.split("model_")[-1][:-4] for p in MATRIX_GOLDEN])
def test_mlp_kernel_matches_reference_network(built_lib, path):
    """fp32 kernel vs the reference's own outputs: same maths, different summation order -> 1e-5 relative on the hidden
    state / logits (the north star's fp32 tolerance), 1e-4 on the scalars behind the steep inverse transform."""
    z, _, sd, (n, a, h, b) = load_model_golden(path)
    inf = _inference(z, sd, n, a, h)
    dev = inf.device
    hidden = torch.from_numpy(z["hidden"]).to(dev)
    act = torch.from_numpy(z["action"]).to(dev)
    pool = torch.stack([torch.zeros_like(hidden), hidden])      # parent rows live at pool index 1
    idx = torch.ones(b, dtype=torch.int32, device=dev)
    nan = lambda *s: torch.full(s, float("nan"), device=dev)
    nxt, rew, val, probs, beta, logits = nan(b, n * h), nan(b), nan(b), nan(b, n, a), nan(b, n, a), nan(b, n, a)
    greedy = torch.full((b, n), -1, dtype=torch.int32, device=dev)
    inf.recurrent_fused(b, pool, idx, act, nxt, rew, val, probs, beta, greedy, logits)
    torch.cuda.synchronize()
    tol = dict(rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(nxt.cpu().numpy(), z["rec_hidden"], **tol)
    np.testing.assert_allclose(logits.cpu().numpy(), z["rec_policy_logits"], **tol)
    np.testing.assert_allclose(rew.cpu().numpy(), z["rec_reward"].reshape(-1), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(val.cpu().numpy(), z["rec_value"].reshape(-1), rtol=1e-4, atol=1e-5)
    p_ref = torch.softmax(torch.from_numpy(z["rec_policy_logits"]), -1).numpy()
    np.testing.assert_allclose(probs.cpu().numpy(), p_ref, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(beta.cpu().numpy(), p_ref / p_ref.sum(-1, keepdims=True), rtol=1e-5, atol=1e-6)
    assert np.array_equal(greedy.cpu().numpy(), z["rec_policy_logits"].argmax(-1))
    # torch-op twin on the device (roots / cross-check) and prediction()
    t_nxt, t_rew, t_val, t_log = inf.recurrent(hidden, act)
    np.testing.assert_allclose(t_nxt.cpu().numpy(), z["rec_hidden"], **tol)
    np.testing.assert_allclose(t_val.cpu().numpy(), z["rec_value"].reshape(-1), rtol=1e-4, atol=1e-5)
    pol, vlog = inf.prediction(hidden)
    np.testing.assert_allclose(pol.cpu().numpy(), z["pred_policy_logits"], **tol)
    np.testing.assert_allclose(vlog.cpu().numpy(), z["pred_value_logits"], **tol)
    # sequential mode: agent `cur` only, temperature 2
    p1, b1 = nan(b, 1, a), nan(b, 1, a)
    inf.recurrent_fused(b, pool, idx, act, nxt, rew, val, p1, b1, None, None, tree_agents=1, cur=1, inv_tau=0.5)
    torch.cuda.synchronize()
    np.testing.assert_allclose(p1[:, 0].cpu().numpy(), p_ref[:, 1], rtol=1e-5, atol=1e-6)
    bt = p_ref[:, 1] ** 0.5
    np.testing.assert_allclose(b1[:, 0].cpu().numpy(), bt / bt.sum(-1, keepdims=True), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("cur", [None, 0, 1])
@pytest.mark.parametrize("kind", ["matrix_vec", "matrix_scalar"])
def test_matrix_search_on_device_replays_bit_exact(built_lib, oracle_built, kind, cur):
    """BASELINE configs[0] shape through the on-device search (reference: CPU ctree plumbing run)."""
    from oracle.search_oracle import NetworkOutput

    path = [p for p in MATRIX_GOLDEN if kind in p][0]
    z, net, sd, (n, a, h, _) = load_model_golden(path)
    inf = _inference(z, sd, n, a, h)
    B, K, S = 16, 5, 50
    hidden = torch.randn(B, n * h, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        pol, v = net.prediction(hidden)
        value = net._inv(v, net.value_support)
    out0 = NetworkOutput(hidden.cuda(), np.zeros((B, 1), np.float32), value.numpy().reshape(B, 1), pol.numpy())
    o, _ = device_path_replay(inf, out0, n, a, B, K, S, cur, oracle_built)
    assert (o.marginal_visit_count.sum(axis=(1, 2)) == S * (n if cur is None else 1)).all()


def test_reference_style_matrix_module_is_adapted(built_lib):
    """A torch module with the matrix network's parameter names is recognised by `SampledMCTS` (device path)."""
    from mazero_b200.inference_mlp import MlpInference
    from mazero_b200.mcts_sampled import SampledMCTS
    from oracle.model_oracle import OracleMatrixMuZeroNet
    from oracle.search_oracle import NetworkOutput
    from _mock import MockConfig

    n, a, B, K, S = 2, 3, 16, 5, 20
    net = OracleMatrixMuZeroNet(n, a).init_like_reference(0).eval().cuda()
    hidden = torch.randn(B, n * 64, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        pol, v = net.prediction(hidden)
        value = net._inv(v, net.value_support)
    out0 = NetworkOutput(hidden, np.zeros((B, 1), np.float32), value.cpu().numpy().reshape(B, 1), pol.cpu().numpy())
    mcts = SampledMCTS(MockConfig(n, a, S, K), np.random.RandomState(3))
    o = mcts.batch_search(net, out0, None, None, n, None, torch.device("cuda:0"), add_noise=True)
    assert isinstance(next(iter(mcts._inference.values())), MlpInference) and len(mcts._plans) == 1
    assert (o.marginal_visit_count.sum(axis=2) == S).all()


@pytest.mark.parametrize("path", MODEL_GOLDEN, ids=[p.split("model_")[-1][:-4] for p in MODEL_GOLDEN])
def test_initial_inference_on_device_matches_reference_network(built_lib, path):
    """`initial_inference` without leaving the GPU (row-wise MLP kernel for the representation network + prediction heads +
    inverse value transform) against the REAL reference networks' outputs, SMAC and matrix families; and a search started
    from those device tensors equals the search started from the same values as host arrays."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS
    from oracle.search_oracle import NetworkOutput
    from _mock import MockConfig

    z, _, sd, (n, a, h, b) = load_model_golden(path)
    tsd = {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}
    if "supports" in z.files:
        inf = _inference(z, sd, n, a, h)
    else:
        inf = SmacInference(tsd, n, a, h, device="cuda:0", mode="fp32")
    obs = torch.from_numpy(z["obs"]).cuda()
    out = inf.initial_inference(obs)
    assert all(t.is_cuda for t in (out.hidden_state, out.reward, out.value, out.policy_logits))
    tol = dict(rtol=1e-5, atol=3e-6)
    np.testing.assert_allclose(out.hidden_state.cpu().numpy(), z["init_hidden"], **tol)
    np.testing.assert_allclose(out.policy_logits.cpu().numpy(), z["init_policy_logits"], **tol)
    np.testing.assert_allclose(out.value.cpu().numpy().reshape(-1), z["init_value"].reshape(-1), rtol=1e-4, atol=1e-5)
    # kernel == its torch twin
    x = obs.reshape(b * n, -1).float()
    np.testing.assert_allclose(inf.rep(x).cpu().numpy(), inf.rep.torch_forward(x).cpu().numpy(), **tol)
    # search from device tensors == search from the same values on the host
    cfg = MockConfig(n, a, 12, 5)
    dev_res = SampledMCTS(cfg, np.random.RandomState(4)).batch_search(inf, out, 0, None, n, None, "cuda:0", add_noise=True)
    host_out = NetworkOutput(out.hidden_state, out.reward.cpu().numpy(), out.value.cpu().numpy(), out.policy_logits.cpu().numpy())
    host_res = SampledMCTS(cfg, np.random.RandomState(4)).batch_search(inf, host_out, 0, None, n, None, "cuda:0", add_noise=True)
    for f in dev_res._fields:
        x, y = getattr(dev_res, f), getattr(host_res, f)
        assert np.array_equal(x, y) if isinstance(y, np.ndarray) else x == y, f
