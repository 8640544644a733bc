"""GPU: `SmacInference.initial_inference(obs, fused=True)` -- the bf16 root-inference kernel (csrc/infer_initial.cuh,
`maz_infer_initial`): feature_norm + representation mlp + prediction heads + inverse value transform in one launch.

Right-hand side of the accuracy asserts: a float64 restatement, `OracleMAMuZeroNet.initial_inference` run in float64.  Its
representation network and heads are the reference's (oracle/model_oracle.py, pinned to the real network by
tests/test_model_oracle.py).  Tolerances: `TOL_BF16` of tests/test_infer128_gpu.py, as a fraction of max(1, max|ref|)."""
import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_infer128_gpu import TOL_BF16, _relerr
from test_search_native_gpu import _equal

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAMES = ("hidden", "policy_logits", "value")


def _net(N, A, obs, seed=0):
    """Reference-initialised network with non-zero biases and LayerNorm affines, and output heads scaled to O(1) logits, so
    that every bias and every head weight shows in the outputs."""
    from oracle.model_oracle import OracleMAMuZeroNet

    net = OracleMAMuZeroNet(N, A, obs_size=obs).init_like_reference(seed)
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith("bias"):
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
            elif p.dim() == 1:                                   # LayerNorm weights
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
        net.prediction_network.fc_policy[-1].weight.mul_(2000.0)
        net.prediction_network.value_predictor.V.weight.mul_(300.0)
    return net


def _obs(B, N, obs, seed=0):
    """Observations with per-row offsets and scales (1, 50 / 500 offset / 0.05 at -20): feature_norm has work to do."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B * N, obs, generator=g)
    sel = torch.arange(B * N) % 4
    scale = torch.tensor([1.0, 50.0, 1.0, 0.05])[sel]
    offset = torch.tensor([0.0, 0.0, 500.0, -20.0])[sel]
    return (x * scale[:, None] + offset[:, None]).view(B, N, obs)


def _reference(net, obs):
    """float64 restatement on the device: (hidden, policy_logits, value)"""
    import copy

    ref = copy.deepcopy(net).double().to(DEV)
    h, v, p = ref.initial_inference(obs.to(DEV, torch.float64))
    return h, p, v


def _fused(inf, obs):
    out = inf.initial_inference(obs.to(DEV), fused=True)
    torch.cuda.synchronize()
    return out.hidden_state, out.policy_logits, out.value


def _check(got, ref, what, factor=1.0):
    errs = {}
    for name, x, y in zip(NAMES, got, ref):
        assert torch.isfinite(x).all(), f"{what} {name}"
        e = _relerr(x.double(), y.cpu().numpy())
        errs[name] = e
        print(f"{what} {name}: {e:.3g} (tol {TOL_BF16[name] * factor:.3g})")
        assert e <= TOL_BF16[name] * factor, f"{what} {name}: {e}"
    return errs


# (N, A, obs_dim, B): every team shape of the issue, every obs_dim, B = 1, ragged last tiles, 1536 (reanalyze), 20 000
CASES = [
    (3, 9, 16, 1), (3, 9, 285, 1536), (3, 9, 640, 20000),
    (5, 11, 37, 13), (5, 11, 640, 1536),
    (10, 18, 285, 77), (10, 18, 16, 1),
    (27, 36, 640, 1536), (27, 36, 37, 3),
    (2, 70, 37, 20000), (2, 70, 640, 37),
    (2, 128, 640, 1536), (2, 128, 16, 1), (2, 128, 285, 999),
]


@pytest.mark.parametrize("N,A,obs,B", CASES, ids=[f"N{n}-A{a}-obs{o}-B{b}" for n, a, o, b in CASES])
def test_fused_initial_inference_matches_float64_restatement(built_lib, N, A, obs, B):
    from mazero_b200.inference import SmacInference

    net = _net(N, A, obs, seed=N + A + obs)
    inf = SmacInference(net.state_dict(), N, A, device=DEV, mode="bf16")
    x = _obs(B, N, obs, seed=B)
    got = _fused(inf, x)
    assert got[0].shape == (B, N * 128) and got[1].shape == (B, N, A) and got[2].shape == (B, 1)
    _check(got, _reference(net, x), f"N{N} A{A} obs{obs} B{B}")


@pytest.mark.parametrize("control", ["feature_norm_bias", "last_representation_bias"])
def test_negative_controls(built_lib, control):
    """A packing without feature_norm.bias, or without mlp.6.bias, must miss the restatement's hidden state by more than twice
    the tolerance: the comparison above can see a dropped bias."""
    from mazero_b200.inference import SmacInference

    N, A, obs, B = 3, 9, 37, 300
    net = _net(N, A, obs, seed=7)
    inf = SmacInference(net.state_dict(), N, A, device=DEV, mode="bf16")
    x = _obs(B, N, obs, seed=3)
    ref = _reference(net, x)
    _check(_fused(inf, x), ref, "intact")
    kp = (obs + 15) // 16 * 16
    if control == "feature_norm_bias":
        inf.fused.rep_vec[kp:2 * kp].zero_()
    else:
        inf.fused.rep_vec[2 * kp + 6 * 128:].zero_()
    e = _relerr(_fused(inf, x)[0].double(), ref[0].cpu().numpy())
    print(f"{control} dropped: hidden error {e:.3g} (tol {TOL_BF16['hidden']:.3g})")
    assert e > 2 * TOL_BF16["hidden"]


@pytest.mark.parametrize("N,A,obs,B", [(3, 9, 37, 1536), (27, 36, 285, 300), (2, 70, 640, 1024), (2, 128, 16, 77)])
def test_same_answer_as_the_fp32_path(built_lib, N, A, obs, B):
    from mazero_b200.inference import SmacInference

    net = _net(N, A, obs, seed=11)
    sd = net.state_dict()
    x = _obs(B, N, obs, seed=5).to(DEV)
    f = SmacInference(sd, N, A, device=DEV, mode="fp32").initial_inference(x)
    ref = (f.hidden_state, f.policy_logits, f.value)
    got = _fused(SmacInference(sd, N, A, device=DEV, mode="bf16"), x)
    _check(got, ref, f"vs fp32 N{N} A{A}")
    # greedy action per (root, agent) wherever the fp32 top-2 logit gap is clear of the bf16 tolerance
    ref_logits = ref[1]
    top2 = ref_logits.topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 2 * TOL_BF16["policy_logits"] * max(1.0, ref_logits.abs().max().item())
    print(f"clear top-2 gap for {100 * clear.float().mean().item():.1f}% of (root, agent)")
    assert torch.equal(got[1].argmax(-1)[clear], ref_logits.argmax(-1)[clear])
    assert clear.float().mean().item() > 0.25


@pytest.mark.parametrize("N,A,obs,B", [(27, 36, 285, 1536), (2, 128, 640, 999)])
def test_deterministic(built_lib, N, A, obs, B):
    from mazero_b200.inference import SmacInference

    inf = SmacInference(_net(N, A, obs, seed=2).state_dict(), N, A, device=DEV, mode="bf16")
    x = _obs(B, N, obs, seed=9).to(DEV)
    first = [t.clone() for t in _fused(inf, x)]
    for _ in range(50):
        out = inf.initial_inference(x, fused=True)
        for a, b in zip(first, (out.hidden_state, out.policy_logits, out.value)):
            assert torch.equal(a, b)
    torch.cuda.synchronize()


def test_weight_update_reaches_the_kernel(built_lib):
    """`load_state_dict` of new weights: the inference object SampledMCTS caches for the model notices (change signature),
    refreshes, and the next fused=True call computes with the new weights."""
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches

    N, A, obs, B = 5, 11, 37, 200
    model = _net(N, A, obs, seed=21).to(DEV)
    mcts = SampledMCTS(MockConfig(N, A, 10, 5), np.random.RandomState(0), inference_mode="bf16")
    x = _obs(B, N, obs, seed=4)
    inf = mcts._device_inference(model, DEV)
    before = _fused(inf, x)
    _check(before, _reference(model, x), "before")
    model.load_state_dict(_net(N, A, obs, seed=22).state_dict())
    inf2 = mcts._device_inference(model, DEV)
    assert inf2 is inf                                       # the cached object, refreshed in place
    after = _fused(inf2, x)
    _check(after, _reference(model, x), "after")
    assert not torch.equal(before[0], after[0])
    clear_caches()


@pytest.mark.parametrize("turn", ["greedy", "sample"])
@pytest.mark.parametrize("shape", ["3m", "2c_vs_64zg"])
def test_fused_roots_feed_search_agents(built_lib, shape, turn):
    """search_agents started from the fused outputs as CUDA tensors equals search_agents started from the same values as host
    numpy arrays, bit for bit: every agent's SearchOutput, the turn results and the generator state."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS, clear_caches
    from mazero_b200.synthetic import WORKLOADS, NetworkOutput

    N, A, _, _, K = WORKLOADS[shape]
    B, S, obs = 64, 20, 64
    inf = SmacInference(_net(N, A, obs, seed=31).state_dict(), N, A, device=DEV, mode="bf16")
    root = inf.initial_inference(_obs(B, N, obs, seed=6).to(DEV), fused=True)
    host = NetworkOutput(root.hidden_state.clone(), root.reward.cpu().numpy(), root.value.cpu().numpy(),
                         root.policy_logits.cpu().numpy())
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1
    rng = np.random.RandomState(9)
    eps_u = rng.rand(N, B).astype(np.float32)
    rand_act = np.stack([[rng.choice(np.where(legal[b, k] > 0)[0]) for b in range(B)] for k in range(N)]).astype(np.int32)
    kw = dict(add_noise=True, sampled_tau=1.0, turn=turn, temperature=0.5, greedy_epsilon=0.3,
              eps_randoms=(eps_u, rand_act) if turn == "sample" else None)
    outs, states = [], []
    for r in (root, host):
        mcts = SampledMCTS(MockConfig(N, A, S, K), np.random.RandomState(21))
        outs.append(mcts.search_agents(inf, r, N, legal, DEV, **kw))
        states.append(mcts.np_random.get_state()[1])
        clear_caches()
    a, b = outs
    for f in ("actions", "policy_dist", "prob", "entropy"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    for k in range(N):
        _equal(a.search_outputs[k], b.search_outputs[k], f"agent {k}: ")
    assert np.array_equal(states[0], states[1])


def test_default_path_is_untouched(built_lib):
    """initial_inference(obs) without `fused`: the row-wise kernel for the representation and torch ops for the heads, bit for
    bit, also on a bf16 object."""
    from mazero_b200.inference import SmacInference

    N, A, obs, B = 5, 11, 37, 300
    sd = _net(N, A, obs, seed=41).state_dict()
    x = _obs(B, N, obs, seed=8).to(DEV)
    for mode in ("fp32", "bf16"):
        inf = SmacInference(sd, N, A, device=DEV, mode=mode)
        out = inf.initial_inference(x)
        hidden = inf.rep(x.reshape(B * N, obs)).view(B, N * 128)
        pol, vlog = inf.prediction(hidden)
        value = inf._inv_transform(vlog, inf.vsup).reshape(B, 1)
        torch.cuda.synchronize()
        assert torch.equal(out.hidden_state, hidden) and torch.equal(out.policy_logits, pol) and torch.equal(out.value, value)
        assert not out.reward.any()


def test_fused_needs_bf16_and_a_supported_representation(built_lib):
    from mazero_b200.inference import SmacInference

    N, A, obs = 3, 9, 37
    sd = _net(N, A, obs).state_dict()
    x = _obs(2, N, obs).to(DEV)
    with pytest.raises(ValueError, match="bf16"):
        SmacInference(sd, N, A, device=DEV, mode="fp32").initial_inference(x, fused=True)
    sd2 = {k: v for k, v in sd.items() if "feature_norm" not in k}
    with pytest.raises(ValueError, match="feature_norm"):
        SmacInference(sd2, N, A, device=DEV, mode="bf16").initial_inference(x, fused=True)
