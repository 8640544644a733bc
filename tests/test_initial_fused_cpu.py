"""CPU: the root-inference kernel's host side (`maz_infer_initial`, csrc/infer_initial.cuh).

* `fused.supported_initial` takes the reference representation network (feature_norm + mlp([obs, 128, 128, 128])) on top of the
  heads `fused.supported` takes, and rejects each deviation;
* the representation packing (bf16 column blocks of mlp.0, mlp.3, mlp.6; one fp32 vector) round-trips to the state dict;
* the C entry checks its arguments before any CUDA call and, without a GPU, fails with MAZ_ERR_CUDA (no CPU fallback)."""
import ctypes

import pytest
import torch

from mazero_b200 import _lib, fused
from oracle.model_oracle import OracleMAMuZeroNet

H = 128
SLOT_BYTES = 128 * (H + 8) * 2


def _sd(N, A, obs, hidden=H, layers=None, seed=0):
    net = OracleMAMuZeroNet(N, A, hidden_state_size=hidden, obs_size=obs, fc_representation_layers=layers)
    return net.init_like_reference(seed).state_dict()


def test_supported_initial_accepts_the_reference_shape():
    assert fused.supported_initial(_sd(3, 9, 37), 3, 9, H)
    assert fused.supported_initial(_sd(2, 128, 640), 2, 128, H)


@pytest.mark.parametrize("case", ["hidden64", "no_feature_norm", "layer_too_many", "layer_too_few", "A129", "obs641"])
def test_supported_initial_rejects(case):
    N, A, obs, h = 3, 9, 37, H
    if case == "hidden64":
        h = 64
        sd = _sd(N, A, obs, hidden=64)
    elif case == "no_feature_norm":
        sd = _sd(N, A, obs)
        del sd["representation_network.feature_norm.weight"], sd["representation_network.feature_norm.bias"]
    elif case == "layer_too_many":
        sd = _sd(N, A, obs, layers=(128, 128, 128))
    elif case == "layer_too_few":
        sd = _sd(N, A, obs, layers=(128,))
    elif case == "A129":
        A = 129
        sd = _sd(2, A, obs)
        N = 2
    else:
        sd = _sd(N, A, 641)
    assert not fused.supported_initial(sd, N, A, h)
    assert fused.initial_unsupported_reason(sd, N, A, h)


@pytest.mark.parametrize("A", [9, 70, 128])
@pytest.mark.parametrize("obs", [16, 37, 640])
def test_representation_packing_roundtrip(built_lib, A, obs):
    N = 2
    sd = _sd(N, A, obs, seed=A + obs)
    fp = fused.FusedParams(sd, N, A, "cpu")
    assert fp.obs_dim == obs
    kp = (obs + 15) // 16 * 16
    g = lambda k: sd["representation_network." + k].float()
    raw, o = fp.rep_wpk, 0
    blocks = []
    for k0 in range(0, kp, 128):
        kc = min(128, kp - k0)
        t = raw[o: o + 128 * (kc + 8)].view(128, kc + 8)
        assert not t[:, kc:].any()                                  # the ldmatrix padding
        blocks.append(t[:, :kc])
        o += 128 * (kc + 8)
    w0 = torch.cat(blocks, 1)
    assert torch.equal(w0[:, :obs], g("mlp.0.weight").to(torch.bfloat16)) and not w0[:, obs:].any()
    for name in ("mlp.3.weight", "mlp.6.weight"):
        t = raw[o: o + 128 * 136].view(128, 136)
        assert torch.equal(t[:, :128], g(name).to(torch.bfloat16)) and not t[:, 128:].any()
        o += 128 * 136
    assert o == raw.numel()
    v = fp.rep_vec
    assert v.numel() == 2 * kp + 7 * 128
    assert torch.equal(v[:obs], g("feature_norm.weight")) and not v[obs:kp].any()
    assert torch.equal(v[kp:kp + obs], g("feature_norm.bias")) and not v[kp + obs:2 * kp].any()
    rest = torch.cat([g(k) for k in ("mlp.0.bias", "mlp.1.weight", "mlp.1.bias", "mlp.3.bias", "mlp.4.weight", "mlp.4.bias",
                                     "mlp.6.bias")])
    assert torch.equal(v[2 * kp:], rest)
    # the heads half of the descriptor is the small-batch packing: chunks 27, 28, 30, 31 and vec[o_vg:]
    dsc = fp.initial_desc(5, None, None, None, None)
    assert (dsc.B, dsc.N, dsc.A, dsc.H, dsc.obs_dim) == (5, N, A, H, obs)
    for c in (27, 28, 30, 31):
        assert 0 < dsc.chunk_bytes[c] <= SLOT_BYTES and dsc.chunk_bytes[c] % 16 == 0 and dsc.chunk_off[c] % 16 == 0
    vp = "prediction_network.value_predictor."
    assert torch.equal(fp.vec[dsc.o_vg:dsc.o_vg + 64], sd[vp + "gc1.lin_layer.bias"].float())
    assert torch.equal(fp.vec[dsc.o_pol + 96:dsc.o_pol + 96 + A], sd["prediction_network.fc_policy.3.bias"].float())


def test_repack_refreshes_the_representation_in_place(built_lib):
    N, A, obs = 3, 9, 37
    sd = _sd(N, A, obs, seed=1)
    fp = fused.FusedParams(sd, N, A, "cpu")
    wpk, vec = fp.rep_wpk, fp.rep_vec
    sd2 = _sd(N, A, obs, seed=2)
    sd2["representation_network.feature_norm.bias"] += 0.5
    fp.repack(sd2)
    assert fp.rep_wpk is wpk and fp.rep_vec is vec                    # same storage (captured graphs keep their addresses)
    ref = fused.pack_representation(sd2, "cpu")
    assert torch.equal(wpk, ref[0]) and torch.equal(vec, ref[1])


def _desc(**kw):
    N, A, obs = kw.pop("N", 3), kw.pop("A", 9), kw.pop("obs", 37)
    fp = fused.FusedParams(_sd(min(N, 30), min(A, 128), obs), min(N, 30), min(A, 128), "cpu")
    dsc = fp.initial_desc(4, None, None, None, None)
    dsc.obs = dsc.hidden = dsc.value = dsc.policy_logits = 4096          # never dereferenced: the checks come first
    dsc.N, dsc.A = N, A
    for k, v in kw.items():
        setattr(dsc, k, v)
    return dsc, fp


@pytest.mark.parametrize("change,code", [
    (dict(obs_dim=641), _lib.MAZ_ERR_UNSUPPORTED),
    (dict(N=31), _lib.MAZ_ERR_INVALID),
    (dict(N=0), _lib.MAZ_ERR_INVALID),
    (dict(A=129), _lib.MAZ_ERR_UNSUPPORTED),
    (dict(H=64), _lib.MAZ_ERR_UNSUPPORTED),
    (dict(B=0), _lib.MAZ_ERR_INVALID),
    (dict(hidden=None), _lib.MAZ_ERR_INVALID),
    (dict(value=None), _lib.MAZ_ERR_INVALID),
    (dict(policy_logits=None), _lib.MAZ_ERR_INVALID),
    (dict(obs=None), _lib.MAZ_ERR_INVALID),
], ids=["obs641", "N31", "N0", "A129", "H64", "B0", "hidden_null", "value_null", "logits_null", "obs_null"])
def test_arguments_checked_before_any_cuda_call(built_lib, change, code):
    dsc, _fp = _desc(**change)
    assert _lib.lib.maz_infer_initial(ctypes.byref(dsc), None) == code
    assert "maz_infer_initial" in _lib.last_error()
    assert _lib.lib.maz_infer_initial(None, None) == _lib.MAZ_ERR_INVALID


def test_no_cpu_fallback(built_lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    dsc, _fp = _desc()
    assert _lib.lib.maz_infer_initial(ctypes.byref(dsc), None) == _lib.MAZ_ERR_CUDA
    assert "CUDA" in _lib.last_error() or "device" in _lib.last_error()
