"""CPU: networks with 49 to 128 actions per agent (e.g. 2c_vs_64zg, 70 actions) on the fused path.

* `fused.supported` accepts up to 128 actions;
* the weight packings of the small-batch kernel (row-major, one 34 816-byte ring slot per chunk) and of the twin kernel (K-pieces of
  <= 64 features, bf16 one-hot tables) hold the one-hot blocks and fc_policy.3 at 70 and 128 actions;
* the large-batch kernel choice is the twin kernel above 48 actions, and the first-generation kernel is refused there;
* the launch entries reject 129 actions, and the first-generation layout (tc_layout 0) at 70 actions, before any CUDA call."""
import ctypes

import pytest
import torch

from mazero_b200 import fused
from mazero_b200.synthetic import exact_state_dict, random_state_dict

H, PH = 128, 32
SLOT_BYTES = 128 * (H + 8) * 2          # one weight-ring slot of the small-batch kernel (csrc/infer_hmma.cuh)


def _unpack_operand(flat, rows, k):
    """inverse of fused.pack_operand (no swizzle): [rows/8][k/8][8][8] -> [rows, k]"""
    return flat.view(rows // 8, k // 8, 8, 8).permute(0, 2, 1, 3).reshape(rows, k)


def _onehot_blocks(sd, A):
    g = lambda k: sd[k].float()
    d = "dynamics_network."
    r = d + "reward_predictor."
    w_in = g(d + "attention_stack.0.weight")
    wd1 = g(d + "fc_dynamic.0.weight")
    wr1 = torch.cat([g(r + "gc1.lin_layer.weight"), g(r + "nn_gc1.weight")], 0)
    pol3 = g("prediction_network.fc_policy.3.weight")
    return w_in[:, H:H + A], wd1[:, H:H + A], wr1[:, H:H + A], pol3


@pytest.mark.parametrize("A", [49, 70, 128, 129])
def test_supported_up_to_128_actions(A):
    assert fused.supported(random_state_dict(2, A, seed=0), 2, A, H) == (A <= 128)


@pytest.mark.parametrize("A", [70, 128])
def test_small_batch_packing_roundtrip(built_lib, A):
    N = 2
    sd = random_state_dict(N, A, seed=4)
    fp = fused.FusedParams(sd, N, A, "cpu")
    KA = fp.KA
    assert KA == (A + 15) // 16 * 16
    assert len(fp.chunk_bytes_h) == fused.NCHUNK
    for off, nbytes in zip(fp.chunk_off_h, fp.chunk_bytes_h):
        assert off % 16 == 0 and nbytes % 16 == 0 and 0 < nbytes <= SLOT_BYTES
    raw = fp.wpk_h

    def chunk(i, rows, k):
        assert fp.chunk_bytes_h[i] == rows * (k + 8) * 2
        t = raw[fp.chunk_off_h[i] // 2: fp.chunk_off_h[i] // 2 + rows * (k + 8)].view(rows, k + 8)
        assert not t[:, k:].any()                             # the ldmatrix padding
        return t[:, :k]

    w_in, wd1, wr1, pol3 = _onehot_blocks(sd, A)
    pad = lambda w: torch.cat([w, torch.zeros(w.shape[0], KA - A)], 1)
    assert torch.equal(chunk(1, H, KA), pad(w_in).to(torch.bfloat16))           # in-proj, one-hot block
    assert torch.equal(chunk(21, H, KA), pad(wd1).to(torch.bfloat16))           # fc_dynamic.0, one-hot block
    nq = fused.lib.maz_infer_small_nq()
    fw = 64 // nq
    inter = torch.cat([torch.cat([wr1[fw * q:fw * (q + 1)], wr1[64 + fw * q:64 + fw * (q + 1)]]) for q in range(nq)])
    assert torch.equal(chunk(26, H, KA), pad(inter).to(torch.bfloat16))        # reward graph net layer 1, one-hot block
    pol = torch.zeros(KA, PH)
    pol[:A] = pol3
    assert torch.equal(chunk(31, KA, PH), pol.to(torch.bfloat16))               # fc_policy.3, KA rows
    bp2 = fp.vec[fp.off["pol"] + 96: fp.off["pol"] + 96 + KA]
    assert torch.equal(bp2[:A], sd["prediction_network.fc_policy.3.bias"].float()) and not bp2[A:].any()


@pytest.mark.parametrize("A", [70, 128])
def test_twin_packing_roundtrip(built_lib, A):
    N = 2
    sd = random_state_dict(N, A, seed=5)
    fp = fused.FusedParams(sd, N, A, "cpu")
    KA = fp.KA
    raw = fp.wpk_t
    # fc_policy.3 (the last matrix): KA x 32, one K-piece of 32 features
    i = fused.NCHUNK - 1
    assert fp.chunk_bytes_t[i] == KA * PH * 2 <= 16384
    pol = torch.zeros(KA, PH)
    pol[:A] = _onehot_blocks(sd, A)[3]
    assert torch.equal(_unpack_operand(raw[fp.chunk_off_t[i] // 2: fp.chunk_off_t[i] // 2 + KA * PH], KA, PH), pol.to(torch.bfloat16))
    # no other matrix depends on A: every K-piece is <= 64 features and <= 16 KB
    for off, nbytes in zip(fp.chunk_off_t, fp.chunk_bytes_t):
        assert off % 16 == 0 and nbytes <= 2 * 16384
    # one-hot blocks: [A][128] bf16 tables behind the parameter vector
    for off, w in zip(fp.off_oh, _onehot_blocks(sd, A)[:3]):
        assert off % 8 == 0
        tab = fp.vec_t[off:off + A * H // 2].contiguous().view(torch.bfloat16).view(A, H)
        assert torch.equal(tab, w.to(torch.bfloat16).t())
    assert fp.vec_t.numel() == fp.off_oh[2] + A * H // 2


def test_wide_networks_select_the_twin_kernel(built_lib, monkeypatch):
    monkeypatch.delenv("MAZ_INFER_TC", raising=False)
    # the cost model alone would take the first-generation kernel for these (B, N): not above 48 actions
    assert not fused.use_twin(16384, 3) and not fused.use_twin(16384, 3, 48) and not fused.use_twin(1024, 10, 18)
    assert fused.use_twin(16384, 3, 49) and fused.use_twin(1024, 10, 70) and fused.use_twin(16384, 2, 128)
    monkeypatch.setenv("MAZ_INFER_TC", "twin")
    assert fused.use_twin(16384, 2, 70)
    monkeypatch.setenv("MAZ_INFER_TC", "v1")
    assert not fused.use_twin(16384, 3, 48)
    with pytest.raises(ValueError, match="at most 48 actions"):
        fused.use_twin(16384, 2, 70)
    monkeypatch.delenv("MAZ_INFER_TC")
    fp = fused.FusedParams(exact_state_dict(2, 70, seed=0), 2, 70, "cpu")
    d = fp.desc(16384, None, None, None, None, None, None, None, None)
    assert d.tc_layout == 1 and d.KA == d.NAP == 80
    with pytest.raises(ValueError, match="at most 48 actions"):
        fp.desc(16384, None, None, None, None, None, None, None, None, twin=False)
    assert fp.desc(64, None, None, None, None, None, None, None, None, small=True).tc_layout == 0


def _desc(N, A, tc_layout):
    d = fused.InferDesc()
    d.B, d.N, d.A = 64, N, A
    d.KA = d.NAP = (A + 15) // 16 * 16
    d.Nt, d.cur, d.inv_tau = N, -1, 1.0
    d.tc_layout = tc_layout
    return d


def test_launch_entries_reject_unsupported_action_counts(built_lib):
    from mazero_b200 import _lib

    lib = _lib.lib
    for tc_layout in (0, 1):
        assert lib.maz_infer_recurrent(ctypes.byref(_desc(2, 129, tc_layout)), None) == _lib.MAZ_ERR_UNSUPPORTED
        assert "128" in _lib.last_error()
    assert lib.maz_infer_recurrent_small(ctypes.byref(_desc(2, 129, 0)), None) == _lib.MAZ_ERR_UNSUPPORTED
    assert "128" in _lib.last_error()
    assert lib.maz_infer_recurrent(ctypes.byref(_desc(2, 70, 0)), None) == _lib.MAZ_ERR_UNSUPPORTED
    assert "first-generation" in _lib.last_error()
    # inside the limits the shape passes and the (NULL) buffers are what is refused
    assert lib.maz_infer_recurrent(ctypes.byref(_desc(2, 70, 1)), None) == _lib.MAZ_ERR_INVALID
    assert lib.maz_infer_recurrent_small(ctypes.byref(_desc(2, 128, 0)), None) == _lib.MAZ_ERR_INVALID
