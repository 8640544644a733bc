"""GPU: the fused tensor-core inference path against a plain PyTorch fp32 reference."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


from mazero_b200.fused import pack_operand  # noqa: E402  (host-side packing under test as well)


@pytest.mark.parametrize("n,k", [(128, 128), (64, 64), (256, 128), (16, 32), (128, 272), (32, 144)])
def test_umma_gemm_stage(built_lib, n, k):
    from mazero_b200 import _lib

    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(n * 1000 + k)
    a = torch.randn(128, k, generator=g).to(dev)
    w = (torch.randn(n, k, generator=g) / k ** 0.5).to(dev)
    out = torch.full((128, n), float("nan"), device=dev)
    wp = pack_operand(w).contiguous()
    _lib.check(_lib.lib.maz_dbg_umma_gemm(a.data_ptr(), wp.data_ptr(), out.data_ptr(), n, k,
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    ref = a.to(torch.bfloat16).float() @ w.to(torch.bfloat16).float().t()   # bf16 operands, fp32 accumulate
    err = (out - ref).abs().max().item()
    assert err < 2e-3, f"max abs err {err}"     # fp32 accumulation-order noise only


NARROW = [(3, 9, 100), (5, 11, 70), (10, 18, 33), (27, 36, 9), (1, 5, 130), (2, 3, 16), (2, 40, 20),
          (30, 17, 5), (3, 9, 1), (27, 36, 1300),    # 1300 x 27: 325 tiles = more than one wave of tile pairs
          (8, 12, 40), (16, 6, 10)]                  # teams that fill a 32-row warp exactly
# 49 to 128 actions (KA > 48): the wide instances of the twin and small-batch kernels (the first generation refuses them)
WIDE = [(2, 49, 301),       # the smallest wide KA (64)
        (2, 70, 301),       # 2c_vs_64zg
        (3, 113, 70),       # KA = 128 with 15 padding columns; 30-row quadrants
        (27, 65, 30),       # KA = 80: the twin's column part 2 has one TMEM block; one root per quadrant
        (8, 100, 40), (1, 128, 130),
        (2, 128, 20000)]    # 313 twin tiles: more than one wave of tile pairs
CASES = [(*s, k) for s in NARROW for k in ("twin", "tcgen05", "small")] + [(*s, k) for s in WIDE for k in ("twin", "small")]


def _close64(name, got, want, rtol, atol=1e-30):
    """A kernel output against a float64 restatement from the kernel's own logits; prints the largest relative error."""
    got, want = got.double(), want.double()
    big = want.abs() > atol
    rel = ((got - want).abs() / want.abs())[big].max().item()
    print(f"{name}: max rel err {rel:.3g} (rtol {rtol:g})")
    assert torch.allclose(got, want, rtol=rtol, atol=atol), f"{name}: max rel err {rel}"


@pytest.mark.parametrize("N,A,B,kernel", CASES)
def test_fused_recurrent_inference_matches_fp32_reference(built_lib, N, A, B, kernel):
    """bf16 tensor-core kernels (tcgen05 128-row tiles; small-batch 32-row tiles on warp-level MMAs) vs the plain fp32 torch
    forward (same weights).  Tolerance: bf16 operand
    rounding (2^-8 relative) through ~20 chained GEMMs -> 2% of each tensor's dynamic range (max |ref|,
    at least 1); probabilities 1e-2 absolute.  The epilogue (softmax, beta, greedy) is fp32 arithmetic on the kernel's own
    logits: it is checked in float64 from those logits, in joint mode and in sequential mode for the first and the last agent."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import random_state_dict

    dev = torch.device("cuda:0")
    sd = random_state_dict(N, A, seed=N, head_scale=30.0)   # heads large enough to give non-uniform policies
    ref = SmacInference(sd, N, A, device=dev, mode="fp32")
    fus = SmacInference(sd, N, A, device=dev, mode="bf16")
    g = torch.Generator().manual_seed(B)
    S = 3
    pool = torch.randn(S, B, N * 128, generator=g).to(dev)
    idx = torch.randint(0, S, (B,), generator=g).to(torch.int32).to(dev)
    act = torch.randint(0, A, (B, N), generator=g).to(torch.int32).to(dev)
    act[0] = 0                     # the one-hot edges: the first and the last action of every agent
    act[1:2] = A - 1
    h = pool.view(-1, N * 128).index_select(0, idx.long() * B + torch.arange(B, device=dev))
    nxt_ref, rew_ref, val_ref, log_ref = ref.recurrent(h, act)

    nxt = torch.full((B, N * 128), float("nan"), device=dev)
    rew = torch.full((B,), float("nan"), device=dev)
    val = torch.full((B,), float("nan"), device=dev)
    probs = torch.full((B, N, A), float("nan"), device=dev)
    beta = torch.full((B, N, A), float("nan"), device=dev)
    logits = torch.full((B, N, A), float("nan"), device=dev)
    greedy = torch.full((B, N), -1, dtype=torch.int32, device=dev)
    fus.recurrent_fused(B, pool, idx, act, nxt, rew, val, probs, beta, greedy, logits, kernel=kernel)
    torch.cuda.synchronize()
    for name, x, y, rel in (("next_hidden", nxt, nxt_ref, 2e-2), ("policy_logits", logits, log_ref, 2e-2),
                            ("reward", rew, rew_ref, 4e-2), ("value", val, val_ref, 4e-2),   # + the steep inv_h transform
                            ("probs", probs, torch.softmax(log_ref, -1), 1e-2)):
        assert torch.isfinite(x).all(), name
        err = (x - y).abs().max().item()
        tol = rel * max(1.0, y.abs().max().item())
        print(f"{name}: max abs err {err:.4g} (tol {tol:.3g}, ref range {y.abs().max().item():.3g})")
        assert err < tol, f"{name}: max abs err {err} > {tol}"
    assert torch.allclose(beta, probs / probs.sum(-1, keepdim=True), atol=1e-6)
    assert torch.allclose(probs.sum(-1), torch.ones(B, N, device=dev), atol=1e-5)
    # greedy = argmax of the kernel's own logits
    assert torch.equal(greedy.long(), logits.argmax(-1))
    # the epilogue in float64 from the kernel's own logits (at ~1/128 per action the 1e-2 bound above cannot see a wrong column)
    p64, b64 = torch.softmax(logits.double(), -1), torch.softmax(logits.double() * 0.5, -1)
    _close64("probs vs softmax(own logits)", probs, p64, 2e-5)
    assert (probs.double().sum(-1) - 1).abs().max().item() <= 1e-5
    # negative control: the next-hidden comparison above sees every action shifted by one
    nxt_bad = torch.full_like(nxt, float("nan"))
    fus.recurrent_fused(B, pool, idx, (act + 1) % A, nxt_bad, rew.clone(), val.clone(), probs.clone(), beta.clone(), kernel=kernel)
    torch.cuda.synchronize()
    bad = (nxt_bad - nxt_ref).abs().max().item() / max(1.0, nxt_ref.abs().max().item())
    print(f"next_hidden with every action shifted by one: {bad:.4g} of the range (tol 2e-2)")
    assert bad >= 2 * 2e-2
    # sequential mode: only agent `cur` is written, as (B,1,A)
    for cur in sorted({0, N - 1}):
        p1 = torch.full((B, 1, A), float("nan"), device=dev)
        b1 = torch.full((B, 1, A), float("nan"), device=dev)
        fus.recurrent_fused(B, pool, idx, act, nxt, rew, val, p1, b1, None, None, tree_agents=1, cur=cur, inv_tau=0.5, kernel=kernel)
        torch.cuda.synchronize()
        assert torch.allclose(p1[:, 0], probs[:, cur], atol=1e-6)
        bt = probs[:, cur] ** 0.5
        assert torch.allclose(b1[:, 0], bt / bt.sum(-1, keepdim=True), atol=1e-4)
        _close64(f"sequential cur={cur}: probs", p1[:, 0], p64[:, cur], 2e-5)
        _close64(f"sequential cur={cur}: beta at tau 2", b1[:, 0], b64[:, cur], 1e-4)
    # joint mode with a sampling temperature: every agent's beta = probs^(1/tau) renormalised (mcts_sampled.py:160)
    p2 = torch.full((B, N, A), float("nan"), device=dev)
    b2 = torch.full((B, N, A), float("nan"), device=dev)
    fus.recurrent_fused(B, pool, idx, act, nxt, rew, val, p2, b2, None, None, inv_tau=0.5, kernel=kernel)
    torch.cuda.synchronize()
    assert torch.allclose(p2, probs, atol=1e-6)
    bt = probs ** 0.5
    assert torch.allclose(b2, bt / bt.sum(-1, keepdim=True), atol=1e-4)
    _close64("joint beta at tau 2", b2, b64, 1e-4)
    assert (b2.double().sum(-1) - 1).abs().max().item() <= 1e-5


# joint mode keeps the ids it always had; sequential mode (tree_agents = 1, last agent, tau = 2) is the "-seq" twin of each shape
DET = [(27, 36, 300), (5, 11, 1000), (10, 18, 500), (2, 70, 20000), (27, 65, 300)]


@pytest.mark.parametrize("N,A,B,seq", [pytest.param(*s, q, id="-".join(map(str, s)) + ("-seq" if q else ""))
                                       for s in DET for q in (False, True)])
def test_twin_kernel_is_deterministic(built_lib, N, A, B, seq):
    """Race guard for the two-tiles-in-flight kernel (compute-sanitizer is closed on this pool): its epilogue warps are not
    synchronised per stage any more (mbarrier hand-off, quadrant barriers, two CTA-wide barriers), so a shared-memory hazard
    would show as run-to-run differences.  200 launches on the same inputs, interleaved with launches of another size (different
    timing), must give bit-identical outputs.  Sequential mode returns from the policy epilogue without the joint-mode staging
    barriers: the quadrant barrier at its end keeps tile 1's exchange writes behind every warp's reads of tile 0's."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.synthetic import random_state_dict

    dev = torch.device("cuda:0")
    fus = SmacInference(random_state_dict(N, A, seed=7, head_scale=30.0), N, A, device=dev, mode="bf16")
    g = torch.Generator().manual_seed(B)
    pool = torch.randn(2, B, N * 128, generator=g).to(dev)
    idx = torch.zeros(B, dtype=torch.int32, device=dev)
    act = torch.randint(0, A, (B, N), generator=g).to(torch.int32).to(dev)

    Nt = 1 if seq else N
    mode = dict(tree_agents=1, cur=N - 1, inv_tau=0.5) if seq else {}

    def launch(b):
        out = [torch.zeros(b, N * 128, device=dev), torch.zeros(b, device=dev), torch.zeros(b, device=dev),
               torch.zeros(b, Nt, A, device=dev), torch.zeros(b, Nt, A, device=dev), torch.zeros(b, N, dtype=torch.int32, device=dev)]
        fus.recurrent_fused(b, pool[:, :b].contiguous() if b != B else pool, idx[:b], act[:b], *out[:5], out[5], None, kernel="twin",
                            **mode)
        return out

    first = launch(B)
    torch.cuda.synchronize()
    for it in range(200):
        if it % 3 == 1:
            launch(max(1, B // 7))                    # a short launch in between: the next one starts on a differently warm GPU
        cur = launch(B)
        torch.cuda.synchronize()
        for a, b in zip(first, cur):
            assert torch.equal(a, b), f"launch {it} differs"
