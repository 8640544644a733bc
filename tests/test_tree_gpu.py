"""GPU parity tests of the tree engine, through the C ABI (mazero_b200.cytree.Tree_batch -> libmaz_b200.so).

Bit-exact against the CPU oracle on identical injected network outputs and identical RNG seeds:
selected actions, hidden-state indices, sampled action sets, visit counts AND every float readout."""
import glob
import os

import numpy as np
import pytest

from _harness import MCTS, SHAPES, Inputs, assert_same, drive, drive_fused
from test_oracle import GOLDEN, check_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cytree(built_lib):
    from mazero_b200 import cytree

    return cytree


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[5:-4] for p in GOLDEN])
def test_cuda_tree_matches_golden(cytree, path):
    check_golden(lambda *a: cytree.Tree_batch(*a), path)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("mode", ["random", "mock", "quantized"])
def test_cuda_tree_matches_oracle(cytree, oracle_built, shape, mode):
    B, N, A, K, S = SHAPES[shape]
    for seed in (0, 1):
        inp = Inputs(B, N, A, S, seed=seed, mode=mode, legal_frac=0.7 if seed else None)
        ours = cytree.Tree_batch(B, N, A, K, S, MCTS["delta_lb"], 3 + seed, MCTS["rho"], MCTS["lam"])
        orc = oracle_built.OracleTreeBatch(B, N, A, K, S, MCTS["delta_lb"], 3 + seed, MCTS["rho"], MCTS["lam"], kind="port")
        assert_same(drive(ours, inp, K), drive(orc, inp, K), exact=True, what=f"{shape}/{mode}/{seed}: ")
        tot, sl, _, _ = ours.stats()
        otot, osl = orc.stats()
        assert np.array_equal(tot, otot) and np.array_equal(sl, osl)


@pytest.mark.parametrize("rho,lam,K", [(0.25, 0.8, 5), (0.0, 1.0, 1), (0.9, 0.5, 10), (0.75, 0.8, 32)])
def test_cuda_tree_other_hyperparameters(cytree, oracle_built, rho, lam, K):
    B, N, A, S = 32, 2, 5, 40
    inp = Inputs(B, N, A, S, seed=5, mode="random")
    mcts = dict(MCTS, rho=rho, lam=lam)
    ours = cytree.Tree_batch(B, N, A, K, S, 0.01, 99, rho, lam)
    orc = oracle_built.OracleTreeBatch(B, N, A, K, S, 0.01, 99, rho, lam, kind="port")
    assert_same(drive(ours, inp, K, mcts=mcts), drive(orc, inp, K, mcts=mcts), exact=True)


@pytest.mark.parametrize("B,N,A,K,S", [(1, 1, 2, 1, 1), (3, 1, 2, 1, 120), (2, 32, 3, 2, 20), (5, 2, 200, 7, 15), (40, 2, 6, 3, 90)])
def test_cuda_tree_edge_shapes(cytree, oracle_built, B, N, A, K, S):
    """Single root / single simulation; K=1 chains (paths longer than a warp, logs longer than the register cache);
    32 agents; large action spaces; many simulations."""
    inp = Inputs(B, N, A, S, seed=B + S, mode="random")
    ours = cytree.Tree_batch(B, N, A, K, S, 0.01, 41, 0.75, 0.8)
    orc = oracle_built.OracleTreeBatch(B, N, A, K, S, 0.01, 41, 0.75, 0.8, kind="port")
    assert_same(drive(ours, inp, K), drive(orc, inp, K), exact=True)


def test_cuda_tree_long_rng_stream(cytree, oracle_built):
    """Many draws per expansion: crosses the 624-word mt19937 block boundary at every position parity."""
    B, N, A, K, S = 8, 13, 7, 9, 60
    inp = Inputs(B, N, A, S, seed=2, mode="random")
    ours = cytree.Tree_batch(B, N, A, K, S, 0.01, 1234567, 0.75, 0.8)
    orc = oracle_built.OracleTreeBatch(B, N, A, K, S, 0.01, 1234567, 0.75, 0.8, kind="port")
    assert_same(drive(ours, inp, K), drive(orc, inp, K), exact=True)


# The fused step of the on-device loop (k_expand_backup_select2) holds the wide selection (tree_step.cuh: select_path_wide), taken
# when the previous path had at least wide_min_len = 3 + 2 ceil((S+1)/32) nodes; MAZ_SELECT_WIDE=1 takes it at every selection
# (except where the RNG words it needs straddle the end of the mt19937 block), =0 never.
# name: (B, N, A, K, S, seed of the injected arrays, tree seed, what the oracle must show the case reaches)
FUSED_CASES = {
    **{f"{s}/{m}": (*SHAPES[s], 1, 4, ()) for s in SHAPES for m in ("random", "quantized")},
    # K = 1 chains: the last path has S nodes (longer than a warp), the value log fills to within 8 entries of its capacity
    "chain_s120": (3, 1, 2, 1, 120, 123, 41, ("deep", "chain")),
    "chain_s200": (24, 3, 9, 1, 200, 224, 41, ("deep", "chain")),
    "k2_s150": (16, 2, 6, 2, 150, 166, 41, ("wide",)),          # two children per node: the wide form's UCB choice matters
    "long_rng": (8, 13, 7, 9, 60, 2, 1234567, ()),             # 2 K N = 234 draws per expansion
    "slots": (2, 3, 6, 32, 2045, 2047, 41, ("slots",)),         # K (S+2) = 65504 node slots: slot indices above 32767
    "wpb2": (lambda sms: 8 * sms + 317, 2, 5, 3, 12, 3, 41, ("wide",)),       # two trees per block, the last block ragged (1501 on a B200)
    "wpb4": (lambda sms: 16 * sms + 133, 2, 5, 3, 12, 4, 41, ("wide",)),      # four trees per block, the last block ragged (2501 on a B200)
}
_FUSED_ORACLE = {}


class _PathLog:
    """A tree batch that records its per-tree path length (`stats()[1]`) after every selection."""

    def __init__(self, tree):
        self.tree, self.lens = tree, []

    def __getattr__(self, name):
        return getattr(self.tree, name)

    def batch_selection(self, *a):
        r = self.tree.batch_selection(*a)
        self.lens.append(self.tree.stats()[1].copy())
        return r


def _fused_case(name, oracle_built):
    import torch

    B, N, A, K, S, seed, tree_seed, reach = FUSED_CASES[name]
    if callable(B):
        B = B(torch.cuda.get_device_properties(0).multi_processor_count)
    mode = name.split("/")[1] if "/" in name else "random"
    inp = Inputs(B, N, A, S, seed=seed, mode=mode, legal_frac=0.7 if "/" in name else None)
    if name not in _FUSED_ORACLE:
        orc = _PathLog(oracle_built.OracleTreeBatch(B, N, A, K, S, MCTS["delta_lb"], tree_seed, MCTS["rho"], MCTS["lam"], kind="port"))
        want = drive(orc, inp, K)
        lens = np.stack(orc.lens)                                       # (S, B)
        tot = orc.stats()[0]
        log_len = 1 + (lens + 1).sum(axis=0)                            # root entry + one entry per path level and simulation
        wide_min_len = 3 + 2 * ((S + 1 + 31) // 32)
        above = int((lens[:-1] >= wide_min_len).sum())                  # selections after which the next one is wide by default
        print(f"{name}: B={B} largest path {lens.max()}, longest value log {log_len.max()} (capacity {1 + S * (S + 3) // 2 + 8}), "
              f"selections at or above wide_min_len {wide_min_len}: {above}, most nodes {tot.max()}")
        if "deep" in reach:
            assert lens.max() > 32 and log_len.max() > 256
        if "chain" in reach:
            assert K == 1 and (lens[-1] == S).all() and (log_len == 1 + S * (S + 3) // 2).all()
        if "deep" in reach or "wide" in reach:
            assert above > 0
        if "slots" in reach:
            assert tot.max() > 32768
        _FUSED_ORACLE[name] = want
    return (B, N, A, K, S, tree_seed), inp, _FUSED_ORACLE[name]


@pytest.mark.parametrize("select_wide", [None, "0", "1"], ids=["default", "wide0", "wide1"])
@pytest.mark.parametrize("name", list(FUSED_CASES))
def test_fused_step_matches_oracle(cytree, oracle_built, monkeypatch, name, select_wide):
    """The on-device loop's launch order (prepare, selection, S-1 fused expansion + backup + selection, the last expansion +
    backup, readouts) on injected arrays, bit for bit against the oracle, with the wide selection at its default threshold,
    forced off and forced on."""
    (B, N, A, K, S, tree_seed), inp, want = _fused_case(name, oracle_built)
    if select_wide is None:
        monkeypatch.delenv("MAZ_SELECT_WIDE", raising=False)
    else:
        monkeypatch.setenv("MAZ_SELECT_WIDE", select_wide)              # read by the tree layout when the batch is created
    ours = cytree.Tree_batch(B, N, A, K, S, MCTS["delta_lb"], tree_seed, MCTS["rho"], MCTS["lam"])
    assert_same(drive_fused(ours, inp, K), want, exact=True, what=f"{name}/{select_wide}: ")


def test_root_index_offset_makes_shards_equal_to_the_whole(cytree):
    """Sharding invariance (multi-GPU): trees [4,8) of an 8-root batch == a 4-root batch with offset 4."""
    B, N, A, K, S = 8, 3, 9, 10, 30
    inp = Inputs(B, N, A, S, seed=4, mode="random")
    whole = drive(cytree.Tree_batch(B, N, A, K, S, 0.01, 17, 0.75, 0.8), inp, K)

    class Half:
        pass

    half = Half()
    half.B, half.N, half.A, half.S, half.noise_eps = 4, N, A, S, inp.noise_eps
    half.rewards, half.values = inp.rewards[:, 4:], inp.values[:, 4:]
    half.probs, half.beta, half.noises = inp.probs[:, 4:], inp.beta[:, 4:], inp.noises[4:]
    part = drive(cytree.Tree_batch(4, N, A, K, S, 0.01, 17, 0.75, 0.8, device=0, root_index_offset=4), half, K)
    assert np.array_equal(part["value"], whole["value"][4:])
    assert np.array_equal(part["marginal_visit_count"], whole["marginal_visit_count"][4:])
    assert np.array_equal(part["sel_act"], whole["sel_act"][:, 4:])


def test_device_pointer_entry_points(cytree, oracle_built):
    """The `_dev` entry points (torch CUDA tensors, asynchronous) give the same result as the host ones."""
    import torch

    B, N, A, K, S = 64, 3, 9, 10, 20
    inp = Inputs(B, N, A, S, seed=9, mode="random")
    host = drive(cytree.Tree_batch(B, N, A, K, S, 0.01, 5, 0.75, 0.8), inp, K)
    t = cytree.Tree_batch(B, N, A, K, S, 0.01, 5, 0.75, 0.8)
    dev = torch.device("cuda:0")
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    t.set_puct(MCTS["pb_c_base"], MCTS["pb_c_init"])
    t.prepare(d(inp.rewards[0]), d(inp.values[0]), d(inp.probs[0]), d(inp.beta[0]), K, float(inp.noise_eps), d(inp.noises))
    ix = torch.empty(B, dtype=torch.int32, device=dev)
    iy = torch.empty(B, dtype=torch.int32, device=dev)
    act = torch.empty(B, N, dtype=torch.int32, device=dev)
    acts = []
    for s in range(S):
        t.batch_selection_device(MCTS["pb_c_base"], MCTS["pb_c_init"], MCTS["discount"], ix, iy, act)
        acts.append(act.clone())
        t.batch_expansion_and_backup(s + 1, MCTS["discount"], K, d(inp.rewards[s + 1]), d(inp.values[s + 1]),
                                     d(inp.probs[s + 1]), d(inp.beta[s + 1]))
    t.check()
    assert np.array_equal(torch.stack(acts).cpu().numpy(), host["sel_act"])
    assert np.array_equal(t.get_roots_values(), host["value"])
    assert np.array_equal(t.get_roots_marginal_visit_count(), host["marginal_visit_count"])


def test_reset_reuses_arena(cytree):
    B, N, A, K, S = 16, 2, 4, 5, 25
    inp = Inputs(B, N, A, S, seed=3, mode="random")
    t = cytree.Tree_batch(B, N, A, K, S, 0.01, 21, 0.75, 0.8)
    a = drive(t, inp, K)
    t.reset(22, 0.01, 0.75, 0.8)
    b = drive(t, inp, K)
    t.reset(21, 0.01, 0.75, 0.8)
    c = drive(t, inp, K)
    assert_same(a, c, exact=True)
    assert not np.array_equal(a["sel_act"], b["sel_act"])


def test_errors_are_runtime_errors(cytree):
    with pytest.raises(RuntimeError):
        cytree.Tree_batch(4, 1, 3, 64, 5, 0.01, 0, 0.75, 0.8)  # K > 32
    with pytest.raises(RuntimeError):
        cytree.Tree_batch(2, 3, 6, 32, 2046, 0.01, 0, 0.75, 0.8)  # K (S+2) = 65536 node slots: more than 16-bit slots address
    t = cytree.Tree_batch(4, 1, 3, 2, 5, 0.01, 0, 0.75, 0.8)
    with pytest.raises(RuntimeError):
        t.batch_selection(19652.0, 1.25, 0.99)  # before prepare
    z = np.zeros(4)
    with pytest.raises(ValueError):  # float64 input, as the typed memoryview in cytree.pyx:25
        t.prepare(z, z, np.zeros((4, 1, 3)), np.zeros((4, 1, 3)), 2, 0.0, np.zeros((4, 1, 3)))
