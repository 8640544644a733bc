"""CPU tests of the checker itself: the plain-C restatement (oracle/maz_oracle.c) against
(a) the committed golden vectors generated from the compiled reference and
(b) the compiled reference (oracle/_ref/libmazref.so) when it is present."""
import glob
import os

import numpy as np
import pytest

from _harness import MCTS, SHAPES, Inputs, assert_same, drive, pack

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "tree_*.npz")))


class GoldenInputs:
    def __init__(self, z):
        self.B, self.N, self.A, self.K, self.S = [int(x) for x in z["dims"]]
        self.rewards, self.values, self.probs, self.beta = z["in_rewards"], z["in_values"], z["in_probs"], z["in_beta"]
        self.noises, self.noise_eps = z["in_noises"], z["in_noise_eps"]
        m = z["mcts"]
        self.mcts = dict(pb_c_base=float(m[0]), pb_c_init=float(m[1]), discount=float(m[2]), rho=float(m[3]),
                         lam=float(m[4]), delta_lb=float(m[5]))
        self.seed = int(z["tree_seed"])
        self.expected = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
        self.tot_nodes = z["tot_nodes"]


def check_golden(make_tree, path, exact=True):
    g = GoldenInputs(np.load(path))
    tree = make_tree(g.B, g.N, g.A, g.K, g.S, g.mcts["delta_lb"], g.seed, g.mcts["rho"], g.mcts["lam"])
    out = pack(drive(tree, g, g.K, mcts=g.mcts))
    exp = g.expected
    assert set(out) == set(exp)
    for k in exp:
        a, b = out[k], exp[k]
        assert a.shape == b.shape and a.dtype == b.dtype, (k, a.shape, b.shape, a.dtype, b.dtype)
        if exact or a.dtype.kind in "iu":
            assert np.array_equal(a.view(np.int32) if a.dtype == np.float32 else a,
                                  b.view(np.int32) if b.dtype == np.float32 else b), f"{os.path.basename(path)}:{k}"
        else:
            np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-7, err_msg=k)
    assert np.array_equal(tree.stats()[0], g.tot_nodes), f"{os.path.basename(path)}: node counts"
    return tree


def test_golden_present():
    assert len(GOLDEN) >= 8


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[5:-4] for p in GOLDEN])
def test_oracle_port_matches_golden(oracle_built, path):
    check_golden(lambda *a: oracle_built.OracleTreeBatch(*a, kind="port"), path)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("mode", ["random", "mock", "quantized"])
def test_oracle_port_matches_compiled_reference(oracle_built, shape, mode):
    if not oracle_built.available("reference"):
        pytest.skip("oracle/_ref/libmazref.so not built (no /root/reference on this box)")
    B, N, A, K, S = SHAPES[shape]
    B = min(B, 16)
    for seed in (0, 1):
        inp = Inputs(B, N, A, S, seed=seed, mode=mode, legal_frac=0.7 if seed else None)
        ref = oracle_built.OracleTreeBatch(B, N, A, K, S, MCTS["delta_lb"], 3 + seed, MCTS["rho"], MCTS["lam"], kind="reference")
        port = oracle_built.OracleTreeBatch(B, N, A, K, S, MCTS["delta_lb"], 3 + seed, MCTS["rho"], MCTS["lam"], kind="port")
        assert_same(drive(ref, inp, K), drive(port, inp, K), exact=True, what=f"{shape}/{mode}/{seed}: ")
        assert np.array_equal(ref.stats()[0], port.stats()[0])


def test_oracle_known_answer_depth1_value():
    """Hand-checkable KAT (SURVEY section 4): one root, value .5, three sims returning value .6 / reward .1,
    rho=.75, lam=.8: root sets are depth0={.5}, depth1={.694 x3} -> top-25% keeps one -> (0.5+0.8*0.694)/1.8."""
    from oracle.pyoracle import OracleTreeBatch

    B, N, A, K, S = 1, 1, 3, 5, 3
    inp = Inputs(B, N, A, S, seed=0, mode="mock")
    t = OracleTreeBatch(B, N, A, K, S, 0.01, 7, 0.75, 0.8)
    out = drive(t, inp, K)
    nc = len(out["sampled_visit_count"][0])
    if nc >= 3:  # all three sims were forced round-robin visits of distinct root children
        assert abs(out["value"][0] - (0.5 + 0.8 * 0.694) / 1.8) < 1e-6


def test_oracle_wrong_dtype_raises(oracle_built):
    t = oracle_built.OracleTreeBatch(2, 1, 3, 2, 2, 0.01, 0, 0.75, 0.8)
    z = np.zeros(2)
    with pytest.raises(ValueError):
        t.prepare(z, z, np.zeros((2, 1, 3)), np.zeros((2, 1, 3)), 2, 0.0, np.zeros((2, 1, 3)))
