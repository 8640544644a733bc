"""CPU: the restated per-agent turn logic (oracle/turn_oracle.py) against known answers produced by the reference's
own `select_action` / `eps_greedy_action` (tests/golden/turns_kat.npz, made by tests/golden/make_golden_turns.py),
and -- in the build container, where /root/reference exists -- against those functions called live."""
import os

import numpy as np
import pytest
import torch

KAT = os.path.join(os.path.dirname(__file__), "golden", "turns_kat.npz")
REF = os.environ.get("MAZ_REFERENCE", "/root/reference")


def test_select_action_reproduces_reference_known_answers():
    from oracle.turn_oracle import select_action

    z = np.load(KAT)
    for i in range(len(z["lens"])):
        c = z["counts"][i, : z["lens"][i]]
        pos, ent = select_action(c, temperature=float(z["temps"][i]), deterministic=False, uniform=float(z["uniforms"][i]))
        assert pos == z["pos"][i], i
        assert ent == z["entropy"][i], i          # same float64 operations in the same order: bit-identical
    assert select_action(np.array([3, 9, 9, 1]), deterministic=True)[0] == 1


def test_eps_greedy_reproduces_reference_known_answers():
    from oracle.turn_oracle import eps_greedy_action

    z = np.load(KAT)
    for i in range(len(z["greedy"])):
        assert eps_greedy_action(z["greedy"][i], float(z["eps"]), z["eps_u"][i], z["rand_act"][i]) == z["eps_result"][i]


def test_turn_draws_from_seeds_reproduce_reference_known_answers():
    """The draws of the live comparison below, made here from the seeds the known answers were recorded with:
    np.random.RandomState(1000 + i) for select_action; for eps_greedy_action torch.manual_seed(i), then one rand_like draw,
    then Categorical(mask).sample(), the order in which the reference consumes torch's global generator."""
    from oracle.turn_oracle import eps_greedy_action, select_action

    z = np.load(KAT)
    for i in range(len(z["lens"])):
        c = z["counts"][i, : z["lens"][i]]
        u = np.random.RandomState(1000 + i).random_sample()
        pos, ent = select_action(c, temperature=float(z["temps"][i]), deterministic=False, uniform=u)
        assert pos == z["pos"][i] and ent == z["entropy"][i], i
    for i in range(len(z["greedy"])):
        torch.manual_seed(i)
        m = torch.from_numpy(z["masks"][i])
        u = float(torch.rand_like(m[..., 0].float()))
        ra = int(torch.distributions.Categorical(m).sample())
        assert eps_greedy_action(int(z["greedy"][i]), float(z["eps"]), u, ra) == z["eps_result"][i], i


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "core", "utils.py")), reason="reference sources not present on this box")
def test_turn_functions_equal_reference_live():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_golden_turns as mt
    from oracle.turn_oracle import eps_greedy_action, select_action

    ru = mt.reference_utils()
    rng = np.random.RandomState(5)
    for i in range(200):
        n = rng.randint(1, 11)
        c = rng.randint(0, 30, size=n).astype(np.int32)
        c[rng.randint(n)] += 1
        t = float(rng.choice([1.0, 0.5, 0.25, 0.9]))
        ref = ru.select_action(c, temperature=t, deterministic=False, np_random=np.random.RandomState(i))
        mine = select_action(c, temperature=t, deterministic=False, uniform=np.random.RandomState(i).random_sample())
        assert ref[0] == mine[0] and ref[1] == mine[1]
        mask = (rng.rand(7) < 0.5).astype(np.float32)
        mask[0] = 1
        torch.manual_seed(i)
        r = int(ru.eps_greedy_action(3, mask, 0.4)[0])
        torch.manual_seed(i)
        m = torch.from_numpy(mask)
        u = float(torch.rand_like(m[..., 0].float()))
        ra = int(torch.distributions.Categorical(m).sample())
        assert r == eps_greedy_action(3, 0.4, u, ra)


def test_root_prepare_equals_restated_driver_arrays(oracle_built):
    """turn_oracle.root_prepare is the block of oracle/search_oracle.py (pinned to the reference's own driver by
    tests/test_reference_driver_cpu.py) factored out: identical arrays reach Tree_batch.prepare."""
    from oracle import pyoracle, turn_oracle

    B, N, A = 6, 3, 5
    rng = np.random.RandomState(0)
    logits = rng.randn(B, N, A).astype(np.float32)
    legal = (rng.rand(B, N, A) < 0.7).astype(np.float64)
    legal[..., 1] = 1
    for cur in (None, 0, 2):
        Nt = N if cur is None else 1
        noises = np.random.RandomState(1).dirichlet([0.3] * A, B * Nt).astype(np.float32).reshape(B, Nt, A)
        p, b, n = turn_oracle.root_prepare(logits, cur, legal, noises, 0.25, 1.0)
        assert p.dtype == b.dtype == n.dtype == np.float32 and p.shape == (B, Nt, A)
        np.testing.assert_allclose(p.sum(-1), 1, rtol=1e-6)
        np.testing.assert_allclose(b.sum(-1), 1, rtol=1e-6)
        m = legal if cur is None else legal[:, cur:cur + 1]
        assert ((p > 0) == (m > 0)).all() and ((b > 0) == (m > 0)).all()
