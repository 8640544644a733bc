"""Shared helpers for the parity tests: seeded synthetic network outputs, and a driver that runs one
whole search through any object with the ``cytree.Tree_batch`` method set (ours, the C oracle, or the
compiled reference) with IDENTICAL injected arrays, recording everything observable.

The step order is the reference's simulation loop (core/mcts/tree_search/mcts_sampled.py:89-191).
"""
import numpy as np

MCTS = dict(pb_c_base=19652.0, pb_c_init=1.25, discount=0.99, rho=0.75, lam=0.8, delta_lb=0.01)

# BASELINE.json configs, scaled so the CPU oracle finishes in seconds
SHAPES = {
    # name: (B, N, A, K, S)
    "matrix": (16, 2, 3, 5, 50),
    "matrix_seq": (16, 1, 3, 5, 50),
    "3m": (64, 3, 9, 10, 50),
    "3m_seq": (64, 1, 9, 10, 50),
    "2s3z": (32, 5, 11, 10, 100),
    "mmm2": (16, 10, 18, 10, 50),
    "27m": (8, 27, 36, 10, 50),
}


def softmax(x):
    e = np.exp(x - np.max(x, axis=-1, keepdims=True))
    return e / np.sum(e, axis=-1, keepdims=True)


class Inputs:
    """Injected network outputs for a whole search: index 0 = root, s+1 = simulation s."""

    def __init__(self, B, N, A, S, seed=0, mode="random", tau=1.0, noise_eps=0.25, legal_frac=None, logit_scale=1.0):
        rng = np.random.RandomState(seed)
        self.B, self.N, self.A, self.S = B, N, A, S
        self.noise_eps = np.float32(noise_eps)
        if mode == "random":
            logits = (rng.randn(S + 1, B, N, A) * logit_scale).astype(np.float32)
            self.values = (rng.randn(S + 1, B) * 0.5).astype(np.float32)
            self.rewards = (rng.randn(S + 1, B) * 0.3).astype(np.float32)
            self.rewards[0] = 0
        elif mode == "mock":
            # the reference's MockModel (unit_test_mcts.py:68-130): zero logits, value .5 -> .6, reward .1
            logits = np.zeros((S + 1, B, N, A), dtype=np.float32)
            self.values = np.full((S + 1, B), 0.6, dtype=np.float32)
            self.values[0] = 0.5
            self.rewards = np.full((S + 1, B), 0.1, dtype=np.float32)
            self.rewards[0] = 0
        elif mode == "quantized":
            # few distinct values/logits: forces exact ties in UCB scores, value sets and min-max stats
            logits = (rng.randint(-1, 2, size=(S + 1, B, N, A)) * 0.5).astype(np.float32)
            self.values = (rng.randint(-2, 3, size=(S + 1, B)) * 0.25).astype(np.float32)
            self.rewards = (rng.randint(-1, 2, size=(S + 1, B)) * 0.5).astype(np.float32)
            self.rewards[0] = 0
        else:
            raise ValueError(mode)
        probs = softmax(logits).astype(np.float32)
        noises = rng.dirichlet([0.3] * A, (B, N)).astype(np.float32)
        if legal_frac is not None:
            mask = (rng.rand(B, N, A) < legal_frac).astype(np.float32)
            mask[..., min(1, A - 1)] = 1.0
            p0 = probs[0] * mask
            p0 += mask * 1e-4
            probs[0] = p0 / p0.sum(-1, keepdims=True)
            noises = noises * mask + mask * 1e-4
            noises = (noises / noises.sum(-1, keepdims=True)).astype(np.float32)
        else:
            mask = np.ones((B, N, A), dtype=np.float32)
        self.mask = mask
        self.probs = probs
        self.noises = noises
        beta = probs.copy()
        beta[0] = probs[0] * (1 - self.noise_eps) + noises * self.noise_eps
        beta = beta ** np.float32(1.0 / tau)
        beta[0] *= mask
        self.beta = (beta / beta.sum(-1, keepdims=True)).astype(np.float32)


def drive(tree, inp, K, sims=None, mcts=MCTS, record_steps=True):
    """Run prepare + S simulations + all readouts; return a dict of everything observable."""
    S = inp.S if sims is None else sims
    out = {}
    tree.prepare(inp.rewards[0], inp.values[0], inp.probs[0], inp.beta[0], K, float(inp.noise_eps), inp.noises)
    ixs, acts = [], []
    for s in range(S):
        ix, iy, act = tree.batch_selection(mcts["pb_c_base"], mcts["pb_c_init"], mcts["discount"])
        assert list(iy) == list(range(inp.B))
        if record_steps:
            ixs.append(np.asarray(ix, dtype=np.int32))
            acts.append(np.asarray(act, dtype=np.int32).copy())
        tree.batch_expansion_and_backup(s + 1, mcts["discount"], K, inp.rewards[s + 1], inp.values[s + 1],
                                        inp.probs[s + 1], inp.beta[s + 1])
    if record_steps:
        out["sel_idx"] = np.stack(ixs) if ixs else np.zeros((0, inp.B), np.int32)
        out["sel_act"] = np.stack(acts) if acts else np.zeros((0, inp.B, inp.N), np.int32)
    out.update(readouts(tree, mcts["discount"]))
    return out


def drive_fused(tree, inp, K, mcts=MCTS):
    """`drive` in the launch order of the on-device loop (maz_search.cu: enqueue_loop), on torch CUDA copies of the arrays:
    prepare, the selection of simulation 0, then for s < S-1 the fused expansion + backup of s and selection of s+1 (the
    two-warp kernel, which holds the wide selection), the last expansion + backup alone, the readouts.  Same dict as `drive`."""
    import torch

    B, N, S = inp.B, inp.N, inp.S
    dev = torch.device("cuda:0")
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    rewards, values, probs, beta = d(inp.rewards), d(inp.values), d(inp.probs), d(inp.beta)
    ix = torch.empty(S, B, dtype=torch.int32, device=dev)
    iy = torch.empty(B, dtype=torch.int32, device=dev)
    act = torch.empty(S, B, N, dtype=torch.int32, device=dev)
    c_base, c_init, discount = mcts["pb_c_base"], mcts["pb_c_init"], mcts["discount"]
    tree.prepare(rewards[0], values[0], probs[0], beta[0], K, float(inp.noise_eps), d(inp.noises))
    if S > 0:
        tree.batch_selection_device(c_base, c_init, discount, ix[0], iy, act[0])
    for s in range(S - 1):
        tree.expansion_backup_selection_device(s + 1, discount, K, rewards[s + 1], values[s + 1], probs[s + 1], beta[s + 1],
                                               c_base, c_init, ix[s + 1], iy, act[s + 1])
    if S > 0:
        tree.batch_expansion_and_backup(S, discount, K, rewards[S], values[S], probs[S], beta[S])
    tree.check()
    if S > 0:
        assert iy.cpu().tolist() == list(range(B))
    out = {"sel_idx": ix.cpu().numpy(), "sel_act": act.cpu().numpy()}
    out.update(readouts(tree, discount))
    return out


LIST_FIELDS = ("sampled_actions", "sampled_visit_count", "sampled_pred_probs", "sampled_beta", "sampled_beta_hat",
               "sampled_priors", "sampled_imp_ratio", "sampled_pred_values", "sampled_mcts_values", "sampled_rewards",
               "sampled_qvalues")


def readouts(tree, discount):
    out = {
        "value": tree.get_roots_values(),
        "marginal_visit_count": tree.get_roots_marginal_visit_count(),
        "marginal_priors": tree.get_roots_marginal_priors(),
        "sampled_actions": tree.get_roots_sampled_actions(),
        "sampled_visit_count": tree.get_roots_sampled_visit_count(),
        "sampled_pred_probs": tree.get_roots_sampled_pred_probs(),
        "sampled_beta": tree.get_roots_sampled_beta(),
        "sampled_beta_hat": tree.get_roots_sampled_beta_hat(),
        "sampled_priors": tree.get_roots_sampled_priors(),
        "sampled_imp_ratio": tree.get_roots_sampled_imp_ratio(),
        "sampled_pred_values": tree.get_roots_sampled_pred_values(),
        "sampled_mcts_values": tree.get_roots_sampled_mcts_values(),
        "sampled_rewards": tree.get_roots_sampled_rewards(),
        "sampled_qvalues": tree.get_roots_sampled_qvalues(discount),
    }
    return out


def pack(out):
    """Flatten the ragged per-root lists into padded arrays so a result fits in one .npz."""
    res = {}
    for k, v in out.items():
        if isinstance(v, list):
            n = np.array([len(x) for x in v], dtype=np.int32)
            res["num_children"] = n
            kmax = int(n.max()) if len(n) else 0
            first = np.asarray(v[0])
            pad = np.zeros((len(v), kmax) + first.shape[1:], dtype=first.dtype)
            for b, x in enumerate(v):
                pad[b, : len(x)] = x
            res[k] = pad
        else:
            res[k] = np.asarray(v)
    return res


def assert_same(a, b, exact=True, rtol=1e-5, what=""):
    """a, b: dicts from drive(). Integer outputs bit-exact always; float outputs bit-exact (exact=True)
    or within rtol (the north star's 1e-5 relative for root values / Q statistics)."""
    a, b = pack(a), pack(b)
    assert a.keys() == b.keys(), (a.keys(), b.keys())
    for k in a:
        x, y = a[k], b[k]
        assert x.shape == y.shape, f"{what}{k}: shape {x.shape} vs {y.shape}"
        assert x.dtype == y.dtype, f"{what}{k}: dtype {x.dtype} vs {y.dtype}"
        if x.dtype.kind in "iu" or exact:
            if not np.array_equal(x.view(np.int32) if x.dtype == np.float32 else x,
                                  y.view(np.int32) if y.dtype == np.float32 else y):
                bad = np.argwhere(x != y)
                raise AssertionError(f"{what}{k}: {len(bad)} mismatches, first at {bad[:3].tolist()}: "
                                     f"{x[tuple(bad[0])]} vs {y[tuple(bad[0])]}")
        else:
            np.testing.assert_allclose(x, y, rtol=rtol, atol=1e-7, err_msg=f"{what}{k}")
