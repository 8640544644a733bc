"""Synthetic SMAC-shaped problems for benchmarks and smoke tests (there is no StarCraft, dataset or
checkpoint in the image): random-init weights with the reference network's parameter names and shapes
(config/smac/model.py:397-470 with the sizes of config/smac/__init__.py:15-27), random root hidden states.
"""
import math
from collections import namedtuple

import numpy as np
import torch

NetworkOutput = namedtuple("NetworkOutput", ["hidden_state", "reward", "value", "policy_logits"])  # core/model.py:14-19

# BASELINE.json configs: name -> (agents N, actions A, roots B, simulations S, sampled_times K)
WORKLOADS = {
    "matrix": (2, 3, 16, 50, 5),
    "3m": (3, 9, 1024, 50, 10),
    "2s3z": (5, 11, 4096, 100, 10),
    "mmm2": (10, 18, 8192, 50, 10),
    "27m": (27, 36, 16384, 50, 10),
    "2c_vs_64zg": (2, 70, 1024, 50, 10),      # 6 + 64 actions per agent: the wide instances of the fused kernels
}


class SearchConfig:
    """The attributes `SampledMCTS` reads from the reference's BaseConfig (core/config.py:76-91,246-255)."""

    def __init__(self, action_space_size, num_simulations=50, sampled_action_times=10, discount=0.99, pb_c_base=19652.0,
                 pb_c_init=1.25, mcts_rho=0.75, mcts_lambda=0.8, root_dirichlet_alpha=0.3, root_exploration_fraction=0.25,
                 tree_value_stat_delta_lb=0.01):
        self.action_space_size = action_space_size
        self.num_simulations = num_simulations
        self.sampled_action_times = sampled_action_times
        self.discount = discount
        self.pb_c_base, self.pb_c_init = pb_c_base, pb_c_init
        self.mcts_rho, self.mcts_lambda = mcts_rho, mcts_lambda
        self.root_dirichlet_alpha, self.root_exploration_fraction = root_dirichlet_alpha, root_exploration_fraction
        self.tree_value_stat_delta_lb = tree_value_stat_delta_lb


def random_state_dict(num_agents, action_space_size, hidden=128, gnn_hidden=64, policy_hidden=32, support=11, seed=0,
                      head_scale=1.0):
    """Search-path parameters of a MAMuZeroNet: scaled-normal linears, unit LayerNorms, ~0 output heads
    (the reference zero-ish initialises its reward / value / policy heads: model.py:60-69,131-133)."""
    g = torch.Generator().manual_seed(seed)
    H, A = hidden, action_space_size
    sd = {}

    def lin(name, out_f, in_f, scale=None):
        s = math.sqrt(2.0 / in_f) if scale is None else scale
        w = torch.randn(out_f, in_f, generator=g) * s if scale is None else (torch.rand(out_f, in_f, generator=g) * 2 - 1) * s
        sd[name + ".weight"], sd[name + ".bias"] = w, torch.zeros(out_f)

    def ln(name, n):
        sd[name + ".weight"], sd[name + ".bias"] = torch.ones(n), torch.zeros(n)

    d = "dynamics_network."
    lin(d + "attention_stack.0", H, H + A)
    tab = np.array([[p / np.power(10000, 2 * (j // 2) / H) for j in range(H)] for p in range(30)])
    tab[:, 0::2], tab[:, 1::2] = np.sin(tab[:, 0::2]), np.cos(tab[:, 1::2])
    sd[d + "attention_stack.2.pos_embed.pos_table"] = torch.FloatTensor(tab).unsqueeze(0)
    for i in range(3):
        p = f"{d}attention_stack.2.encoder.layers.{i}."
        sd[p + "self_attn.in_proj_weight"] = torch.randn(3 * H, H, generator=g) * math.sqrt(1.0 / H)
        sd[p + "self_attn.in_proj_bias"] = torch.zeros(3 * H)
        lin(p + "self_attn.out_proj", H, H, )
        lin(p + "linear1", H, H)
        lin(p + "linear2", H, H)
        ln(p + "norm1", H)
        ln(p + "norm2", H)
    lin(d + "fc_dynamic.0", H, 2 * H + A)
    ln(d + "fc_dynamic.1", H)
    lin(d + "fc_dynamic.3", H, H)
    ln(d + "fc_dynamic.4", H)
    lin(d + "fc_dynamic.6", H, H)

    def gnn(prefix, in_dim):
        lin(prefix + "gc1.lin_layer", gnn_hidden, in_dim)
        lin(prefix + "nn_gc1", gnn_hidden, in_dim)
        lin(prefix + "gc2.lin_layer", gnn_hidden, gnn_hidden)
        lin(prefix + "nn_gc2", gnn_hidden, gnn_hidden)
        lin(prefix + "V", support, gnn_hidden, scale=3e-3 * head_scale)
        sd[prefix + "adj"] = torch.ones(num_agents, num_agents)

    gnn(d + "reward_predictor.", H + A)
    p = "prediction_network."
    gnn(p + "value_predictor.", H)
    lin(p + "fc_policy.0", policy_hidden, H)
    ln(p + "fc_policy.1", policy_hidden)
    lin(p + "fc_policy.3", A, policy_hidden, scale=1e-3 * head_scale)
    return sd


def root_hidden(batch, num_agents, hidden=128, seed=0, pinned=False):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(batch, num_agents * hidden, generator=g)
    return h.pin_memory() if pinned else h


def exact_state_dict(num_agents, action_space_size, hidden=128, gnn_hidden=64, policy_hidden=32, support=11, seed=0,
                     head_scale=30.0):
    """Search-path parameters of a MAMuZeroNet that are BIT-IDENTICAL on every machine: each value is an MT19937 integer
    in [-2^15, 2^15) divided by 2^15 (exact in fp32) times one fp32 scale (one correctly rounded multiply) -- no libm, no
    vectorised normal sampler.  Used where a fixture generated in the build container (outputs of the REAL reference
    network for these weights, tests/golden/make_golden_model128.py) must meet the same weights regenerated on the GPU box.
    Non-trivial biases, LayerNorm affines and output heads, so every parameter of the path is exercised."""
    rng = np.random.RandomState(seed)
    H, A = hidden, action_space_size
    sd = {}

    def u(*shape):
        return torch.from_numpy((rng.randint(-32768, 32768, size=shape).astype(np.float32) / np.float32(32768.0)))

    def lin(name, out_f, in_f, scale=None):
        s = np.float32(math.sqrt(3.0 / in_f) if scale is None else scale)
        sd[name + ".weight"] = u(out_f, in_f) * s
        sd[name + ".bias"] = u(out_f) * np.float32(0.1)

    def ln(name, n):
        sd[name + ".weight"] = u(n) * np.float32(0.25) + 1.0
        sd[name + ".bias"] = u(n) * np.float32(0.1)

    d = "dynamics_network."
    lin(d + "attention_stack.0", H, H + A)
    tab = np.array([[p / np.power(10000, 2 * (j // 2) / H) for j in range(H)] for p in range(30)])
    tab[:, 0::2], tab[:, 1::2] = np.sin(tab[:, 0::2]), np.cos(tab[:, 1::2])
    # (the table is a buffer of the reference module: the golden fixture stores the reference's own copy)
    sd[d + "attention_stack.2.pos_embed.pos_table"] = torch.FloatTensor(tab).unsqueeze(0)
    for i in range(3):
        p = f"{d}attention_stack.2.encoder.layers.{i}."
        sd[p + "self_attn.in_proj_weight"] = u(3 * H, H) * np.float32(math.sqrt(3.0 / H))
        sd[p + "self_attn.in_proj_bias"] = u(3 * H) * np.float32(0.1)
        lin(p + "self_attn.out_proj", H, H)
        lin(p + "linear1", H, H)
        lin(p + "linear2", H, H)
        ln(p + "norm1", H)
        ln(p + "norm2", H)
    lin(d + "fc_dynamic.0", H, 2 * H + A)
    ln(d + "fc_dynamic.1", H)
    lin(d + "fc_dynamic.3", H, H)
    ln(d + "fc_dynamic.4", H)
    lin(d + "fc_dynamic.6", H, H)

    def gnn(prefix, in_dim):
        lin(prefix + "gc1.lin_layer", gnn_hidden, in_dim)
        lin(prefix + "nn_gc1", gnn_hidden, in_dim)
        lin(prefix + "gc2.lin_layer", gnn_hidden, gnn_hidden)
        lin(prefix + "nn_gc2", gnn_hidden, gnn_hidden)
        lin(prefix + "V", support, gnn_hidden, scale=3e-3 * head_scale)
        sd[prefix + "adj"] = torch.ones(num_agents, num_agents)

    gnn(d + "reward_predictor.", H + A)
    p = "prediction_network."
    gnn(p + "value_predictor.", H)
    lin(p + "fc_policy.0", policy_hidden, H)
    ln(p + "fc_policy.1", policy_hidden)
    lin(p + "fc_policy.3", A, policy_hidden, scale=1e-2 * head_scale)
    return sd


def state_dict_digest(sd):
    """sha256 over the raw fp32 bytes of a state dict in key order (fixtures pin the weights they were generated with)."""
    import hashlib

    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(np.ascontiguousarray(sd[k].detach().cpu().numpy().astype(np.float32)).tobytes())
    return h.hexdigest()
