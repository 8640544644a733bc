"""Device-resident forward of the network the search calls: `prediction` and `recurrent_inference` of
the reference's SMAC `MAMuZeroNet` (config/smac/model.py:494-501, 562-574) with NO host round trip:
reward / value come back as device scalars (the reference's eval mode does `.cpu().numpy()` on every
simulation, config/smac/model.py:568-572).

`SmacInference.from_model(model)` reads the weights of a reference-style module tree (same parameter
names: dynamics_network.*, prediction_network.*).

mode="fp32": parity mode -- plain fp32 torch ops on the device, the floating-point reference for the fused
kernels.  mode="bf16": the fused tensor-core path (see csrc/), when built.
"""
import math

import torch
import torch.nn.functional as F


def _get(sd, key, device, dtype=torch.float32, registry=None):
    t = sd[key].detach().to(device=device, dtype=dtype).contiguous()
    if registry is not None:
        registry[key] = t
    return t


class _GraphNetW:
    def __init__(self, sd, prefix, device, registry=None):
        g = lambda k: _get(sd, prefix + k, device, registry=registry)
        self.gc1_w, self.gc1_b = g("gc1.lin_layer.weight"), g("gc1.lin_layer.bias")
        self.nn1_w, self.nn1_b = g("nn_gc1.weight"), g("nn_gc1.bias")
        self.gc2_w, self.gc2_b = g("gc2.lin_layer.weight"), g("gc2.lin_layer.bias")
        self.nn2_w, self.nn2_b = g("nn_gc2.weight"), g("nn_gc2.bias")
        self.v_w, self.v_b = g("V.weight"), g("V.bias")

    def __call__(self, x):
        """x (B,N,D) -> logits (B,support).  All-ones adjacency: bmm(adj, f) == sum over agents
        (config/smac/model.py:84,151-163)."""
        f = F.linear(x, self.gc1_w, self.gc1_b).sum(dim=1, keepdim=True) + F.linear(x, self.nn1_w, self.nn1_b)
        f = F.layer_norm(F.relu(f), [f.size(-1)])
        o = F.linear(f, self.gc2_w, self.gc2_b).sum(dim=1, keepdim=True) + F.linear(f, self.nn2_w, self.nn2_b)
        o = F.layer_norm(F.relu(o), [o.size(-1)])
        return F.linear(o.mean(dim=1), self.v_w, self.v_b)


class SmacInference:
    def __init__(self, state_dict, num_agents, action_space_size, hidden_state_size=128, reward_support=(-5, 5),
                 value_support=(-5, 5), device="cuda", mode="fp32", nhead=8):
        self.N, self.A, self.H = int(num_agents), int(action_space_size), int(hidden_state_size)
        self.device = torch.device(device)
        self.mode = mode
        self.nhead = nhead
        sd = state_dict
        dev = self.device
        self._params = {}   # state-dict key -> device tensor (refreshed in place by `refresh`)
        g = lambda k: _get(sd, k, dev, registry=self._params)
        d = "dynamics_network."
        self.in_w, self.in_b = g(d + "attention_stack.0.weight"), g(d + "attention_stack.0.bias")
        self.pos = g(d + "attention_stack.2.pos_embed.pos_table")[0, : self.N]  # (N,H) view
        self.layers = []
        i = 0
        while f"{d}attention_stack.2.encoder.layers.{i}.self_attn.in_proj_weight" in sd:
            p = f"{d}attention_stack.2.encoder.layers.{i}."
            self.layers.append(dict(
                qkv_w=g(p + "self_attn.in_proj_weight"), qkv_b=g(p + "self_attn.in_proj_bias"),
                out_w=g(p + "self_attn.out_proj.weight"), out_b=g(p + "self_attn.out_proj.bias"),
                l1_w=g(p + "linear1.weight"), l1_b=g(p + "linear1.bias"),
                l2_w=g(p + "linear2.weight"), l2_b=g(p + "linear2.bias"),
                n1_w=g(p + "norm1.weight"), n1_b=g(p + "norm1.bias"),
                n2_w=g(p + "norm2.weight"), n2_b=g(p + "norm2.bias")))
            i += 1
        # fc_dynamic: Linear, LN, ReLU, ..., Linear   (mlp(): config/smac/model.py:52-58)
        self.dyn = []
        idx = 0
        while f"{d}fc_dynamic.{idx}.weight" in sd:
            lin = (g(f"{d}fc_dynamic.{idx}.weight"), g(f"{d}fc_dynamic.{idx}.bias"))
            ln = None
            if f"{d}fc_dynamic.{idx + 1}.weight" in sd:
                ln = (g(f"{d}fc_dynamic.{idx + 1}.weight"), g(f"{d}fc_dynamic.{idx + 1}.bias"))
            self.dyn.append((lin, ln))
            idx += 3
        self.reward_gnn = _GraphNetW(sd, d + "reward_predictor.", dev, self._params)
        p = "prediction_network."
        self.value_gnn = _GraphNetW(sd, p + "value_predictor.", dev, self._params)
        self.pol = []
        idx = 0
        while f"{p}fc_policy.{idx}.weight" in sd:
            lin = (g(f"{p}fc_policy.{idx}.weight"), g(f"{p}fc_policy.{idx}.bias"))
            ln = None
            if f"{p}fc_policy.{idx + 1}.weight" in sd:
                ln = (g(f"{p}fc_policy.{idx + 1}.weight"), g(f"{p}fc_policy.{idx + 1}.bias"))
            self.pol.append((lin, ln))
            idx += 3
        self.rsup = torch.arange(reward_support[0], reward_support[1] + 1, dtype=torch.float32, device=dev)
        self.vsup = torch.arange(value_support[0], value_support[1] + 1, dtype=torch.float32, device=dev)
        # representation network (initial_inference): row-wise MLP kernel, when the state dict holds it and a GPU is there.
        # (Built first: its parameters join the registry that the fused path packs for the root-inference kernel.)
        self.rep = None
        if "representation_network.mlp.0.weight" in sd and dev.type == "cuda":
            from .inference_mlp import RowMlp

            self.rep = RowMlp(sd, dev, self._params)
        # fused tensor-core path (bf16 operands, fp32 accumulate): csrc/infer_fused.cuh
        self.fused = None
        if mode == "bf16":
            from . import fused

            if dev.type != "cuda":
                raise RuntimeError("mode='bf16' needs a CUDA device (no CPU fallback)")
            if tuple(reward_support) != (-5, 5) or tuple(value_support) != (-5, 5) or nhead != 8 or \
                    not fused.supported(sd, self.N, self.A, self.H):
                raise RuntimeError("mode='bf16': network shape not supported by the fused kernel "
                                   "(needs the reference SMAC architecture: hidden 128, 3 layers, 8 heads, support 11)")
            self.fused = fused.FusedParams(self._params, self.N, self.A, dev)

    @classmethod
    def from_model(cls, model, device="cuda", mode="fp32", **kw):
        """`model`: a reference-style MAMuZeroNet (attributes num_agents, action_space_size,
        hidden_state_size_per_agent or hidden; state_dict with the reference's parameter names)."""
        n = int(getattr(model, "num_agents"))
        a = int(getattr(model, "action_space_size"))
        h = int(getattr(model, "hidden_state_size_per_agent", getattr(model, "hidden", 128)))
        return cls(model.state_dict(), n, a, h, device=device, mode=mode, **kw)

    def refresh(self, state_dict):
        """Copy new weights into the existing device tensors (addresses stay valid for captured graphs).
        Tensors that alias the module's own parameters (model already on this device) need no copy."""
        for k, t in self._params.items():
            src = state_dict[k]
            if src.data_ptr() != t.data_ptr():
                t.copy_(src, non_blocking=True)
        if self.fused is not None:
            self.fused.repack(self._params)
        if self.rep is not None:
            self.rep.retranspose()

    def initial_inference(self, observation, fused=False):
        """`MAMuZeroNet.initial_inference` (config/smac/model.py:542-559) without leaving the device: observation
        (B, N, ...) -> NetworkOutput(hidden (B, N*H), reward zeros (B,1), value (B,1), policy_logits (B,N,A)) as CUDA tensors
        with no synchronisation (the reference's eval mode does `.cpu().numpy()` on value and logits).
        fused=False: fp32, the row-wise MLP kernel for the representation and torch ops for the heads.  fused=True: one launch
        of the bf16 root-inference kernel (csrc/infer_initial.cuh, `maz_infer_initial`); needs mode="bf16" and the reference
        representation network (`fused.supported_initial`), else ValueError."""
        from .synthetic import NetworkOutput
        if fused:
            return NetworkOutput(*self._initial_fused(observation))
        if self.rep is None:
            raise RuntimeError("the state dict holds no representation network (or no CUDA device)")
        from .inference_mlp import initial_inference_device
        return NetworkOutput(*initial_inference_device(self, self.rep, observation))

    def _initial_fused(self, observation, stream=None):
        from . import fused

        if self.fused is None:
            raise ValueError(f"initial_inference(fused=True) needs SmacInference(mode='bf16'), this object has mode={self.mode!r}")
        if self.fused.rep_wpk is None:
            raise ValueError("initial_inference(fused=True): " + (fused.initial_unsupported_reason(self._params, self.N, self.A, self.H)
                                                                  or "representation network not packed"))
        B = observation.shape[0]
        x = observation.reshape(B * self.N, -1).to(device=self.device, dtype=torch.float32).contiguous()
        if x.shape[1] != self.fused.obs_dim:
            raise ValueError(f"initial_inference(fused=True): {x.shape[1]} observation features per agent, the representation "
                             f"network takes {self.fused.obs_dim}")
        hidden = torch.empty(B, self.N * self.H, dtype=torch.float32, device=self.device)
        value = torch.empty(B, 1, dtype=torch.float32, device=self.device)
        logits = torch.empty(B, self.N, self.A, dtype=torch.float32, device=self.device)
        dsc = self.fused.initial_desc(B, x, hidden, value, logits)
        fused.launch_initial(dsc, (stream if stream is not None else torch.cuda.current_stream(self.device)).cuda_stream)
        return hidden, torch.zeros(B, 1, dtype=torch.float32, device=self.device), value, logits

    def recurrent_fused(self, B, pool, idx_x, actions, next_hidden, reward, value, probs, beta, greedy=None,
                        logits_out=None, tree_agents=None, cur=-1, inv_tau=1.0, stream=None, dbg_clock=None, kernel=None):
        """One launch of the fused kernel: gather parent hidden from `pool` by `idx_x`, recurrent_inference,
        inverse support transforms, softmax / beta of the tree agents.  Everything stays on the device."""
        from . import fused

        small = fused.use_small(int(B), self.N) if kernel is None else (kernel == "small")
        twin = None if kernel is None else (kernel == "twin")       # "tcgen05": first-generation one-tile-per-CTA kernel
        dsc = self.fused.desc(B, pool, idx_x, actions, next_hidden, reward, value, probs, beta, greedy, logits_out,
                              tree_agents, cur, inv_tau, dbg_clock, small=small, twin=twin)
        fused.launch(dsc, (stream if stream is not None else torch.cuda.current_stream(self.device)).cuda_stream, small)

    # ---- pieces ----------------------------------------------------------------------------------------
    @staticmethod
    def _mlp(x, layers):
        for (w, b), ln in layers:
            x = F.linear(x, w, b)
            if ln is not None:
                x = F.relu(F.layer_norm(x, [x.size(-1)], ln[0], ln[1]))
        return x

    @staticmethod
    def _inv_transform(logits, sup):
        """softmax . support -> inv_h (core/config.py:430-442, 463-499), without boolean-mask indexing
        (which would synchronise) so that it can be captured in a CUDA graph."""
        eps = 0.001
        x = (torch.softmax(logits, dim=-1) * sup).sum(dim=-1)
        out = ((torch.sqrt(1 + 4 * eps * (torch.abs(x) + 1 + eps)) - 1) / (2 * eps)) ** 2 - 1
        out = torch.where(x < 0, -out, out)
        out = torch.where(torch.isnan(out), torch.zeros_like(out), out)
        return torch.where(torch.abs(out) < eps, torch.zeros_like(out), out)

    def _encoder_layer(self, x, L):
        """Post-LN nn.TransformerEncoderLayer (relu, eval) over the agent axis.  x: (B,N,H)."""
        B, N, H = x.shape
        nh, hd = self.nhead, H // self.nhead
        qkv = F.linear(x, L["qkv_w"], L["qkv_b"]).view(B, N, 3, nh, hd).permute(2, 0, 3, 1, 4)  # (3,B,nh,N,hd)
        att = torch.softmax(torch.matmul(qkv[0], qkv[1].transpose(-1, -2)) / math.sqrt(hd), dim=-1)
        sa = torch.matmul(att, qkv[2]).permute(0, 2, 1, 3).reshape(B, N, H)
        x = F.layer_norm(x + F.linear(sa, L["out_w"], L["out_b"]), [H], L["n1_w"], L["n1_b"])
        ff = F.linear(F.relu(F.linear(x, L["l1_w"], L["l1_b"])), L["l2_w"], L["l2_b"])
        return F.layer_norm(x + ff, [H], L["n2_w"], L["n2_b"])

    # ---- the two calls the search makes ---------------------------------------------------------------------
    @torch.no_grad()
    def prediction(self, hidden):
        """hidden (B,N*H) -> (policy_logits (B,N,A), value_logits (B,support))."""
        B = hidden.shape[0]
        hs = hidden.view(B, self.N, self.H)
        return self._mlp(hs, self.pol), self.value_gnn(hs)

    @torch.no_grad()
    def recurrent(self, hidden, action, out_hidden=None):
        """hidden (B,N*H) fp32, action (B,N) int -> next_hidden (B,N*H), reward (B,), value (B,),
        policy_logits (B,N,A); all on the device, no synchronisation."""
        B = hidden.shape[0]
        hs = hidden.view(B, self.N, self.H)
        onehot = F.one_hot(action.long(), num_classes=self.A).to(hs.dtype)
        x = F.relu(F.linear(torch.cat([hs, onehot], dim=2), self.in_w, self.in_b)) + self.pos
        for L in self.layers:
            x = self._encoder_layer(x, L)
        upd = self._mlp(torch.cat([hs, onehot, x], dim=2), self.dyn)
        nxt = upd + hs
        reward = self._inv_transform(self.reward_gnn(torch.cat([nxt, onehot], dim=2)), self.rsup)
        value = self._inv_transform(self.value_gnn(nxt), self.vsup)
        policy_logits = self._mlp(nxt, self.pol)
        nxt = nxt.reshape(B, self.N * self.H)
        if out_hidden is not None:
            out_hidden.copy_(nxt)
            nxt = out_hidden
        return nxt, reward, value, policy_logits
