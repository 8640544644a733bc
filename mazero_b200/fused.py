"""Host side of the fused tensor-core inference kernel (include/maz_infer.h, csrc/infer_fused.cuh):
packs a reference-named state dict into (a) bf16 weight chunks in the tcgen05 shared-memory operand layout,
in the order the kernel consumes them, and (b) one fp32 vector of biases / LayerNorm affines / positional
table / value & reward heads; fills the launch descriptor.
"""
import ctypes as C
import os

import torch

from ._lib import check, lib

NCHUNK = 32
A_MAX = 128       # actions per agent of the fused kernels: the wide instances above A_NARROW (csrc/infer_hmma.cuh, csrc/infer_twin.cuh)
A_NARROW = 48     # ... and of the first-generation tcgen05 kernel (csrc/infer_fused.cuh)
SWIZZLE = False   # must match MAZ_SWIZZLE in csrc/umma.cuh (128-byte swizzled operand tiles; measured slower)
H, GH, PH, SUP = 128, 64, 32, 11


class InferDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("N", C.c_int), ("A", C.c_int), ("KA", C.c_int), ("NAP", C.c_int), ("Nt", C.c_int), ("cur", C.c_int),
        ("inv_tau", C.c_float),
        ("pool", C.c_void_p), ("idx_x", C.c_void_p), ("actions", C.c_void_p), ("next_hidden", C.c_void_p),
        ("reward", C.c_void_p), ("value", C.c_void_p), ("probs", C.c_void_p), ("beta", C.c_void_p), ("greedy", C.c_void_p),
        ("logits_out", C.c_void_p), ("wpk", C.c_void_p), ("vec", C.c_void_p), ("vec_floats", C.c_int),
        ("chunk_off", C.c_uint * NCHUNK), ("chunk_bytes", C.c_uint * NCHUNK),
        ("o_bin", C.c_int), ("o_pos", C.c_int), ("o_layer", C.c_int), ("o_dyn", C.c_int), ("o_rg", C.c_int),
        ("o_vg", C.c_int), ("o_pol", C.c_int), ("dbg_clock", C.c_void_p), ("dbg_flags", C.c_int),
        ("roots_per_tile", C.c_int), ("factor", C.c_void_p), ("greedy_pool", C.c_void_p),
        ("tc_layout", C.c_int), ("o_oh_in", C.c_int), ("o_oh_dyn", C.c_int), ("o_oh_rg", C.c_int),
    ]


class InitialDesc(C.Structure):      # include/maz_infer.h: maz_initial_desc
    _fields_ = [
        ("B", C.c_int), ("N", C.c_int), ("A", C.c_int), ("H", C.c_int), ("obs_dim", C.c_int),
        ("obs", C.c_void_p), ("hidden", C.c_void_p), ("value", C.c_void_p), ("policy_logits", C.c_void_p),
        ("rep_wpk", C.c_void_p), ("rep_vec", C.c_void_p), ("wpk", C.c_void_p), ("vec", C.c_void_p), ("vec_floats", C.c_int),
        ("chunk_off", C.c_uint * NCHUNK), ("chunk_bytes", C.c_uint * NCHUNK), ("o_vg", C.c_int), ("o_pol", C.c_int),
    ]


OBS_MAX = 640     # observation features per agent of the root-inference kernel (csrc/infer_initial.cuh)
REP = "representation_network."


def _pad16(n):
    return (n + 15) // 16 * 16


def pack_operand(w):
    """[rows, K] fp32 -> bf16 in the kernels' shared-memory operand layout (csrc/umma.cuh).
    K % 64 == 0: SWIZZLE_128B, K-major -- atoms of 8 rows x 64 elements stored [K/64][rows/8]; inside an atom the
    16-byte chunk j of row r sits at chunk position j ^ (r % 8).
    otherwise:   no swizzle, 8x8 core matrices: W.view(rows/8, 8, K/8, 8).permute(0, 2, 1, 3)."""
    r, k = w.shape
    assert r % 8 == 0 and k % 16 == 0, (r, k)
    wb = w.to(torch.bfloat16)
    if SWIZZLE and k % 64 == 0:
        t = wb.view(r // 8, 8, k // 64, 8, 8).permute(2, 0, 1, 3, 4)           # [kb, rg, r8, j, e]
        ar = torch.arange(8, device=w.device)
        src_chunk = ar[None, :] ^ ar[:, None]                                    # [r8, position] -> chunk j = position ^ r8
        return t[:, :, ar[:, None], src_chunk, :].contiguous().view(-1)
    return wb.view(r // 8, 8, k // 8, 8).permute(0, 2, 1, 3).contiguous().view(-1)


def pack_rowmajor(w):
    """[rows, K] fp32 -> bf16 [rows][K + 8]: the small-batch kernel's weight layout (csrc/infer_hmma.cuh): row-major with 16
    bytes of padding per row so that ldmatrix reads are bank-conflict free."""
    r, k = w.shape
    assert r % 16 == 0 and k % 16 == 0, (r, k)
    out = torch.zeros(r, k + 8, dtype=torch.bfloat16, device=w.device)
    out[:, :k] = w.to(torch.bfloat16)
    return out.view(-1)


def _interleave_gnn(stacked):
    """Stacked GraphNetNN weight [gc (64 rows); nn (64 rows)] -> column group q of the small-batch kernel gets, in its
    128 / nq output columns, gc[fw*q : fw*(q+1)] then nn[fw*q : fw*(q+1)] (both halves of the fw = 64 / nq features it
    normalises); nq = column groups the kernel was compiled for."""
    nq = lib.maz_infer_small_nq()
    fw = GH // nq
    gc, nn = stacked[:GH], stacked[GH:]
    return torch.cat([torch.cat([gc[fw * q:fw * (q + 1)], nn[fw * q:fw * (q + 1)]]) for q in range(nq)])


def _padcols(w, k):
    out = torch.zeros(w.shape[0], k, dtype=w.dtype, device=w.device)
    out[:, : w.shape[1]] = w
    return out


def _padrows(w, r):
    out = torch.zeros(r, w.shape[1], dtype=w.dtype, device=w.device)
    out[: w.shape[0]] = w
    return out


def supported(sd, num_agents, action_space_size, hidden):
    d = "dynamics_network."
    try:
        return (hidden == H and num_agents <= 30 and action_space_size <= A_MAX   # 30 = positional table (attention.py:35)
                and f"{d}attention_stack.2.encoder.layers.2.linear1.weight" in sd
                and f"{d}attention_stack.2.encoder.layers.3.linear1.weight" not in sd
                and sd[f"{d}attention_stack.2.encoder.layers.0.linear1.weight"].shape == (H, H)
                and sd[f"{d}fc_dynamic.3.weight"].shape == (H, H) and f"{d}fc_dynamic.6.weight" in sd
                and f"{d}fc_dynamic.9.weight" not in sd
                and sd[f"{d}reward_predictor.gc1.lin_layer.weight"].shape[0] == GH
                and sd[f"{d}reward_predictor.V.weight"].shape[0] == SUP
                and sd["prediction_network.value_predictor.V.weight"].shape[0] == SUP
                and sd["prediction_network.fc_policy.0.weight"].shape[0] == PH
                and "prediction_network.fc_policy.3.weight" in sd and "prediction_network.fc_policy.6.weight" not in sd)
    except KeyError:
        return False


def supported_initial(sd, num_agents, action_space_size, hidden):
    """The root-inference kernel (csrc/infer_initial.cuh, `maz_infer_initial`) takes the reference representation network
    (config/smac/model.py:176-195, use_feature_norm): feature_norm, then mlp([obs, 128, 128, 128]) = Linear, LayerNorm, ReLU,
    Linear, LayerNorm, ReLU, Linear (mlp.{0,1,3,4,6}), 1 <= obs <= 640, on top of the heads `supported` takes."""
    return initial_unsupported_reason(sd, num_agents, action_space_size, hidden) is None


def initial_unsupported_reason(sd, num_agents, action_space_size, hidden):
    if not supported(sd, num_agents, action_space_size, hidden):
        return ("the network is not the reference SMAC architecture the fused kernels take (hidden 128, 3 x 8-head encoder "
                "layers, support 11, <= 30 agents, <= 128 actions)")
    m = REP + "mlp."
    if f"{m}0.weight" not in sd:
        return "the state dict holds no representation network"
    if f"{REP}feature_norm.weight" not in sd or f"{REP}feature_norm.bias" not in sd:
        return "the representation network has no feature_norm (use_feature_norm=False)"
    layers = sorted(int(k[len(m):].split(".")[0]) for k in sd if k.startswith(m) and k.endswith(".weight"))
    if layers != [0, 1, 3, 4, 6]:
        return f"the representation mlp must be Linear, LN, ReLU, Linear, LN, ReLU, Linear (mlp.0/1/3/4/6), not layers {layers}"
    obs = sd[f"{m}0.weight"].shape[1]
    shapes = {f"{REP}feature_norm.weight": (obs,), f"{REP}feature_norm.bias": (obs,), f"{m}0.weight": (H, obs), f"{m}0.bias": (H,),
              f"{m}1.weight": (H,), f"{m}1.bias": (H,), f"{m}3.weight": (H, H), f"{m}3.bias": (H,), f"{m}4.weight": (H,),
              f"{m}4.bias": (H,), f"{m}6.weight": (H, H), f"{m}6.bias": (H,)}
    for k, shp in shapes.items():
        if k not in sd or tuple(sd[k].shape) != shp:
            return f"representation parameter {k}: expected shape {shp} (widths [obs, 128, 128, 128])"
    if not 1 <= obs <= OBS_MAX:
        return f"observation size {obs} outside 1..{OBS_MAX}"
    return None


def pack_representation(sd, device):
    """The representation network in the layout of maz_initial_desc (include/maz_infer.h): bf16 row-major chunks with 8 elements
    of padding -- mlp.0 (zero columns up to kp = obs rounded up to 16) as column blocks of <= 128 features, then mlp.3, mlp.6 --
    and one fp32 vector: feature_norm weight / bias (zero padded to kp), mlp.0 bias, mlp.1 w / b, mlp.3 bias, mlp.4 w / b,
    mlp.6 bias.  Returns (wpk bf16 flat, vec fp32, obs)."""
    g = lambda k: sd[REP + k].detach().to(device=device, dtype=torch.float32)
    w0 = g("mlp.0.weight")
    obs = w0.shape[1]
    kp = _pad16(obs)
    w0 = _padcols(w0, kp)
    chunks = [w0[:, k0:k0 + 128] for k0 in range(0, kp, 128)] + [g("mlp.3.weight"), g("mlp.6.weight")]
    wpk = torch.cat([pack_rowmajor(c.contiguous()) for c in chunks])
    pad = lambda v: torch.cat([v, torch.zeros(kp - obs, device=v.device)])
    vec = torch.cat([pad(g("feature_norm.weight")), pad(g("feature_norm.bias")), g("mlp.0.bias"), g("mlp.1.weight"),
                     g("mlp.1.bias"), g("mlp.3.bias"), g("mlp.4.weight"), g("mlp.4.bias"), g("mlp.6.bias")]).contiguous()
    return wpk, vec, obs


class FusedParams:
    """Device-resident packed parameters + the constant half of the launch descriptor."""

    def __init__(self, sd, num_agents, action_space_size, device):
        self.N, self.A = int(num_agents), int(action_space_size)
        self.KA = _pad16(self.A)
        self.device = torch.device(device)
        self.wpk = None
        self.vec = None
        self.rep_wpk = self.rep_vec = None     # representation network (root inference), when the state dict has a supported one
        self.repack(sd)

    def repack(self, sd):
        dev, N, A, KA = self.device, self.N, self.A, self.KA
        g = lambda k: sd[k].detach().to(device=dev, dtype=torch.float32)
        d, p = "dynamics_network.", "prediction_network."
        chunks = []
        w_in = g(d + "attention_stack.0.weight")                       # (128, 128 + A)
        chunks += [w_in[:, :H], _padcols(w_in[:, H:H + A], KA)]
        for l in range(3):
            e = f"{d}attention_stack.2.encoder.layers.{l}."
            qkv = g(e + "self_attn.in_proj_weight")
            chunks += [qkv[0:H], qkv[H:2 * H], qkv[2 * H:3 * H], g(e + "self_attn.out_proj.weight"),
                       g(e + "linear1.weight"), g(e + "linear2.weight")]
        wd1 = g(d + "fc_dynamic.0.weight")                             # (128, 128 + A + 128)
        chunks += [wd1[:, :H], _padcols(wd1[:, H:H + A], KA), wd1[:, H + A:], g(d + "fc_dynamic.3.weight"),
                   g(d + "fc_dynamic.6.weight")]
        r = d + "reward_predictor."
        wr1 = torch.cat([g(r + "gc1.lin_layer.weight"), g(r + "nn_gc1.weight")], 0)      # (128, 128 + A)
        chunks += [wr1[:, :H], _padcols(wr1[:, H:H + A], KA)]                            # chunks 25, 26
        chunks.append(torch.cat([g(r + "gc2.lin_layer.weight"), g(r + "nn_gc2.weight")], 0))
        v = p + "value_predictor."
        chunks.append(torch.cat([g(v + "gc1.lin_layer.weight"), g(v + "nn_gc1.weight")], 0))
        chunks.append(torch.cat([g(v + "gc2.lin_layer.weight"), g(v + "nn_gc2.weight")], 0))
        chunks.append(g(p + "fc_policy.0.weight"))                     # (32, 128)
        chunks.append(_padrows(g(p + "fc_policy.3.weight"), KA))       # (KA, 32)
        assert len(chunks) == NCHUNK
        # small-batch kernel: same 32 matrices, row-major padded, heads merged into two stages
        # (L1: reward h / reward onehot / value / policy.0; L2: reward / value / policy.3), GNN rows interleaved
        c = chunks
        hm = c[:25] + [_interleave_gnn(c[25]), _interleave_gnn(c[26]), _interleave_gnn(c[28]), c[30],
                       _interleave_gnn(c[27]), _interleave_gnn(c[29]), c[31]]
        hp = [pack_rowmajor(t.contiguous()) for t in hm]
        offs_h, o = [], 0
        for t in hp:
            offs_h.append(o)
            o += t.numel() * 2
        wpk_h = torch.cat(hp)
        self.chunk_off_h, self.chunk_bytes_h = offs_h, [t.numel() * 2 for t in hp]
        if getattr(self, "wpk_h", None) is None:
            self.wpk_h = wpk_h
        else:
            self.wpk_h.copy_(wpk_h)
        packed = [pack_operand(c.contiguous()) for c in chunks]
        offs, o = [], 0
        for t in packed:
            offs.append(o)
            o += t.numel() * 2
        wpk = torch.cat(packed)
        self.chunk_off = offs
        self.chunk_bytes = [t.numel() * 2 for t in packed]

        # two-tiles-in-flight kernel (csrc/infer_twin.cuh): 32 matrices in the order of its stage table (per layer [Q|K] and V of
        # heads 0-3, of heads 4-7, out-proj, linear1, linear2; no one-hot blocks), each stored as K-halves (<= 64 input features, <= 16 KB)
        tw = [c[0]]
        for l in range(3):
            b = 2 + 6 * l
            wq, wk, wv = c[b], c[b + 1], c[b + 2]
            for h in (0, 1):                  # four heads per stage: [Q rows | K rows] stacked (128 x 128), V rows (64 x 128)
                tw += [torch.cat([wq[64 * h:64 * h + 64], wk[64 * h:64 * h + 64]], 0), wv[64 * h:64 * h + 64]]
            tw += [c[b + 3], c[b + 4], c[b + 5]]
        tw += [c[20], c[22], c[23], c[24], c[25], c[27], c[28], c[29], c[30], c[31]]
        assert len(tw) == NCHUNK
        tp = []
        for m in tw:
            m = m.contiguous()
            tp.append(torch.cat([pack_operand(m[:, k0:k0 + 64].contiguous()) for k0 in range(0, m.shape[1], 64)]))
        offs_t, o = [], 0
        for t in tp:
            offs_t.append(o)
            o += t.numel() * 2
        wpk_t = torch.cat(tp)
        self.chunk_off_t, self.chunk_bytes_t = offs_t, [t.numel() * 2 for t in tp]
        if getattr(self, "wpk_t", None) is None:
            self.wpk_t = wpk_t
        else:
            self.wpk_t.copy_(wpk_t)
        # the one-hot blocks as bf16 [A][128] tables (what the one-hot MMA would have added), stored as [A][64] 32-bit words
        oh = [w[:, H:H + A].t().contiguous().to(torch.bfloat16).view(torch.float32) for w in (w_in, wd1, wr1)]

        vec, self.off = [], {}

        def put(name, *ts):
            self.off[name] = sum(t.numel() for t in vec)
            for t in ts:
                vec.append(t.reshape(-1))

        z16 = torch.zeros(16, device=dev)
        put("bin", g(d + "attention_stack.0.bias"))
        put("pos", g(d + "attention_stack.2.pos_embed.pos_table")[0, :N].contiguous())
        self.off["layer"] = sum(t.numel() for t in vec)
        for l in range(3):
            e = f"{d}attention_stack.2.encoder.layers.{l}."
            qb = g(e + "self_attn.in_proj_bias")
            vec += [qb, g(e + "self_attn.out_proj.bias"), g(e + "norm1.weight"), g(e + "norm1.bias"), g(e + "linear1.bias"),
                    g(e + "linear2.bias"), g(e + "norm2.weight"), g(e + "norm2.bias")]
        put("dyn", g(d + "fc_dynamic.0.bias"), g(d + "fc_dynamic.1.weight"), g(d + "fc_dynamic.1.bias"),
            g(d + "fc_dynamic.3.bias"), g(d + "fc_dynamic.4.weight"), g(d + "fc_dynamic.4.bias"), g(d + "fc_dynamic.6.bias"))
        for name, pre in (("rg", r), ("vg", v)):
            put(name, g(pre + "gc1.lin_layer.bias"), g(pre + "nn_gc1.bias"), g(pre + "gc2.lin_layer.bias"), g(pre + "nn_gc2.bias"),
                g(pre + "V.weight"), torch.cat([g(pre + "V.bias"), z16[: 16 - SUP]]))
        bp2 = torch.cat([g(p + "fc_policy.3.bias"), torch.zeros(KA - A, device=dev)])
        put("pol", g(p + "fc_policy.0.bias"), g(p + "fc_policy.1.weight"), g(p + "fc_policy.1.bias"), bp2)
        vecf = torch.cat(vec)
        if vecf.numel() % 8:      # (a multiple of 4 for the bulk copy; of 8 so that the tables behind it are 32-byte aligned)
            vecf = torch.cat([vecf, torch.zeros(8 - vecf.numel() % 8, device=dev)])
        vecf = vecf.contiguous()
        assert all(o % 4 == 0 for o in self.off.values())
        self.off_oh = [vecf.numel() + i * A * (H // 2) for i in range(3)]
        vec_t = torch.cat([vecf] + [t.reshape(-1) for t in oh]).contiguous()
        if self.wpk is None:
            self.wpk, self.vec, self.vec_t = wpk, vecf, vec_t
        else:                      # keep addresses stable for captured CUDA graphs
            self.wpk.copy_(wpk)
            self.vec.copy_(vecf)
            self.vec_t.copy_(vec_t)
        if supported_initial(sd, N, A, H):
            rw, rv, self.obs_dim = pack_representation(sd, dev)
            if self.rep_wpk is None or self.rep_wpk.shape != rw.shape:
                self.rep_wpk, self.rep_vec = rw, rv
            else:
                self.rep_wpk.copy_(rw)
                self.rep_vec.copy_(rv)

    def initial_desc(self, B, obs, hidden, value, policy_logits):
        """maz_initial_desc for `maz_infer_initial`: obs (B*N, obs_dim) fp32, outputs hidden (B, N*128), value (B,),
        policy_logits (B, N, A); device tensors (or None for a bare descriptor)."""
        ptr = lambda t: (t.data_ptr() if t is not None else None)
        dsc = InitialDesc()
        dsc.B, dsc.N, dsc.A, dsc.H = int(B), self.N, self.A, H
        dsc.obs_dim = int(self.obs_dim) if self.rep_wpk is not None else 0
        dsc.obs, dsc.hidden, dsc.value, dsc.policy_logits = ptr(obs), ptr(hidden), ptr(value), ptr(policy_logits)
        dsc.rep_wpk, dsc.rep_vec = ptr(self.rep_wpk), ptr(self.rep_vec)
        dsc.wpk, dsc.vec, dsc.vec_floats = self.wpk_h.data_ptr(), self.vec.data_ptr(), self.vec.numel()
        for i in range(NCHUNK):
            dsc.chunk_off[i], dsc.chunk_bytes[i] = self.chunk_off_h[i], self.chunk_bytes_h[i]
        dsc.o_vg, dsc.o_pol = self.off["vg"], self.off["pol"]
        return dsc

    def desc(self, B, pool, idx_x, actions, next_hidden, reward, value, probs, beta, greedy=None, logits_out=None,
             tree_agents=None, cur=-1, inv_tau=1.0, dbg_clock=None, small=False, factor=None, greedy_pool=None, roots_per_tile=0,
             twin=None):
        ptr = lambda t: (t.data_ptr() if t is not None else None)
        dsc = InferDesc()
        dsc.B, dsc.N, dsc.A, dsc.KA, dsc.NAP = int(B), self.N, self.A, self.KA, self.KA
        dsc.Nt = self.N if tree_agents is None else int(tree_agents)
        dsc.cur, dsc.inv_tau = int(cur), float(inv_tau)
        dsc.pool, dsc.idx_x, dsc.actions, dsc.next_hidden = ptr(pool), ptr(idx_x), ptr(actions), ptr(next_hidden)
        dsc.reward, dsc.value, dsc.probs, dsc.beta = ptr(reward), ptr(value), ptr(probs), ptr(beta)
        dsc.greedy, dsc.logits_out = ptr(greedy), ptr(logits_out)
        dsc.dbg_clock = ptr(dbg_clock)
        dsc.factor, dsc.greedy_pool, dsc.roots_per_tile = ptr(factor), ptr(greedy_pool), int(roots_per_tile)
        import os as _os
        dsc.dbg_flags = int(_os.environ.get('MAZ_DBG_FLAGS', '0'))
        if twin is not None and not twin and not small and self.A > A_NARROW:
            raise ValueError(f"the first-generation tcgen05 kernel supports at most {A_NARROW} actions per agent (this network has {self.A})")
        twin = (not small) and (use_twin(B, self.N, self.A) if twin is None else bool(twin))
        dsc.wpk, dsc.vec, dsc.vec_floats = (self.wpk_h if small else self.wpk).data_ptr(), self.vec.data_ptr(), self.vec.numel()
        co, cb = (self.chunk_off_h, self.chunk_bytes_h) if small else (self.chunk_off, self.chunk_bytes)
        if twin:
            dsc.tc_layout = 1
            dsc.wpk, dsc.vec, dsc.vec_floats = self.wpk_t.data_ptr(), self.vec_t.data_ptr(), self.vec_t.numel()
            co, cb = self.chunk_off_t, self.chunk_bytes_t
            dsc.o_oh_in, dsc.o_oh_dyn, dsc.o_oh_rg = self.off_oh
        for i in range(NCHUNK):
            dsc.chunk_off[i], dsc.chunk_bytes[i] = co[i], cb[i]
        o = self.off
        dsc.o_bin, dsc.o_pos, dsc.o_layer, dsc.o_dyn = o["bin"], o["pos"], o["layer"], o["dyn"]
        dsc.o_rg, dsc.o_vg, dsc.o_pol = o["rg"], o["vg"], o["pol"]
        return dsc


def _weights_desc(self, B, small):
    """The weight half of a descriptor (buffers NULL): what maz_search_create copies."""
    return self.desc(B, None, None, None, None, None, None, None, None, small=small)


FusedParams.weights_desc = _weights_desc


# Which kernel: the tcgen05 kernel needs 128-row tiles (a CTA per 4*floor(32/N) roots), the small-batch kernel 32-row tiles
# (a CTA per floor(32/N) roots) but re-reads the 0.9 MB of weights from L2 once per CTA.  MAZ_INFER_KERNEL=small|tcgen05
# forces one; "auto" takes the small-batch kernel while its grid stays within SMALL_MAX_TILES.
SMALL_MAX_TILES = int(os.environ.get("MAZ_INFER_SMALL_MAX_TILES", "222"))   # 1.5 waves of 148 SMs (measured cross-over, profiles/prof_infer_cmp.py)


def use_twin(B=None, N=None, A=None):
    """Which large-batch kernel: two tiles in flight per CTA (csrc/infer_twin.cuh) or the first generation, one tile per CTA
    (csrc/infer_fused.cuh).  MAZ_INFER_TC=twin|v1 forces one.  With more than A_NARROW actions per agent (A given) only the twin
    kernel has a (wide) instance: the answer is True, and MAZ_INFER_TC=v1 raises ValueError.  Cost model from profiles/r02_infer_cmp.log (per launch, B200): a wave
    of tile PAIRS takes ~141-146 us whatever the team size, a wave of single first-generation tiles 88 us (N = 3), 96 (N = 5),
    117 (N = 10), 166 (N = 27) ~ 80 + 3.2 N; the kernel with the shorter sum of waves on 148 SMs is taken (e.g. 3m-shaped 16 384
    roots: 3 x 88 us of single tiles beat 2 x 141 us of pairs; 2s3z 4096 roots: one wave of pairs beats two of single tiles)."""
    mode = os.environ.get("MAZ_INFER_TC", "auto")
    if A is not None and int(A) > A_NARROW:
        if mode == "v1":
            raise ValueError(f"MAZ_INFER_TC=v1: the first-generation tcgen05 kernel supports at most {A_NARROW} actions per agent "
                             f"(this network has {int(A)}); unset MAZ_INFER_TC or set it to twin")
        return True
    if mode in ("twin", "v1"):
        return mode == "twin"
    if B is None or N is None:
        return True
    sms = 148
    tiles = -(-int(B) // (4 * (32 // int(N))))
    pairs = (tiles + 1) // 2
    t_pairs = -(-pairs // sms) * (141.0 + 0.2 * int(N))
    t_tiles = -(-tiles // sms) * (80.0 + 3.2 * int(N))
    return t_pairs < t_tiles


def use_small(B, N):
    mode = os.environ.get("MAZ_INFER_KERNEL", "auto")
    if mode in ("small", "tcgen05"):
        return mode == "small"
    rpt = 32 // N
    return (B + rpt - 1) // rpt <= SMALL_MAX_TILES


def launch_initial(dsc, stream_ptr):
    check(lib.maz_infer_initial(C.byref(dsc), C.c_void_p(stream_ptr)))


def launch(dsc, stream_ptr, small=False):
    fn = lib.maz_infer_recurrent_small if small else lib.maz_infer_recurrent
    check(fn(C.byref(dsc), C.c_void_p(stream_ptr)))
