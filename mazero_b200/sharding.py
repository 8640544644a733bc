"""Root sharding across the GPUs of one box (SURVEY 8e).

Trees are independent (private RNG seeded by the GLOBAL root index, cnode.cpp:571-576), so rank r owns the
contiguous root slice `shard_range(B, r, world)` and passes `root_index_offset = start` to the search:
results are identical to one `Tree_batch` over all B roots, whatever the number of ranks.  There is no
collective inside the simulation loop; the only exchange is ONE all-gather of the packed readouts per
search (root values, visit counts, sampled actions ...) so that the learner rank sees every root.  The per-agent loop of one
environment step (`SampledMCTS.search_agents_sharded`) exchanges once per step: every agent's readouts and the turn results
travel in one buffer (`merge_turn_shards`).
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(total_roots, rank, world):
    """Contiguous slice [start, start + count) of rank `rank`; the first `total % world` ranks get one extra."""
    base, extra = divmod(int(total_roots), int(world))
    count = base + (1 if rank < extra else 0)
    start = rank * base + min(rank, extra)
    return start, count


def pack_readout(readout, keys=None):
    """dict of per-root arrays (leading dim = local roots) -> (int32 matrix (roots, words), layout)."""
    keys = sorted(readout) if keys is None else list(keys)
    cols, layout = [], []
    for k in keys:
        a = np.ascontiguousarray(readout[k])
        if a.dtype not in (np.int32, np.float32):
            raise ValueError(f"{k}: only int32 / float32 readouts can be packed, got {a.dtype}")
        flat = a.reshape(a.shape[0], -1).view(np.int32)
        layout.append((k, a.dtype, a.shape[1:], flat.shape[1]))
        cols.append(flat)
    return np.concatenate(cols, axis=1), layout


def unpack_readout(mat, layout):
    out, o = {}, 0
    for k, dt, shp, w in layout:
        out[k] = np.ascontiguousarray(mat[:, o:o + w]).view(dt).reshape((mat.shape[0],) + tuple(shp))
        o += w
    return out


def all_gather_readouts(readout, total_roots, group=None, device=None):
    """Every rank contributes the readouts of its root slice; returns the dict for ALL roots in global root
    order (on every rank; the learner is rank 0).  One collective.  Works with NCCL (device tensors) and gloo."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    mat, layout = pack_readout(readout)
    start, count = shard_range(total_roots, rank, world)
    if mat.shape[0] != count:
        raise ValueError(f"rank {rank}: expected {count} local roots, got {mat.shape[0]}")
    max_count = shard_range(total_roots, 0, world)[1]
    buf = torch.zeros(max_count, mat.shape[1], dtype=torch.int32, device=device)
    buf[:count] = torch.from_numpy(mat).to(buf.device)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf, group=group)
    rows = [parts[r][: shard_range(total_roots, r, world)[1]].cpu().numpy() for r in range(world)]
    return unpack_readout(np.concatenate(rows, axis=0), layout)


# ---- the product-level sharded search: device tensors end to end ------------------------------------------------------------
def pad_rows(x, rows):
    """Repeat the last row of a per-root array (numpy or torch) up to `rows` rows: ranks with one root less than the largest shard
    search a dummy copy of their last root, whose results are dropped after the exchange."""
    n = x.shape[0]
    if n == rows:
        return x
    if torch.is_tensor(x):
        return torch.cat([x, x[-1:].expand(rows - n, *x.shape[1:])], dim=0)
    return np.concatenate([x, np.repeat(x[-1:], rows - n, axis=0)], axis=0)


def split_packed(words, spec, roots):
    """One rank's packed readout block (1-D int32, field-major as `_DevicePlan` lays it out) -> dict of per-root arrays."""
    out, o = {}, 0
    for name, dt, shp in spec:
        n = int(np.prod(shp))
        out[name] = words[o:o + n].view(dt).reshape(shp)
        o += n
    assert all(v.shape[0] == roots for v in out.values())
    return out


def merge_shards(blocks, spec_of, total_roots, world):
    """blocks[r] = rank r's packed readouts (padded to the largest shard); returns the dict for ALL roots in global order."""
    parts = []
    for r in range(world):
        _, count = shard_range(total_roots, r, world)
        d = split_packed(blocks[r], spec_of, shard_range(total_roots, 0, world)[1])
        parts.append({k: v[:count] for k, v in d.items()})
    return {k: np.concatenate([p[k] for p in parts], axis=0) for k in parts[0]}


# ---- the sharded environment step (`SampledMCTS.search_agents_sharded`): ONE buffer per rank holds every agent's readouts and the
# turn results, and ONE all-gather exchanges it -------------------------------------------------------------------------------------
def split_turn_block(words, layout, roots):
    """One rank's step buffer (1-D int32, `_DevicePlan.res_flat`) -> (per-agent readout dicts, dict of the turn fields).
    layout = (readout_spec, agent_offsets, turn_fields) as `_DevicePlan.turn_layout()` gives it: the word offset of each agent's
    packed readout block, and (name, dtype, shape, word offset) of every turn field.  8-byte fields are copied out of the int32 words
    (never viewed at a 4-byte boundary), so their bits are kept whatever the buffer's alignment."""
    readout_spec, agent_offsets, turn_fields = layout
    n = sum(int(np.prod(shp)) for _, _, shp in readout_spec)
    agents = [split_packed(words[o:o + n], readout_spec, roots) for o in agent_offsets]
    turns = {}
    for name, dt, shp, o in turn_fields:
        dt = np.dtype(dt)
        w = int(np.prod(shp)) * dt.itemsize // 4
        assert dt.itemsize == 4 or o % 2 == 0, f"{name}: {dt} field at the odd word offset {o}"
        assert o + w <= len(words), f"{name}: past the end of the block"
        turns[name] = np.ascontiguousarray(words[o:o + w]).view(dt).reshape(shp)
        assert turns[name].shape[0] == roots
    return agents, turns


def merge_turn_shards(blocks, layout, total_roots, world):
    """blocks[r] = rank r's step buffer (padded to the largest shard); returns (per-agent readout dicts, turn-field dict) for ALL
    roots in global root order, the padding rows dropped."""
    rows = shard_range(total_roots, 0, world)[1]
    assert len(blocks) == world and all(len(b) % 2 == 0 for b in blocks), "step buffers are whole 8-byte words"
    parts = []
    for r in range(world):
        _, count = shard_range(total_roots, r, world)
        agents, turns = split_turn_block(blocks[r], layout, rows)
        parts.append(([{k: v[:count] for k, v in d.items()} for d in agents], {k: v[:count] for k, v in turns.items()}))
    cat = lambda ds: {k: np.concatenate([d[k] for d in ds], axis=0) for k in ds[0]}
    agents = [cat([p[0][t] for p in parts]) for t in range(len(parts[0][0]))]
    return agents, cat([p[1] for p in parts])
