"""CPU: host-side logic of `SampledMCTS.search_agents_sharded` -- every rank's whole step buffer (each agent's packed readouts +
the turn results, float64 fields included), padded to the largest shard, merged in global root order bit for bit
(`mazero_b200.sharding.merge_turn_shards`), directly and through a gloo world-size-2 all-gather."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mazero_b200.sharding import merge_turn_shards, pad_rows, shard_range

T, N, A, K = 3, 3, 5, 3      # agents (= turns), team size, actions, sampled actions


def _readout_spec(rows):
    return [("value", np.float32, (rows,)), ("num_children", np.int32, (rows,)), ("visit_count", np.int32, (rows, K))]


def _turn_spec(rows):
    return [("turn_actions", np.int32, (rows, N)), ("prob_prod", np.float64, (rows,)), ("policy_dist", np.float64, (rows, N, A)),
            ("entropy", np.float64, (rows, N))]


def _layout(rows):
    """The word layout of a sequential-agent plan's step buffer, restated: T readout blocks rounded to an even word count, then
    the turn fields with every float64 field at an even word offset; the whole buffer an even number of words."""
    words = sum(int(np.prod(s)) for _, _, s in _readout_spec(rows))
    words += words & 1
    o, fields = T * words, []
    for name, dt, shp in _turn_spec(rows):
        if np.dtype(dt).itemsize == 8 and o % 2:
            o += 1
        fields.append((name, dt, shp, o))
        o += int(np.prod(shp)) * np.dtype(dt).itemsize // 4
    return (_readout_spec(rows), [t * words for t in range(T)], fields), o + (o & 1)


def _fake_step(start, count):
    """Deterministic per-root step results keyed by the GLOBAL root index; the float64 fields carry non-trivial bit patterns
    (1/3, subnormals, -0.0, neighbours one ulp apart)."""
    g = np.arange(start, start + count)
    agents = [{"value": (g * 0.5 + t).astype(np.float32), "num_children": ((g + t) % 7).astype(np.int32),
               "visit_count": (g[:, None] * 10 + np.arange(K)[None] + 100 * t).astype(np.int32)} for t in range(T)]
    sub = np.float64(5e-324)
    gg = g.astype(np.float64)
    turns = {"turn_actions": ((g[:, None] * 3 + np.arange(N)[None]) % A).astype(np.int32),
             "prob_prod": 1.0 / (3.0 + gg),
             "policy_dist": ((gg[:, None, None] + 1) / 3.0 + np.arange(N * A).reshape(1, N, A) * sub),
             "entropy": np.stack([np.nextafter(1.0 / 3.0, gg + 1), (gg + 1) * sub, np.where(g % 2 == 0, -0.0, 2.0 / 3.0)], axis=1)}
    return agents, turns


def _block(start, count, rows):
    """One rank's padded step buffer as int32 words, written at the offsets of `_layout`."""
    (rspec, aoffs, fields), total = _layout(rows)
    words = np.zeros(total, dtype=np.int32)
    agents, turns = _fake_step(start, count)
    for t, o in enumerate(aoffs):
        for name, _, shp in rspec:
            a = np.ascontiguousarray(pad_rows(agents[t][name], rows)).reshape(-1).view(np.int32)
            words[o:o + a.size] = a
            o += a.size
    for name, _, _, o in fields:
        a = np.ascontiguousarray(pad_rows(turns[name], rows)).reshape(-1).view(np.int32)
        words[o:o + a.size] = a
    return words


def _check_merged(agents, turns, total):
    want_a, want_t = _fake_step(0, total)
    assert len(agents) == T
    for t in range(T):
        for k, v in want_a[t].items():
            assert agents[t][k].dtype == v.dtype and np.array_equal(agents[t][k], v), (t, k)
    for k, v in want_t.items():
        assert turns[k].dtype == v.dtype and turns[k].shape == v.shape, k
        assert np.array_equal(turns[k].view(np.uint8), v.view(np.uint8)), k        # bit for bit (-0.0 and subnormals included)


@pytest.mark.parametrize("total,world", [(7, 1), (7, 2), (7, 3), (8, 2), (11, 3), (9, 4)])
def test_merge_turn_shards_returns_every_field_in_global_order_bit_for_bit(total, world):
    rows = shard_range(total, 0, world)[1]
    blocks = np.stack([_block(*shard_range(total, r, world), rows) for r in range(world)])
    agents, turns = merge_turn_shards(blocks, _layout(rows)[0], total, world)
    _check_merged(agents, turns, total)


def test_layout_puts_a_float64_field_behind_an_odd_word_count():
    """7 roots over 3 ranks: 3 rows x 3 agents of int32 actions = 9 words before prob_prod, so a pad word keeps it 8-byte aligned;
    a layout that would place it at the odd offset is refused."""
    (rspec, aoffs, fields), _ = _layout(3)
    offs = {n: o for n, _, _, o in fields}
    assert offs["prob_prod"] == offs["turn_actions"] + 9 + 1
    bad = [(n, dt, s, o - 1 if n == "prob_prod" else o) for n, dt, s, o in fields]
    blocks = np.stack([_block(*shard_range(7, r, 3), 3) for r in range(3)])
    with pytest.raises(AssertionError):
        merge_turn_shards(blocks, (rspec, aoffs, bad), 7, 3)


def _worker(rank, world, port, total, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rows = shard_range(total, 0, world)[1]
    mine = torch.from_numpy(_block(*shard_range(total, rank, world), rows))
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    agents, turns = merge_turn_shards(np.stack([p.numpy() for p in parts]), _layout(rows)[0], total, world)
    q.put((rank, [{k: (v.dtype.str, v.shape, v.tobytes()) for k, v in d.items()} for d in agents],
           {k: (v.dtype.str, v.shape, v.tobytes()) for k, v in turns.items()}))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("total", [7, 8])
def test_step_buffers_merge_through_a_gloo_all_gather_world2(total):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, total, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    back = lambda d: {k: np.frombuffer(b, dtype=np.dtype(dt)).reshape(shp) for k, (dt, shp, b) in d.items()}
    assert sorted(r for r, _, _ in results) == [0, 1]
    for _, agents, turns in results:
        _check_merged([back(d) for d in agents], back(turns), total)
