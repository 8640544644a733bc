"""GPU: `SampledMCTS.search_agents_sharded` -- the N sequential per-agent searches of one environment step with the roots sharded
over the ranks -- equals single-process `search_agents` over all roots bit for bit, and leaves `np_random` in the same state.

* emulated ranks (one GPU): the per-rank body `_search_agents_rank` for every rank of a world, each with its own copy of the
  generator; the ranks' local slices concatenated, and their raw step buffers merged as the all-gather path merges them;
* real ranks (>= 2 GPUs, NCCL): the public entry with gather=True, one `all_gather_into_tensor` per environment step."""
import os
import socket

import numpy as np
import pytest
import torch

from _mock import MockConfig
from test_search_gpu import root_output, smac_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, K, S = 37, 10, 20
SHAPES = {"3m": (3, 9), "2s3z": (5, 11)}


def _inputs(N, A, dev):
    model = smac_model(N, A)
    out0 = root_output(model, B)
    out0 = out0._replace(hidden_state=out0.hidden_state.to(dev))
    legal = (np.random.RandomState(6).rand(B, N, A) < 0.7).astype(np.float32)
    legal[..., 1] = 1
    rng = np.random.RandomState(9)
    eps_u = rng.rand(N, B).astype(np.float32)
    rand_act = np.stack([[rng.choice(np.where(legal[b, k] > 0)[0]) for b in range(B)] for k in range(N)]).astype(np.int32)
    return model, out0, legal, (eps_u, rand_act)


def _slice(out0, legal, eps, start, count):
    sl = slice(start, start + count)
    return out0._replace(hidden_state=out0.hidden_state[sl], reward=out0.reward[sl], value=out0.value[sl],
                         policy_logits=out0.policy_logits[sl]), legal[sl], (eps[0][:, sl], eps[1][:, sl])


def _kwargs(turn, eps):
    return dict(add_noise=True, sampled_tau=1.0, turn=turn, temperature=0.5, greedy_epsilon=0.3 if turn == "sample" else 0.0,
                eps_randoms=eps if turn == "sample" else None)


def _concat(parts):
    """Local AgentTurnsOutputs of consecutive root slices -> (turn arrays, per-agent list of {field: per-root arrays})."""
    turns = {f: np.concatenate([getattr(p, f) for p in parts]) for f in ("actions", "policy_dist", "prob", "entropy")}
    agents = []
    for k in range(len(parts[0].search_outputs)):
        fields = {}
        for f in parts[0].search_outputs[k]._fields:
            xs = [getattr(p.search_outputs[k], f) for p in parts]
            fields[f] = np.concatenate(xs) if isinstance(xs[0], np.ndarray) else [a for x in xs for a in x]
        agents.append(fields)
    return turns, agents


def _assert_equal(got_turns, got_agents, ref):
    for f, v in got_turns.items():
        r = getattr(ref, f)
        assert v.dtype == r.dtype and v.shape == r.shape and np.array_equal(v.view(np.uint8), r.view(np.uint8)), f
    assert len(got_agents) == len(ref.search_outputs)
    for k, fields in enumerate(got_agents):
        for f, v in fields.items():
            r = getattr(ref.search_outputs[k], f)
            if isinstance(r, np.ndarray):
                assert v.dtype == r.dtype and np.array_equal(v, r), (k, f)
            else:
                assert len(v) == len(r) and all(np.array_equal(a, b) for a, b in zip(v, r)), (k, f)


def _same_state(a, b):
    sa, sb = a.get_state(), b.get_state()
    return sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


@pytest.mark.parametrize("turn", ["greedy", "sample"])
@pytest.mark.parametrize("shape", ["3m", "2s3z"])
@pytest.mark.parametrize("world", [2, 3])
def test_emulated_ranks_equal_single_process_search_agents(built_lib, world, shape, turn):
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import AgentTurnsOutput, SampledMCTS, _local_agent_turns, _output_from_readout
    from mazero_b200.sharding import merge_turn_shards, shard_range

    N, A = SHAPES[shape]
    cfg = MockConfig(N, A, S, K)
    model, out0, legal, eps = _inputs(N, A, DEV)
    inf = SmacInference.from_model(model, device=DEV, mode="bf16")
    ref_rs = np.random.RandomState(21)
    ref = SampledMCTS(cfg, ref_rs).search_agents(inf, out0, N, legal, DEV, **_kwargs(turn, eps))

    parts, blocks, states = [], [], []
    for r in range(world):
        start, count = shard_range(B, r, world)
        o, lg, ep = _slice(out0, legal, eps, start, count)
        rs = np.random.RandomState(21)
        plan, n = SampledMCTS(cfg, rs)._search_agents_rank(inf, o, N, B, r, world, lg, DEV, **_kwargs(turn, ep))
        assert n == count
        torch.cuda.synchronize()
        blocks.append(plan.res_flat.cpu().numpy())          # what this rank contributes to the all-gather
        layout = plan.turn_layout()
        parts.append(_local_agent_turns(plan, count))
        states.append(rs)
    _assert_equal(*_concat(parts), ref)
    # the gather path's merge of the raw step buffers, with the plan's own layout
    outs, t = merge_turn_shards(np.stack(blocks), layout, B, world)
    merged = AgentTurnsOutput(t["turn_actions"], t["policy_dist"], t["prob_prod"], t["entropy"], [_output_from_readout(x) for x in outs])
    _assert_equal(*_concat([merged]), ref)
    # every rank's generator ends where the single-process one does
    assert all(_same_state(rs, ref_rs) for rs in states)


def test_wrong_local_row_count_is_refused(built_lib):
    from mazero_b200.inference import SmacInference
    from mazero_b200.mcts_sampled import SampledMCTS

    N, A = SHAPES["3m"]
    model, out0, legal, eps = _inputs(N, A, DEV)
    inf = SmacInference.from_model(model, device=DEV, mode="bf16")
    m = SampledMCTS(MockConfig(N, A, S, K), np.random.RandomState(0))
    o, lg, ep = _slice(out0, legal, eps, 0, 19)           # rank 0 of 2 owns 19 roots
    with pytest.raises(ValueError, match="rank 1: expected 18 local roots, got 19"):
        m._search_agents_rank(inf, o, N, B, 1, 2, lg, DEV)
    with pytest.raises(ValueError, match="rank 0: expected 19 local roots"):
        m._search_agents_rank(inf, o, N, B, 0, 2, lg, DEV, turn="sample", eps_randoms=(eps[0][:, :18], eps[1][:, :18]))


# ---- real ranks: one process per GPU, NCCL -----------------------------------------------------------------------------------------
def _worker(rank, world, port, q):
    import torch.distributed as dist

    try:
        os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
        dev = torch.device("cuda", rank)
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        from mazero_b200.inference import SmacInference
        from mazero_b200.mcts_sampled import SampledMCTS
        from mazero_b200.sharding import shard_range

        calls = [0]
        gather = dist.all_gather_into_tensor

        def counted(*a, **kw):
            calls[0] += 1
            return gather(*a, **kw)

        dist.all_gather_into_tensor = counted
        N, A = SHAPES["3m"]
        cfg = MockConfig(N, A, S, K)
        model, out0, legal, eps = _inputs(N, A, dev)
        inf = SmacInference.from_model(model, device=dev, mode="bf16")
        start, count = shard_range(B, rank, world)
        o, lg, ep = _slice(out0, legal, eps, start, count)
        rs, ref_rs = np.random.RandomState(21), np.random.RandomState(21)
        m, ref_m = SampledMCTS(cfg, rs), SampledMCTS(cfg, ref_rs)
        msgs = []
        for step, turn in enumerate(("greedy", "sample")):           # two environment steps, one generator
            got = m.search_agents_sharded(inf, o, N, B, lg, dev, group=None, gather=True, **_kwargs(turn, ep))
            if calls[0] != step + 1:
                msgs.append(f"{turn}: {calls[0]} all_gather_into_tensor calls after {step + 1} steps")
            if rank == 0:                                             # the single-process reference, in lockstep
                ref = ref_m.search_agents(inf, out0, N, legal, dev, **_kwargs(turn, eps))
                try:
                    _assert_equal(*_concat([got]), ref)
                except AssertionError as e:
                    msgs.append(f"{turn}: rank 0 output differs from search_agents: {e}")
                if not _same_state(rs, ref_rs):
                    msgs.append(f"{turn}: generator state differs from the single-process run")
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, msgs))
    except Exception as e:  # reported to the parent, which fails the test
        q.put((rank, [f"{type(e).__name__}: {e}"]))
        raise


@pytest.mark.parametrize("world", [2, 4, 8])
def test_real_ranks_gather_equals_single_process_search_agents(built_lib, world):
    import torch.multiprocessing as mp

    have = torch.cuda.device_count()
    if have < world:
        pytest.skip(f"needs {world} GPUs for {world} NCCL ranks (one per GPU); this machine has {have}")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = dict(q.get(timeout=600) for _ in procs)
        for p in procs:
            p.join(timeout=120)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    assert sorted(results) == list(range(world))
    assert all(not msgs for msgs in results.values()), results
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
