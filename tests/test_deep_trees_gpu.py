"""GPU: deep trees through the whole device search, replayed bit for bit through the CPU oracle tree.

The network-driven searches of the other tests build shallow trees (K = 10: paths of 5 to 11 nodes are rare).  Here K = 1 chains
make every path one node longer than the last, up to S: paths longer than a warp, value logs far longer than the 256 entries the
backup caches in registers (tree_step.cuh: kLogRegs), and the persistent kernel's shared-memory tree tables filled to their
S + 2 entries.  Every case runs both loops (the persistent kernel at a pinned number of roots per CTA, and the CUDA-graph loop
of the two-warp fused tree step), with the wide selection at its default threshold, forced off and forced on
(MAZ_SELECT_WIDE); the three give identical results, each equal to the oracle.  Each case also checks, from the oracle's side,
that it reached what it is there for."""
import numpy as np
import pytest

from test_search_gpu import device_path_replay, root_output, smac_model
from test_search_native_gpu import _equal

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# name: (N, A, K, S, roots per CTA of the persistent kernel, B)
ROWS = {
    "3m_k1_s200": (3, 9, 1, 200, 3, 20),
    "3m_k2_s150": (3, 9, 2, 150, 4, 23),             # two children per node: the selection's UCB choice matters
    "2c_vs_64zg_k1_s100": (2, 70, 1, 100, 8, 47),    # the wide instance; its last CTA holds 7 of 8 trees
}


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ("MAZ_SEARCH_STRATEGY", "MAZ_SEARCH_PERSIST_MAX_CTAS", "MAZ_INFER_KERNEL", "MAZ_INFER_TC", "MAZ_SELECT_WIDE"):
        monkeypatch.delenv(k, raising=False)


def _network(row):
    """One network and its roots per test: the runs a test compares must see the same network (smac_model draws some of its
    weights from torch's global generator)."""
    from mazero_b200.inference import SmacInference

    N, A, K, S, rpt, B = ROWS[row]
    model = smac_model(N, A)
    out0 = root_output(model, B)
    return SmacInference.from_model(model, device=DEV, mode="bf16"), out0._replace(hidden_state=out0.hidden_state.cuda())


def _search(row, net, cur, strategy, select_wide, oracle_built, monkeypatch):
    from mazero_b200 import mcts_sampled

    N, A, K, S, rpt, B = ROWS[row]
    inf, out0 = net
    monkeypatch.setenv("MAZ_SEARCH_RPT", str(rpt))
    if select_wide is None:
        monkeypatch.delenv("MAZ_SELECT_WIDE", raising=False)
    else:
        monkeypatch.setenv("MAZ_SELECT_WIDE", select_wide)
    # the tree layout reads MAZ_SELECT_WIDE when the plan is created, and the plan cache key does not hold it
    mcts_sampled.clear_caches()
    try:
        out, lens = device_path_replay(inf, out0, N, A, B, K, S, cur, oracle_built, strategy=strategy)
        plans = list(mcts_sampled._PLAN_CACHE.values())
        assert len(plans) == 1 and plans[0].native is not None
        assert plans[0].native.strategy == strategy
        assert plans[0].native.roots_per_cta() == (rpt if strategy == "persistent" else 0)
    finally:
        mcts_sampled.clear_caches()
    # what the case reaches, from the oracle's side
    log_len = 1 + (lens + 1).sum(axis=0)             # root entry + one entry per path level and simulation
    wide_min_len = 3 + 2 * ((S + 1 + 31) // 32)
    above = int((lens[:-1] >= wide_min_len).sum())   # selections after which the next one is wide by default
    print(f"{row} cur={cur} {strategy} MAZ_SELECT_WIDE={select_wide}: largest path {lens.max()}, longest value log {log_len.max()}, "
          f"selections at or above wide_min_len {wide_min_len}: {above}")
    assert log_len.max() > 256
    if K == 1:
        assert (lens[-1] == S).all() and lens.max() > 32 and above > 0
    return out


@pytest.mark.parametrize("strategy", ["persistent", "graph"])
@pytest.mark.parametrize("row", list(ROWS))
def test_deep_trees_joint(built_lib, oracle_built, monkeypatch, row, strategy):
    net = _network(row)
    outs = [_search(row, net, None, strategy, w, oracle_built, monkeypatch) for w in (None, "0", "1")]
    _equal(outs[1], outs[0], "MAZ_SELECT_WIDE=0 vs default: ")
    _equal(outs[2], outs[0], "MAZ_SELECT_WIDE=1 vs default: ")


@pytest.mark.parametrize("strategy", ["persistent", "graph"])
@pytest.mark.parametrize("turn", ["first", "last"])
@pytest.mark.parametrize("row", list(ROWS))
def test_deep_trees_sequential(built_lib, oracle_built, monkeypatch, row, turn, strategy):
    N = ROWS[row][0]
    _search(row, _network(row), 0 if turn == "first" else N - 1, strategy, None, oracle_built, monkeypatch)


def test_persistent_kernel_refuses_deep_narrow_trees_at_8_roots_per_cta(built_lib):
    """3m at K = 1, S = 200: 8 trees per CTA need 8 x 7296 bytes of tree-step scratch, more than the 27648 bytes the narrow
    instance aliases (search_persist.cuh: TREE_SCRATCH_BYTES).  The persistent strategy is refused and "auto" takes the graph loop."""
    from mazero_b200.inference import SmacInference
    from mazero_b200.search_native import NativeSearch

    N, A, K, S, B = 3, 9, 1, 200, 20
    inf = SmacInference.from_model(smac_model(N, A), device=DEV, mode="bf16")
    with pytest.raises(RuntimeError, match="persistent kernel does not support"):
        NativeSearch(inf, B, K, S, True, strategy="persistent")
    ns = NativeSearch(inf, B, K, S, True)
    assert ns.strategy == "graph"
    del ns
