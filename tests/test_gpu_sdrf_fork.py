"""Forked states, batched edits, seed sweeps from an edited graph and the device export (DESIGN §4.11).

``DynamicCurvature.fork`` copies a device-resident SDRF state on the device (``dcr_sdrf_fork``), ``dcr.dynamic.edit_batch``
edits many states in one launch (``dcr_sdrf_edit_batch``), ``DynamicCurvature.rewire_batch`` runs B continuations of
SDRF from the current graph in one launch, and ``SdrfState.edge_index`` exports ``from_networkx(G).edge_index`` on the
device (``dcr_sdrf_export_edge_index``).  Every GPU comparison is bit for bit against the oracle dicts of
``tests/test_gpu_sdrf_edit.py``, a fresh full pass, or the single-state path the batched one stands for."""
from unittest import mock

import numpy as np
import pytest

from test_gpu_sdrf_edit import (MODE_IDS, MODES, OracleGraph, _oracle_log_tuples, check_state, graphs_for,
                                oracle_loop_from, random_edits, same_bits)

INF = float("inf")
NEW_SYMBOLS = ("dcr_sdrf_fork", "dcr_sdrf_edit_batch", "dcr_sdrf_edit_batch_workspace_bytes",
               "dcr_sdrf_export_edge_index")


def _bound(curv_type):
    return 0.2 if curv_type in ("bfc", "bfc_paper") else 2.0


def _oracle_loop(og, loops, bound, tau, uniforms, remove_edges):
    """``oracle_loop_from`` (which always removes) with the oracle loop's ``remove_edges`` argument set."""
    import oracle.sdrf as osd
    import oracle.sdrf_classical as oc
    if remove_edges:
        return oracle_loop_from(og, loops, bound, tau, uniforms)
    loop_b, loop_c = osd.sdrf_oracle, oc.sdrf_classical_oracle
    with mock.patch.object(osd, "sdrf_oracle", lambda e, n, k, _rm, *a, **kw: loop_b(e, n, k, False, *a, **kw)), \
            mock.patch.object(oc, "sdrf_classical_oracle",
                              lambda e, n, ct, k, _rm, *a, **kw: loop_c(e, n, ct, k, False, *a, **kw)):
        return oracle_loop_from(og, loops, bound, tau, uniforms)


def _snapshot(dc):
    rp, od = dc.insertion_order()
    return rp, od, dc.edge_index(), dc.curvature()


def _same_snapshot(a, b):
    return all(same_bits(x, y) if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y) for x, y in zip(a, b))


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_new_symbols_are_declared_and_bound():
    import ctypes

    from dcr import lib as L
    from test_host import _declared_symbols
    declared = set(_declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared and name in L.SIGNATURES
    assert ctypes.sizeof(L.SdrfEditRun) == 32       # dcr_sdrf_edit_run: pointer, pointer, int64, pointer


class _NoState:
    """Stands in for a device state: any use of it fails the test (the checks must come before any launch)."""

    def __getattr__(self, name):
        raise AssertionError(f"the device state was used ({name}) before the argument checks")


def _fake(mode=0, capacity=10, edit_adds=0, loop_adds=0):
    from dcr.dynamic import DynamicCurvature
    dc = DynamicCurvature.__new__(DynamicCurvature)
    dc.mode, dc.capacity, dc._edit_adds, dc._loop_adds, dc._state = mode, capacity, edit_adds, loop_adds, _NoState()
    return dc


def test_edit_batch_checks_before_any_launch():
    from dcr.dynamic import edit_batch
    a, b = _fake(0), _fake(0)
    with pytest.raises(ValueError, match="empty"):
        edit_batch([], [])
    with pytest.raises(ValueError, match="edit lists"):
        edit_batch([a, b], [[[1, 0, 1]]])
    with pytest.raises(ValueError, match="twice"):
        edit_batch([a, b, a], [[[1, 0, 1]]] * 3)
    with pytest.raises(ValueError, match="modes"):
        edit_batch([a, _fake(2)], [[[1, 0, 1]]] * 2)
    with pytest.raises(ValueError, match=r"\[m, 3\]"):
        edit_batch([a, b], [[[1, 0, 1]], [[1, 0]]])


def test_rewire_batch_checks_before_any_launch():
    dc = _fake(capacity=20, edit_adds=6, loop_adds=4)
    with pytest.raises(ValueError, match=r"run 1: 11 iterations exceed the remaining additions budget \(10\)"):
        dc.rewire_batch([10, 11], True, 0.5, INF, uniforms=np.zeros((2, 11)))
    with pytest.raises(ValueError, match="exceed"):
        dc.rewire_batch(11, True, 0.5, INF, uniforms=np.zeros((3, 11)))
    with pytest.raises(ValueError, match="batch of 2 runs"):
        dc.rewire_batch([1, 2, 3], True, 0.5, INF, uniforms=np.zeros((2, 3)))
    with pytest.raises(ValueError, match="uniforms"):
        dc.rewire_batch(1, True, 0.5, INF, uniforms=np.zeros(3))
    with pytest.raises(ValueError, match="empty"):
        dc.rewire_batch(1, True, 0.5, INF, uniforms=[])


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_fork_copies_are_exact_and_deep(mode):
    """Forks after 0, 1 and 300 edits and after a partial rewire equal the source; edits that relocate rows in one copy
    and a rewire of another leave the source and the siblings unchanged."""
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(21)
    for ei, n in graphs_for(curv_type, und)[1:3]:
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=900) as dc:
            for count in (0, 1, 300):
                dc.edit(random_edits(og, count, rng))
                ref = _snapshot(dc)
                copies = dc.fork(3)
                try:
                    for c in copies:
                        assert c.remaining == dc.remaining and c.mode == dc.mode
                        assert _same_snapshot(_snapshot(c), ref)
                    # copy 0: many adds at one node (its row outgrows its slack and moves); copy 1: SDRF
                    u = int(np.argmin([len(a) for a in og.adj]))
                    adds = [(1, u, v) for v in range(n) if v != u and not og.has(u, v)][:40]
                    copies[0].edit(adds)
                    copies[1].rewire(10, True, _bound(curv_type), INF, uniforms=np.zeros(10))
                    assert _same_snapshot(_snapshot(dc), ref) and _same_snapshot(_snapshot(copies[2]), ref)
                    c0 = OracleGraph(np.zeros((2, 0), dtype=np.int64), n, curv_type, und)
                    c0.adj, c0.pred = [dict(a) for a in og.adj], og.pred and [dict(p) for p in og.pred]
                    for op, a, b in adds:
                        c0.apply(op, a, b)
                    check_state(copies[0], c0)
                finally:
                    for c in copies:
                        c.close()
            check_state(dc, og)
            # a fork after a partial rewire carries the rewired graph and what is left of the budget
            dc.rewire(5, True, _bound(curv_type), INF, uniforms=np.zeros(5))
            ref = _snapshot(dc)
            (c,) = dc.fork()
            with c:
                assert c.remaining == dc.remaining and _same_snapshot(_snapshot(c), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_fork_more_copies_than_sms(mode):
    from dcr.dynamic import DynamicCurvature, edit_batch
    curv_type, und = mode
    ei, n = graphs_for(curv_type, und)[0]
    og = OracleGraph(ei, n, curv_type, und)
    with DynamicCurvature(ei, n, curv_type, und, capacity=50) as dc:
        dc.edit(random_edits(og, 20, np.random.default_rng(1)))
        ref = _snapshot(dc)
        copies = dc.fork(300)
        try:
            assert len(copies) == 300 and len({c._state.handle.value for c in copies}) == 300
            for c in copies[::37] + copies[-1:]:
                assert _same_snapshot(_snapshot(c), ref)
            # 300 different single edits in one launch, each copy checked against its own oracle graph
            rng = np.random.default_rng(2)
            ops = []
            for _ in copies:
                g = OracleGraph(np.zeros((2, 0), dtype=np.int64), n, curv_type, und)
                g.adj, g.pred = [dict(a) for a in og.adj], og.pred and [dict(p) for p in og.pred]
                ops.append((g, random_edits(g, 3, rng)))
            assert edit_batch(copies, [e for _, e in ops]) == [len(e) for _, e in ops]
            for i in (0, 150, 299):
                check_state(copies[i], ops[i][0])
            assert _same_snapshot(_snapshot(dc), ref)
        finally:
            for c in copies:
                c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("tau", [INF, 3.0], ids=["greedy", "stochastic"])
def test_rewire_batch_equals_forked_rewire_and_the_oracle(mode, tau):
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(13)
    loops = 15
    bound = _bound(curv_type)
    for ei, n in graphs_for(curv_type, und)[:3]:
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=60 + loops) as dc:
            dc.edit(random_edits(og, 60, rng))
            U = np.random.RandomState(n).random_sample((3, loops))
            per_loops = [loops, 9, loops]
            for remove in (True, False):
                outs, logs = dc.rewire_batch(per_loops, remove, bound, tau, uniforms=U, return_log=True)
                for r in range(3):
                    (f,) = dc.fork()
                    with f:
                        want, wlog = f.rewire(per_loops[r], remove, bound, tau, uniforms=U[r], return_log=True)
                    assert np.array_equal(outs[r], want) and np.array_equal(logs[r], wlog)
                    oe, olog = _oracle_loop(og, per_loops[r], bound, tau, U[r], remove)
                    assert np.array_equal(outs[r], oe)
                    assert [tuple(int(v) for v in x) for x in logs[r]] == _oracle_log_tuples(olog)
                    assert remove or not np.any(logs[r][:, 6] >= 0)
                check_state(dc, og)                    # the parent is unchanged
                assert dc.remaining == 75 - int(dc._edit_adds)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_rewire_batch_on_a_fresh_object_equals_sdrf_batch(mode):
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import named_graph
    curv_type, und = mode
    ei, n = named_graph("wisconsin")
    if not und:
        ei = ei[:, ei[0] < ei[1]]
    loops = 40
    U = np.random.RandomState(3).random_sample((5, loops))
    taus = [INF, 2.0, 8.0, 0.5, 30.0]
    bound = 0.5 if curv_type in ("bfc", "bfc_paper") else 2.0
    want, wlog = sdrf.sdrf_batch(ei, n, loops, True, bound, taus, uniforms=U, return_log=True, is_undirected=und,
                                 curv_type=curv_type)
    with DynamicCurvature(ei, n, curv_type, und, capacity=loops) as dc:
        got, glog = dc.rewire_batch(loops, True, bound, taus, uniforms=U, return_log=True)
        assert dc.remaining == loops
    for a, b, la, lb in zip(got, want, glog, wlog):
        assert np.array_equal(a, b) and np.array_equal(la, lb)


@pytest.mark.gpu
def test_rewire_batch_host_path_for_every_draw():
    """guard = 1 hands every stochastic draw back to the host: the same runs as the on-device draws."""
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    ei, n = graphs_for("bfc", True)[1]
    og = OracleGraph(ei, n, "bfc", True)
    U = np.random.RandomState(8).random_sample((3, 12))
    with DynamicCurvature(ei, n, capacity=80) as dc:
        dc.edit(random_edits(og, 40, np.random.default_rng(4)))
        calls = []
        choice = sdrf.host_choice

        def counted(*a):
            calls.append(1)
            return choice(*a)

        with mock.patch.object(sdrf, "host_choice", counted):
            host, hlog = dc.rewire_batch(12, True, 0.2, 3.0, uniforms=U, guard=1.0, return_log=True)
            host_draws = len(calls)
            dev, dlog = dc.rewire_batch(12, True, 0.2, 3.0, uniforms=U, return_log=True)
        # with guard = 1 every iteration that draws (has candidates) stops with NEED_HOST and is decided on the host;
        # the default guard hands back (almost) none
        assert host_draws == sum(int(np.count_nonzero(lg[:, 2] > 0)) for lg in hlog) > 0
        assert len(calls) - host_draws < host_draws
    for r in range(3):
        want, wlog = oracle_loop_from(og, 12, 0.2, 3.0, U[r])
        assert np.array_equal(host[r], want) and np.array_equal(dev[r], want)
        assert np.array_equal(hlog[r], dlog[r])


@pytest.mark.gpu
def test_rewire_batch_failing_run_fails_alone():
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import named_graph
    ei, n = named_graph("texas")
    U = np.full((3, 5), 0.5)
    taus = [2.0, 1e6, 2.0]                       # exp(a * 1e6) overflows: run 1 raises what sdrf() raises
    with DynamicCurvature(ei, n, capacity=10) as dc:
        ref = _snapshot(dc)
        outs, logs = dc.rewire_batch(5, True, 0.5, taus, uniforms=U, return_log=True, return_exceptions=True)
        assert isinstance(outs[1], ValueError) and ("NaN" in str(outs[1]) or "sum to 1" in str(outs[1]))
        (f,) = dc.fork()
        with f:
            want = f.rewire(5, True, 0.5, 2.0, uniforms=U[0])
        assert np.array_equal(outs[0], want) and np.array_equal(outs[2], want)
        with pytest.raises(ValueError, match="sum to 1|NaN"):
            dc.rewire_batch(5, True, 0.5, taus, uniforms=U)
        assert _same_snapshot(_snapshot(dc), ref) and dc.remaining == 10


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_edit_batch_equals_sequential_edits(mode):
    """Different edit lists on forks in one launch equal the same lists applied by ``edit`` on other forks, including
    the stops: a bad edit, a remove of a non-edge and the budget, each with the same index and exception."""
    from dcr import lib as L
    from dcr.dynamic import DynamicCurvature, edit_batch
    curv_type, und = mode
    rng = np.random.default_rng(5)
    ei, n = graphs_for(curv_type, und)[3]
    og = OracleGraph(ei, n, curv_type, und)
    with DynamicCurvature(ei, n, curv_type, und, capacity=120) as dc:
        dc.edit(random_edits(og, 30, rng))
        lists = []
        for count in (0, 1, 25, 100, 60, 60, 60):
            g = OracleGraph(np.zeros((2, 0), dtype=np.int64), n, curv_type, und)
            g.adj, g.pred = [dict(a) for a in og.adj], og.pred and [dict(p) for p in og.pred]
            lists.append(random_edits(g, count, rng))
        u = int(np.argmin([len(a) for a in og.adj]))
        absent = next(v for v in range(n) if v != u and not og.has(u, v))
        lists[4] = np.concatenate([lists[4][:20], [[1, u, u]], lists[4][20:]])                 # bad edit
        lists[5] = np.concatenate([lists[5][:20], [[0, u, absent]], lists[5][20:]])            # non-edge
        room = [(1, u, v) for v in range(n) if v != u and not og.has(u, v)]
        lists[6] = np.array((room * 10)[: dc.remaining + 3], dtype=np.int64)                    # over the budget
        batch, seq = dc.fork(len(lists)), dc.fork(len(lists))
        try:
            got = edit_batch(batch, lists, return_exceptions=True)
            for b, (x, y, ops) in enumerate(zip(batch, seq, lists)):
                try:
                    want = y.edit(ops)
                except Exception as e:          # noqa: BLE001  the exception is the result here
                    want = e
                if isinstance(want, Exception):
                    assert type(got[b]) is type(want) and str(got[b]) == str(want)
                else:
                    assert got[b] == want == len(ops)
                assert x.remaining == y.remaining
                assert _same_snapshot(_snapshot(x), _snapshot(y))
            assert [isinstance(g, Exception) for g in got] == [False] * 4 + [True] * 3
            assert type(got[4]) is ValueError and type(got[6]) is L.DcrError
            assert type(got[5]).__name__ in ("NetworkXError", "KeyError")
            assert batch[6].remaining == 0
            with pytest.raises(ValueError, match=f"edit \\({u}, {u}\\)"):     # the lowest-index failure is raised
                edit_batch([batch[4], batch[6]], [[[1, u, u]], [[1, u, absent]]])
            with pytest.raises(L.DcrError, match="budget"):
                edit_batch([batch[6], batch[4]], [[[1, u, absent]], [[1, u, u]]])
        finally:
            for c in batch + seq:
                c.close()


@pytest.mark.gpu
def test_edit_batch_rejects_mixed_modes_and_repeats_at_the_c_entry_point():
    from dcr import lib as L
    from dcr.dynamic import DynamicCurvature, edit_batch
    from dcr.sdrf import edit_batch_states
    ei, n = graphs_for("bfc", True)[0]
    with DynamicCurvature(ei, n, capacity=4) as a, DynamicCurvature(ei, n, capacity=4) as b, \
            DynamicCurvature(ei, n, "augmented", capacity=4) as c:
        one = np.zeros((0, 3), dtype=np.int64)
        with pytest.raises(L.DcrError, match="one mode per call"):
            edit_batch_states([a._state, c._state], [one, one])
        with pytest.raises(L.DcrError, match="twice"):
            edit_batch_states([a._state, b._state, a._state], [one] * 3)
        with pytest.raises(ValueError, match="modes"):
            edit_batch([a, c], [one, one])
        with pytest.raises(ValueError, match="twice"):
            edit_batch([a, a], [one, one])
        assert a.remaining == b.remaining == c.remaining == 4
        assert edit_batch([a, b], [one, one]) == [0, 0]


def _host_edge_index(state, directed):
    from dcr import graph as G
    rp, od = state.export()
    return (G.from_digraph_order if directed else G.from_networkx_order)(rp, od)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_device_export_equals_the_host_conversion(mode):
    import torch
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(9)
    for ei, n in graphs_for(curv_type, und):
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=400) as dc:
            for _ in range(2):
                got = dc._state.edge_index()
                assert got.is_cuda and got.dtype == torch.int64
                got = got.cpu().numpy()
                assert np.array_equal(got, _host_edge_index(dc._state, not und))
                assert np.array_equal(got, og.edge_index())
                dc.edit(random_edits(og, 150, rng))


@pytest.mark.gpu
def test_device_export_edge_cases():
    import torch
    from dcr import lib as L
    from dcr.dynamic import DynamicCurvature
    # the classical loop removes the loop edge (0, 0): the state then has one column fewer than it had self entries
    e = [(0, i) for i in range(1, 7)] + [(0, 0), (7, 8), (8, 9), (1, 7)]
    ei = np.array(e).T
    ei = np.concatenate([ei, ei[::-1]], axis=1)
    with DynamicCurvature(ei, 10, "haantjes", capacity=1) as dc:
        _, log = dc.rewire(1, True, 1.0, INF, uniforms=np.zeros(1), return_log=True)
        assert (log[0, 6], log[0, 7]) == (0, 0)
        got = dc.edge_index()
        assert got.shape[1] == dc._state.nnz() and not np.any(got[0] == got[1])
        assert np.array_equal(got, _host_edge_index(dc._state, False))
    # an empty graph, and a single node with and without its self-loop
    for curv_type, und in MODES[:5]:
        with DynamicCurvature(np.zeros((2, 0), dtype=np.int64), 5, curv_type, und, capacity=2) as dc:
            assert dc.edge_index().shape == (2, 0)
            dc.add_edges([(3, 1)])
            assert np.array_equal(dc.edge_index(), _host_edge_index(dc._state, not und))
        with DynamicCurvature(np.array([[0], [0]]), 1, curv_type, und, capacity=0) as dc:
            assert dc.edge_index().tolist() == [[0], [0]]
        with DynamicCurvature(np.zeros((2, 0), dtype=np.int64), 1, curv_type, und, capacity=0) as dc:
            assert dc.edge_index().shape == (2, 0)
    # a capacity that is too short: nothing at or beyond it is written, everything before it is the full export's
    ei, n = graphs_for("bfc", True)[1]
    with DynamicCurvature(ei, n, capacity=0) as dc:
        full = dc.edge_index()
        st = dc._state
        m = full.shape[1]
        for cap in (0, 1, m - 3):
            rowptr = torch.empty(n + 1, dtype=torch.int32, device=st.device)
            out = torch.full((2, m + 8), -7, dtype=torch.int64, device=st.device)
            L.check(st.lib.dcr_sdrf_export_edge_index(st.handle, rowptr.data_ptr(), out[0].data_ptr(),
                                                      out[1].data_ptr(), cap, L.current_stream()))
            o = out.cpu().numpy()
            assert int(rowptr[-1]) == m
            assert np.array_equal(o[:, :cap], full[:, :cap]) and np.all(o[:, cap:] == -7)
