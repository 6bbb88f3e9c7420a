"""Caller edits on the device-resident SDRF state (``dcr_sdrf_edit``, ``dcr.dynamic.DynamicCurvature``, DESIGN §4.10).

An edit is the networkx operation on the loop's ``G``: ``add_edge`` appends to both rows (a present edge keeps its
position), ``remove_edge`` deletes in place.  The CPU tests pin those semantics on the oracle's adjacency dicts against
networkx itself, the alignment of sorted-order values to ``edge_index()`` columns and the argument checks.  The GPU
tests compare, in every loop mode, the edited state with the same edits made on the oracle's dicts: insertion order,
``edge_index()``, curvature bit for bit against a fresh full pass, SDRF resumed from the edited graph, the replay of
an SDRF log, and the stops before a failing edit."""
import copy
from unittest import mock

import numpy as np
import pytest

from helpers import gnp

INF = float("inf")
# (curv_type, is_undirected) of every loop mode
MODES = [("bfc", True), ("bfc", False), ("1d", True), ("augmented", True), ("haantjes", True), ("bfc_paper", True)]
MODE_IDS = ["bfc", "bfc_directed", "1d", "augmented", "haantjes", "bfc_paper"]


# ---------------------------------------------------------------------------------------------------------------------
# the oracle side: the loop's G as adjacency dicts, and the same edits on it
# ---------------------------------------------------------------------------------------------------------------------
class OracleGraph:
    """The graph each loop mode starts from (``oracle.sdrf`` / ``oracle.sdrf_classical`` set-up), edited the networkx
    way.  ``adj`` are the neighbour (directed: successor) dicts, ``pred`` the predecessor dicts of the directed mode."""

    def __init__(self, ei, n, curv_type, is_undirected):
        from oracle.sdrf import networkx_adjacency, networkx_digraph
        from oracle.sdrf_classical import networkx_adjacency_classical
        self.n, self.curv_type, self.directed = n, curv_type, not is_undirected
        self.pred = None
        if self.directed:
            self.adj, self.pred = networkx_digraph(ei, n)
        elif curv_type == "bfc":
            self.adj = networkx_adjacency(ei, n)
        else:
            self.adj = networkx_adjacency_classical(ei, n)

    def has(self, u, v):
        return v in self.adj[u]

    def apply(self, op, u, v):
        if op == 1:
            self.adj[u][v] = None                  # dict assignment: a present key keeps its position
            (self.pred[v] if self.directed else self.adj[v])[u] = None
        else:
            del self.adj[u][v]
            del (self.pred[v] if self.directed else self.adj[v])[u]

    def rows(self):
        rowptr = np.zeros(self.n + 1, dtype=np.int64)
        rowptr[1:] = np.cumsum([len(a) for a in self.adj])
        order = np.array([v for a in self.adj for v in a], dtype=np.int64)
        return rowptr, order

    def edge_index(self):
        from oracle.sdrf import edge_index_from_adjacency, edge_index_from_digraph
        return edge_index_from_digraph(self.adj) if self.directed else edge_index_from_adjacency(self.adj)


def random_edits(og: OracleGraph, count, rng, hub_share=0.25):
    """``count`` valid mixed edits made on ``og`` as they are drawn: adds of non-edges, re-adds of removed edges,
    no-op adds of present edges and removes, a share of them at the highest-degree node."""
    n = og.n
    hub = int(np.argmax([len(a) for a in og.adj]))
    removed, out = [], []
    for _ in range(count):
        kind = rng.random()
        u = hub if rng.random() < hub_share else int(rng.integers(n))
        if kind < 0.15 and removed:                                    # re-add a removed edge
            u, v = removed.pop(int(rng.integers(len(removed))))
            op = 1
        elif kind < 0.25:                                              # no-op add of a present edge
            nb = [w for w in og.adj[u] if w != u]
            if not nb:
                continue
            op, v = 1, nb[int(rng.integers(len(nb)))]
        elif kind < 0.6:                                               # remove
            nb = [w for w in og.adj[u] if w != u]
            if not nb:
                continue
            op, v = 0, nb[int(rng.integers(len(nb)))]
            removed.append((u, v))
        else:                                                          # add
            v = int(rng.integers(n))
            if v == u:
                continue
            op = 1
        og.apply(op, u, v)
        out.append((op, u, v))
    return np.array(out, dtype=np.int64).reshape(-1, 3)


def _with_self_loops(ei, n, k, seed):
    rng = np.random.default_rng(seed)
    who = rng.choice(n, size=min(k, n), replace=False)
    out = np.concatenate([ei, np.stack([who, who])], axis=1)
    return out[:, rng.permutation(out.shape[1])]


def _random_digraph(n, m, seed):
    rng = np.random.default_rng(seed)
    ei = rng.integers(0, n, size=(2, m))
    ei = np.unique(ei[:, ei[0] != ei[1]], axis=1)
    return ei[:, rng.permutation(ei.shape[1])]


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_dict_edits_follow_networkx():
    """Append on add, in-place delete, a re-add goes to the end, an add of a present edge keeps its position."""
    nx = pytest.importorskip("networkx")
    rng = np.random.default_rng(3)
    for directed in (False, True):
        n = 12
        og = OracleGraph(np.zeros((2, 0), dtype=np.int64), n, "bfc", not directed)
        g = (nx.DiGraph if directed else nx.Graph)()
        g.add_nodes_from(range(n))
        for u, v in zip(rng.integers(0, n, 40).tolist(), rng.integers(0, n, 40).tolist()):
            if u != v:
                og.apply(1, u, v)
                g.add_edge(u, v)
        edits = random_edits(og, 200, rng)
        assert {0, 1} <= set(edits[:, 0].tolist())
        for op, u, v in edits.tolist():
            (g.add_edge if op else g.remove_edge)(u, v)
        assert [list(g.adj[u]) for u in range(n)] == [list(a) for a in og.adj]
        if directed:
            assert [list(g.pred[u]) for u in range(n)] == [list(p) for p in og.pred]


def test_align_to_columns():
    from dcr import graph as G
    from dcr.dynamic import align_to_columns, classical_loop_values
    from oracle.sdrf_classical import curvature_edge, networkx_adjacency_classical
    rng = np.random.default_rng(1)
    n = 30
    ei = _with_self_loops(gnp(n, 0.2, 8), n, 4, 2)
    rowptr_o, order = G.networkx_order(ei, n, keep_self_loops=True)
    cols = G.from_networkx_order(rowptr_o, order)
    keep = ei[0] != ei[1]
    rowptr, col = G.undirected_csr(ei[:, keep], n)
    vals = rng.standard_normal(col.size).astype(np.float32)
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    want = {(int(a), int(b)): v for a, b, v in zip(rows, col, vals)}
    got = align_to_columns(rowptr, col, vals, cols)
    assert got.dtype == np.float32
    for (a, b), v in zip(cols.T.tolist(), got):
        assert v == (0 if a == b else want[(a, b)])
    adj = networkx_adjacency_classical(ei, n)
    deg = np.array([len([w for w in adj[u] if w != u]) for u in range(n)])
    for ct in ("1d", "augmented", "haantjes"):
        lv = classical_loop_values(deg, ct)
        for u in range(n):
            if u in adj[u]:
                assert lv[u] == curvature_edge(adj, (u, u), ct)
    with pytest.raises(ValueError, match="not an entry"):
        absent = next((a, b) for a in range(n) for b in range(n) if a != b and (a, b) not in want)
        align_to_columns(rowptr, col, vals, np.array(absent).reshape(2, 1))


def test_edit_argument_checks():
    import torch
    from dcr import lib as L
    from dcr.dynamic import edit_array, pair_array
    from dcr.sdrf import _raise_for_status
    assert edit_array([]).shape == (0, 3)
    assert edit_array(torch.tensor([[1, 2, 3]])).tolist() == [[1, 2, 3]]
    assert edit_array([[1, -4, 2**40]]).tolist() == [[1, -4, 2**40]]    # ids are checked on the device, in order
    for bad in ([1, 2, 3], [[1, 2]], np.zeros((2, 3, 1), dtype=np.int64)):
        with pytest.raises(ValueError, match=r"\[m, 3\]"):
            edit_array(bad)
    with pytest.raises(ValueError, match="op must be"):
        edit_array([[1, 0, 1], [2, 0, 1]])
    with pytest.raises(ValueError, match="integer"):
        edit_array(np.array([[1.0, 0, 1]]))
    with pytest.raises(ValueError, match=r"\[m, 2\]"):
        pair_array([[0, 1, 2]])
    with pytest.raises(ValueError, match="self-loop or a node id"):
        _raise_for_status(L.SDRF_BAD_EDIT, (3, 3))
    with pytest.raises(Exception, match="The edge 4-7 is not in the graph"):
        _raise_for_status(L.SDRF_REMOVE_NONEDGE, (4, 7))


def test_edit_tensor_checks_the_int32_range():
    import torch
    from dcr.sdrf import edit_tensor
    assert edit_tensor(np.array([[1, 2, 3]], dtype=np.int64)).dtype == torch.int32
    assert edit_tensor([]).shape == (0, 3)
    assert edit_tensor([[0, -2**31, 2**31 - 1]]).tolist() == [[0, -2**31, 2**31 - 1]]
    for bad in ([[1, 0, 2**31]], [[1, -2**31 - 1, 0]], np.array([[1, 0, 2**32 + 5]])):
        with pytest.raises(ValueError, match="fit int32"):           # the int32 cast would wrap 2**32 + 5 to 5
            edit_tensor(bad)
    with pytest.raises(ValueError, match="integer"):
        edit_tensor(np.array([[1.0, 0, 1]]))
    with pytest.raises(ValueError, match=r"\[m, 3\]"):
        edit_tensor([1, 2, 3])


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def fresh_curvature(ei, n, curv_type, directed, og=None):
    """A fresh full pass on the graph ``ei`` (columns of ``edge_index()``), one value per column."""
    import torch
    from dcr import bfc
    from dcr import graph as G
    u, v = ei
    loop = u == v
    if curv_type in ("1d", "augmented", "haantjes"):
        from oracle.sdrf_classical import curvature_edge
        return np.array([curvature_edge(og.adj, (a, b), curv_type) for a, b in ei.T.tolist()], dtype=np.int64)
    e = ei[:, ~loop]
    if directed:
        d = bfc.DirectedCSR.from_edge_index(e, n)
        c = bfc.cuda_flavour_directed(d, want_fields=False)["c32"].cpu().numpy()
        rowptr, col = d.out.rowptr.cpu().numpy(), d.out.colidx.cpu().numpy()
    else:
        rowptr, col = G.undirected_csr(e, n)
        csr = bfc.DeviceCSR.from_host(rowptr, col)
        if curv_type == "bfc":
            c = bfc.cuda_flavour(csr, want_fields=False, tri=bfc.support(csr))["c32"].cpu().numpy()
        else:
            rows = np.repeat(np.arange(n), np.diff(rowptr))
            up = rows < col
            p = bfc.paper_flavour(csr, edges=(torch.from_numpy(rows[up].astype(np.int32)).cuda(),
                                              torch.from_numpy(col[up].astype(np.int32)).cuda()))
            vals = p["bfc"].cpu().numpy()
            both = {}
            for a, b, x in zip(rows[up].tolist(), col[up].tolist(), vals):
                both[(a, b)] = both[(b, a)] = x
            return np.array([both[(a, b)] for a, b in ei.T.tolist()], dtype=np.float64)
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    at = {(a, b): x for a, b, x in zip(rows.tolist(), col.tolist(), c)}
    return np.array([0.0 if a == b else at[(a, b)] for a, b in ei.T.tolist()], dtype=np.float32)


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    return np.array_equal(a.view(np.int64 if a.itemsize == 8 else np.int32).ravel() if a.dtype.kind == "f" else a,
                          b.view(np.int64 if b.itemsize == 8 else np.int32).ravel() if b.dtype.kind == "f" else b)


def check_state(dc, og, ei_start=None):
    """insertion order, edge_index() and curvature() of ``dc`` against the oracle graph ``og`` and a fresh pass"""
    rp, od = dc.insertion_order()
    wrp, wod = og.rows()
    assert np.array_equal(rp, wrp) and np.array_equal(od, wod)
    ei = dc.edge_index()
    assert ei.dtype == np.int64 and np.array_equal(ei, og.edge_index())
    got = dc.curvature()
    want = fresh_curvature(ei, og.n, dc.curv_type, dc.directed, og)
    assert same_bits(got, want)


def graphs_for(curv_type, is_undirected):
    from dcr.synth import named_graph
    out = []
    for s in range(2):
        n = 30 + 17 * s
        if not is_undirected:
            ei = _random_digraph(n, 5 * n, 40 + s)
        else:
            ei = gnp(n, 0.15, 40 + s)
        if curv_type != "bfc_paper" and s == 1:
            ei = _with_self_loops(ei, n, 5, s)
        out.append((ei, n))
    for name in ("cornell", "wisconsin"):
        ei, n = named_graph(name)
        if not is_undirected:      # a directed view of the shape: one direction of each pair, shuffled
            ei = ei[:, ei[0] < ei[1]]
            ei = ei[:, np.random.default_rng(n).permutation(ei.shape[1])]
        if curv_type != "bfc_paper" and name == "cornell":   # (directed: the node lists itself as successor and
            ei = _with_self_loops(ei, n, 6, 3)                 #  as predecessor)
        out.append((ei, n))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_edits_values_and_order_are_exact(mode):
    """1 … 300 random mixed edits; after each batch the state equals the oracle dicts and a fresh full pass."""
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(7)
    looped = 0
    for gi, (ei, n) in enumerate(graphs_for(curv_type, und)):
        og = OracleGraph(ei, n, curv_type, und)
        looped += sum(u in og.adj[u] for u in range(n))
        with DynamicCurvature(ei, n, curv_type, und, capacity=600) as dc:
            check_state(dc, og)
            for count in (1, 7, 40, 300):
                edits = random_edits(og, count, rng, hub_share=0.4 if gi else 0.2)
                assert dc.edit(edits) == len(edits)
                check_state(dc, og)
            # add_edges / remove_edges: the same operations
            u = int(np.argmax([len(a) for a in og.adj]))
            nb = [w for w in og.adj[u] if w != u][:3]
            dc.remove_edges([(u, w) for w in nb])
            for w in nb:
                og.apply(0, u, w)
            dc.add_edges([(w, u) for w in nb[::-1]])
            for w in nb[::-1]:
                og.apply(1, w, u)
            check_state(dc, og)
    assert looped > 0 if curv_type != "bfc_paper" else looped == 0     # self-loops wherever the mode keeps them


def _oracle_log_tuples(log):
    return [(r["x"], r["y"], r["n_candidates"], r["k"], r["l"], r["choice"],
             -1 if r["removed"] is None else r["removed"][0], -1 if r["removed"] is None else r["removed"][1])
            for r in log]


def oracle_loop_from(og, loops, bound, tau, uniforms):
    """The oracle loop of ``og``'s mode started from ``og``'s dicts (its set-up from an edge_index replaced by them)."""
    import oracle.sdrf as osd
    import oracle.sdrf_classical as oc
    ei = og.edge_index()
    adj, pred = copy.deepcopy(og.adj), copy.deepcopy(og.pred)
    if og.curv_type == "bfc":
        target = ("networkx_digraph", lambda e, n: (adj, pred)) if og.directed else \
            ("networkx_adjacency", lambda e, n: adj)
        with mock.patch.object(osd, target[0], target[1]):
            return osd.sdrf_oracle(ei, og.n, loops, True, bound, tau, uniforms, is_undirected=not og.directed)
    patches = [mock.patch.object(oc, "networkx_adjacency_classical", lambda e, n: adj)]
    if og.curv_type == "bfc_paper":
        from oracle.paper_flavour import bfc_edge_fields

        class KeySets:
            def __init__(self, a):
                self.a = a

            def __getitem__(self, v):
                return self.a[v].keys()

        patches.append(mock.patch.object(oc, "curvature_edge", lambda a, e, ct: bfc_edge_fields(KeySets(a), *e)[6]))
    with patches[0]:
        if len(patches) == 1:
            return oc.sdrf_classical_oracle(ei, og.n, og.curv_type, loops, True, bound, tau, uniforms)
        with patches[1]:
            return oc.sdrf_classical_oracle(ei, og.n, og.curv_type, loops, True, bound, tau, uniforms)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("tau", [INF, 3.0], ids=["greedy", "stochastic"])
def test_rewire_resumes_exactly_from_the_edited_graph(mode, tau):
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(11)
    loops = 15
    bound = 0.2 if curv_type in ("bfc", "bfc_paper") else 2.0
    for ei, n in graphs_for(curv_type, und)[:3]:
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=60 + loops) as dc:
            edits = random_edits(og, 60, rng)
            dc.edit(edits)
            # a fresh state from the edited state's insertion-order rows (the directed mode's predecessor rows from
            # the oracle, which the successor side above was checked against)
            rp, od = dc.insertion_order()
            extra = ()
            if not und:
                prp = np.zeros(n + 1, dtype=np.int64)
                prp[1:] = np.cumsum([len(p) for p in og.pred])
                extra = (prp, np.array([v for p in og.pred for v in p], dtype=np.int64))
            fresh = sdrf.SdrfState(rp, od, loops, dc.mode, *extra)
            uni = np.random.RandomState(5).random_sample(loops)
            got, glog = dc.rewire(loops, True, bound, tau, uniforms=uni, return_log=True)
            try:
                flog = sdrf._run_state(fresh, loops, True, bound, tau, uni, 1e-9)
                frp, fod = fresh.export()
            finally:
                fresh.close()
            want, wlog = oracle_loop_from(og, loops, bound, tau, uni)
            assert [tuple(int(v) for v in r) for r in glog] == _oracle_log_tuples(wlog)
            assert np.array_equal(got, want)
            assert np.array_equal(glog, flog)
            assert np.array_equal((sdrf.G.from_digraph_order if not und else sdrf.G.from_networkx_order)(frp, fod), got)
            assert dc.remaining == 60 + loops - int(np.count_nonzero(edits[:, 0] == 1)) - int(np.count_nonzero(glog[:, 3] >= 0))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_replaying_an_sdrf_log_gives_the_sdrf_state(mode):
    """The adds (k, l) and removes (xr, yr) of an SDRF run, replayed as edits on a fresh state of the same input, give
    the run's final graph and bit-identical curvature (runs whose log removes a self-loop are left out)."""
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import SDRF_PARAMS
    curv_type, und = mode
    replayed = 0
    for gi, (ei, n) in enumerate(graphs_for(curv_type, und)):
        loops, tau, bound = SDRF_PARAMS["cornell"] if gi >= 2 else (40, 4.0, 0.3)
        if curv_type in ("1d", "augmented", "haantjes"):
            bound = 1.0
        keep = []
        _, log = sdrf.sdrf(ei, n, loops, True, bound, tau, uniforms=np.random.RandomState(gi).random_sample(loops),
                           return_log=True, state_out=keep, is_undirected=und, curv_type=curv_type)
        st = keep[0]
        try:
            if np.any((log[:, 6] >= 0) & (log[:, 6] == log[:, 7])):
                continue
            ops = []
            for r in log.tolist():
                if r[3] >= 0:
                    ops.append((1, r[3], r[4]))
                if r[6] >= 0:
                    ops.append((0, r[6], r[7]))
            ops = np.array(ops, dtype=np.int64).reshape(-1, 3)
            with DynamicCurvature(ei, n, curv_type, und, capacity=int(np.count_nonzero(ops[:, 0] == 1))) as dc:
                dc.edit(ops)
                assert dc.remaining == 0
                for a, b in zip(dc._state.export(), st.export()):
                    assert np.array_equal(a, b)
                for a, b in zip(dc._state.export(with_curvature=True), st.export(with_curvature=True)):
                    assert (a is None and b is None) or same_bits(a, b)
            replayed += 1
        finally:
            st.close()
    assert replayed >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_failing_edits_stop_before_themselves(mode):
    import torch
    from dcr import lib as L
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(2)
    ei, n = graphs_for(curv_type, und)[1]
    og = OracleGraph(ei, n, curv_type, und)
    with DynamicCurvature(ei, n, curv_type, und, capacity=40) as dc:
        u = int(np.argmin([len(a) for a in og.adj]))          # room for many adds at u
        absent = next(v for v in range(n) if v != u and not og.has(u, v))
        for bad, exc in (((0, u, absent), Exception), ((1, u, u), ValueError), ((0, 3, 3), ValueError),
                         ((1, u, n), ValueError), ((0, -4, u), ValueError), ((1, u, 2**40), ValueError)):
            good = random_edits(og, 5, rng)
            tail = np.array([[1, u, (u + 1) % n]], dtype=np.int64)
            with pytest.raises(exc) as info:
                dc.edit(np.concatenate([good, [bad], tail]))
            if exc is ValueError:                   # the pair as the caller gave it
                assert f"({bad[1]}, {bad[2]})" in str(info.value)
            else:
                assert type(info.value).__name__ == "NetworkXError" and f"{u}-{absent}" in str(info.value)
            check_state(dc, og)                     # the five edits before it applied, nothing after it
        # the budget: the device stops before the first add beyond max_additions ...
        left = dc.remaining
        adds = np.array([[1, u, v] for v in range(n) if v != u and not og.has(u, v)][: left + 2], dtype=np.int64)
        assert adds.shape[0] == left + 2
        with pytest.raises(L.DcrError):
            dc.edit(adds)
        for op, a, b in adds[:left].tolist():
            og.apply(op, a, b)
        check_state(dc, og)
        assert dc.remaining == 0
        dc.edit(np.array([[0, u, int(adds[0, 2])]]))   # removes need no budget
        og.apply(0, u, int(adds[0, 2]))
        check_state(dc, og)
        with pytest.raises(ValueError, match="budget"):
            dc.rewire(1, True, 0.5, INF, uniforms=np.zeros(1))
        check_state(dc, og)
    # ... and so does the C entry point itself, reporting the offending pair
    with DynamicCurvature(ei, n, curv_type, und, capacity=2) as dc:
        st = dc._state
        og = OracleGraph(ei, n, curv_type, und)
        free = [v for v in range(n) if v != u and not og.has(u, v)][:3]
        res = st.edit(torch.tensor([[1, u, v] for v in free]))
        assert res["status"] == L.SDRF_ARENA_FULL and res["iterations_done"] == 2
        assert (res["pending_x"], res["pending_y"]) == (u, free[2])
        res = st.edit(np.zeros((0, 3), dtype=np.int64))
        assert res["status"] == L.SDRF_OK and res["iterations_done"] == 0
        for v in free[:2]:
            og.apply(1, u, v)
        check_state(dc, og)


@pytest.mark.gpu
def test_rewire_host_protocol_and_errors():
    """``rewire`` draws from numpy's global generator like ``sdrf()`` and raises what ``sdrf()`` raises."""
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import named_graph
    ei, n = named_graph("texas")
    np.random.seed(4)
    want = sdrf.sdrf(ei, n, 30, True, 1.64, 22)
    after_sdrf = np.random.random_sample()
    np.random.seed(4)
    with DynamicCurvature(ei, n, capacity=30) as dc:
        got = dc.rewire(30, True, 1.64, 22)
    assert np.array_equal(got, want) and np.random.random_sample() == after_sdrf
    with pytest.raises(Exception, match="not available"):
        DynamicCurvature(ei, n, curv_type="nope")
    with pytest.raises(NotImplementedError):
        DynamicCurvature(ei, n, curv_type="bfc_paper", is_undirected=False)
    with DynamicCurvature(ei, n, capacity=10) as dc:
        with pytest.raises(ValueError, match="sum to 1|NaN"):
            dc.rewire(5, True, 0.5, 1e6, uniforms=np.full(5, 0.5))
        dc.edit([[1, 0, 1]])                           # still usable afterwards
