"""SDRF with the paper-flavour Balanced Forman curvature (``curv_type='bfc_paper'``): ``sdrf_no_cuda``'s loop with
``bfc_naive.bfc_edge`` as the curvature, on the device loop's LOOP_PAPER flavour (DESIGN §4.9).

The CPU tests pin the two identities the device loop relies on against ``oracle.paper_flavour.bfc_edge_fields``: the
closed form of an interior candidate's improvement and the dirty-set rule of the incremental refresh.  The GPU tests run
the loop against ``paper_sdrf_oracle``: the classical oracle loop (``oracle.sdrf_classical``, run unchanged) with
``bfc_edge_fields`` as its curvature."""
from unittest import mock

import numpy as np
import pytest

from helpers import gnp, toy_graphs

INF = float("inf")


class _KeySets:
    """``adj[v]`` of the oracle's adjacency dicts as the set-like key view ``bfc_edge_fields`` operates on."""

    def __init__(self, adj):
        self.adj = adj

    def __getitem__(self, v):
        return self.adj[v].keys()


def paper_sdrf_oracle(ei, n, loops, remove_edges, bound, tau, uniforms):
    """``sdrf_no_cuda``'s loop (``oracle.sdrf_classical.sdrf_classical_oracle``) with ``bfc_naive.bfc_edge``
    (``bfc_edge_fields(...)[6]``: the int 0 where deg_min == 1, else a Python float) as ``compute_curvature_edge``."""
    import oracle.sdrf_classical as oc
    from oracle.paper_flavour import bfc_edge_fields

    def curvature_edge(adj, e, curv_type):
        return bfc_edge_fields(_KeySets(adj), *e)[6]

    with mock.patch.object(oc, "curvature_edge", curvature_edge):
        return oc.sdrf_classical_oracle(ei, n, "bfc_paper", loops, remove_edges, bound, tau, uniforms)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the identities behind the scoring and the refresh
# ---------------------------------------------------------------------------------------------------------------------
def _adj_sets(ei, n):
    from oracle.paper_flavour import adjacency_sets
    return adjacency_sets(ei, n)


def _value(d1, d2, tri, sq1, sq2, gamma):
    """bfc_naive.py:31-32 / :39-40 from the fields, as ``bfc_edge_fields`` evaluates them."""
    if min(d1, d2) == 1:
        return 0
    dmax, dmin = max(d1, d2), min(d1, d2)
    v = 2 / d1 + 2 / d2 - 2 + 2 * tri / dmax + tri / dmin
    if sq1 and sq2:
        v = v + 1 / gamma / dmax * (sq1 + sq2)
    return v


def _c(adj, a, b, k):
    """c(k) = |N(k) ∩ (N(b) \\ N(a) \\ {a})| for k in M_a = N(a) \\ N(b) \\ {b}, else None."""
    if k == b or k in adj[b]:
        return None
    return len(adj[k] & (adj[b] - adj[a] - {a}))


def _random_graphs(count, seed):
    rng = np.random.default_rng(seed)
    for g in range(count):
        n = int(rng.integers(6, 24))
        yield gnp(n, float(rng.uniform(0.12, 0.45)), 1000 * seed + g), n


def test_closed_form_of_interior_cells_matches_bfc_edge():
    from oracle.paper_flavour import bfc_edge_fields
    checked = zero = 0
    for ei, n in _random_graphs(120, 1):
        adj = _adj_sets(ei, n)
        edges = [(int(a), int(b)) for a, b in ei.T if a < b]
        for x, y in edges[:: max(1, len(edges) // 6)]:
            before = bfc_edge_fields(adj, x, y)[6]
            cx = {k: _c(adj, x, y, k) for k in adj[x]}
            cy = {k: _c(adj, y, x, k) for k in adj[y]}
            tri = len(adj[x] & adj[y])
            sq_x = sum(1 for v in cx.values() if v)
            sq_y = sum(1 for v in cy.values() if v)
            gam = max([v for v in list(cx.values()) + list(cy.values()) if v is not None] + [0])
            for i in adj[x]:
                for j in adj[y]:
                    if i == j or j in adj[i]:
                        continue
                    adj[i].add(j)
                    adj[j].add(i)
                    after = bfc_edge_fields(adj, x, y)[6]
                    adj[i].discard(j)
                    adj[j].discard(i)
                    if cx[i] is None or cy[j] is None:          # a common neighbour (or y / x): nothing bfc reads moves
                        assert after - before == 0
                        zero += 1
                        continue
                    want = _value(len(adj[x]), len(adj[y]), tri, sq_x + (cx[i] == 0), sq_y + (cy[j] == 0),
                                  max(gam, cx[i] + 1, cy[j] + 1))
                    assert float(after) == float(want)
                    checked += 1
    assert checked > 1000 and zero > 100


def test_dirty_set_rule_covers_every_changed_edge():
    from oracle.paper_flavour import bfc_edge_fields
    rng = np.random.default_rng(3)
    toggles = 0
    for ei, n in _random_graphs(80, 2):
        adj = _adj_sets(ei, n)
        for _ in range(5):
            k, l = (int(v) for v in rng.choice(n, 2, replace=False))
            present = l in adj[k]
            if not present:
                adj[k].add(l)
                adj[l].add(k)
            edges = [(a, b) for a in range(n) for b in adj[a] if a < b]
            # the rule on the graph WITH the edge {k,l}: edges at k or l, edges between N(k) and N(l)
            dirty = {e for e in edges if k in e or l in e}
            dirty |= {(min(a, b), max(a, b)) for a in adj[k] for b in adj[a] if b in adj[l]}
            with_edge = {e: bfc_edge_fields(adj, *e)[6] for e in edges}
            adj[k].discard(l)
            adj[l].discard(k)
            without = {e: bfc_edge_fields(adj, *e)[6] for e in edges if e != (min(k, l), max(k, l))}
            for e, v in without.items():
                if float(v) != float(with_edge[e]):
                    assert e in dirty, (e, k, l)
            if present:
                adj[k].add(l)
                adj[l].add(k)
            toggles += 1
    assert toggles == 400


def test_oracle_loop_on_toy_graphs():
    from oracle.paper_flavour import bfc_edge_fields
    for name, (ei, n) in toy_graphs().items():
        out, log = paper_sdrf_oracle(ei, n, 5, True, 0.5, 2, np.random.RandomState(4).random_sample(5))
        assert log and out.shape[0] == 2, name
        adj = _adj_sets(ei, n)
        x, y = log[0]["x"], log[0]["y"]
        first = min(((a, b) for a in range(n) for b in sorted(adj[a]) if a < b),
                    key=lambda e: bfc_edge_fields(adj, *e)[6])
        assert bfc_edge_fields(adj, x, y)[6] == bfc_edge_fields(adj, *first)[6], name
    # SURVEY App. G: the paper flavour of the Petersen graph is -2/3 on every edge; of the cube 2/3
    ei, n = toy_graphs()["petersen"]
    assert bfc_edge_fields(_adj_sets(ei, n), 0, 1)[6] == pytest.approx(-2 / 3)
    _, log = paper_sdrf_oracle(ei, n, 1, False, 0.5, INF, np.zeros(1))
    assert (log[0]["x"], log[0]["y"]) == (0, 1)


def test_loop_mode_and_errors():
    from dcr import lib as L
    from dcr import sdrf
    mode, order = sdrf._loop_mode("bfc_paper", True)
    assert mode == L.SDRF_MODE_BFC_PAPER == 5
    ei, n = toy_graphs()["c5"]
    rp, od = order(ei, n)
    rp2, od2 = sdrf._loop_mode("haantjes", True)[1](ei, n)
    assert np.array_equal(rp, rp2) and np.array_equal(od, od2)          # the classical loop's order
    with pytest.raises(NotImplementedError):
        order(np.concatenate([ei, [[2], [2]]], axis=1), n)
    with pytest.raises(NotImplementedError):
        sdrf._loop_mode("bfc_paper", False)
    with pytest.raises(Exception, match="Method ollivier not available."):
        sdrf._loop_mode("ollivier", True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_log_tuples(log):
    return [(r["x"], r["y"], r["n_candidates"], r["k"], r["l"], r["choice"],
             -1 if r["removed"] is None else r["removed"][0], -1 if r["removed"] is None else r["removed"][1])
            for r in log]


def _run_both(ei, n, loops, bound, tau, seed, remove_edges=True, guard=1e-9):
    from dcr import sdrf
    uni = np.random.RandomState(seed).random_sample(loops)
    got, glog = sdrf.sdrf(ei, n, loops, remove_edges, bound, tau, uniforms=uni, return_log=True, curv_type="bfc_paper",
                          guard=guard)
    want, wlog = paper_sdrf_oracle(ei, n, loops, remove_edges, bound, tau, uni)
    assert [tuple(int(v) for v in r) for r in glog] == _oracle_log_tuples(wlog)
    assert np.array_equal(got, want)
    return glog


@pytest.mark.gpu
@pytest.mark.parametrize("tau", [INF, 2])
def test_paper_toy_and_random_graphs_match_oracle(tau):
    for name, (ei, n) in toy_graphs().items():          # symmetric graphs: every min / max is a tie
        _run_both(ei, n, 6, 0.5, tau, 3)
        _run_both(ei, n, 6, 0.5, tau, 3, remove_edges=False)
    for seed in range(4):
        n = 16 + 7 * seed
        _run_both(gnp(n, 0.25, 900 + seed), n, 20, -0.2 + 0.3 * seed, tau, 40 + seed)


@pytest.mark.gpu
def test_paper_webkb_shapes_full_length_and_exits():
    from dcr.synth import SDRF_PARAMS, named_graph
    for name in ("cornell", "texas", "wisconsin"):
        ei, n = named_graph(name)
        loops, tau, bound = SDRF_PARAMS[name]
        _run_both(ei, n, loops, bound, tau, 5)
        _run_both(ei, n, loops, bound, INF, 6)
    ei, n = named_graph("cornell")
    _run_both(ei, n, 40, 0.5, 3, 7, remove_edges=False)
    ei, n = toy_graphs()["k5"]                          # complete graph: no candidates -> both exits
    log = _run_both(ei, n, 5, 100.0, INF, 1)
    assert len(log) == 1
    log = _run_both(ei, n, 5, 100.0, INF, 1, remove_edges=False)
    assert len(log) == 1
    _run_both(ei, n, 5, -5.0, INF, 1)                   # removal only, until the graph has candidates again


@pytest.mark.gpu
def test_paper_cora_shape_prefix():
    from dcr.synth import named_graph
    ei, n = named_graph("cora")
    _run_both(ei, n, 100, 0.95, 163, 12)


@pytest.mark.gpu
def test_paper_improvements_bit_for_bit_through_the_host():
    """guard = 1.0: every finite-tau draw is handed to the host with the improvements of its iteration."""
    import torch
    from dcr import lib as L
    from dcr import sdrf
    from dcr.synth import named_graph
    cases = [(named_graph("texas"), 30, 1.64, 22), ((gnp(30, 0.2, 77), 30), 25, 0.3, 2)]
    for (ei, n), loops, bound, tau in cases:
        uni = np.random.RandomState(9).random_sample(loops)
        _, wlog = paper_sdrf_oracle(ei, n, loops, True, bound, tau, uni)
        mode, order = sdrf._loop_mode("bfc_paper", True)
        state = sdrf._new_state(mode, order(ei, n), loops)
        u_dev = torch.from_numpy(uni).to(state.device)
        done = draws = 0
        forced = -1
        hosted = 0
        try:
            while done < loops:
                res, _ = state.run(loops - done, True, bound, tau, u_dev[draws:], forced_choice=forced, guard=1.0)
                forced = -1
                done += res["iterations_done"]
                draws += res["draws_used"]
                if res["status"] == L.SDRF_OK:
                    break
                assert res["status"] == L.SDRF_NEED_HOST
                imp = state.pending_improvements(res["pending_n"])
                want = wlog[done]["improvements"]
                assert imp.dtype == np.float64 and np.array_equal(imp.view(np.int64), want.view(np.int64))
                forced = sdrf.host_choice(imp, tau, float(uni[draws]))
                hosted += 1
        finally:
            state.close()
        assert done == len(wlog) and hosted == sum(1 for r in wlog if r["n_candidates"])


@pytest.mark.gpu
def test_paper_incremental_values_equal_a_fresh_paper_pass():
    import torch
    from dcr import bfc, sdrf
    from dcr.synth import named_graph
    ei, n = named_graph("wisconsin")
    for loops in (1, 7, 60, 200):
        keep = []
        sdrf.sdrf(ei, n, loops, True, 1.2, 4, uniforms=np.random.RandomState(loops).random_sample(loops),
                  state_out=keep, curv_type="bfc_paper")
        rowptr, order, col, c64, tri = keep[0].export(with_curvature=True)
        keep[0].close()
        assert tri is None and c64.dtype == np.float64
        rows = np.repeat(np.arange(n), np.diff(rowptr))
        pos = {(int(a), int(b)): p for p, (a, b) in enumerate(zip(rows, col))}
        assert all(c64[p] == c64[pos[(b, a)]] for (a, b), p in pos.items())
        up = rows < col
        csr = bfc.DeviceCSR.from_host(rowptr, col)
        fresh = bfc.paper_flavour(csr, edges=(torch.from_numpy(rows[up].astype(np.int32)).cuda(),
                                              torch.from_numpy(col[up].astype(np.int32)).cuda()))
        assert np.array_equal(c64[up].view(np.int64), fresh["bfc"].cpu().numpy().view(np.int64)), loops


@pytest.mark.gpu
def test_paper_batch_equals_single_runs():
    import torch
    from dcr import compat, sdrf
    from dcr.synth import SDRF_PARAMS, named_graph
    ei, n = named_graph("texas")
    loops, tau, bound = SDRF_PARAMS["texas"]
    count = 160                                           # more runs than the B200 has SMs
    uni = np.random.RandomState(21).random_sample((count, loops))
    taus = [tau if r % 3 else INF for r in range(count)]
    outs, logs = sdrf.sdrf_batch(ei, n, loops, True, bound, taus, uniforms=uni, return_log=True, curv_type="bfc_paper")
    for r in list(range(0, count, 23)) + [count - 1]:
        got, glog = sdrf.sdrf(ei, n, loops, True, bound, taus[r], uniforms=uni[r], return_log=True,
                              curv_type="bfc_paper")
        assert np.array_equal(outs[r], got) and np.array_equal(logs[r], glog), r
    compat.ensure_torch_geometric()
    from rewiring.rewire import rewire, rewire_batch
    from torch_geometric.data import Data
    wei, wn = named_graph("wisconsin")
    wl, wt, wb = SDRF_PARAMS["wisconsin"]
    data = Data(edge_index=torch.from_numpy(wei))
    data.num_nodes = wn
    seeds = [0, 1, 2, 3]
    batch = rewire_batch(data, "bfc_paper", wl, wb, wt, seeds=seeds)
    for s, out in zip(seeds, batch):
        np.random.seed(s)
        assert torch.equal(out, rewire(data, "bfc_paper", wl, wb, wt)), s


@pytest.mark.gpu
def test_paper_rejections():
    import torch
    from dcr import lib as L
    from dcr import sdrf
    ei, n = toy_graphs()["c5"]
    rp, od = sdrf.G.classical_order(np.concatenate([ei, [[2], [2]]], axis=1), n, keep_self_loops=True)
    with pytest.raises(L.DcrError, match="lists itself"):
        sdrf.SdrfState(rp, od, 4, L.SDRF_MODE_BFC_PAPER)
    with pytest.raises(NotImplementedError):
        sdrf.sdrf(np.concatenate([ei, [[2], [2]]], axis=1), n, 3, True, 0.5, 2, uniforms=np.zeros(3),
                  curv_type="bfc_paper")
    with pytest.raises(ValueError):                       # no edges: min() of an empty sequence
        sdrf.sdrf(np.zeros((2, 0), dtype=np.int64), 4, 3, True, 0.5, 2, uniforms=np.zeros(3), curv_type="bfc_paper")
    a = sdrf._new_state(L.SDRF_MODE_BFC_PAPER, sdrf._loop_mode("bfc_paper", True)[1](ei, n), 4)
    b = sdrf._new_state(L.SDRF_MODE_HAANTJES, sdrf._loop_mode("haantjes", True)[1](ei, n), 4)
    try:
        dev = a.device
        u = torch.zeros(4, dtype=torch.float64, device=dev)
        logs = [torch.empty((4, L.SDRF_LOG_INTS), dtype=torch.int32, device=dev) for _ in range(2)]
        with pytest.raises(L.DcrError, match="one mode per call"):
            sdrf.run_batch([a, b], [4, 4], [0.5, 0.5], [2, 2], [u, u], [-1, -1], logs, True, 1e-9,
                           torch.zeros((2, 8), dtype=torch.int32, device=dev), sdrf.batch_workspace(2, dev))
        with pytest.raises(L.DcrError, match="only DCR_SDRF_MODE_BFC_PAPER"):
            L.check(a.lib.dcr_sdrf_export_c64(b.handle, logs[0].data_ptr(), u.data_ptr(), L.current_stream()),
                    "dcr_sdrf_export_c64")
    finally:
        a.close()
        b.close()
