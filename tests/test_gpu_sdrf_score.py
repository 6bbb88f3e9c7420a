"""Candidate scoring of many pairs on a device-resident SDRF state (``dcr_sdrf_score``, DESIGN §4.12).

``DynamicCurvature.improvements`` / ``best_additions`` run the loop's own scoring step for caller-chosen pairs, one CTA
per pair.  The GPU tests check, in every loop mode, that a query at the pair the loop picked gives the loop's own
improvements bit for bit (every draw handed to the host with guard = 1) and its greedy choice, that queries at other
pairs match the oracles, that batched queries equal single ones, that queries change nothing, and the rejections.  The
CPU tests cover the Python argument checks and the symbol table."""
import types

import numpy as np
import pytest

from test_gpu_sdrf_edit import MODE_IDS, MODES, OracleGraph, graphs_for, random_edits, same_bits

CLASSICAL = ("1d", "augmented", "haantjes")
NEW_SYMBOLS = ("dcr_sdrf_score_sizes", "dcr_sdrf_score_workspace_bytes", "dcr_sdrf_score")


def _bound(curv_type):
    return 0.2 if curv_type in ("bfc", "bfc_paper") else 2.0


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_score_symbols_and_status():
    import os
    import re
    from dcr import lib as L
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "dcr.h")).read()
    for name in NEW_SYMBOLS:
        assert name in L.SIGNATURES and re.search(rf"\b{name}\s*\(", header)
    assert L.SDRF_BAD_QUERY == 10 and re.search(r"#define DCR_SDRF_BAD_QUERY 10\b", header)


def test_query_argument_checks():
    """Shape, type and id range are checked on the host, before anything reaches the device; no pairs, no launch."""
    from dcr.dynamic import DynamicCurvature

    def never(*a, **k):
        raise AssertionError("no launch expected")

    dc = object.__new__(DynamicCurvature)
    dc.n = 10
    dc._state = types.SimpleNamespace(device="cpu", score=never)
    for bad, match in (([[0, 1, 2]], r"\[m, 2\]"), (np.array([[0.0, 1.0]]), "integer"),
                       ([[0, 1], [3, 10]], r"pairs\[1\] = \(3, 10\)"), ([[-1, 2]], r"pairs\[0\] = \(-1, 2\)"),
                       ([[1, 2], [2, 1], [2**40, 1]], rf"pairs\[2\] = \({2**40}, 1\)")):
        for call in (dc.improvements, dc.best_additions):
            with pytest.raises(ValueError, match=match):
                call(bad)
    assert dc.improvements(np.zeros((0, 2), dtype=np.int64)) == []
    pairs, imp, cnt = dc.best_additions([])
    assert pairs.shape == (0, 2) and imp.shape == (0,) and cnt.shape == (0,)
    dc._state = None                                  # closed: as every other method
    with pytest.raises(AttributeError):
        dc.improvements([[0, 1]])


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _cora(und):
    from dcr.synth import named_graph
    ei, n = named_graph("cora")
    if not und:
        ei = ei[:, ei[0] < ei[1]]
        ei = ei[:, np.random.default_rng(n).permutation(ei.shape[1])]
    return ei, n


def _lists(og, x, y):
    """the loop's candidate lists of (x, y) from the oracle dicts: x's row then x, y's row (directed: predecessors) then y"""
    return list(og.adj[x]) + [x], list((og.pred if og.directed else og.adj)[y]) + [y]


def dense_of_oracle(og):
    """``(A, C)``: the dense adjacency of ``og`` without self-loops and its cuda-flavour curvature (BFC modes)"""
    from oracle.cuda_flavour import bfc_cuda_dense
    A = np.zeros((og.n, og.n), dtype=np.float32)
    for u in range(og.n):
        for v in og.adj[u]:
            if u != v:
                A[u, v] = 1
    return A, bfc_cuda_dense(A)["C"]


def oracle_improvements(og, x, y, dense=None):
    """``(candidates [m, 2], improvements [m])`` of the pair (x, y) from the oracles, masked cells dropped; ``dense``:
    ``dense_of_oracle(og)`` in the BFC modes"""
    from oracle.cuda_flavour import post_delta_dense
    rows, cols = _lists(og, x, y)
    cand, vals = [], []
    if og.curv_type == "bfc":
        A, C = dense
        cxy = C[x, y]
        D = post_delta_dense(A, x, y, rows, cols)
        for I, i in enumerate(rows):
            for J, j in enumerate(cols):
                if D[I, J] != np.float32(-1000):
                    cand.append((i, j))
                    vals.append(np.float64(np.float32(D[I, J] - cxy)))
        return np.array(cand, dtype=np.int64).reshape(-1, 2), np.array(vals, dtype=np.float64)
    if og.curv_type in CLASSICAL:
        from oracle.sdrf_classical import curvature_edge
        before = curvature_edge(og.adj, (x, y), og.curv_type)
    else:
        from oracle.paper_flavour import bfc_edge_fields
        sets = [set(a) for a in og.adj]
        before = bfc_edge_fields(sets, x, y)[6]
    for i in rows:
        for j in cols:
            if i == j or j in og.adj[i]:
                continue
            if og.curv_type in CLASSICAL:
                adj = [dict(a) for a in og.adj]
                adj[i][j] = adj[j][i] = None
                after = curvature_edge(adj, (x, y), og.curv_type)
            else:
                sets[i].add(j), sets[j].add(i)
                after = bfc_edge_fields(sets, x, y)[6]
                sets[i].discard(j), sets[j].discard(i)
            cand.append((i, j))
            vals.append(float(after - before))
    return np.array(cand, dtype=np.int64).reshape(-1, 2), np.array(vals, dtype=np.float64)


def valid_pairs(og, rng, count, curv_type):
    """``count`` pairs the mode's loop can score: edges in both orientations, hub edges, self-loop pairs and, in the
    BFC modes, non-edges, x == y and (0, 0)"""
    edges = [(u, v) for u in range(og.n) for v in og.adj[u] if u != v]
    hubs = np.argsort([-len(a) for a in og.adj])[:3].tolist()
    hub_edges = [(u, v) for u in hubs for v in og.adj[u] if u != v]
    loops = [(u, u) for u in range(og.n) if u in og.adj[u]]
    out = []
    for _ in range(count):
        r = rng.random()
        if r < 0.1 and loops and curv_type != "bfc_paper":
            out.append(loops[rng.integers(len(loops))] if curv_type in CLASSICAL else
                       (loops[rng.integers(len(loops))][0], int(rng.integers(og.n))))
        elif r < 0.3 and hub_edges:
            out.append(hub_edges[rng.integers(len(hub_edges))])
        elif r < 0.4 and curv_type == "bfc":
            out.append((int(rng.integers(og.n)), int(rng.integers(og.n))) if rng.random() < 0.8 else (0, 0))
        else:
            u, v = edges[rng.integers(len(edges))]
            out.append((v, u) if rng.random() < 0.5 else (u, v))
    if curv_type == "bfc":
        out[:3] = [(0, 0), (hubs[0], hubs[0]), (hubs[0], hubs[1])]
    return np.array(out, dtype=np.int64)


def snapshot(dc):
    rp, od = dc.insertion_order()
    return rp, od, dc.edge_index(), dc.curvature()


def same_snapshot(a, b):
    return all(same_bits(x, y) if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y) for x, y in zip(a, b))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_query_at_the_loops_pair_gives_its_improvements(mode):
    """guard = 1: every draw stops with NEED_HOST.  A query at the stop's (x, y) gives pending_improvements bit for bit,
    queries at other pairs in between change nothing, and the run equals one without queries."""
    import torch
    from dcr import lib as L
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(21)
    checked = 0
    for gi, (ei, n) in enumerate(graphs_for(curv_type, und)[:3] + [_cora(und)]):
        loops = 100 if gi == 3 else 40
        tau, bound = 3.0, _bound(curv_type)
        uni = np.random.RandomState(gi).random_sample(loops)
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=loops + 40) as dc, \
                DynamicCurvature(ei, n, curv_type, und, capacity=loops + 40) as ref:
            edits = random_edits(og, 30, rng) if gi == 1 else np.zeros((0, 3), dtype=np.int64)
            dc.edit(edits)
            ref.edit(edits)
            st = dc._state
            u_dev = torch.from_numpy(uni).to(st.device)
            done = draws = 0
            forced = -1
            logs = []
            while done < loops:
                res, log = st.run(loops - done, True, bound, tau, u_dev[draws:], forced_choice=forced, guard=1.0)
                forced = -1
                done += res["iterations_done"]
                draws += res["draws_used"]
                logs.append(log.cpu().numpy())
                if res["status"] != L.SDRF_NEED_HOST:
                    assert res["status"] == L.SDRF_OK
                    break
                want = st.pending_improvements(res["pending_n"])
                x, y = res["pending_x"], res["pending_y"]
                dc.best_additions([(y, x), (x, y)])       # queries between the stop and the re-entry
                (cand, got), = dc.improvements([(x, y)])
                assert got.size == res["pending_n"] and same_bits(got, want)
                assert cand.shape == (got.size, 2)
                checked += 1
                forced = sdrf.host_choice(want, tau, float(uni[draws]))
            log = np.concatenate(logs)
            got_ei = dc.edge_index()
            want_ei, want_log = ref.rewire(loops, True, bound, tau, uniforms=uni, return_log=True)
            assert np.array_equal(log, want_log) and np.array_equal(got_ei, want_ei)
    assert checked >= 100


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_queries_match_the_oracles(mode):
    """Random edges, hubs, self-loop nodes, both orientations and (BFC) non-edges and x == y, on the input, after 300
    mixed edits (rows relocated) and after a partial rewire."""
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(5)
    for gi, (ei, n) in enumerate(graphs_for(curv_type, und)[1:4]):
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=400) as dc:
            for stage in range(3 if und else 2):      # (directed: the oracle dicts have no loop-run counterpart)
                if stage == 1:
                    dc.edit(random_edits(og, 300, rng, hub_share=0.4))
                if stage == 2:
                    dc.rewire(20, True, _bound(curv_type), 3.0, uniforms=np.random.RandomState(gi).random_sample(20))
                    rp, od = dc.insertion_order()       # (checked against the oracle loop in test_gpu_sdrf_edit)
                    og.adj = [dict.fromkeys(od[rp[u]:rp[u + 1]].tolist()) for u in range(n)]
                dense = dense_of_oracle(og) if curv_type == "bfc" else None
                pairs = valid_pairs(og, rng, 12, curv_type)
                got = dc.improvements(pairs)
                for (x, y), (gc, gv) in zip(pairs.tolist(), got):
                    wc, wv = oracle_improvements(og, x, y, dense)
                    assert np.array_equal(gc, wc), (x, y)
                    assert same_bits(gv, wv), (x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_best_addition_is_the_greedy_choice(mode):
    """best_additions at the loop's (x, y) is the (k, l, choice) of one tau = inf iteration on a fork"""
    import torch
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(8)
    hits = 0
    for ei, n in graphs_for(curv_type, und):
        og = OracleGraph(ei, n, curv_type, und)
        with DynamicCurvature(ei, n, curv_type, und, capacity=200) as dc:
            for _ in range(4):
                dc.edit(random_edits(og, 20, rng))
                (f,) = dc.fork()
                with f:
                    _, log = f.rewire(1, False, 0.0, float("inf"), uniforms=np.zeros(1), return_log=True)
                x, y, n_cand, k, l, choice = (int(v) for v in log[0, :6])
                pairs, imp, cnt = dc.best_additions([(x, y)])
                best = dc._state.score(torch.tensor([[x, y]], dtype=torch.int32, device=dc._state.device))["best"]
                best = best.cpu().numpy()
                assert cnt[0] == n_cand
                if n_cand == 0:
                    assert pairs[0].tolist() == [-1, -1] and np.isnan(imp[0]) and best[0, 1] == -1
                    continue
                want = [k, l]
                got = pairs[0].tolist() if curv_type == "bfc" else sorted(pairs[0].tolist())
                assert got == want and best[0, 1] == choice
                cand, vals = dc.improvements([(x, y)])[0]
                assert same_bits(imp[:1], vals[choice:choice + 1]) and vals.max() == imp[0]
                hits += 1
    assert hits >= 8


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_batched_queries_equal_single_queries(mode):
    """Q = 1, 148 and 1000 queries (duplicates and hub-hub pairs among them) in one call equal Q single calls."""
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(3)
    ei, n = graphs_for(curv_type, und)[3]
    og = OracleGraph(ei, n, curv_type, und)
    with DynamicCurvature(ei, n, curv_type, und, capacity=100) as dc:
        pool = valid_pairs(og, rng, 400, curv_type)
        singles = {}
        for q in (1, 148, 1000):
            pairs = pool[rng.integers(len(pool), size=q)]           # duplicates
            batch = dc.improvements(pairs)
            bp, bi, bn = dc.best_additions(pairs)
            for t, (x, y) in enumerate(pairs.tolist()):
                if (x, y) not in singles:
                    singles[(x, y)] = (dc.improvements([(x, y)])[0], dc.best_additions([(x, y)]))
                (sc, sv), (sp, si, sn) = singles[(x, y)]
                assert np.array_equal(batch[t][0], sc) and same_bits(batch[t][1], sv)
                assert np.array_equal(bp[t], sp[0]) and same_bits(bi[t:t + 1], si) and bn[t] == sn[0]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_queries_leave_the_object_unchanged(mode):
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    rng = np.random.default_rng(9)
    ei, n = graphs_for(curv_type, und)[2]
    og = OracleGraph(ei, n, curv_type, und)
    with DynamicCurvature(ei, n, curv_type, und, capacity=200) as dc:
        dc.edit(random_edits(og, 60, rng))
        (fresh,) = dc.fork()
        before = snapshot(dc)
        remaining = dc.remaining
        pairs = valid_pairs(og, rng, 300, curv_type)
        dc.improvements(pairs)
        dc.best_additions(pairs)
        assert same_snapshot(snapshot(dc), before) and dc.remaining == remaining
        uni = np.random.RandomState(2).random_sample(30)
        with fresh:
            want = fresh.rewire(30, True, _bound(curv_type), 3.0, uniforms=uni, return_log=True)
        got = dc.rewire(30, True, _bound(curv_type), 3.0, uniforms=uni, return_log=True)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_rejected_queries(mode):
    import torch
    from dcr import lib as L
    from dcr.dynamic import DynamicCurvature
    curv_type, und = mode
    ei, n = graphs_for(curv_type, und)[1]
    og = OracleGraph(ei, n, curv_type, und)
    dc = DynamicCurvature(ei, n, curv_type, und, capacity=10)
    edge = next((u, v) for u in range(n) for v in og.adj[u] if u != v)
    bad = [(n, 0), (0, -1), (2**40, 1)]
    if curv_type != "bfc":
        non_edge = next((u, v) for u in range(n) for v in range(n) if u != v and v not in og.adj[u])
        plain = next(u for u in range(n) if u not in og.adj[u])
        bad += [non_edge, (plain, plain)]
    before = snapshot(dc)
    for b in bad:
        for call in (dc.improvements, dc.best_additions):
            with pytest.raises(ValueError, match=rf"pairs\[1\] = \({b[0]}, {b[1]}\)"):
                call([edge, b, edge])
    with pytest.raises(ValueError, match="max_cells"):
        dc.improvements([edge], max_cells=1)
    assert same_snapshot(snapshot(dc), before)
    # the C entry points: count < 1, null pointers, a short workspace
    lib, st = L.load(), dc._state
    dev = st.device
    p = torch.tensor([edge], dtype=torch.int32, device=dev)
    s = torch.zeros((1, 2), dtype=torch.int32, device=dev)
    stat = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = L.current_stream()
    assert lib.dcr_sdrf_score_sizes(st.handle, p.data_ptr(), 0, s.data_ptr(), stat.data_ptr(), stream) == 1
    assert lib.dcr_sdrf_score_sizes(None, p.data_ptr(), 1, s.data_ptr(), stat.data_ptr(), stream) == 1
    assert lib.dcr_sdrf_score_sizes(st.handle, p.data_ptr(), 1, 0, stat.data_ptr(), stream) == 1
    assert lib.dcr_sdrf_score_workspace_bytes(st.handle, 0) == 0
    need = lib.dcr_sdrf_score_workspace_bytes(st.handle, 1)
    assert need > 0
    off = torch.zeros(2, dtype=torch.int64, device=dev)
    cand = torch.zeros(4096, dtype=torch.int32, device=dev)
    imp = torch.zeros(1 << 20, dtype=torch.float64, device=dev)
    best = torch.zeros((1, 4), dtype=torch.int64, device=dev)
    ws = torch.zeros(need // 4 + 1, dtype=torch.int32, device=dev)
    args = [st.handle, p.data_ptr(), 1, off.data_ptr(), off.data_ptr(), cand.data_ptr(), imp.data_ptr(),
            best.data_ptr(), ws.data_ptr(), need, stream]
    for k, v in ((2, 0), (1, 0), (3, 0), (4, 0), (5, 0), (6, 0), (7, 0), (8, 0), (9, need - 1), (0, None)):
        a = list(args)
        a[k] = v
        assert lib.dcr_sdrf_score(*a) == 1, k
    assert lib.dcr_sdrf_score(*args) == 0
    torch.cuda.synchronize()
    assert best[0, 0].item() == dc.best_additions([edge])[2][0]
    dc.close()
    with pytest.raises(AttributeError):
        dc.improvements([edge])
