"""SDRF over a batched dataset (DESIGN §4.13): ``dcr.sdrf.sdrf_dataset`` and ``rewiring.rewire.rewire_dataset``.

The dataset is in the PyG batch layout: one ``edge_index`` in global node ids and ``ptr``.  Its insertion order is
computed once on the disjoint union, all states are set up by one ``dcr_sdrf_create_batch`` and exported by one
``dcr_sdrf_export_edge_index_batch``.  Every GPU comparison is bit for bit against ``sdrf()`` on each graph alone and
against ``sdrf_batch`` on the list of graphs."""
import ctypes

import numpy as np
import pytest

from test_gpu_sdrf_edit import MODE_IDS, MODES

INF = float("inf")
NEW_SYMBOLS = ("dcr_sdrf_create_batch", "dcr_sdrf_export_edge_index_batch",
               "dcr_sdrf_export_edge_index_batch_workspace_bytes")
LOG_NODE_FIELDS = [0, 1, 3, 4, 6, 7]


def _bound(curv_type):
    return 0.2 if curv_type in ("bfc", "bfc_paper") else 2.0


def _undirected(pairs, rng):
    """both directions of every pair, a few listed one way only, columns shuffled"""
    if not pairs:
        return np.zeros((2, 0), dtype=np.int64)
    a = np.array(sorted(pairs), dtype=np.int64).T
    keep_back = rng.random(a.shape[1]) > 0.1
    ei = np.concatenate([a, a[::-1][:, keep_back]], axis=1)
    return ei[:, rng.permutation(ei.shape[1])]


def random_graph(rng, kind, curv_type, und):
    """One graph ``(edge_index, n)`` in local ids.  Kinds: 0 a single node (with its self-loop where the mode keeps them),
    1 no edges, 2 a hub, 3 random with trailing isolated nodes, 4 random with self-loops, 5 a cycle."""
    loops_ok = curv_type != "bfc_paper"
    if kind == 0:
        n = 1
        ei = np.array([[0], [0]]) if loops_ok and rng.random() < 0.5 else np.zeros((2, 0), dtype=np.int64)
        return ei.astype(np.int64), n
    if kind == 1:
        return np.zeros((2, 0), dtype=np.int64), int(rng.integers(2, 6))
    n = int(rng.integers(6, 45))
    pairs = set()
    if kind == 2:
        for v in range(1, n):
            if rng.random() < 0.8:
                pairs.add((0, v))
    if kind == 5:
        pairs |= {(min(v, (v + 1) % n), max(v, (v + 1) % n)) for v in range(n)}
    active = n - 3 if kind == 3 else n
    for _ in range(int(rng.integers(n // 2, 2 * n))):
        a, b = rng.integers(0, active, size=2)
        if a != b:
            pairs.add((int(min(a, b)), int(max(a, b))))
    if und:
        ei = _undirected(pairs, rng)
    else:
        d = {(a, b) if rng.random() < 0.5 else (b, a) for a, b in pairs}
        d |= {(b, a) for a, b in list(d) if rng.random() < 0.3}
        ei = np.array(sorted(d), dtype=np.int64).T.reshape(2, -1)
        ei = ei[:, rng.permutation(ei.shape[1])]
    if kind == 4 and loops_ok:
        who = rng.choice(active, size=3, replace=False)
        ei = np.concatenate([ei, np.stack([who, who])], axis=1)
        ei = ei[:, rng.permutation(ei.shape[1])]
    return ei.astype(np.int64), n


def random_dataset(curv_type, und, count, seed, kinds=6):
    rng = np.random.default_rng(seed)
    return [random_graph(rng, int(k), curv_type, und) for k in rng.permutation(np.arange(count) % kinds)]


def concat(graphs, seed=0):
    """The PyG layout of ``graphs``: global ids, ``ptr``; the columns of different graphs are interleaved at random,
    each graph's own columns keep their order."""
    rng = np.random.default_rng(seed)
    ptr = np.concatenate([[0], np.cumsum([n for _, n in graphs])]).astype(np.int64)
    cols, keys = [], []
    for g, (ei, _) in enumerate(graphs):
        cols.append(ei + ptr[g])
        keys.append(np.sort(rng.random(ei.shape[1])))
    ei = np.concatenate(cols, axis=1) if cols else np.zeros((2, 0), dtype=np.int64)
    return ei[:, np.argsort(np.concatenate(keys), kind="stable")], ptr


def _unshift_log(log, base):
    out = np.array(log, copy=True)
    node = out[:, LOG_NODE_FIELDS]
    out[:, LOG_NODE_FIELDS] = np.where(node >= 0, node - base, node)
    return out


def _same_error(a, b):
    return type(a) is type(b) and str(a) == str(b)


def check_dataset(curv_type, und, graphs, loops, remove, taus, uniforms, guard=1e-9, seed=0, per_graph=None):
    """sdrf_dataset against sdrf_batch on the list and against sdrf() on every graph in ``per_graph`` (default all)."""
    import torch

    from dcr import sdrf
    ei, ptr = concat(graphs, seed)
    bound = _bound(curv_type)
    got, gptr, glogs, errs = sdrf.sdrf_dataset(torch.from_numpy(ei), torch.from_numpy(ptr), loops, remove, bound, taus,
                                               uniforms=uniforms, guard=guard, return_log=True, is_undirected=und,
                                               curv_type=curv_type, return_exceptions=True)
    assert got.is_cuda and got.dtype == torch.int64 and gptr.dtype == torch.int64 and gptr.numel() == len(graphs) + 1
    got, gptr = got.cpu().numpy(), gptr.cpu().numpy()
    assert gptr[0] == 0 and gptr[-1] == got.shape[1] and np.all(np.diff(gptr) >= 0)
    bt, blogs = sdrf.sdrf_batch([e for e, _ in graphs], [n for _, n in graphs], loops, remove, bound, taus,
                                uniforms=uniforms, guard=guard, return_log=True, is_undirected=und,
                                curv_type=curv_type, return_exceptions=True)
    loops_g = sdrf._per_run("loops", loops, len(graphs))
    taus_g = sdrf._per_run("tau", taus, len(graphs))
    for g, (eg, n) in enumerate(graphs):
        cols = got[:, gptr[g]:gptr[g + 1]]
        if isinstance(bt[g], Exception):
            assert _same_error(errs[g], bt[g]) and cols.shape[1] == 0, g
        else:
            assert errs[g] is None, (g, errs[g])
            assert np.all((cols >= ptr[g]) & (cols < ptr[g + 1]))
            assert np.array_equal(cols - ptr[g], bt[g]), g
            assert np.array_equal(_unshift_log(glogs[g], ptr[g]), blogs[g]), g
        if per_graph is not None and g not in per_graph:
            continue
        try:
            want, wlog = sdrf.sdrf(eg, n, loops_g[g], remove, bound, taus_g[g], uniforms=uniforms[g], guard=guard,
                                   return_log=True, is_undirected=und, curv_type=curv_type)
        except Exception as e:      # noqa: BLE001  the exception is the result here
            assert _same_error(errs[g], e), (g, errs[g], e)
            continue
        assert np.array_equal(cols - ptr[g], want) and np.array_equal(_unshift_log(glogs[g], ptr[g]), wlog), g
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_new_symbols_are_declared_and_bound():
    from dcr import lib as L
    from test_host import _declared_symbols
    declared = set(_declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared and name in L.SIGNATURES


@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_union_order_equals_per_graph_order(mode):
    """The order function of each mode on the disjoint union, in local ids, equals its result on every graph alone."""
    from dcr import sdrf
    curv_type, und = mode
    for seed in range(4):
        graphs = random_dataset(curv_type, und, 40, seed)
        ei, ptr = concat(graphs, seed)
        m, order = sdrf._loop_mode(curv_type, und)
        gid = sdrf._column_graphs(ei, ptr)
        union = sdrf._dataset_order(order, m, ei, ptr, gid)
        assert union[0].dtype == np.int64 and union[1].dtype == np.int32
        for half in range(len(union) // 2):
            rp, od = union[2 * half], union[2 * half + 1]
            for g, (eg, n) in enumerate(graphs):
                want = order(eg, n)
                wrp, wod = np.asarray(want[2 * half], dtype=np.int64), want[2 * half + 1]
                lo, hi = ptr[g], ptr[g + 1]
                assert np.array_equal(rp[lo:hi + 1] - rp[lo], wrp), (g, half)
                assert np.array_equal(od[rp[lo]:rp[hi]], wod), (g, half)


def test_python_input_validation():
    from dcr import sdrf
    u = np.zeros((3, 2))
    ei = np.array([[0, 1, 2, 3, 4, 5], [1, 0, 3, 2, 5, 4]])
    run = lambda e, p, **kw: sdrf.sdrf_dataset(e, p, 2, True, 0.5, INF, uniforms=kw.pop("uni", u), **kw)  # noqa: E731
    with pytest.raises(ValueError, match=r"column 1 = \(1, 2\) joins graph 0 and graph 1"):
        run(np.array([[0, 1], [1, 2]]), [0, 2, 4, 6])
    with pytest.raises(ValueError, match=r"column 0 = \(5, 6\) has a node outside \[0, 6\).*graph 2"):
        run(np.array([[5], [6]]), [0, 2, 4, 6])
    with pytest.raises(ValueError, match=r"outside"):
        run(np.array([[-1], [0]]), [0, 2, 4, 6])
    with pytest.raises(ValueError, match=r"graph 1: ptr is not monotone"):
        run(ei, [0, 4, 2, 6])
    with pytest.raises(ValueError, match=r"graph 1 has no nodes"):
        run(ei, [0, 4, 4, 6])
    with pytest.raises(ValueError, match=r"ptr\[0\]"):
        run(ei, [1, 2, 4, 6])
    with pytest.raises(ValueError, match="3 graphs, the batch has 2"):
        run(ei, [0, 2, 4, 6], uni=np.zeros((2, 2)))
    with pytest.raises(ValueError, match="empty"):
        run(ei, [0, 6], uni=[])
    with pytest.raises(ValueError, match="1-d integer"):
        run(ei, np.array([0.0, 3.0, 6.0, 6.0]))
    # the mode input errors name the graph
    loop = np.array([[0, 1, 3, 4, 4], [1, 0, 4, 3, 4]])
    with pytest.raises(NotImplementedError, match="graph 1: curv_type='bfc_paper' does not take graphs with self-loops"):
        run(loop, [0, 2, 5, 6], curv_type="bfc_paper")
    rep = np.array([[0, 2, 3, 3], [1, 3, 2, 2]])
    with pytest.raises(NotImplementedError, match="graph 1: directed SDRF: repeated"):
        run(rep, [0, 2, 4, 6], is_undirected=False)
    with pytest.raises(NotImplementedError, match="undirected graphs only"):
        run(ei, [0, 2, 4, 6], curv_type="bfc_paper", is_undirected=False)


def _create_batch(lib, count, mode, nn, rp, od, ma, irp=None, iod=None):
    handles = (ctypes.c_void_p * max(count, 1))()
    ptr = lambda a: a.ctypes.data if a is not None else 0  # noqa: E731
    rc = lib.dcr_sdrf_create_batch(count, mode, ptr(nn), ptr(rp), ptr(od), ptr(irp), ptr(iod), ptr(ma), handles)
    return rc, handles


def test_create_batch_rejects_bad_input_before_any_allocation():
    """Every rejection of dcr_sdrf_create_batch comes before the device is touched, so it is checked without one; no
    handle is written."""
    from dcr import lib as L
    lib = L.load()
    nn = np.array([2, 3], dtype=np.int32)
    rp = np.array([0, 1, 2, 3, 4, 4], dtype=np.int64)
    od = np.array([1, 0, 1, 0], dtype=np.int32)
    ma = np.array([1, 1], dtype=np.int64)

    def rejected(count=2, mode=L.SDRF_MODE_BFC, nn=nn, rp=rp, od=od, ma=ma, match=""):
        rc, handles = _create_batch(lib, count, mode, nn, rp, od, ma)
        assert rc == 1 and all(h is None for h in handles[:max(count, 1)])
        assert match in L.last_error(), L.last_error()

    rejected(count=0, match="count must be >= 1")
    rejected(mode=9, match="unknown mode")
    rejected(nn=np.array([2, 0], dtype=np.int32), match="graph 1 has 0 nodes")
    rejected(rp=np.array([1, 1, 2, 3, 4, 4], dtype=np.int64), match="start at 0")
    rejected(rp=np.array([0, 1, 2, 1, 4, 4], dtype=np.int64), match="graph 1: the row offsets decrease at node 0")
    rejected(od=np.array([1, 0, 1, 7], dtype=np.int32), match="graph 1: bad neighbour id")
    rejected(rp=np.array([0, 1, 2, 4, 4, 4], dtype=np.int64), od=np.array([1, 0, 0, 0], dtype=np.int32),
             match="graph 1: node 0 lists itself more than once")
    rejected(mode=L.SDRF_MODE_BFC_PAPER, od=np.array([1, 0, 0, 1], dtype=np.int32),
             match="graph 1: node 0 lists itself (the paper-flavour loop takes no self-loops)")
    rejected(mode=L.SDRF_MODE_BFC_DIRECTED, match="the directed mode needs the predecessor lists")
    rejected(ma=np.array([1, -1], dtype=np.int64), match="graph 1: max_additions < 0")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("count", [1, 7, 300])
def test_dataset_equals_sdrf_per_graph_and_sdrf_batch(mode, count):
    """Mixed graphs (a single node, no edges, hubs, trailing isolated nodes, self-loops where the mode keeps them),
    columns interleaved across graphs, greedy and stochastic runs of different lengths, with and without removal."""
    curv_type, und = mode
    graphs = random_dataset(curv_type, und, count, seed=count)
    rng = np.random.default_rng(count + 1)
    loops = [int(v) for v in rng.integers(0, 14, size=count)]
    taus = [INF if g % 2 else 3.0 for g in range(count)]
    uniforms = [rng.random(m) for m in loops]
    for remove in (True, False):
        errs = check_dataset(curv_type, und, graphs, loops, remove, taus, uniforms, seed=count)
        if curv_type != "bfc" and count > 1:      # the classical and paper loops raise on a graph without edges
            assert any(isinstance(e, ValueError) for e in errs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [MODES[0], MODES[2], MODES[5]], ids=[MODE_IDS[0], MODE_IDS[2], MODE_IDS[5]])
def test_dataset_host_path_for_every_draw(mode):
    """guard = 1 hands every stochastic draw back to the host; the results are those of sdrf() and sdrf_batch."""
    from unittest import mock

    from dcr import sdrf
    curv_type, und = mode
    graphs = random_dataset(curv_type, und, 12, seed=5)
    rng = np.random.default_rng(6)
    uniforms = [rng.random(10) for _ in graphs]
    calls = []
    choice = sdrf.host_choice

    def counted(*a):
        calls.append(1)
        return choice(*a)

    with mock.patch.object(sdrf, "host_choice", counted):
        check_dataset(curv_type, und, graphs, 10, True, 2.0, uniforms, guard=1.0)
    assert calls


@pytest.mark.gpu
def test_dataset_of_2000_small_graphs():
    """More states than one wave of CTAs; every graph against sdrf_batch, a sample against sdrf()."""
    graphs = random_dataset("bfc", True, 2000, seed=11)
    rng = np.random.default_rng(12)
    uniforms = [rng.random(6) for _ in graphs]
    check_dataset("bfc", True, graphs, 6, True, [INF, 4.0] * 1000, uniforms, per_graph=set(range(0, 2000, 97)))


def _state_image(st):
    """everything a state exports before any run: insertion order (self entries included), sorted columns, curvature,
    supports, nnz and the device edge_index"""
    from dcr import lib as L
    out = [st.nnz(), st.n_self]
    out += [np.asarray(a) for a in st.export() if a is not None]
    out += [np.asarray(a) for a in st.export(with_curvature=True) if a is not None]
    out.append(st.edge_index().cpu().numpy())
    if st.mode == L.SDRF_MODE_BFC_PAPER:
        out.append(st.export(with_curvature=True)[3])
    return out


def _same_image(a, b):
    return len(a) == len(b) and all(np.asarray(x).dtype == np.asarray(y).dtype and np.array_equal(
        np.asarray(x).view(np.uint8) if np.asarray(x).ndim else x, np.asarray(y).view(np.uint8) if np.asarray(y).ndim else y)
        for x, y in zip(a, b))


def _batch_states(curv_type, und, graphs, budgets):
    from dcr import sdrf
    ei, ptr = concat(graphs, 1)
    mode, order = sdrf._loop_mode(curv_type, und)
    lists = sdrf._dataset_order(order, mode, ei, ptr, sdrf._column_graphs(ei, ptr))
    return sdrf.SdrfState.create_batch(mode, np.diff(ptr), lists[0], lists[1], budgets, *lists[2:]), mode, order


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_create_batch_states_equal_single_states(mode):
    """Before any run: curvature (bits), supports, insertion order and nnz of every batched state equal those of the
    state dcr_sdrf_create_mode makes for the graph alone."""
    from dcr import sdrf
    curv_type, und = mode
    graphs = random_dataset(curv_type, und, 60, seed=3)
    budgets = [g % 5 for g in range(len(graphs))]
    states, m, order = _batch_states(curv_type, und, graphs, budgets)
    try:
        for g, (eg, n) in enumerate(graphs):
            single = sdrf._new_state(m, order(eg, n), budgets[g])
            try:
                assert states[g].n == n and states[g].mode == m
                assert _same_image(_state_image(states[g]), _state_image(single)), g
            finally:
                single.close()
    finally:
        for s in states:
            s.close()


@pytest.mark.gpu
def test_pool_life_cycle():
    """States of one pool closed in any order, some run after their siblings are closed, and a fork of a pooled state
    that outlives the whole pool."""
    from dcr import sdrf
    graphs = [random_graph(np.random.default_rng(s), 2 + s % 4, "bfc", True) for s in range(9)]
    loops = 8
    U = np.random.RandomState(2).random_sample((9, loops))
    want = sdrf.sdrf_batch([e for e, _ in graphs], [n for _, n in graphs], loops, True, 0.2, 3.0, uniforms=U)
    states, m, order = _batch_states("bfc", True, graphs, [2 * loops] * 9)
    (fork,) = states[4].fork(1)
    from dcr import graph as G

    def result(st, g):
        sdrf._run_state(st, loops, True, 0.2, 3.0, U[g], 1e-9)
        return G.from_networkx_order(*st.export())

    for g in (7, 0, 2):
        states[g].close()
    for g in (1, 8):
        assert np.array_equal(result(states[g], g), want[g])
    for g in (3, 5, 6, 4, 1, 8):
        states[g].close()
    assert all(s.handle is None for s in states)
    # the fork owns its slab: it runs (twice its source's budget) and exports after the pool is gone
    assert np.array_equal(result(fork, 4), want[4])
    fork.close()


@pytest.mark.gpu
def test_failing_graphs_fail_alone():
    """Softmax overflow in one graph and a classical graph without edges: each fails alone, with sdrf()'s exception,
    its graph empty in edge_ptr; the others are unaffected; without return_exceptions the lowest-index one is raised."""
    import torch

    from dcr import sdrf
    graphs = [g for g in random_dataset("augmented", True, 12, seed=8) if g[1] >= 6][:6]
    graphs.insert(3, (np.zeros((2, 0), dtype=np.int64), 4))
    taus = [2.0] * 7
    taus[5] = 1e6
    uniforms = [np.full(6, 0.5)] * 7
    errs = check_dataset("augmented", True, graphs, 6, True, taus, uniforms)
    assert [e is not None for e in errs] == [False, False, False, True, False, True, False]
    assert "empty" in str(errs[3]) and ("NaN" in str(errs[5]) or "sum to 1" in str(errs[5]))
    ei, ptr = concat(graphs)
    with pytest.raises(ValueError, match="empty sequence"):
        sdrf.sdrf_dataset(ei, ptr, 6, True, 2.0, taus, uniforms=uniforms, curv_type="augmented")
    # every graph failing leaves an empty output
    out, eptr, errs = sdrf.sdrf_dataset(ei[:, :0], ptr, 6, True, 2.0, 2.0, uniforms=uniforms, curv_type="augmented",
                                        return_exceptions=True)
    assert out.shape == (2, 0) and torch.all(eptr == 0) and all(isinstance(e, ValueError) for e in errs)


@pytest.mark.gpu
@pytest.mark.parametrize("curv_type", ["bfc", "1d", "bfc_paper"])
def test_rewire_dataset_equals_rewire_batch(curv_type):
    import torch

    from rewiring.rewire import rewire_batch, rewire_dataset
    from torch_geometric.data import Data       # (the stand-in, when PyG is absent, once rewiring is imported)
    graphs = [g for g in random_dataset(curv_type, True, 20, seed=9) if g[0].shape[1] > 0]
    data = [Data(edge_index=torch.from_numpy(e)) for e, _ in graphs]
    for d, (_, n) in zip(data, graphs):
        d.num_nodes = n
    seeds = list(range(100, 100 + len(data)))
    iters = [5 + g % 7 for g in range(len(data))]
    want = rewire_batch(data, curv_type, iters, 0.3, 4.0, seeds=seeds)
    got, eptr = rewire_dataset(data, curv_type, iters, 0.3, 4.0, seeds=seeds)
    ptr = np.concatenate([[0], np.cumsum([n for _, n in graphs])])
    got, eptr = got.cpu(), eptr.cpu()
    for g in range(len(data)):
        assert torch.equal(got[:, eptr[g]:eptr[g + 1]] - int(ptr[g]), want[g]), g
    # a Batch-like input gives the same; curv_type None gives the input back
    class Batch:
        pass
    b = Batch()
    b.edge_index, b.ptr = rewire_dataset(data, None, iters, 0.3, 4.0, seeds=seeds)[0], torch.from_numpy(ptr)
    again, eptr2 = rewire_dataset(b, curv_type, iters, 0.3, 4.0, seeds=seeds)
    assert torch.equal(again.cpu(), got) and torch.equal(eptr2.cpu(), eptr)
    same, sptr = rewire_dataset(b, None, iters, 0.3, 4.0, seeds=seeds)
    assert same is b.edge_index or torch.equal(same, b.edge_index)
    assert sptr.tolist() == np.concatenate([[0], np.cumsum([e.shape[1] for e, _ in graphs])]).tolist()
    with pytest.raises(TypeError, match="exactly one"):
        rewire_dataset(b, curv_type, 5, 0.3, 4.0)


@pytest.mark.gpu
def test_export_batch_rejections_and_short_capacity():
    import torch

    from dcr import lib as L
    from dcr import sdrf
    graphs = [random_graph(np.random.default_rng(s), 3, "bfc", True) for s in range(5)]
    states, _, _ = _batch_states("bfc", True, graphs, [1] * 5)
    (other,) = _batch_states("1d", True, graphs[:1], [1])[0]
    lib = L.load()

    def call(sts, offs, capacity, count=None, ws=True):
        h = (ctypes.c_void_p * max(len(sts), 1))(*[s.handle.value for s in sts])
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        o = torch.full((2, capacity + 8), -7, dtype=torch.int64, device="cuda")
        e = torch.empty(len(sts) + 1, dtype=torch.int64, device="cuda")
        nb = int(lib.dcr_sdrf_export_edge_index_batch_workspace_bytes(h, len(sts)))
        w = torch.empty(max(nb // 8, 1), dtype=torch.int64, device="cuda")
        rc = lib.dcr_sdrf_export_edge_index_batch(h, len(sts) if count is None else count, offs.ctypes.data,
                                                  o[0].data_ptr(), o[1].data_ptr(), capacity, e.data_ptr(),
                                                  w.data_ptr(), nb if ws else 8, L.current_stream())
        return rc, o, e

    try:
        ptr = np.concatenate([[0], np.cumsum([n for _, n in graphs])])
        full, eptr = sdrf.export_edge_index_batch(states, ptr[:-1], 10**4)
        total = int(eptr[-1])
        for g, st in enumerate(states):
            assert torch.equal(full[:, eptr[g]:eptr[g + 1]] - int(ptr[g]), st.edge_index())
        # a short capacity: nothing at or beyond it is written, everything before it is the full export's
        for cap in (0, 1, total - 5):
            rc, o, e = call(states, ptr[:-1], cap)
            assert rc == 0 and torch.equal(e, eptr)
            assert torch.equal(o[:, :cap], full[:, :cap]) and bool(torch.all(o[:, cap:] == -7))
        assert call(states, ptr[:-1], 8, count=0)[0] == 1 and "count must be >= 1" in L.last_error()
        assert call(states[:2], [0, 1], 8)[0] == 1 and "overlaps" in L.last_error()
        assert call(states[:2], [-1, 10], 8)[0] == 1 and "negative" in L.last_error()
        assert call([states[0], other], [0, 10], 8)[0] == 1 and "one mode per call" in L.last_error()
        assert call(states, ptr[:-1], 8, ws=False)[0] == 1 and "workspace" in L.last_error()
    finally:
        for s in states + [other]:
            s.close()
