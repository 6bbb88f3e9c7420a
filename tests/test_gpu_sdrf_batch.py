"""Batched SDRF (``dcr.sdrf.sdrf_batch``, ``rewiring.rewire.rewire_batch``): B independent loops in one launch, one CTA
per run, must compute exactly what B separate ``sdrf`` / ``rewire`` calls compute.  Argument validation runs without a
device; everything else is marked ``gpu``."""
import ctypes as C

import numpy as np
import pytest

from helpers import gnp, golden, toy_graphs

INF = float("inf")


def _uni(seed, k):
    return np.random.RandomState(seed).random_sample(k)


def _singles(runs, remove_edges=True, **kw):
    """runs: (edge_index, n, loops, bound, tau, uniforms) tuples -> [(edge_index, log)] of separate sdrf calls."""
    from dcr import sdrf
    return [sdrf.sdrf(ei, n, loops, remove_edges, bound, tau, uniforms=uni, return_log=True, **kw)
            for ei, n, loops, bound, tau, uni in runs]


def _batch(runs, remove_edges=True, **kw):
    from dcr import sdrf
    cols = list(zip(*runs))
    return sdrf.sdrf_batch(list(cols[0]), list(cols[1]), list(cols[2]), remove_edges, list(cols[3]), list(cols[4]),
                           uniforms=list(cols[5]), return_log=True, **kw)


def _assert_batch_equals_singles(runs, remove_edges=True, guard=1e-9, **kw):
    outs, logs = _batch(runs, remove_edges, guard=guard, **kw)
    want = _singles(runs, remove_edges, **kw)
    assert len(outs) == len(logs) == len(runs)
    for r, (o, lg, (wo, wl)) in enumerate(zip(outs, logs, want)):
        assert np.array_equal(lg, wl), r
        assert np.array_equal(o, wo), r
    return outs, logs


# ---------------------------------------------------------------------------------------------------------------
# validation (no device)
# ---------------------------------------------------------------------------------------------------------------
def test_sdrf_batch_rejects_length_mismatches_before_touching_cuda():
    from dcr import sdrf
    ei = gnp(10, 0.3, 1)
    uni = np.zeros((3, 4))
    with pytest.raises(ValueError, match="loops"):
        sdrf.sdrf_batch(ei, 10, [4, 4], True, 0.5, 3, uniforms=uni)
    with pytest.raises(ValueError, match="edge_indices"):
        sdrf.sdrf_batch([ei, ei], 10, 4, True, 0.5, 3, uniforms=uni)
    with pytest.raises(ValueError, match="tau"):
        sdrf.sdrf_batch(ei, 10, 4, True, 0.5, [3, 4, 5, 6], uniforms=uni)
    with pytest.raises(ValueError, match="removal_bound"):
        sdrf.sdrf_batch(ei, 10, 4, True, [0.5], 3, uniforms=uni)
    with pytest.raises(ValueError, match="num_nodes"):
        sdrf.sdrf_batch(ei, [10, 10], 4, True, 0.5, 3, uniforms=uni)
    with pytest.raises(ValueError, match="uniforms"):
        sdrf.sdrf_batch(ei, 10, 4, True, 0.5, 3, uniforms=np.zeros(4))
    with pytest.raises(ValueError, match="empty"):
        sdrf.sdrf_batch(ei, 10, 4, True, 0.5, 3, uniforms=[])


def test_rewire_batch_needs_exactly_one_of_seeds_and_uniforms():
    import torch
    from dcr import compat
    compat.ensure_torch_geometric()
    from rewiring.rewire import rewire_batch
    from torch_geometric.data import Data
    data = Data(edge_index=torch.from_numpy(gnp(10, 0.3, 1)))
    data.num_nodes = 10
    with pytest.raises(TypeError):
        rewire_batch(data, "bfc", 4, 0.5, 3)
    with pytest.raises(TypeError):
        rewire_batch(data, "bfc", 4, 0.5, 3, seeds=[0, 1], uniforms=np.zeros((2, 4)))
    with pytest.raises(ValueError, match="datasets"):
        rewire_batch([data, data, data], "bfc", 4, 0.5, 3, seeds=[0, 1])
    with pytest.raises(ValueError, match="max_iterations"):
        rewire_batch(data, "bfc", [4, 4, 4], 0.5, 3, seeds=[0, 1])


# ---------------------------------------------------------------------------------------------------------------
# parity with single runs (B200)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batch_bfc_mixed_graphs_match_single_runs_and_oracle():
    from dcr.synth import SDRF_PARAMS, named_graph
    from oracle.sdrf import sdrf_oracle
    taus = [INF, 3, 12, 60]
    runs, oracle_runs = [], []
    for s in range(8):                                   # gnp graphs of different sizes
        n = 14 + 4 * s
        run = (gnp(n, 0.2 + 0.01 * s, 300 + s), n, 8 + 2 * s, [0.5, 0.3, 1.2, 0.05][s % 4], taus[s % 4],
               _uni(40 + s, 8 + 2 * s))
        runs.append(run)
        oracle_runs.append(len(runs) - 1)
    for name in ("cornell", "texas", "wisconsin"):       # reference hyper-parameters
        ei, n = named_graph(name)
        loops, tau, bound = SDRF_PARAMS[name]
        runs.append((ei, n, loops, bound, tau, _uni(5, loops)))
        runs.append((ei, n, 40, bound, INF, _uni(6, 40)))
    for t, (name, (ei, n)) in enumerate(sorted(toy_graphs().items())):   # tie-heavy
        runs.append((ei, n, 8, 0.4, taus[t % 4], _uni(7, 8)))
        if taus[t % 4] == INF:
            oracle_runs.append(len(runs) - 1)
    outs, logs = _assert_batch_equals_singles(runs)
    for r in oracle_runs:
        ei, n, loops, bound, tau, uni = runs[r]
        want, wlog = sdrf_oracle(ei, n, loops, True, bound, tau, uni, rounding="compiled")
        assert np.array_equal(outs[r], want), r
        assert [(int(a[3]), int(a[4])) for a in logs[r]] == [(w["k"], w["l"]) for w in wlog], r


@pytest.mark.gpu
def test_batch_with_more_runs_than_sms_and_long_cora_runs():
    import torch
    from dcr import sdrf
    from dcr.synth import named_graph
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 30
    ei = gnp(n, 0.2, 11)
    count = 2 * sms
    uni = np.stack([_uni(s, 16) for s in range(count)])
    outs, logs = sdrf.sdrf_batch(ei, n, 16, True, 0.6, 12, uniforms=uni, return_log=True)   # one input, repeated
    for s in range(count):
        want, wlog = sdrf.sdrf(ei, n, 16, True, 0.6, 12, uniforms=uni[s], return_log=True)
        assert np.array_equal(logs[s], wlog), s
        assert np.array_equal(outs[s], want), s
    ei, n = named_graph("cora")
    runs = [(ei, n, 1000, 0.95, 163, _uni(s, 1000)) for s in range(8)]
    outs, logs = _assert_batch_equals_singles(runs)
    assert all(len(lg) == 1000 for lg in logs)


@pytest.mark.gpu
def test_batch_directed_and_classical_flavours_match_single_runs():
    taus = [INF, 4, 2, 20]
    runs = []
    for s in range(6):
        n = 16 + 3 * s
        ei = gnp(n, 0.25, 500 + s)
        dei = ei[:, (ei[0] < ei[1]) | ((ei[0] + s) % 3 == 0)]          # drop most reverse directions
        runs.append((dei, n, 10, [0.5, 0.2, 1.0][s % 3], taus[s % 4], _uni(60 + s, 10)))
    _assert_batch_equals_singles(runs, is_undirected=False)
    for ct, bound in (("1d", -4.0), ("augmented", 0.5), ("haantjes", 1.5)):
        runs = [(gnp(14 + 4 * s, 0.22, 700 + s), 14 + 4 * s, 12, bound + s, taus[s % 4], _uni(80 + s, 12))
                for s in range(5)]
        _assert_batch_equals_singles(runs, curv_type=ct)


@pytest.mark.gpu
def test_batch_self_loop_goldens_one_batch_per_flavour():
    for fname, kw in (("sdrf_selfloop_seq.npz", {}), ("sdrf_directed_selfloop_seq.npz", {"is_undirected": False})):
        z = golden(fname)
        runs = [(z[f"{m}/edge_index"], int(z[f"{m}/n"]), int(z[f"{m}/loops"]), float(z[f"{m}/bound"]),
                 float(z[f"{m}/tau"]), z[f"{m}/uniforms"]) for m in (str(s) for s in z["names"])]
        _assert_batch_equals_singles(runs, **kw)
    z = golden("sdrf_classical_selfloop_seq.npz")
    names = [str(s) for s in z["names"]]
    for ct in sorted({str(z[f"{m}/curv_type"]) for m in names}):
        mine = [m for m in names if str(z[f"{m}/curv_type"]) == ct]
        runs = [(z[f"{m}/edge_index"], int(z[f"{m}/n"]), int(z[f"{m}/loops"]), float(z[f"{m}/bound"]),
                 float(z[f"{m}/tau"]), z[f"{m}/uniforms"]) for m in mine]
        outs, _ = _assert_batch_equals_singles(runs, curv_type=ct)
        for m, o in zip(mine, outs):
            assert np.array_equal(o, z[f"{m}/out"]), m


@pytest.mark.gpu
def test_batch_mixed_exits_and_host_redecisions():
    # early stops (complete graph; a bound nothing reaches), runs that exhaust `loops`, greedy and stochastic runs;
    # guard = 2 hands every stochastic draw to the host, so those runs re-enter across many interleaved launches
    k5, n5 = toy_graphs()["k5"]
    for remove_edges in (False, True):
        runs = [(k5, n5, 5, 0.5 if not remove_edges else 100.0, INF, _uni(1, 5))]
        for s in range(5):
            n = 18 + 3 * s
            runs.append((gnp(n, 0.2, 40 + s), n, 6 + 3 * s, 0.4, [7, INF, 3, 12, 5][s], _uni(90 + s, 6 + 3 * s)))
        runs.append((k5, n5, 3, 100.0, 4, _uni(2, 3)))
        a, alog = _assert_batch_equals_singles(runs, remove_edges=remove_edges, guard=1e-9)
        b, blog = _assert_batch_equals_singles(runs, remove_edges=remove_edges, guard=2.0)
        for r in range(len(runs)):
            assert np.array_equal(a[r], b[r]) and np.array_equal(alog[r], blog[r]), r
        assert len(alog[0]) <= 1 and len(alog[-1]) <= 1     # the complete-graph runs stopped at once


@pytest.mark.gpu
def test_batch_isolates_failing_runs():
    from dcr import lib as L
    from dcr import sdrf
    bar, nb = toy_graphs()["barbell41"]
    runs = [(gnp(20, 0.2, 3), 20, 10, 0.5, 6, _uni(3, 10)),
            (bar, nb, 3, 0.5, 5000, np.array([0.3, 0.3, 0.3])),             # softmax overflow -> ValueError (NaN)
            (gnp(24, 0.2, 4), 24, 12, 0.4, INF, _uni(4, 12)),
            (gnp(22, 0.25, 5), 22, 10, 0.4, 8, _uni(5, 2)),                   # too few uniforms -> DcrError
            (gnp(26, 0.2, 6), 26, 9, 0.3, 12, _uni(6, 9))]
    single = []
    for ei, n, loops, bound, tau, uni in runs:
        try:
            single.append(sdrf.sdrf(ei, n, loops, True, bound, tau, uniforms=uni, return_log=True))
        except Exception as e:
            single.append(e)
    assert isinstance(single[1], ValueError) and "probabilities contain NaN" in str(single[1])
    assert isinstance(single[3], L.DcrError)
    cols = list(zip(*runs))
    outs, logs = sdrf.sdrf_batch(list(cols[0]), list(cols[1]), list(cols[2]), True, list(cols[3]), list(cols[4]),
                                 uniforms=list(cols[5]), return_log=True, return_exceptions=True)
    for r, want in enumerate(single):
        if isinstance(want, Exception):
            assert type(outs[r]) is type(want) and str(outs[r]) == str(want), r
        else:
            assert np.array_equal(outs[r], want[0]) and np.array_equal(logs[r], want[1]), r
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        sdrf.sdrf_batch(list(cols[0]), list(cols[1]), list(cols[2]), True, list(cols[3]), list(cols[4]),
                        uniforms=list(cols[5]))
    with pytest.raises(L.DcrError, match="ran out of uniforms"):
        sdrf.sdrf_batch(list(cols[0][2:]), list(cols[1][2:]), list(cols[2][2:]), True, list(cols[3][2:]),
                        list(cols[4][2:]), uniforms=list(cols[5][2:]))
    _assert_batch_equals_singles([runs[0], runs[2], runs[4]])              # the device is still fine


@pytest.mark.gpu
def test_run_batch_c_abi_rejections():
    import torch
    from dcr import graph
    from dcr import lib as L
    from dcr import sdrf
    lib = L.load()
    ei = gnp(16, 0.3, 2)
    rp, od = graph.networkx_order(ei, 16, keep_self_loops=True)
    crp, cod = graph.classical_order(ei, 16, keep_self_loops=True)
    a = sdrf.SdrfState(rp, od, 4)
    b = sdrf.SdrfState(rp, od, 4)
    c = sdrf.SdrfState(crp, cod, 4, mode=L.SDRF_MODE_1D)
    try:
        dev = a.device
        uni = torch.from_numpy(_uni(0, 4)).to(dev)
        log = torch.empty((3, 4, 8), dtype=torch.int32, device=dev)
        res = torch.zeros((3, 8), dtype=torch.int32, device=dev)
        ws = sdrf.batch_workspace(3, dev)
        wsb = ws.numel() * ws.element_size()

        def call(states, nbytes=wsb, count=None):
            runs = (L.SdrfBatchRun * max(len(states), 1))()
            for i, s in enumerate(states):
                runs[i] = L.SdrfBatchRun(s.handle if s is not None else None, 4, -1, 0.5, 3.0, uni.data_ptr(), 4,
                                         log[i].data_ptr(), res[i].data_ptr())
            return lib.dcr_sdrf_run_batch(runs, len(states) if count is None else count, 1, 1e-9, ws.data_ptr(),
                                          nbytes, L.current_stream())

        assert call([a, c]) == 1 and "mode" in L.last_error()
        assert call([a, b, a]) == 1 and "twice" in L.last_error()
        assert call([a], count=0) == 1 and "count" in L.last_error()
        assert call([a, None]) == 1 and "no state" in L.last_error()
        assert call([a, b], nbytes=lib.dcr_sdrf_batch_workspace_bytes(2) - 1) == 1 and "workspace" in L.last_error()
        assert lib.dcr_sdrf_batch_workspace_bytes(2) > 0
        assert call([a, b]) == 0                                              # and the valid call runs
        torch.cuda.synchronize()
        assert res[:2, 0].tolist() == [L.SDRF_OK, L.SDRF_OK]
        assert torch.equal(log[0], log[1])
    finally:
        for s in (a, b, c):
            s.close()


@pytest.mark.gpu
def test_rewire_batch_with_seeds_equals_seeded_rewire_and_leaves_global_rng_alone():
    import torch
    from dcr import compat
    from dcr.synth import SDRF_PARAMS, named_graph
    compat.ensure_torch_geometric()
    from rewiring.rewire import rewire, rewire_batch
    from torch_geometric.data import Data
    ei, n = named_graph("wisconsin")
    loops, tau, bound = SDRF_PARAMS["wisconsin"]
    data = Data(edge_index=torch.from_numpy(ei))
    data.num_nodes = n
    seeds = list(range(6))
    for curv, b in (("bfc", bound), ("augmented", 2.5)):
        np.random.seed(2024)
        before = np.random.get_state()
        got = rewire_batch(data, curv, loops, b, tau, seeds=seeds)
        after = np.random.get_state()
        assert before[0] == after[0] and np.array_equal(before[1], after[1]) and before[2:] == after[2:]
        for s, g in zip(seeds, got):
            np.random.seed(s)
            want = rewire(data, curv, loops, b, tau)
            assert g.dtype == torch.long and torch.equal(g, want), (curv, s)
    # per-run datasets and hyper-parameters with explicit uniforms; None returns the inputs
    g2 = gnp(30, 0.2, 9)
    d2 = Data(edge_index=torch.from_numpy(g2))
    d2.num_nodes = 30
    uni = [_uni(1, 20), _uni(2, 10)]
    got = rewire_batch([data, d2], "bfc", [20, 10], [bound, 0.5], [tau, INF], uniforms=uni)
    for d, m, b, t, u, g in zip([data, d2], [20, 10], [bound, 0.5], [tau, INF], uni, got):
        from rewiring.sdrf_cuda_bfc import sdrf_cuda_bfc
        assert torch.equal(g, sdrf_cuda_bfc(d, m, True, b, t, True, uniforms=u).edge_index)
    assert all(e is data.edge_index for e in rewire_batch(data, None, 5, 0.5, 3, seeds=[1, 2]))
