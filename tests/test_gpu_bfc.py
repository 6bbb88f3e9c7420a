"""GPU parity, BFC: the CUDA kernels (through the C ABI) against the oracle and the golden fixtures.

Bars: integer counts bit-exact; paper-flavour fp64 value bit-exact (same operation order, explicit rounding);
cuda-flavour fp32 image bit-exact against the compiled-dataflow oracle and within 1e-6 of the simulator goldens.
"""
import numpy as np
import pytest

from helpers import dense_of, gnp, golden, sym_edge_index, toy_graphs

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["auto", "hashed"])
def paper_mode(request):
    """Both membership structures of the paper-flavour kernels: ``auto`` picks the exact shared-memory bitmap of
    N(a) (every graph here has n <= DENSE_MAX_N), ``hashed`` forces the hashed-bitmap + table kernels that graphs
    with more nodes take (``dcr_bfc_paper_set_mode``, per call — no environment variable involved)."""
    from dcr import bfc
    old = bfc.set_paper_mode(request.param)
    yield request.param
    bfc.set_paper_mode(old)


def _csr(ei, n):
    from dcr import bfc, graph
    rowptr, col = graph.undirected_csr(ei, n)
    return bfc.DeviceCSR.from_host(rowptr, col)


def _paper_gpu(ei, n):
    from dcr import bfc
    csr = _csr(ei, n)
    out = bfc.paper_flavour(csr)
    f = {k: out[k].cpu().numpy() for k in ("tri", "sq_i", "sq_j", "gamma", "bfc")}
    f["edges"] = np.stack([out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()], axis=1).astype(np.int64)
    return f


def _check_paper(ei, n, tag):
    from oracle.paper_flavour import bfc_paper
    got = _paper_gpu(ei, n)
    ref = bfc_paper(ei, n, got["edges"])
    for k in ("tri", "sq_i", "sq_j", "gamma"):
        assert np.array_equal(got[k], ref[k]), (tag, k, np.flatnonzero(got[k] != ref[k])[:5])
    assert np.array_equal(got["bfc"], ref["bfc"]), (tag, np.abs(got["bfc"] - ref["bfc"]).max())
    return got


def test_paper_flavour_golden_reference_values(paper_mode):
    z = golden("paper_kat.npz")
    for name in (str(s) for s in z["names"]):
        ei, n = z[f"{name}/edge_index"], int(z[f"{name}/n"])
        if ei.shape[1] == 0:
            continue
        got = _paper_gpu(ei, n)
        assert np.array_equal(got["edges"], z[f"{name}/edges"]), name
        assert np.array_equal(got["bfc"], z[f"{name}/bfc"]), name     # unmodified bfc_naive.bfc_edge, bit for bit


@pytest.mark.parametrize("seed", range(8))
def test_paper_flavour_random_graphs(seed, paper_mode):
    n = 20 + 17 * seed
    _check_paper(gnp(n, [0.05, 0.1, 0.2, 0.4][seed % 4], seed), n, f"gnp{seed}")


def test_paper_flavour_edge_cases(paper_mode):
    # single edge, star (deg_min == 1 everywhere), disjoint union with isolated nodes, complete graph
    _check_paper(sym_edge_index([(0, 1)], 2), 2, "k2")
    _check_paper(sym_edge_index([(0, i) for i in range(1, 40)], 45), 45, "star+isolated")
    _check_paper(sym_edge_index([(i, j) for i in range(24) for j in range(i + 1, 24)], 24), 24, "k24")
    for name, (ei, n) in toy_graphs().items():
        _check_paper(ei, n, name)


def test_paper_flavour_cta_team_and_global_table_paths(paper_mode):
    # hubs: tested endpoints of degree ~700-900 (group kernel G1 / dense group) and ~17000 (hashed: class X, the
    # CTA-team kernel with its table in global memory; dense: still the group kernel), cooperative edges included
    rng = np.random.default_rng(5)
    n = 3000
    pairs = [(0, i) for i in range(1, 700)] + [(1, i) for i in range(2, 900)]
    extra = rng.integers(0, n, size=(6000, 2))
    ei = sym_edge_index(pairs + [tuple(p) for p in extra.tolist()], n)
    _check_paper(ei, n, "hubs-cta")
    n = 20000
    pairs = [(0, i) for i in range(1, 17000)] + [(1, i) for i in range(2, 9000)]
    extra = rng.integers(0, n, size=(30000, 2))
    ei = sym_edge_index(pairs + [tuple(p) for p in extra.tolist()], n)
    from dcr import bfc
    from oracle.paper_flavour import adjacency_sets, bfc_edge_fields
    csr = _csr(ei, n)
    out = bfc.paper_flavour(csr)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    adj = adjacency_sets(ei, n)
    pick = np.concatenate([np.flatnonzero((es == 0) & (ed == 1)), rng.choice(es.size, 60, replace=False)])
    got = {k: out[k].cpu().numpy() for k in ("tri", "sq_i", "sq_j", "gamma", "bfc")}
    for e in pick.tolist():
        f = bfc_edge_fields(adj, int(es[e]), int(ed[e]))
        assert (got["tri"][e], got["sq_i"][e], got["sq_j"][e], got["gamma"][e]) == f[2:6], e
        assert got["bfc"][e] == float(f[6])


def _many_distinct_matches(n_k, n_m, per_m):
    """Edge (0,1): 0 has n_k pure neighbours, 1 has n_m; every pure neighbour of 1 is adjacent to per_m DISTINCT pure
    neighbours of 0 -> #squares at 0 is n_m*per_m distinct vertices although the stream is short."""
    a, b = 0, 1
    ks = list(range(2, 2 + n_k))
    ms = list(range(2 + n_k, 2 + n_k + n_m))
    pairs = [(a, b)] + [(a, k) for k in ks] + [(b, m) for m in ms]
    for q, m in enumerate(ms):
        pairs += [(m, ks[q * per_m + r]) for r in range(per_m)]
    n = 2 + n_k + n_m
    return sym_edge_index(pairs, n), n


def test_paper_flavour_match_hash_overflow_paths(paper_mode):
    # 500 distinct matched neighbours: more than one warp's match hash holds -> retried by the whole CTA;
    # 2400: more than the CTA-wide hash holds -> global overflow list -> CTA-team kernel
    for n_k, n_m, per_m in ((600, 10, 50), (2600, 40, 60)):
        ei, n = _many_distinct_matches(n_k, n_m, per_m)
        got = _check_paper(ei, n, f"distinct{n_m * per_m}")
        e01 = np.flatnonzero((got["edges"][:, 0] == 0) & (got["edges"][:, 1] == 1))[0]
        assert max(got["sq_i"][e01], got["sq_j"][e01]) == n_m * per_m


def test_paper_flavour_split_hub_hub_edge(paper_mode):
    """Two hubs with ~3000 neighbours each (500 shared: triangles are frequent in the stream) over a random background
    of average degree ~20: the stream of edge (0,1) exceeds SPLIT_STREAM, so it is cut into parts processed by
    different CTAs and merged through the global match hash."""
    from oracle.paper_flavour import adjacency_sets, bfc_edge_fields
    rng = np.random.default_rng(11)
    n = 6000
    pairs = [(0, 1)] + [(0, i) for i in range(2, 3002)] + [(1, i) for i in range(2502, 5502)]
    extra = rng.integers(2, n, size=(60000, 2))
    ei = sym_edge_index(pairs + [tuple(q) for q in extra.tolist()], n)
    from dcr import bfc
    csr = _csr(ei, n)
    out = bfc.paper_flavour(csr)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    adj = adjacency_sets(ei, n)
    assert sum(len(adj[m]) for m in adj[1]) > 49152        # the streamed side of (0,1), whichever it is
    pick = np.concatenate([np.flatnonzero((es == 0) & (ed == 1)), np.flatnonzero(es == 0)[:40],
                           np.flatnonzero(es == 1)[:40], rng.choice(es.size, 80, replace=False)])
    got = {k: out[k].cpu().numpy() for k in ("tri", "sq_i", "sq_j", "gamma", "bfc")}
    for e in pick.tolist():
        f = bfc_edge_fields(adj, int(es[e]), int(ed[e]))
        assert (got["tri"][e], got["sq_i"][e], got["sq_j"][e], got["gamma"][e]) == f[2:6], (e, es[e], ed[e])
        assert got["bfc"][e] == float(f[6])


def test_paper_flavour_named_shapes_vs_oracle(paper_mode):
    from dcr.synth import named_graph
    for name in ("cornell", "wisconsin", "cora"):
        ei, n = named_graph(name)
        _check_paper(ei, n, name)


def test_paper_flavour_strided_shards_reassemble():
    from dcr import bfc
    from dcr.synth import named_graph
    ei, n = named_graph("cora")
    csr = _csr(ei, n)
    full = bfc.paper_flavour(csr)
    E = full["count"]
    for world in (2, 3, 8):
        for key in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
            merged = np.zeros(E, dtype=full[key].cpu().numpy().dtype)
            for r in range(world):
                part = bfc.paper_flavour(csr, rank=r, world=world)
                merged[r::world] = part[key].cpu().numpy()
            assert np.array_equal(merged, full[key].cpu().numpy()), (world, key)


def _cuda_gpu(ei, n):
    import torch
    from dcr import bfc
    csr = _csr(ei, n)
    out = bfc.cuda_flavour(csr)
    C = torch.full((n, n), 7.0, device="cuda")
    bfc.scatter_dense(csr, out["c32"], C)
    return csr, out, C.cpu().numpy()


def _check_cuda(ei, n, tag):
    from oracle.cuda_flavour import bfc_cuda_dense
    csr, out, C = _cuda_gpu(ei, n)
    ref = bfc_cuda_dense(dense_of(ei, n), "compiled")
    assert np.array_equal(C.view(np.uint32), ref["C"].view(np.uint32)), (tag, np.abs(C - ref["C"]).max())
    rows = np.repeat(np.arange(n), np.diff(csr.rowptr.cpu().numpy()))
    cols = csr.colidx.cpu().numpy()
    assert np.array_equal(out["tri"].cpu().numpy(), ref["a2"][rows, cols].astype(np.int32)), tag
    assert np.array_equal(out["sharp"].cpu().numpy(), ref["sharp"][rows, cols].astype(np.int32)), tag
    assert np.array_equal(out["lam"].cpu().numpy(), ref["lam"][rows, cols].astype(np.int32)), tag
    c64 = out["c64"].cpu().numpy()
    assert np.allclose(c64, ref["C"][rows, cols], rtol=1e-6, atol=1e-7)
    return C


def test_cuda_flavour_golden_simulator_values():
    z = golden("cuda_kat.npz")
    for name in (str(s) for s in z["names"]):
        ei, n = z[f"{name}/edge_index"], int(z[f"{name}/n"])
        C = _check_cuda(ei, n, name)
        assert np.abs(C - z[f"{name}/C"]).max() <= 1e-6, name     # simulator (all-fp32) within fp32 noise


@pytest.mark.parametrize("seed", range(6))
def test_cuda_flavour_random_graphs(seed):
    n = 16 + 23 * seed
    _check_cuda(gnp(n, [0.08, 0.15, 0.3][seed % 3], 50 + seed), n, f"gnp{seed}")


def test_cuda_flavour_named_shapes_vs_oracle():
    from dcr.synth import named_graph
    for name in ("cornell", "wisconsin"):
        ei, n = named_graph(name)
        _check_cuda(ei, n, name)


def test_post_delta_golden_and_oracle():
    import torch
    from dcr import bfc
    from oracle.cuda_flavour import post_delta_dense
    z = golden("cuda_kat.npz")
    for name in (str(s) for s in z["names"]):
        ei, n = z[f"{name}/edge_index"], int(z[f"{name}/n"])
        csr = _csr(ei, n)
        tri = bfc.support(csr)
        A = dense_of(ei, n)
        for q in range(int(z[f"{name}/npd"])):
            x, y = (int(v) for v in z[f"{name}/pd{q}/xy"])
            xn, yn = z[f"{name}/pd{q}/xn"], z[f"{name}/pd{q}/yn"]
            D = torch.zeros(len(xn), len(yn), device="cuda")
            bfc.post_delta(csr, tri, x, y, torch.from_numpy(xn.astype(np.int32)).cuda(),
                           torch.from_numpy(yn.astype(np.int32)).cuda(), D)
            ref = post_delta_dense(A, x, y, xn.tolist(), yn.tolist(), "compiled")
            got = D.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (name, q, np.abs(got - ref).max())
            assert np.abs(got - z[f"{name}/pd{q}/D"]).max() <= 1e-6


def test_post_delta_arbitrary_lists_and_non_edges():
    # generic lists (not N(x)+[x]) and (x,y) that is not an edge, incl. the (0,0) fallback of the SDRF loop
    import torch
    from dcr import bfc
    from oracle.cuda_flavour import post_delta_dense
    rng = np.random.default_rng(11)
    for seed in range(6):
        n = 18 + 4 * seed
        ei = gnp(n, 0.22, 200 + seed)
        csr = _csr(ei, n)
        tri = bfc.support(csr)
        A = dense_of(ei, n)
        for _ in range(4):
            x, y = (int(v) for v in rng.integers(0, n, 2))
            if _ == 0:
                x = y = 0
            xn = rng.permutation(n)[: rng.integers(1, n)].astype(np.int32)
            yn = rng.permutation(n)[: rng.integers(1, n)].astype(np.int32)
            D = torch.zeros(len(xn), len(yn), device="cuda")
            bfc.post_delta(csr, tri, x, y, torch.from_numpy(xn).cuda(), torch.from_numpy(yn).cuda(), D)
            ref = post_delta_dense(A, x, y, xn.tolist(), yn.tolist(), "compiled")
            got = D.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (seed, x, y, np.abs(got - ref).max())


def test_dense_roundtrip_and_validation():
    import torch
    from dcr import bfc
    n = 300
    ei = gnp(n, 0.05, 9)
    A = torch.from_numpy(dense_of(ei, n)).cuda()
    csr = bfc.DeviceCSR.from_dense(A)
    from dcr import graph
    rowptr, col = graph.undirected_csr(ei, n)
    assert np.array_equal(csr.rowptr.cpu().numpy(), rowptr)
    assert np.array_equal(csr.colidx.cpu().numpy(), col)
    B = A.clone()
    B[3, 5] = 1.0 - B[3, 5]
    with pytest.raises(NotImplementedError):
        bfc.DeviceCSR.from_dense(B)
    B = A.clone()
    B[7, 7] = 1.0
    with pytest.raises(NotImplementedError):
        bfc.DeviceCSR.from_dense(B)


def test_full_size_squirrel_shape_every_edge_against_c_oracle(paper_mode):
    """Config-4 size: all 198,000 edges against the plain-C restatement of bfc_naive.py, both membership modes."""
    import os
    from dcr import bfc, graph
    from dcr.synth import named_graph
    from oracle.c_port import bfc_paper_c
    ei, n = named_graph("squirrel")
    rowptr, col = graph.undirected_csr(ei, n)
    csr = bfc.DeviceCSR.from_host(rowptr, col)
    out = bfc.paper_flavour(csr)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 4
    ref = bfc_paper_c(rowptr, col, es, ed, threads=threads)
    for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
        got = out[k].cpu().numpy()
        assert np.array_equal(got, ref[k]), (k, int((got != ref[k]).sum()))


def test_global_table_class_every_edge_against_c_oracle(paper_mode):
    """The graph of the CTA-team test (a hub of degree ~17000: hashed mode takes the global-table kernel, class X): every
    edge against the C oracle, not a sample."""
    import os
    from dcr import bfc, graph
    from oracle.c_port import bfc_paper_c
    rng = np.random.default_rng(5)
    n = 20000
    pairs = [(0, i) for i in range(1, 17000)] + [(1, i) for i in range(2, 9000)]
    extra = rng.integers(0, n, size=(30000, 2))
    ei = sym_edge_index(pairs + [tuple(p) for p in extra.tolist()], n)
    rowptr, col = graph.undirected_csr(ei, n)
    csr = bfc.DeviceCSR.from_host(rowptr, col)
    out = bfc.paper_flavour(csr)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 4
    ref = bfc_paper_c(rowptr, col, es, ed, threads=threads)
    for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
        got = out[k].cpu().numpy()
        assert np.array_equal(got, ref[k]), (k, int((got != ref[k]).sum()))


def test_paper_flavour_golden_integer_fields(paper_mode):
    """deg, #triangles, #squares_1, #squares_2, gamma read from the locals of the UNMODIFIED bfc_naive.bfc_edge
    (tests/golden/generate_golden.py::gen_paper_ints) — the integer fields pinned by the reference itself, not only
    through the oracle."""
    z = golden("paper_ints_kat.npz")
    for name in (str(s) for s in z["names"]):
        ei, n = z[f"{name}/edge_index"], int(z[f"{name}/n"])
        if ei.shape[1] == 0:
            continue
        got = _paper_gpu(ei, n)
        assert np.array_equal(got["edges"], z[f"{name}/edges"]), name
        ints = z[f"{name}/ints"]
        assert np.array_equal(got["tri"], ints[:, 2]), name
        assert np.array_equal(got["sq_i"], ints[:, 3]), name
        assert np.array_equal(got["sq_j"], ints[:, 4]), name
        assert np.array_equal(got["gamma"], ints[:, 5]), name
        assert np.array_equal(got["bfc"], z[f"{name}/bfc"]), name


def test_full_size_properties_squirrel_shape():
    """Config-4 size: size-independent properties + oracle spot checks (the dense oracle is too slow here)."""
    from dcr import bfc
    from dcr.synth import named_graph
    from oracle.paper_flavour import adjacency_sets, bfc_edge_fields
    ei, n = named_graph("squirrel")
    csr = _csr(ei, n)
    out = bfc.paper_flavour(csr)
    tri = out["tri"].cpu().numpy().astype(np.int64)
    sq_i, sq_j = out["sq_i"].cpu().numpy(), out["sq_j"].cpu().numpy()
    gamma = out["gamma"].cpu().numpy()
    # every triangle is seen from its three edges; cross-check with the support kernel of the other flavour
    supp = bfc.support(csr).cpu().numpy().astype(np.int64)
    assert tri.sum() % 3 == 0 and supp.sum() == 2 * tri.sum()
    # the bipartite square graph between the pure neighbourhoods is empty on one side iff on the other
    assert np.array_equal(sq_i > 0, sq_j > 0)
    assert np.array_equal(gamma > 0, sq_i > 0)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    adj = adjacency_sets(ei, n)
    rng = np.random.default_rng(0)
    bfcv = out["bfc"].cpu().numpy()
    for e in rng.choice(es.size, 200, replace=False).tolist():
        f = bfc_edge_fields(adj, int(es[e]), int(ed[e]))
        assert (tri[e], sq_i[e], sq_j[e], gamma[e]) == f[2:6], e
        assert bfcv[e] == float(f[6])


def test_sharded_path_single_process_matches_full():
    """The NCCL-route code path (shared result block, gather buffer, unshard kernel) run as W emulated ranks on one GPU."""
    import torch
    from dcr import bfc
    from dcr.dist import chunk_size
    from dcr.synth import named_graph
    ei, n = named_graph("cora")
    csr = _csr(ei, n)
    full = bfc.paper_flavour(csr)
    E = full["count"]
    for world in (2, 8):
        chunk = chunk_size(E, world)
        gathered = torch.zeros(world * chunk * 24, dtype=torch.uint8, device="cuda")
        for r in range(world):
            ws = bfc.PaperWorkspace(csr, bfc.shard_count(E, r, world), chunk=chunk)
            bfc.paper_flavour(csr, rank=r, world=world, ws=ws)
            gathered[r * chunk * 24:(r + 1) * chunk * 24] = ws.block
        out = bfc.unshard(gathered, world, chunk, E, out=bfc.unshard_outputs(E, "cuda"))
        for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
            assert torch.equal(out[k], full[k]), (world, k)


def test_contiguous_ranges_through_the_sharded_entry_point(paper_mode):
    """dcr_bfc_paper_sharded over work-balanced contiguous ranges (the peer-memory route with the peers left out: W
    emulated ranks, one after the other, each writing its range at the edges' own positions of ONE result buffer) ==
    the single pass; also an empty range and the ShardedPaperBFC wrapper at world size 1."""
    import torch
    from dcr import bfc, dist as ddist
    from dcr import lib as L
    from dcr.synth import named_graph
    for name in ("cora", "squirrel"):
        ei, n = named_graph(name)
        csr = _csr(ei, n)
        full = bfc.paper_flavour(csr)
        esrc, edst, _ = csr.undirected_edges()
        E = full["count"]
        cost = ddist.edge_cost(csr, esrc, edst)
        lib = L.load()
        for world in (3, 8):
            b = ddist.balanced_bounds(torch.cumsum(cost, 0), world)
            assert b[0] == 0 and b[-1] == E
            work = [int(cost[b[r]:b[r + 1]].sum()) for r in range(world)]
            assert max(work) <= sum(work) / world + int(cost.max())
            comm = ddist.PeerComm(E, 0, 1)
            nbytes = int(lib.dcr_bfc_paper_scratch_bytes(n, csr.max_degree, E))
            scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            for r in list(range(world)) + [0]:                  # (+ a repeated range: the buffer is simply overwritten)
                L.check(lib.dcr_bfc_paper_sharded(csr.rowptr.data_ptr(), csr.colidx.data_ptr(), n, csr.max_degree,
                                                  esrc.data_ptr(), edst.data_ptr(), b[r], b[r + 1] - b[r], comm.handle,
                                                  scratch.data_ptr(), nbytes, 0, 0, L.current_stream()), "sharded")
            L.check(lib.dcr_bfc_paper_sharded(csr.rowptr.data_ptr(), csr.colidx.data_ptr(), n, csr.max_degree,
                                              esrc.data_ptr(), edst.data_ptr(), b[1], 0, comm.handle,
                                              scratch.data_ptr(), nbytes, 0, 0, L.current_stream()), "sharded (empty)")
            torch.cuda.synchronize()
            for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
                assert torch.equal(comm.views[k], full[k]), (name, world, k)
            assert comm.error() == 0
            comm.close()
        sh = ddist.ShardedPaperBFC(csr)
        assert sh.mode == "peer" and (sh.lo, sh.hi) == (0, E)
        out = sh.run()
        for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
            assert torch.equal(out[k], full[k]), (name, k)
        sh.check()
        sh.close()


def test_host_end_to_end_pass_single_rank():
    """HostShardedPaperBFC (pinned host CSR in, host result block out) at world size 1."""
    import torch
    from dcr import bfc, dist as ddist, graph
    from dcr.synth import named_graph
    ei, n = named_graph("cora")
    rowptr, col = graph.undirected_csr(ei, n)
    m = ei[0] < ei[1]
    esrc, edst = ei[0][m].astype(np.int32), ei[1][m].astype(np.int32)
    csr = bfc.DeviceCSR.from_host(rowptr, col)
    full = bfc.paper_flavour(csr)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    hs = ddist.HostShardedPaperBFC(n, col.size, esrc.size, csr.max_degree)
    lo, hi = hs.run(pin(rowptr.astype(np.int32)), pin(col), pin(esrc), pin(edst))
    torch.cuda.synchronize()
    assert (lo, hi) == (0, esrc.size)
    hv = hs.host_views()
    for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
        assert np.array_equal(hv[k].numpy(), full[k].cpu().numpy()), k
    # the CSR alone: the undirected edge list (row < col entries, CSR order) is derived on the device
    for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
        hv[k].zero_()
    h2d_full = hs.bytes_per_pass()[0]
    hs.d_esrc.fill_(-1)
    hs.d_edst.fill_(-1)
    hs.run(pin(rowptr.astype(np.int32)), pin(col))
    torch.cuda.synchronize()
    assert np.array_equal(hs.d_esrc.cpu().numpy(), esrc) and np.array_equal(hs.d_edst.cpu().numpy(), edst)
    for k in ("tri", "sq_i", "sq_j", "gamma", "bfc"):
        assert np.array_equal(hv[k].numpy(), full[k].cpu().numpy()), k
    assert hs.bytes_per_pass()[0] == h2d_full - 8 * esrc.size
    hs.close()


def test_two_gpus_peer_memory_exchange():
    """The real thing when the box has two GPUs: two ranks under torchrun, peer-memory route and NCCL route, device and
    host forms, every rank's full arrays compared with the single-GPU pass (tests/multi_gpu_worker.py)."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", os.path.join(here, "multi_gpu_worker.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "multi_gpu_worker ok" in r.stdout


def test_tensor_core_support_matches_sparse_support():
    """Dense-regime A·A on tcgen05 (int8, TMA, TMEM) with the fused edge-extraction epilogue == sorted-list supports."""
    import torch
    from dcr import bfc
    from dcr.synth import chung_lu_graph
    for n, e, seed in ((100, 600, 1), (257, 3000, 2), (1000, 30000, 3), (5201, 198000, 5201)):
        ei = chung_lu_graph(n, e, 0.7, 0.3, seed)
        csr = _csr(ei, n)
        want = bfc.support(csr)
        got = bfc.support_tc(csr)
        torch.cuda.synchronize()
        assert torch.equal(got, want), (n, int((got != want).sum()))
    # edge cases: empty rows / isolated nodes, a clique (every tile entry on an edge)
    csr = _csr(sym_edge_index([(0, i) for i in range(1, 40)], 300), 300)
    assert torch.equal(bfc.support_tc(csr), bfc.support(csr))
    csr = _csr(sym_edge_index([(i, j) for i in range(140) for j in range(i + 1, 140)], 140), 140)
    assert torch.equal(bfc.support_tc(csr), bfc.support(csr))


def test_tensor_core_cuda_flavour_matches_sparse_route_and_oracle():
    import torch
    from dcr import bfc
    from dcr.synth import chung_lu_graph
    from oracle.cuda_flavour import bfc_cuda_dense
    for n, e, seed in ((60, 300, 7), (300, 4000, 8), (5201, 198000, 5201)):
        ei = chung_lu_graph(n, e, 0.7, 0.3, seed)
        csr = _csr(ei, n)
        a = bfc.cuda_flavour(csr)
        b = bfc.cuda_flavour_tc(csr)
        torch.cuda.synchronize()
        for k in ("tri", "sharp", "lam"):
            assert torch.equal(a[k], b[k]), (n, k)
        assert torch.equal(a["c32"].view(torch.int32), b["c32"].view(torch.int32)), n     # fp32 bit patterns
        assert torch.equal(a["c64"], b["c64"]), n
        if n <= 300:
            ref = bfc_cuda_dense(dense_of(ei, n), "compiled")
            C = torch.zeros(n, n, device="cuda")
            bfc.scatter_dense(csr, b["c32"], C)
            assert np.array_equal(C.cpu().numpy().view(np.uint32), ref["C"].view(np.uint32))


def test_full_size_arxiv_shape_exact_against_c_oracle(paper_mode):
    """Config 5 at full size: every one of the 1,166,243 edges against the plain-C restatement of bfc_naive.py
    (ints bit-exact, fp64 bit-exact), plus the size-independent properties."""
    import os
    from dcr import bfc
    from dcr.synth import named_graph
    from dcr import graph
    from oracle.c_port import bfc_paper_c
    ei, n = named_graph("arxiv")
    rowptr, col = graph.undirected_csr(ei, n)
    csr = bfc.DeviceCSR.from_host(rowptr, col)
    out = bfc.paper_flavour(csr)
    es, ed = out["esrc"].cpu().numpy(), out["edst"].cpu().numpy()
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 4
    ref = bfc_paper_c(rowptr, col, es, ed, threads=threads)
    for k in ("tri", "sq_i", "sq_j", "gamma"):
        got = out[k].cpu().numpy()
        assert np.array_equal(got, ref[k]), (k, int((got != ref[k]).sum()))
    assert np.array_equal(out["bfc"].cpu().numpy(), ref["bfc"])
    tri = out["tri"].cpu().numpy().astype(np.int64)
    supp = bfc.support(csr).cpu().numpy().astype(np.int64)
    assert tri.sum() % 3 == 0 and supp.sum() == 2 * tri.sum()
    assert np.array_equal(out["sq_i"].cpu().numpy() > 0, out["sq_j"].cpu().numpy() > 0)


def test_bench_runs_the_requested_steps_and_dumps_the_outputs(tmp_path):
    """`bench.py --steps K --dump-outputs DIR`: K timed steps, and DIR holds every field of the last one as float64,
    equal to the C oracle on every edge of the workload."""
    import json
    import os
    import subprocess
    import sys
    from conftest import REPO
    from oracle.c_port import bfc_paper_c
    sys.path.insert(0, REPO)
    import bench
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--workload", "cora", "--steps", "2",
                        "--warmup", "0", "--no-dense", "--no-cpu", "--no-sdrf", "--no-clocks",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and len(d["step_ms"]) == 2
    _, _, rowptr, col, esrc, edst = bench.build_graph("cora")
    ref = bfc_paper_c(rowptr, col, esrc, edst)
    assert sorted(os.listdir(tmp_path)) == sorted(f"{k}.npy" for k in ref)
    for k, want in ref.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, want), k


def test_edge_centric_cuda_flavour_matches_per_entry_kernels_and_oracle():
    """dcr_bfc_cuda_edges (one work item per undirected edge, hub-hub edges by a CTA) against the per-entry kernels at
    every size incl. the arxiv shape, and against the dense oracle on small graphs; a single-GPU dcr_comm run of the
    sharded entry point gives the same arrays."""
    import torch
    from dcr import bfc
    from dcr import dist as ddist
    from dcr.synth import named_graph
    from oracle.cuda_flavour import bfc_cuda_dense
    cases = [(gnp(60, 0.2, 3), 60), toy_graphs()["k5"], toy_graphs()["star5"]]
    cases += [named_graph(nm) for nm in ("cornell", "cora", "squirrel", "arxiv")]
    hub = sym_edge_index([(0, i) for i in range(1, 1500)] + [(1, i) for i in range(2, 1400)] +
                         [(i, i + 1) for i in range(2, 1300)], 1500)          # one edge with a 1398-long shorter row
    cases.append((hub, 1500))
    for ei, n in cases:
        csr = _csr(ei, n)
        per_entry = bfc.cuda_flavour(csr, tri=bfc.support(csr))      # tri given: the per-entry kernels
        esrc, edst, entry = csr.undirected_edges()
        got = bfc.cuda_flavour_edges(csr)
        for k in ("tri", "sharp", "lam"):
            assert torch.equal(got[k], per_entry[k][entry]), (n, k)
        assert torch.equal(got["c64"].view(torch.int64), per_entry["c64"][entry].view(torch.int64)), n
        assert torch.equal(got["c32"].view(torch.int32), per_entry["c32"][entry].view(torch.int32)), n
        if n <= 200:
            C = bfc_cuda_dense(dense_of(ei, n))["C"]
            want = C[esrc.cpu().numpy(), edst.cpu().numpy()]
            assert np.array_equal(got["c32"].cpu().numpy().view(np.uint32), want.view(np.uint32)), n
        # ranges: supports of everything first, then the closing pass in two halves
        e = int(esrc.numel())
        out = bfc.cuda_flavour_edges(csr, phases=1)
        bfc.cuda_flavour_edges(csr, 0, e // 2, phases=2, out=out)
        bfc.cuda_flavour_edges(csr, e // 2, e - e // 2, phases=2, out=out)
        assert torch.equal(out["c32"].view(torch.int32), got["c32"].view(torch.int32)), n
        sc = ddist.ShardedCudaBFC(csr)
        v = sc.run()
        torch.cuda.synchronize()
        assert torch.equal(v["c32"].view(torch.int32), got["c32"].view(torch.int32)) and torch.equal(v["tri"], got["tri"])
        assert torch.equal(v["sharp"], got["sharp"]) and torch.equal(v["lam"], got["lam"])
        sc.close()
