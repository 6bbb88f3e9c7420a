"""Rate of caller edits on the device-resident SDRF state (``dcr_sdrf_edit``, ``dcr.dynamic.DynamicCurvature``,
DESIGN §4.10) against one fresh full curvature pass of the same flavour on the same graph.

Workloads (every batch is valid: ``m`` adds of random pairs, then the removes of the same pairs in the same order,
so the graph ends where it started and every batch does the same work):
  random     both endpoints uniform;
  hub        one endpoint the highest-degree node, the other uniform (a paper-flavour toggle at a hub dirties every
             edge between the hub's neighbours and the other endpoint's);
on the cora shape in every loop mode and on the arxiv shape for ``'bfc'`` and ``'bfc_paper'``.

Edit rate: CUDA events around the ``dcr_sdrf_edit`` launch of one batch, median over the repetitions after one warm-up
batch.  Full pass: CUDA events around ``bfc.cuda_flavour`` (supports + the edge-centric cuda-flavour kernels) or
``bfc.paper_flavour`` on the CSR of the same graph, median after one warm-up.  ``break_even_edits`` = full-pass time
over time per edit: the number of edits per curvature query up to which the incremental route is the faster one.

    python profiles/sdrf_edit_bench.py --out DIR [--reps 5] [--batch 256] [--hub-batch 16]
        # writes DIR/sdrf_edit_bench.json (rewritten after every workload)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(REPO, "discrete-curvature-rewiring_b200"), REPO, os.path.join(REPO, "profiles")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from sdrf_batch_bench import gpu_identity  # noqa: E402

MODES = {"bfc": ("bfc", True), "bfc_directed": ("bfc", False), "1d": ("1d", True), "augmented": ("augmented", True),
         "haantjes": ("haantjes", True), "bfc_paper": ("bfc_paper", True)}


def batches(ei, n, directed, kind, m, count, seed):
    """``count`` batches of ``m`` adds of fresh pairs followed by their removes (device tensors)."""
    import torch
    rng = np.random.default_rng(seed)
    deg = np.bincount(ei[0], minlength=n) + (0 if directed else np.bincount(ei[1], minlength=n))
    hub = int(np.argmax(deg))
    present = set(zip(ei[0].tolist(), ei[1].tolist()))
    out = []
    for _ in range(count):
        pairs = []
        while len(pairs) < m:
            u = hub if kind == "hub" else int(rng.integers(n))
            v = int(rng.integers(n))
            if u == v or (u, v) in present or (v, u) in present or (u, v) in pairs or (v, u) in pairs:
                continue
            pairs.append((u, v))
        p = np.array(pairs, dtype=np.int32)
        e = np.concatenate([np.column_stack([np.ones(m, np.int32), p]), np.column_stack([np.zeros(m, np.int32), p])])
        out.append(torch.from_numpy(e).cuda())
    return out, int(deg[hub])


def edit_rate(torch, dc, edits):
    """Median seconds of one ``dcr_sdrf_edit`` launch over the batches (the first one warms up)."""
    from dcr import lib as L
    st = dc._state
    res = torch.zeros(8, dtype=torch.int32, device="cuda")
    times = []
    for e in edits:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(st.lib.dcr_sdrf_edit(st.handle, e.data_ptr(), int(e.shape[0]), res.data_ptr(), L.current_stream()),
                "dcr_sdrf_edit")
        e1.record()
        torch.cuda.synchronize()
        r = res.cpu().tolist()
        assert r[0] == L.SDRF_OK and r[1] == e.shape[0], r
        times.append(e0.elapsed_time(e1) * 1e-3)
    return statistics.median(times[1:]), times[1:]


def full_pass(torch, ei, n, curv_type, directed, reps):
    """Name and median seconds of one fresh full pass of the flavour on the graph (for the classical types the support
    pass: a classical value needs nothing else but the degrees)."""
    from dcr import bfc
    from dcr import graph as G
    e = ei[:, ei[0] != ei[1]]
    if curv_type in ("1d", "augmented", "haantjes"):
        csr = bfc.DeviceCSR.from_host(*G.undirected_csr(e, n))
        run = lambda: bfc.support(csr)                              # noqa: E731
        name = "dcr_bfc_support"
    elif directed:
        d = bfc.DirectedCSR.from_edge_index(e, n)
        run = lambda: bfc.cuda_flavour_directed(d, want_fields=False)   # noqa: E731
        name = "dcr_bfc_cuda_flavour_directed"
    elif curv_type == "bfc":
        csr = bfc.DeviceCSR.from_host(*G.undirected_csr(e, n))
        run = lambda: bfc.cuda_flavour(csr, want_fields=False)      # noqa: E731
        name = "cuda_flavour (edge-centric)"
    else:
        csr = bfc.DeviceCSR.from_host(*G.undirected_csr(e, n))
        ws = bfc.PaperWorkspace(csr, int(csr.nnz // 2))
        run = lambda: bfc.paper_flavour(csr, ws=ws)                 # noqa: E731
        name = "dcr_bfc_paper"
    times = []
    for _ in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return name, statistics.median(times[1:])


def workload(torch, shape, mode, kind, batch, reps):
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import named_graph
    ei, n = named_graph(shape)
    curv_type, und = MODES[mode]
    if not und:                                   # the directed view of the shape: one direction of every pair
        ei = ei[:, ei[0] < ei[1]]
    edits, hub_deg = batches(ei, n, not und, kind, batch, reps + 1, 7)
    with DynamicCurvature(ei, n, curv_type, und, capacity=batch * (reps + 1)) as dc:
        s, all_s = edit_rate(torch, dc, edits)
    per_edit = s / (2 * batch)
    name, full = full_pass(torch, ei, n, curv_type, not und, reps)
    return {"shape": shape, "mode": mode, "edits": kind, "n": n, "columns": int(ei.shape[1]), "hub_degree": hub_deg,
            "edits_per_batch": 2 * batch, "s_per_batch_median": s, "s_per_batch_all": all_s,
            "edits_per_s": 1.0 / per_edit, "us_per_edit": per_edit * 1e6, "full_pass": name, "full_pass_ms": full * 1e3,
            "break_even_edits": full / per_edit}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256, help="adds per batch (each batch also removes them)")
    ap.add_argument("--hub-batch", type=int, default=16, help="adds per batch of the hub workloads")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "sdrf_edit_bench measures on the GPU; there is no CPU fallback"
    import __graft_entry__
    __graft_entry__.build()
    rec = {"gpu": gpu_identity(torch), "batch_adds": args.batch, "hub_batch_adds": args.hub_batch, "reps": args.reps,
           "results": []}
    plan = [("cora", m, k) for m in MODES for k in ("random", "hub")]
    plan += [("arxiv", m, k) for m in ("bfc", "bfc_paper") for k in ("random", "hub")]
    os.makedirs(args.out, exist_ok=True)
    for shape, mode, kind in plan:
        print(f"{shape:6s} {mode:13s} {kind:6s} ...", flush=True)
        r = workload(torch, shape, mode, kind, args.hub_batch if kind == "hub" else args.batch, args.reps)
        rec["results"].append(r)
        print(f"{shape:6s} {mode:13s} {kind:6s} {r['edits_per_s']:12.0f} edits/s  {r['us_per_edit']:9.2f} us/edit  "
              f"full pass {r['full_pass_ms']:8.3f} ms  break-even {r['break_even_edits']:10.1f} edits", flush=True)
        with open(os.path.join(args.out, "sdrf_edit_bench.json"), "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
