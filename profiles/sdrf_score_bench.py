"""Candidate scoring of many pairs on a device-resident SDRF state (``dcr_sdrf_score``, DESIGN §4.12).

Workloads, every time the median of ``--reps`` windows between CUDA events (each shape warmed up first):
  cora shape, every loop mode: Q = 1 (the first edge), Q = 148 random valid pairs (edges in both orientations) and Q =
      every negatively curved edge, each orientation once;
  arxiv shape, ``'bfc'`` and ``'bfc_paper'``: Q = 148 random edges and Q = 148 edges at the 8 highest-degree nodes,
      oriented hub first (the hub's row has the most candidates).
Per workload three timings:
  batch   ``SdrfState.score`` of all Q pairs: the sizes launch, one read of the totals, the output allocations and the
          scoring launch (what ``DynamicCurvature.improvements`` / ``best_additions`` pay on the device);
  kernel  the ``dcr_sdrf_score`` launch alone, outputs allocated before the window;
  single  Q calls of ``SdrfState.score`` with one pair each.
Rates: queries/s and cells/s (cells = sum of n_i * n_j).  ``batch_equals_single`` compares the cells of the batch with
those of the single calls bit for bit.  On the cora shape, each mode also times ``pending_improvements`` (the read of
the loop's own improvements after a NEED_HOST stop) against a query at the same pair, whose values must be equal.

    python profiles/sdrf_score_bench.py --out DIR [--reps 5]     # writes DIR/sdrf_score_bench_<card>.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(REPO, "discrete-curvature-rewiring_b200"), REPO, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from sdrf_batch_bench import gpu_identity  # noqa: E402

MODES = [("bfc", True), ("bfc", False), ("1d", True), ("augmented", True), ("haantjes", True), ("bfc_paper", True)]
MAX_CELLS = 1 << 31


def _timed(torch, fn, reps):
    """median / min seconds of ``fn()`` between CUDA events over ``reps`` windows"""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / 1e3)
    return {"s_median": statistics.median(out), "s_min": min(out)}


def measure(torch, dc, name, pairs, reps, singles=True):
    from dcr import lib as L
    if len(pairs) == 0:                                   # (e.g. no negatively curved edge in this mode)
        print(json.dumps({"workload": name, "q": 0, "skipped": "no queries"}), flush=True)
        return {"workload": name, "queries": 0, "skipped": "no queries"}
    st = dc._state
    p = torch.from_numpy(np.ascontiguousarray(pairs, dtype=np.int32)).to(st.device)
    q = int(p.shape[0])
    res = st.score(p, MAX_CELLS)                                           # warm-up, and the buffers of `kernel`
    cells = int(res["cell_offsets"][-1])
    nbytes = int(st.lib.dcr_sdrf_score_workspace_bytes(st.handle, q))
    ws = torch.empty(max(nbytes // 4, 1), dtype=torch.int32, device=st.device)

    def kernel():
        L.check(st.lib.dcr_sdrf_score(st.handle, p.data_ptr(), q, res["cell_offsets"].data_ptr(),
                                      res["cand_offsets"].data_ptr(), res["cand"].data_ptr(), res["imp"].data_ptr(),
                                      res["best"].data_ptr(), ws.data_ptr(), nbytes, L.current_stream()), "score")

    out = {"workload": name, "queries": q, "cells": cells, "output_bytes": 8 * cells + 4 * int(res["cand_offsets"][-1]),
           "batch": _timed(torch, lambda: st.score(p, MAX_CELLS), reps), "kernel": _timed(torch, kernel, reps)}
    if singles:
        one = [p[t:t + 1] for t in range(q)]
        out["single"] = _timed(torch, lambda: [st.score(x, MAX_CELLS) for x in one], max(1, reps // 2))
        got = st.score(p, MAX_CELLS)["imp"].cpu().numpy().view(np.int64)
        want = np.concatenate([st.score(x, MAX_CELLS)["imp"].cpu().numpy() for x in one]).view(np.int64)
        out["batch_equals_single"] = bool(np.array_equal(got, want))
    for k in ("batch", "kernel", "single"):
        if k in out:
            s = out[k]["s_median"]
            out[k]["queries_per_s"] = q / s
            out[k]["cells_per_s"] = cells / s
    print(json.dumps({"workload": name, "q": q, "cells": cells, "batch_s": round(out["batch"]["s_median"], 6),
                      "kernel_s": round(out["kernel"]["s_median"], 6),
                      "single_s": round(out["single"]["s_median"], 6) if singles else None,
                      "equal": out.get("batch_equals_single")}), flush=True)
    return out


def pending_vs_query(torch, dc, reps):
    """one stochastic iteration with guard = 1 on a fork: pending_improvements against a query at its (x, y)"""
    from dcr import lib as L
    (f,) = dc.fork()
    with f:
        st = f._state
        u = torch.full((1,), 0.5, dtype=torch.float64, device=st.device)
        res, _ = st.run(1, True, 0.5, 3.0, u, guard=1.0)
        if res["status"] != L.SDRF_NEED_HOST:
            return {"skipped": f"status {res['status']}"}
        n, x, y = res["pending_n"], res["pending_x"], res["pending_y"]
        want = st.pending_improvements(n)
        got = f.improvements([(x, y)], max_cells=MAX_CELLS)[0][1]
        p = torch.tensor([[x, y]], dtype=torch.int32, device=st.device)
        return {"pair": [x, y], "candidates": n, "equal": bool(np.array_equal(got.view(np.int64), want.view(np.int64))),
                "pending_improvements": _timed(torch, lambda: st.pending_improvements(n), reps),
                "score_one_query": _timed(torch, lambda: st.score(p, MAX_CELLS), reps)}


def edges_of(dc):
    ei = dc.edge_index()
    return ei[:, ei[0] != ei[1]]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for sdrf_score_bench_<card>.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-arxiv", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sdrf_score_bench.py needs a CUDA device")
    from dcr.dynamic import DynamicCurvature
    from dcr.synth import named_graph
    record = {"gpu": gpu_identity(torch), "reps": args.reps,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "cora": [], "arxiv": []}
    rng = np.random.default_rng(0)
    cei, cn = named_graph("cora")
    for curv_type, und in MODES:
        ei = cei if und else cei[:, cei[0] < cei[1]]
        with DynamicCurvature(ei, cn, curv_type, und, capacity=16) as dc:
            mode = curv_type if und else "bfc_directed"
            e = edges_of(dc)
            sel = e[:, rng.integers(e.shape[1], size=148)]
            flip = rng.random(148) < 0.5
            sel[:, flip] = sel[::-1, flip]
            neg = e[:, dc.curvature()[dc.edge_index()[0] != dc.edge_index()[1]] < 0]
            if und:
                neg = neg[:, neg[0] < neg[1]]
            rows = [measure(torch, dc, f"cora {mode} Q=1", e[:, :1].T, args.reps),
                    measure(torch, dc, f"cora {mode} Q=148", sel.T, args.reps),
                    measure(torch, dc, f"cora {mode} negative edges", neg.T, args.reps)]
            record["cora"].append({"mode": mode, "rows": rows, "pending": pending_vs_query(torch, dc, args.reps)})
    if not args.skip_arxiv:
        aei, an = named_graph("arxiv")
        for curv_type in ("bfc", "bfc_paper"):
            try:
                dc = DynamicCurvature(aei, an, curv_type, True, capacity=16)
            except Exception as ex:                                    # the record says why a mode is missing
                record["arxiv"].append({"mode": curv_type, "error": repr(ex)})
                continue
            with dc:
                e = edges_of(dc)
                deg = np.bincount(e[0], minlength=an)
                hubs = np.argsort(-deg)[:8]
                at_hub = e[:, np.isin(e[0], hubs)]
                rows = [measure(torch, dc, f"arxiv {curv_type} random edges", e[:, rng.integers(e.shape[1], size=148)].T,
                                args.reps),
                        measure(torch, dc, f"arxiv {curv_type} hub edges", at_hub[:, rng.integers(at_hub.shape[1], size=148)].T,
                                args.reps)]
                record["arxiv"].append({"mode": curv_type, "rows": rows, "max_degree": int(deg.max())})
    os.makedirs(args.out, exist_ok=True)
    card = torch.cuda.get_device_name().split()[-1].lower()          # "NVIDIA B200" -> b200
    path = os.path.join(args.out, f"sdrf_score_bench_{card}.json")
    with open(path, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"written": path}))


if __name__ == "__main__":
    main()
