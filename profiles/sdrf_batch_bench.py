"""Batched SDRF against sequential runs: B independent rewiring loops as B ``SdrfState.run`` launches (one CTA each, one
after the other) versus one ``dcr_sdrf_run_batch`` launch (B CTAs side by side).

Workloads: the cora shape (1000 iterations, tau 163, bound 0.95) for B in {1, 16, 64, 148, 296} with seeds 0..B-1 —
148 is one CTA per SM of a B200, 296 two waves — and the ``redo_rewiring`` case of the reference's
``experiment/save_models.py`` (100 seeds of the wisconsin shape with its ``utils/hyperparams.py`` values).

Per workload and repetition, both paths are timed in the same process, alternated, after a warm-up:
  device   CUDA events around the launches only (states are built before the window; the window ends in a synchronise;
           guard = 0, so every run finishes in its first launch and both paths do the same work);
  e2e      host clock around ``sdrf.sdrf`` per run versus one ``sdrf.sdrf_batch`` (set-up + loop + export, default guard).
Every run's log of the batched launch must equal its sequential log, and the e2e outputs must agree.

    python profiles/sdrf_batch_bench.py --out DIR [--reps 3]      # writes DIR/sdrf_batch_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(REPO, "discrete-curvature-rewiring_b200"), REPO):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def gpu_identity(torch) -> dict:
    out = {"device_name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                           text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip()
    except Exception as e:                              # the record says why the power limit is missing
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def run_workload(torch, name, ei, n, loops, tau, bound, count, reps):
    from dcr import graph, sdrf
    rp, od = graph.networkx_order(ei, n, keep_self_loops=True)
    unis = [np.random.RandomState(s).random_sample(loops) for s in range(count)]
    u_dev = [torch.from_numpy(u).cuda() for u in unis]
    results = torch.zeros((count, 8), dtype=torch.int32, device="cuda")
    workspace = sdrf.batch_workspace(count, "cuda")

    def device_pass(batched):
        states = [sdrf.SdrfState(rp, od, max_additions=loops) for _ in range(count)]
        logs = [torch.empty((loops, 8), dtype=torch.int32, device="cuda") for _ in range(count)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        if batched:
            res = sdrf.run_batch(states, [loops] * count, [bound] * count, [tau] * count, u_dev, [-1] * count, logs,
                                 True, 0.0, results, workspace)
        else:
            res = [s.run(loops, True, bound, tau, u_dev[i], guard=0.0, log=logs[i])[0] for i, s in enumerate(states)]
        e1.record()
        torch.cuda.synchronize()
        for s in states:
            s.close()
        assert all(r["status"] == 0 for r in res), res
        iters = sum(r["iterations_done"] for r in res)
        return e0.elapsed_time(e1) * 1e-3, iters, [lg[: r["iterations_done"]].cpu().numpy() for lg, r in zip(logs, res)]

    def e2e_pass(batched):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if batched:
            outs = sdrf.sdrf_batch(ei, n, loops, True, bound, tau, uniforms=np.stack(unis))
        else:
            outs = [sdrf.sdrf(ei, n, loops, True, bound, tau, uniforms=u) for u in unis]
        torch.cuda.synchronize()
        return time.perf_counter() - t0, outs

    dev = {"sequential": [], "batched": []}
    e2e = {"sequential": [], "batched": []}
    logs_equal = outputs_equal = True
    iters = None
    for rep in range(reps):
        ts, iters, lseq = device_pass(False)
        tb, ib, lbat = device_pass(True)
        assert ib == iters
        logs_equal &= all(np.array_equal(a, b) for a, b in zip(lseq, lbat))
        dev["sequential"].append(ts)
        dev["batched"].append(tb)
        ts, oseq = e2e_pass(False)
        tb, obat = e2e_pass(True)
        outputs_equal &= all(np.array_equal(a, b) for a, b in zip(oseq, obat))
        e2e["sequential"].append(ts)
        e2e["batched"].append(tb)

    def summary(times):
        med = statistics.median(times)
        return {"s_median": med, "s_min": min(times), "s_all": times, "agg_iters_per_s": iters / med}

    out = {"workload": name, "runs": count, "loops": loops, "tau": tau, "removal_bound": bound,
           "total_iterations": iters, "logs_equal": bool(logs_equal), "e2e_outputs_equal": bool(outputs_equal),
           "device": {k: summary(v) for k, v in dev.items()}, "e2e": {k: summary(v) for k, v in e2e.items()}}
    out["device"]["speedup"] = out["device"]["sequential"]["s_median"] / out["device"]["batched"]["s_median"]
    out["e2e"]["speedup"] = out["e2e"]["sequential"]["s_median"] / out["e2e"]["batched"]["s_median"]
    print(json.dumps({"workload": name, "runs": count, "device_speedup": round(out["device"]["speedup"], 2),
                      "batched_agg_iters_per_s": round(out["device"]["batched"]["agg_iters_per_s"]),
                      "logs_equal": out["logs_equal"], "e2e_outputs_equal": out["e2e_outputs_equal"]}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for sdrf_batch_bench.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch-sizes", default="1,16,64,148,296")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sdrf_batch_bench.py needs a CUDA device")
    from dcr.synth import SDRF_PARAMS, named_graph
    record = {"gpu": gpu_identity(torch), "reps": args.reps, "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    cei, cn = named_graph("cora")
    wei, wn = named_graph("wisconsin")
    wloops, wtau, wbound = SDRF_PARAMS["wisconsin"]
    run_workload(torch, "warm-up", cei, cn, 50, 163, 0.95, 4, 1)
    run_workload(torch, "warm-up", wei, wn, 20, wtau, wbound, 4, 1)
    record["results"] = [run_workload(torch, "cora", cei, cn, 1000, 163, 0.95, b, args.reps)
                         for b in (int(v) for v in args.batch_sizes.split(","))]
    record["results"].append(run_workload(torch, "wisconsin redo_rewiring", wei, wn, wloops, wtau, wbound, 100,
                                          args.reps))
    base = next((r for r in record["results"] if r["workload"] == "cora" and r["runs"] == 1), None)
    if base is not None:
        b1 = base["device"]["batched"]["agg_iters_per_s"]
        for r in record["results"]:
            if r["workload"] == "cora":
                r["device"]["agg_rate_over_b1"] = r["device"]["batched"]["agg_iters_per_s"] / b1
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sdrf_batch_bench.json"), "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"written": os.path.join(args.out, "sdrf_batch_bench.json")}))


if __name__ == "__main__":
    main()
