"""Rate of the paper-flavour SDRF loop (``curv_type='bfc_paper'``, DESIGN §4.9) on the device, and of the oracle's Python
loop on the host cores for comparison.

Workloads, all with ``remove_edges=True``:
  cora       the cora shape, 1000 iterations, tau 163, bound 0.95 (the shape and values of the batch benchmark);
  webkb      cornell / texas / wisconsin at the reference's hyper-parameters (``dcr.synth.SDRF_PARAMS``);
  batch      148 seeds of the cora workload in one ``sdrf_batch`` launch (one CTA per SM of a B200);
  oracle     ``paper_sdrf_oracle`` of ``tests/test_gpu_sdrf_paper.py`` (the classical oracle loop with
             ``bfc_edge_fields`` as the curvature) on a prefix of the cora workload, on the host.

Device rates: CUDA events around ``SdrfState.run`` / ``run_batch`` with states built before the window and guard = 0,
so every run finishes in its one launch; the window ends in a synchronise.  Every device log is checked against its
single-run log (batch) and, for the prefix the oracle runs, against the oracle.

    python profiles/sdrf_paper_bench.py --out DIR [--reps 3] [--oracle-iters 20]   # writes DIR/sdrf_paper_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(REPO, "discrete-curvature-rewiring_b200"), REPO, os.path.join(REPO, "profiles")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from sdrf_batch_bench import gpu_identity  # noqa: E402


def single_rate(torch, ei, n, loops, tau, bound, seed, reps):
    """Median iterations/s of one run (one CTA) and its log."""
    from dcr import lib as L
    from dcr import sdrf
    mode, order = sdrf._loop_mode("bfc_paper", True)
    od = order(ei, n)
    u = torch.from_numpy(np.random.RandomState(seed).random_sample(loops)).cuda()
    times, log, iters = [], None, 0
    for _ in range(reps + 1):                          # the first pass warms the module and the shape up
        st = sdrf._new_state(mode, od, loops)
        lg = torch.empty((loops, L.SDRF_LOG_INTS), dtype=torch.int32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        res, _ = st.run(loops, True, bound, tau, u, guard=0.0, log=lg)
        e1.record()
        torch.cuda.synchronize()
        st.close()
        assert res["status"] == L.SDRF_OK, res
        times.append(e0.elapsed_time(e1) * 1e-3)
        iters = res["iterations_done"]
        log = lg[:iters].cpu().numpy()
    med = statistics.median(times[1:])
    return {"iterations": iters, "s_median": med, "s_all": times[1:], "iters_per_s": iters / med}, log


def batch_rate(torch, ei, n, loops, tau, bound, count, reps):
    from dcr import lib as L
    from dcr import sdrf
    mode, order = sdrf._loop_mode("bfc_paper", True)
    od = order(ei, n)
    u = [torch.from_numpy(np.random.RandomState(s).random_sample(loops)).cuda() for s in range(count)]
    results = torch.zeros((count, 8), dtype=torch.int32, device="cuda")
    ws = sdrf.batch_workspace(count, "cuda")
    times, logs, iters = [], None, 0
    for _ in range(reps + 1):
        states = [sdrf._new_state(mode, od, loops) for _ in range(count)]
        lg = [torch.empty((loops, L.SDRF_LOG_INTS), dtype=torch.int32, device="cuda") for _ in range(count)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        res = sdrf.run_batch(states, [loops] * count, [bound] * count, [tau] * count, u, [-1] * count, lg, True, 0.0,
                             results, ws)
        e1.record()
        torch.cuda.synchronize()
        for s in states:
            s.close()
        assert all(r["status"] == L.SDRF_OK for r in res), res
        times.append(e0.elapsed_time(e1) * 1e-3)
        iters = sum(r["iterations_done"] for r in res)
        logs = [g[: r["iterations_done"]].cpu().numpy() for g, r in zip(lg, res)]
    med = statistics.median(times[1:])
    return {"runs": count, "total_iterations": iters, "s_median": med, "s_all": times[1:],
            "agg_iters_per_s": iters / med}, logs


def oracle_rate(ei, n, loops, tau, bound, seed):
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from test_gpu_sdrf_paper import paper_sdrf_oracle
    uni = np.random.RandomState(seed).random_sample(loops)
    t0 = time.perf_counter()
    _, log = paper_sdrf_oracle(ei, n, loops, True, bound, tau, uni)
    dt = time.perf_counter() - t0
    return {"iterations": len(log), "s": dt, "iters_per_s": len(log) / dt, "host_cores": os.cpu_count(),
            "threads_used": 1}, log


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for sdrf_paper_bench.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-iters", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sdrf_paper_bench.py needs a CUDA device")
    from dcr.synth import SDRF_PARAMS, named_graph
    record = {"gpu": gpu_identity(torch), "reps": args.reps,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "results": {}}
    cei, cn = named_graph("cora")
    cora, clog = single_rate(torch, cei, cn, 1000, 163, 0.95, 0, args.reps)
    record["results"]["cora"] = cora
    print(json.dumps({"cora_iters_per_s": round(cora["iters_per_s"], 1)}), flush=True)
    for name in ("cornell", "texas", "wisconsin"):
        ei, n = named_graph(name)
        loops, tau, bound = SDRF_PARAMS[name]
        r, _ = single_rate(torch, ei, n, loops, tau, bound, 5, args.reps)
        r.update(loops=loops, tau=tau, removal_bound=bound)
        record["results"][name] = r
        print(json.dumps({name + "_iters_per_s": round(r["iters_per_s"], 1)}), flush=True)
    b, blogs = batch_rate(torch, cei, cn, 1000, 163, 0.95, 148, args.reps)
    b["log_of_seed0_equals_single_run"] = bool(np.array_equal(blogs[0], clog))
    record["results"]["cora_batch148"] = b
    print(json.dumps({"batch148_agg_iters_per_s": round(b["agg_iters_per_s"], 1)}), flush=True)
    o, olog = oracle_rate(cei, cn, args.oracle_iters, 163, 0.95, 0)
    o["device_prefix_matches"] = [tuple(int(v) for v in r[3:5]) for r in clog[: len(olog)]] == \
        [(r["k"], r["l"]) for r in olog]
    record["results"]["cora_oracle_host"] = o
    o["device_speedup_single"] = cora["iters_per_s"] / o["iters_per_s"]
    print(json.dumps({"oracle_iters_per_s": round(o["iters_per_s"], 3), "prefix_matches": o["device_prefix_matches"]}),
          flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sdrf_paper_bench.json"), "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"written": os.path.join(args.out, "sdrf_paper_bench.json")}))


if __name__ == "__main__":
    main()
