"""Seed sweeps from a forked device state, and batched edits, against the paths they replace.

Seed sweep (cora shape: 1000 iterations, tau 163, bound 0.95, B in {148, 296}; wisconsin shape with its
``SDRF_PARAMS`` values, B = 100), two arms on a host clock that ends in
a synchronise, their order alternated between repetitions:
  sdrf_batch   ``sdrf.sdrf_batch(edge_index, ...)``: B host set-ups, one batched launch, B host exports;
  fork         ``DynamicCurvature(edge_index, capacity=loops).rewire_batch(...)``: one host set-up, B device forks, one
               batched launch, B device exports.
The outputs and logs of the two arms must be equal.  The parts that differ are timed on their own: B host set-ups
(host clock ending in a synchronise) against one ``dcr_sdrf_fork`` of B copies (CUDA events), and B host exports
(``SdrfState.export`` + ``G.from_networkx_order``, host clock) against B ``dcr_sdrf_export_edge_index`` calls (CUDA
events; buffers allocated before the window).

Edit batch (cora shape): 148 forks x 100 random mixed edits, one ``edit_batch`` launch against 148 sequential
``edit`` calls, each timed with CUDA events around the Python call; the curvature and the insertion order of every fork
must be bit-identical between the two.

    python profiles/sdrf_fork_bench.py --out DIR [--reps 3]      # writes DIR/sdrf_fork_bench_<card>.json

On a B200 that is ``sdrf_fork_bench_b200.json``, the record kept in ``profiles/`` and quoted in DESIGN §4.11.
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
for _p in (os.path.join(REPO, "discrete-curvature-rewiring_b200"), REPO, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from sdrf_batch_bench import gpu_identity  # noqa: E402


def _summary(times):
    return {"s_median": statistics.median(times), "s_min": min(times), "s_all": times}


def _events(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def sweep(torch, name, ei, n, loops, tau, bound, count, reps):
    from dcr import graph as G
    from dcr import lib as L
    from dcr import sdrf
    from dcr.dynamic import DynamicCurvature
    U = np.stack([np.random.RandomState(s).random_sample(loops) for s in range(count)])
    times = {"sdrf_batch": [], "fork": []}
    parts = {"host_setup": [], "device_fork": [], "host_export": [], "device_export": []}
    equal = export_equal = True

    def arm_sdrf_batch():
        return sdrf.sdrf_batch(ei, n, loops, True, bound, tau, uniforms=U, return_log=True)

    def arm_fork():
        with DynamicCurvature(ei, n, capacity=loops) as dc:
            return dc.rewire_batch(loops, True, bound, tau, uniforms=U, return_log=True)

    for rep in range(reps):
        res = {}
        for arm, fn in ((("sdrf_batch", arm_sdrf_batch), ("fork", arm_fork))[:: 1 if rep % 2 == 0 else -1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res[arm] = fn()
            torch.cuda.synchronize()
            times[arm].append(time.perf_counter() - t0)
        (want, wlog), (got, glog) = res["sdrf_batch"], res["fork"]
        equal &= all(np.array_equal(a, b) for a, b in zip(got, want))
        equal &= all(np.array_equal(a, b) for a, b in zip(glog, wlog))

        # the parts: B host set-ups against one fork of B copies, B host exports against B device exports
        mode, order = sdrf._loop_mode("bfc", True)
        ordered = order(ei, n)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fresh = [sdrf._new_state(mode, ordered, loops) for _ in range(count)]
        torch.cuda.synchronize()
        parts["host_setup"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for s in fresh:
            G.from_networkx_order(*s.export())
        parts["host_export"].append(time.perf_counter() - t0)
        for s in fresh:
            s.close()
        with DynamicCurvature(ei, n, capacity=loops) as dc:
            e0, e1 = _events(torch)
            torch.cuda.synchronize()
            e0.record()
            forks = dc._state.fork(count)
            e1.record()
            torch.cuda.synchronize()
            parts["device_fork"].append(e0.elapsed_time(e1) * 1e-3)
            cap = forks[0].nnz() + forks[0].n_self
            bufs = [(torch.empty(n + 1, dtype=torch.int32, device="cuda"),
                     torch.empty((2, max(cap, 1)), dtype=torch.int64, device="cuda")) for _ in forks]
            stream = L.current_stream()
            torch.cuda.synchronize()
            e0.record()
            for f, (rp, out) in zip(forks, bufs):
                L.check(f.lib.dcr_sdrf_export_edge_index(f.handle, rp.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                                                         cap, stream))
            e1.record()
            torch.cuda.synchronize()
            parts["device_export"].append(e0.elapsed_time(e1) * 1e-3)
            host = G.from_networkx_order(*dc._state.export())          # the forks are copies of the unrewired graph
            export_equal &= all(np.array_equal(out[:, : int(rp[-1])].cpu().numpy(), host) for rp, out in bufs)
            for f in forks:
                f.close()
    out = {"workload": name, "runs": count, "loops": loops, "tau": tau, "removal_bound": bound,
           "outputs_and_logs_equal": bool(equal), "device_export_equal": bool(export_equal),
           "e2e": {k: _summary(v) for k, v in times.items()},
           "parts": {k: _summary(v) for k, v in parts.items()}}
    out["e2e"]["speedup"] = out["e2e"]["sdrf_batch"]["s_median"] / out["e2e"]["fork"]["s_median"]
    print(json.dumps({"workload": name, "runs": count, "equal": out["outputs_and_logs_equal"],
                      "export_equal": out["device_export_equal"],
                      "sdrf_batch_s": round(out["e2e"]["sdrf_batch"]["s_median"], 4),
                      "fork_s": round(out["e2e"]["fork"]["s_median"], 4),
                      **{k: round(v["s_median"], 5) for k, v in out["parts"].items()}}), flush=True)
    return out


def random_mixed_edits(ei, n, count, rng):
    """``count`` valid edits on the undirected graph ``ei``: removes of present edges and adds of random pairs."""
    edges = {(min(a, b), max(a, b)) for a, b in ei.T.tolist() if a != b}
    present = sorted(edges)
    out = []
    while len(out) < count:
        if rng.random() < 0.5 and present:
            a, b = present.pop(int(rng.integers(len(present))))
            edges.discard((a, b))
            out.append((0, a, b) if rng.random() < 0.5 else (0, b, a))
        else:
            a, b = (int(v) for v in rng.integers(0, n, 2))
            if a == b:
                continue
            if (min(a, b), max(a, b)) not in edges:
                edges.add((min(a, b), max(a, b)))
                present.append((min(a, b), max(a, b)))
            out.append((1, a, b))
    return np.array(out, dtype=np.int64)


def edit_batch_bench(torch, ei, n, count, per, reps):
    from dcr.dynamic import DynamicCurvature, edit_batch
    rng = np.random.default_rng(0)
    lists = [random_mixed_edits(ei, n, per, rng) for _ in range(count)]
    times = {"sequential": [], "batched": []}
    equal = True
    with DynamicCurvature(ei, n, capacity=per) as dc:
        for _ in range(reps):
            seq, bat = dc.fork(count), dc.fork(count)
            e0, e1 = _events(torch)
            torch.cuda.synchronize()
            e0.record()
            for f, e in zip(seq, lists):
                f.edit(e)
            e1.record()
            torch.cuda.synchronize()
            times["sequential"].append(e0.elapsed_time(e1) * 1e-3)
            e0.record()
            applied = edit_batch(bat, lists)
            e1.record()
            torch.cuda.synchronize()
            times["batched"].append(e0.elapsed_time(e1) * 1e-3)
            equal &= applied == [per] * count
            for a, b in zip(seq, bat):
                ra, rb = a.insertion_order(), b.insertion_order()
                equal &= all(np.array_equal(x, y) for x, y in zip(ra, rb))
                ca, cb = a.curvature(), b.curvature()
                equal &= ca.dtype == cb.dtype and np.array_equal(ca.view(np.int32), cb.view(np.int32))
            for f in seq + bat:
                f.close()
    out = {"workload": "cora edit batch", "forks": count, "edits_per_fork": per,
           "curvature_and_order_equal": bool(equal), "events": {k: _summary(v) for k, v in times.items()}}
    out["events"]["speedup"] = out["events"]["sequential"]["s_median"] / out["events"]["batched"]["s_median"]
    out["events"]["batched_edits_per_s"] = count * per / out["events"]["batched"]["s_median"]
    print(json.dumps({"workload": out["workload"], "equal": out["curvature_and_order_equal"],
                      "sequential_s": round(out["events"]["sequential"]["s_median"], 5),
                      "batched_s": round(out["events"]["batched"]["s_median"], 5)}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for sdrf_fork_bench_<card>.json")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sdrf_fork_bench.py needs a CUDA device")
    from dcr.synth import SDRF_PARAMS, named_graph
    record = {"gpu": gpu_identity(torch), "reps": args.reps,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    cei, cn = named_graph("cora")
    wei, wn = named_graph("wisconsin")
    wloops, wtau, wbound = SDRF_PARAMS["wisconsin"]
    sweep(torch, "warm-up", cei, cn, 50, 163, 0.95, 4, 1)
    edit_batch_bench(torch, cei, cn, 4, 10, 1)
    record["sweeps"] = [sweep(torch, "cora", cei, cn, 1000, 163, 0.95, b, args.reps) for b in (148, 296)]
    record["sweeps"].append(sweep(torch, "wisconsin redo_rewiring", wei, wn, wloops, wtau, wbound, 100, args.reps))
    record["edit_batch"] = edit_batch_bench(torch, cei, cn, 148, 100, args.reps)
    os.makedirs(args.out, exist_ok=True)
    card = torch.cuda.get_device_name().split()[-1].lower()          # "NVIDIA B200" -> b200
    path = os.path.join(args.out, f"sdrf_fork_bench_{card}.json")
    with open(path, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"written": path}))


if __name__ == "__main__":
    main()
