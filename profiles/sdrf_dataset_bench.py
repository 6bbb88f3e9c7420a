"""SDRF over a dataset of small graphs: ``sdrf_dataset`` against a loop of ``sdrf()`` and ``sdrf_batch(list)``.

Three datasets built here from a seed, nothing downloaded (BFC, undirected, 16 iterations, tau 4, removal bound 0.5):
  molecules  1000 graphs of 10-40 nodes: a random tree plus a ring closure per ~8 nodes;
  hubby      2000 sparse graphs of ~400 nodes (Chung-Lu, 2 edges per node, power-law degrees);
  ego        5000 dense ego-graphs of ~75 nodes: a centre joined to every node, 15 % of the other pairs.
Three arms, each end to end on a host clock that ends in a synchronise, their order rotated between repetitions:
  loop     ``sdrf.sdrf(ei_g, n_g, ...)`` for every graph;
  batch    ``sdrf.sdrf_batch(list_of_ei, list_of_n, ...)``: B host set-ups, one batched launch, B host exports;
  dataset  ``sdrf.sdrf_dataset(edge_index, ptr, ...)``: one ordering of the union, one ``dcr_sdrf_create_batch``, the
           batched launch, one ``dcr_sdrf_export_edge_index_batch``.
Every graph's columns and log must be equal in the three arms (``equal`` flags).  The dataset arm is split into set-up
(ordering + batched create, host clock ending in its synchronise), launch and export (CUDA events).  For the follow-up
that packs several small runs per SM the record keeps the waves of the batched launch (B CTAs over the SMs), the device
time per wave, and the spread of single-run device times (one ``dcr_sdrf_run`` per graph, CUDA events, a sample of 148).

    python profiles/sdrf_dataset_bench.py --out DIR [--reps 3]     # writes DIR/sdrf_dataset_bench_<card>.json

On a B200 that is ``sdrf_dataset_bench_b200.json``, the record kept in ``profiles/`` and quoted in DESIGN §4.13.
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

LOOPS, TAU, BOUND = 16, 4.0, 0.5


def _sym(pairs):
    a = np.asarray(pairs, dtype=np.int64).reshape(-1, 2).T
    return np.concatenate([a, a[::-1]], axis=1)


def molecules(count, rng):
    out = []
    for _ in range(count):
        n = int(rng.integers(10, 41))
        pairs = [(int(rng.integers(0, v)), v) for v in range(1, n)]
        for _ in range(max(1, n // 8)):
            a, b = rng.choice(n, size=2, replace=False)
            pairs.append((int(a), int(b)))
        out.append((np.unique(_sym(pairs), axis=1), n))
    return out


def hubby(count, rng):
    from dcr.synth import chung_lu_graph
    out = []
    for _ in range(count):
        n = int(rng.integers(380, 421))
        out.append((chung_lu_graph(n, 2 * n, 0.8, 0.1, int(rng.integers(1 << 30))), n))
    return out


def ego(count, rng):
    out = []
    for _ in range(count):
        n = int(rng.integers(65, 86))
        iu = np.triu_indices(n - 1, 1)
        keep = rng.random(iu[0].size) < 0.15
        pairs = np.concatenate([np.stack([np.zeros(n - 1, dtype=np.int64), np.arange(1, n)], 1),
                                np.stack([iu[0][keep] + 1, iu[1][keep] + 1], 1)])
        out.append((_sym(pairs), n))
    return out


def _layout(graphs):
    ptr = np.concatenate([[0], np.cumsum([n for _, n in graphs])]).astype(np.int64)
    return np.concatenate([e + ptr[g] for g, (e, _) in enumerate(graphs)], axis=1), ptr


def _summary(times):
    return {"s_median": statistics.median(times), "s_min": min(times), "s_all": times}


def _split(torch, ei, ptr, uni, count):
    """sdrf_dataset's steps, timed one by one"""
    from dcr import sdrf
    iters = [LOOPS] * count
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    p = sdrf.dataset_ptr(ptr, count)
    gid = sdrf._column_graphs(ei, p)
    mode, order = sdrf._loop_mode("bfc", True)
    lists = sdrf._dataset_order(order, mode, ei, p, gid)
    t1 = time.perf_counter()
    states = sdrf.SdrfState.create_batch(mode, np.diff(p), lists[0], lists[1], iters)
    t2 = time.perf_counter()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    try:
        e[0].record()
        logs, done, errors = sdrf._run_batch_states(states, iters, [BOUND] * count, [TAU] * count, uni, True, 1e-9)
        e[1].record()
        entries = lists[0][p[1:]] - lists[0][p[:-1]]
        cap = int(entries.sum()) + 2 * sum(done)
        e[2].record()
        out, eptr = sdrf.export_edge_index_batch(states, p[:-1], cap)
        total = int(eptr[-1])
        e[3].record()
        torch.cuda.synchronize()
    finally:
        for s in states:
            s.close()
    assert not any(errors) and total <= cap
    return {"order_s": t1 - t0, "create_batch_s": t2 - t1, "launch_ms": e[0].elapsed_time(e[1]),
            "export_ms": e[2].elapsed_time(e[3])}


def _single_runs(torch, graphs, uni, sample):
    """device time of one dcr_sdrf_run per graph (one CTA), for the spread of run lengths"""
    from dcr import sdrf
    mode, order = sdrf._loop_mode("bfc", True)
    ms = []
    for g in sample:
        st = sdrf._new_state(mode, order(*graphs[g]), LOOPS)
        u = torch.from_numpy(uni[g]).cuda()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res, _ = st.run(LOOPS, True, BOUND, TAU, u, guard=0.0)
        e1.record()
        torch.cuda.synchronize()
        st.close()
        ms.append(e0.elapsed_time(e1))
    q = np.percentile(ms, [0, 10, 50, 90, 100]).tolist()
    return {"sample": len(ms), "ms_min_p10_p50_p90_max": q, "ms_mean": float(np.mean(ms))}


def workload(torch, name, graphs, reps, sms):
    from dcr import sdrf
    count = len(graphs)
    ei, ptr = _layout(graphs)
    eis, ns = [e for e, _ in graphs], [n for _, n in graphs]
    uni = [np.random.RandomState(g).random_sample(LOOPS) for g in range(count)]

    def arm_loop():
        return [sdrf.sdrf(eis[g], ns[g], LOOPS, True, BOUND, TAU, uniforms=uni[g], return_log=True) for g in range(count)]

    def arm_batch():
        outs, logs = sdrf.sdrf_batch(eis, ns, LOOPS, True, BOUND, TAU, uniforms=uni, return_log=True)
        return list(zip(outs, logs))

    def arm_dataset():
        out, eptr, logs = sdrf.sdrf_dataset(ei, ptr, LOOPS, True, BOUND, TAU, uniforms=uni, return_log=True)
        return out, eptr, logs

    arms = {"loop": arm_loop, "batch": arm_batch, "dataset": arm_dataset}
    times = {k: [] for k in arms}
    results = {}
    names = list(arms)
    for r in range(reps):
        for k in names[r % 3:] + names[:r % 3]:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = arms[k]()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
            results[k] = res
    out, eptr, dlogs = results["dataset"]
    out, eptr = out.cpu().numpy(), eptr.cpu().numpy()
    eq_loop = eq_batch = True
    for g in range(count):
        cols = out[:, eptr[g]:eptr[g + 1]] - ptr[g]
        log = dlogs[g].copy()
        node = log[:, [0, 1, 3, 4, 6, 7]]
        log[:, [0, 1, 3, 4, 6, 7]] = np.where(node >= 0, node - ptr[g], node)
        le, ll = results["loop"][g]
        be, bl = results["batch"][g]
        eq_loop &= bool(np.array_equal(cols, le) and np.array_equal(log, ll))
        eq_batch &= bool(np.array_equal(cols, be) and np.array_equal(log, bl))
    splits = [_split(torch, ei, ptr, uni, count) for _ in range(reps)]
    split = {k: statistics.median(s[k] for s in splits) for k in splits[0]}
    waves = -(-count // sms)
    rec = {
        "name": name, "graphs": count, "nodes": int(ptr[-1]), "directed_entries": int(ei.shape[1]),
        "nodes_min_median_max": [int(min(ns)), int(statistics.median(ns)), int(max(ns))],
        "loops": LOOPS, "tau": TAU, "removal_bound": BOUND,
        "arms": {k: _summary(v) for k, v in times.items()},
        "equal": {"dataset_vs_loop": eq_loop, "dataset_vs_batch": eq_batch},
        "dataset_split_median": split,
        "waves": waves, "launch_ms_per_wave": split["launch_ms"] / waves,
        "single_run_device_time": _single_runs(torch, graphs, uni, range(0, count, max(1, count // 148))),
    }
    print(json.dumps({k: rec[k] for k in ("name", "equal", "dataset_split_median")}
                     | {"median_s": {k: rec["arms"][k]["s_median"] for k in arms}}), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for sdrf_dataset_bench_<card>.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of every dataset's graph count (rehearsal)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sdrf_dataset_bench.py needs a CUDA device")
    rng = np.random.default_rng(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    record = {"gpu": gpu_identity(torch), "reps": args.reps, "sms": sms}
    sets = [("molecules", molecules(max(1, int(1000 * args.scale)), rng)),
            ("hubby", hubby(max(1, int(2000 * args.scale)), rng)),
            ("ego", ego(max(1, int(5000 * args.scale)), rng))]
    workload(torch, "warm-up", sets[0][1][:40], 1, sms)
    record["workloads"] = [workload(torch, name, graphs, args.reps, sms) for name, graphs in sets]
    os.makedirs(args.out, exist_ok=True)
    card = torch.cuda.get_device_name().split()[-1].lower()          # "NVIDIA B200" -> b200
    path = os.path.join(args.out, f"sdrf_dataset_bench_{card}.json")
    with open(path, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"written": path}))


if __name__ == "__main__":
    main()
