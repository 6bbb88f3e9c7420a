#!/usr/bin/env python
"""bench.py — BFC edges/s (full-graph paper-flavour BFC, arxiv-shaped synthetic graph) and SDRF iterations/s.

    python bench.py --gpus N --steps K --warmup W            # our arm (libdcr.so, sm_100a)
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the oracle's C port on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs as DIR/<name>.npy

One JSON line on stdout (rank 0).  A "step" is one full pass of the hot path over the whole graph: plan + edge
kernels (+ all-gather and re-interleave when N > 1).  Timing: CUDA events per step on the launching stream, an L2
flush (256 MiB memset) between steps outside the events, barrier + synchronize around the timed region, max over
ranks.  See DESIGN.md §Measurement for the definitions of `value`, `e2e`, `roofline` and `cpu_baseline`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "discrete-curvature-rewiring_b200")
for _p in (PKG, REPO):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

DENSE_WORKLOAD = ("squirrel-shaped synthetic graph (N=5201, E=198000): full-graph cuda-flavour BFC in the dense regime — "
                  "supports A2[i,j] on the edges via tcgen05 int8 A·A (TMA, TMEM, fused epilogue), then the per-entry "
                  "closing pass; the sparse sorted-list support kernel is timed beside it")

WORKLOADS = {
    "arxiv": "arxiv-shaped synthetic graph (N=169343, E=1166243, Chung-Lu alpha=0.6, p_tri=0.1, seed 169343): "
             "full-graph paper-flavour BFC (deg, #tri, #sq_i, #sq_j, gamma_max, fp64 value per undirected edge)",
    "squirrel": "squirrel-shaped synthetic graph (N=5201, E=198000): full-graph paper-flavour BFC",
    "cora": "cora-shaped synthetic graph (N=2708, E=5278): full-graph paper-flavour BFC",
}


def load_profile_summary():
    """Counters of the committed ncu capture of the two edge kernels (profiles/r02_edge_kernels_ncu.json, written by
    profiles/summarize_r02.py from the .ncu-rep of `bench.py --steps 1`): DRAM bytes, executed warp instructions and
    streamed entries per pass.  bench.py holds no measured literals of its own."""
    path = os.path.join(REPO, "profiles", "r02_edge_kernels_ncu.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(rowptr: np.ndarray, col: np.ndarray, esrc: np.ndarray, edst: np.ndarray):
    """SURVEY.md §8d: B_gather(e) = 16 + 4(d_i+d_j) + 4((S_i-d_j)+(S_j-d_i)) + 24, S_v = sum of neighbour degrees.
    Also B_compulsory = 4(N+1) + 4*2E + 24E (CSR once + results once)."""
    deg = np.diff(rowptr.astype(np.int64))
    n = deg.size
    rows = np.repeat(np.arange(n), deg)
    S = np.bincount(rows, weights=deg[col].astype(np.float64), minlength=n).astype(np.int64)
    di, dj = deg[esrc], deg[edst]
    per_edge = 16 + 4 * (di + dj) + 4 * ((S[esrc] - dj) + (S[edst] - di)) + 24
    compulsory = 4 * (n + 1) + 4 * col.size + 24 * esrc.size
    return per_edge, int(compulsory)


class ClockSampler:
    """SM clock and throttle reasons for the clocks record of the JSON line.

    * SM clock DURING the timed steps: an in-band probe (`dcr_sm_clock_probe`: one thread, clock64 / globaltimer)
      enqueued on a side stream between the timed steps, so it runs while their kernels run.
    * Throttle reasons: NVML, in-process — but NOT while the timed steps execute.  On these shared hosts every form of
      NVML / nvidia-smi polling tried (nvidia-smi -lms, nvmlDeviceGetClockInfo, nvmlDeviceGetCurrentClocksEventReasons)
      sporadically stalled GPU work for 20-200 ms, turning one 7 ms step into a 170 ms one (step_ms lists in
      profiles/r01_clock_sampling_perturbation.txt; without polling every step is within 0.02 ms of the others).
      The reasons are therefore sampled every 20 ms over an UNTIMED batch of the same steps run back to back right
      after the timed region (`under_load`), i.e. under the identical load."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.masks = []
        self.stop_flag = False
        self.handle = None
        self.nvml = None
        self.max_mhz = None
        self.probe_out = None
        self.probe_stream = None
        self.n_probes = 0
        self.probe_where = "during the timed steps"

    def start(self):
        import torch
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if visible:
                try:
                    idx = int(visible.split(",")[self.gpu])
                except (ValueError, IndexError):
                    idx = self.gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None
        self.probe_out = torch.zeros(64, dtype=torch.float32, device=f"cuda:{self.gpu}")
        self.probe_stream = torch.cuda.Stream(device=self.gpu)

    def _poll(self):
        while not self.stop_flag:
            try:
                try:
                    m = self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    m = self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.masks.append(int(m))
            except Exception:
                pass
            time.sleep(0.02)

    def probe(self):
        """Enqueue one SM-clock probe on the side stream (call between the enqueues of the timed steps)."""
        if self.probe_out is None or self.n_probes >= self.probe_out.numel():
            return
        from dcr import lib as L
        L.check(L.load().dcr_sm_clock_probe(self.probe_out[self.n_probes:].data_ptr(), self.probe_stream.cuda_stream),
                "dcr_sm_clock_probe")
        self.n_probes += 1

    def under_load(self, step_fn, steps: int, exact: bool = False):
        """Poll the throttle reasons while untimed repetitions of the timed step execute (`exact`: exactly `steps`
        of them — needed when the step contains collectives and every rank must run the same count)."""
        import torch
        if self.nvml is None:
            for _ in range(steps if exact else 0):
                step_fn()
            return
        self.stop_flag = False
        th = threading.Thread(target=self._poll, daemon=True)
        th.start()
        t_end = time.perf_counter() + (0.0 if exact else 0.25)
        done = 0
        while done < steps or time.perf_counter() < t_end:       # single GPU: at least a quarter of a second of load
            step_fn()
            done += 1
            if done % 4 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        self.stop_flag = True
        th.join(timeout=3)

    def result(self) -> dict:
        import torch
        torch.cuda.synchronize()
        mhz = [float(v) for v in self.probe_out[: self.n_probes].cpu().tolist() if v > 0] if self.n_probes else []
        mask = 0
        for m in self.masks:
            mask |= m
        return {"sm_mhz": float(np.median(mhz)) if mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": [name for name, bit in self.REASONS if mask & bit],
                "samples": len(mhz), "reason_samples": len(self.masks),
                "source": f"sm_mhz: in-band clock64/globaltimer probes on a side stream {self.probe_where}; reasons: NVML "
                          "every 20 ms over an untimed batch of the same steps run right after the timed region (NVML polling "
                          "inside the region stalls GPU work on these hosts, see profiles/)"}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_bfc_rate(rowptr, col, esrc, edst, threads: int, budget_s: float, seed: int = 0):
    """Time the oracle's C port (bfc_naive restated, pthreads) on a seeded uniform sample of the edges sized for
    about `budget_s` seconds.  Returns (edges/s, sample size, seconds)."""
    from oracle.c_port import bfc_paper_c
    rng = np.random.default_rng(seed)
    perm = rng.permutation(esrc.size)
    probe = perm[: min(esrc.size, 4096)]
    t0 = time.perf_counter()
    bfc_paper_c(rowptr, col, esrc[probe], edst[probe], threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    m = int(min(esrc.size, max(4096, budget_s * probe.size / dt)))
    pick = perm[:m]
    t0 = time.perf_counter()
    bfc_paper_c(rowptr, col, esrc[pick], edst[pick], threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    return m / dt, m, dt


def base_config(workload: str, n: int, E: int, world: int) -> dict:
    """The part of `config` that names the workload — identical in our arm and in the reference arm."""
    return {"workload": WORKLOADS[workload], "nodes": int(n), "undirected_edges": int(E),
            "sharding": ("graph replicated; contiguous edge ranges of equal estimated work, one per GPU; results "
                         "all-gathered (our arm: fused into the closing kernel over NVLink peer memory)") if world > 1
            else "single GPU",
            "l2": "256 MiB memset between steps (outside the per-step CUDA events)",
            "timing": "K steps enqueued back to back, per-step CUDA events, sum over steps, max over ranks"}


def build_graph(workload: str):
    from dcr import graph
    from dcr.synth import named_graph
    ei, n = named_graph(workload)
    rowptr, col = graph.undirected_csr(ei, n)
    m = ei[0] < ei[1]
    esrc = ei[0][m].astype(np.int32)
    edst = ei[1][m].astype(np.int32)
    return ei, n, rowptr, col, esrc, edst


# ------------------------------------------------------------------------------------------------------------
# reference arm: the CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------------------
def build_oracle_only():
    """The reference arm needs the oracle's C library and nothing of ours: it never loads libdcr.so."""
    mk = os.path.join(REPO, "oracle", "c", "Makefile")
    if os.path.exists(mk):
        subprocess.run(["make", "-s", "-C", os.path.dirname(mk)], check=True)


def python_speed_rate(ei, n, esrc, edst, budget_s: float, seed: int = 0):
    """Python-speed stand-in for the reference's own `bfc_naive.bfc` loop (curvature/bfc_naive.py:43-52; the reference
    checkout is not on the GPU box): oracle/paper_flavour.py — the same set arithmetic per edge, one Python thread — on a
    seeded uniform sample of the edges."""
    from oracle.paper_flavour import adjacency_sets, bfc_edge_fields
    adj = adjacency_sets(ei, n)
    rng = np.random.default_rng(seed)
    pick = rng.permutation(esrc.size)
    t0 = time.perf_counter()
    done = 0
    for e in pick.tolist():
        bfc_edge_fields(adj, int(esrc[e]), int(edst[e]))
        done += 1
        if done >= 64 and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    build_oracle_only()
    ei, n, rowptr, col, esrc, edst = build_graph(args.workload)
    threads = host_threads()
    steps = max(1, args.steps)
    budget = min(20.0, 120.0 / (steps + args.warmup))       # whole run stays within a few minutes
    rates, m = [], 0
    for s in range(args.warmup + steps):
        rate, m, dt = cpu_bfc_rate(rowptr, col, esrc, edst, threads, budget, seed=s)
        if s >= args.warmup:
            rates.append((m, dt))
    tot_m = sum(a for a, _ in rates)
    tot_t = sum(b for _, b in rates)
    value = tot_m / tot_t
    sample = (f"oracle C port of curvature/bfc_naive.py (oracle/c/bfc_paper_csr.c), {threads} pthreads, per step a "
              f"seeded uniform sample of {m} of the {esrc.size} undirected edges")
    py_rate, py_m, py_dt = python_speed_rate(ei, n, esrc, edst, 8.0)
    line = {
        "impl": "reference", "metric": "bfc_edges_per_sec", "value": value, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32 counts + f64 value", "data": "synthetic",
        "config": base_config(args.workload, n, esrc.size, world),
        "sample_edges_per_step": m,
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": threads, "kind": "port", "sample": sample},
        "python_speed_baseline": {"value": py_rate, "unit": "edges/s", "cores": 1, "kind": "port",
                                  "sample": f"oracle/paper_flavour.py (set arithmetic of bfc_naive.bfc_edge, one Python "
                                            f"thread), {py_m} sampled edges, {py_dt:.1f} s"},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
def sdrf_bench(args, torch):
    """SDRF iterations/s on the cora-shaped graph (config 3), device loop vs the dense CPU restatement."""
    from dcr import graph, sdrf
    from dcr.synth import named_graph
    from oracle.sdrf import sdrf_oracle
    ei, n = named_graph("cora")
    loops, tau, bound = args.sdrf_loops, 163, 0.95
    uni = np.random.RandomState(3).random_sample(loops)
    out = {"workload": f"cora-shaped synthetic graph (N=2708, E=5278), {loops} iterations, tau={tau}, "
                       f"removal_bound={bound} (utils/hyperparams.py Cora), stochastic draw with host uniforms"}
    # device-resident loop only (state already built): CUDA events around the single persistent-kernel launch
    rowptr_o, order = graph.networkx_order(ei, n)
    best = None
    for rep in range(3):
        st = sdrf.SdrfState(rowptr_o, order, max_additions=loops)
        u_dev = torch.from_numpy(uni).cuda()
        log = torch.empty((loops, 8), dtype=torch.int32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        res, _ = st.run(loops, True, bound, tau, u_dev, log=log)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        done = res["iterations_done"]
        st.close()
        if res["status"] == 0 and (best is None or ms < best[0]):
            best = (ms, done)
    if best is not None:
        out["iters_per_s"] = best[1] / (best[0] * 1e-3)
        out["iterations"] = best[1]
        out["ms_total"] = best[0]
    # end to end through the public entry point: host edge_index in, host edge_index out (set-up + loop + export)
    t0 = time.perf_counter()
    got, glog = sdrf.sdrf(ei, n, loops, True, bound, tau, uniforms=uni, return_log=True)
    dt = time.perf_counter() - t0
    out["e2e_iters_per_s"] = len(glog) / dt
    out["e2e_s"] = dt
    # CPU: dense restatement of bfc_cuda.py + sdrf_cuda_bfc.py (two A@A per iteration, like the reference)
    cpu_iters = args.sdrf_cpu_iters
    t0 = time.perf_counter()
    want, wlog = sdrf_oracle(ei, n, cpu_iters, True, bound, tau, uni, rounding="compiled", incremental_a2=False)
    dt = time.perf_counter() - t0
    out["cpu_baseline"] = {"value": len(wlog) / dt, "unit": "iterations/s", "cores": host_threads(), "kind": "port",
                           "sample": f"first {cpu_iters} iterations of the same run, dense numpy restatement "
                                     "(oracle/sdrf.py, BLAS A@A + per-entry numpy loops)"}
    same = [tuple(int(v) for v in r) for r in glog[:cpu_iters]] == [
        (r["x"], r["y"], r["n_candidates"], r["k"], r["l"], r["choice"],
         -1 if r["removed"] is None else r["removed"][0], -1 if r["removed"] is None else r["removed"][1])
        for r in wlog]
    out["prefix_matches_cpu"] = bool(same)
    if "iters_per_s" in out:
        out["speedup_vs_cpu"] = out["iters_per_s"] / out["cpu_baseline"]["value"]
    # the squirrel shape with the reference's hyper-parameters (utils/hyperparams.py:72-81: 1396 iterations, tau 436,
    # bound 5.88): hub candidate matrices of up to millions of cells; the first --sdrf-squirrel-loops iterations
    try:
        from dcr.synth import SDRF_PARAMS
        sei, sn = named_graph("squirrel")
        lp_full, stau, sbound = SDRF_PARAMS["squirrel"]
        lp = min(lp_full, args.sdrf_squirrel_loops)
        suni = np.random.RandomState(5).random_sample(lp)
        srow, sorder = graph.networkx_order(sei, sn)
        st = sdrf.SdrfState(srow, sorder, max_additions=lp)
        u_dev = torch.from_numpy(suni).cuda()
        slog = torch.empty((lp, 8), dtype=torch.int32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        sres, _ = st.run(lp, True, sbound, stau, u_dev, log=slog)
        e1.record()
        torch.cuda.synchronize()
        st.close()
        out["squirrel"] = {"workload": f"squirrel-shaped synthetic graph (N=5201, E=198000), first {lp} of the reference's "
                                       f"{lp_full} iterations, tau={stau}, removal_bound={sbound}",
                           "iters_per_s": sres["iterations_done"] / (e0.elapsed_time(e1) * 1e-3),
                           "iterations": sres["iterations_done"], "ms_total": e0.elapsed_time(e1), "status": sres["status"]}
    except Exception as exc:
        out["squirrel"] = {"unavailable": repr(exc)[:300]}
    # the other loop flavours (SURVEY.md §8f-3 / §8f-4), same cora-shaped graph
    def loop_rate(state, lp, bnd, tu, un):
        u_dev = torch.from_numpy(un).cuda()
        lg = torch.empty((lp, 8), dtype=torch.int32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        r_, _ = state.run(lp, True, bnd, tu, u_dev, log=lg)
        e1.record()
        torch.cuda.synchronize()
        state.close()
        return r_["iterations_done"] / (e0.elapsed_time(e1) * 1e-3), r_["iterations_done"], r_["status"], lg.cpu().numpy()

    def tuples(wlog_):
        return [(r["x"], r["y"], r["n_candidates"], r["k"], r["l"], r["choice"],
                 -1 if r["removed"] is None else r["removed"][0], -1 if r["removed"] is None else r["removed"][1])
                for r in wlog_]
    try:
        from dcr import lib as L_
        from oracle.sdrf_classical import sdrf_classical_oracle
        cl = {}
        for ct, mode, bnd, tu in (("augmented", L_.SDRF_MODE_AUGMENTED, 0.5, 2), ("1d", L_.SDRF_MODE_1D, -6.0, 2),
                                  ("haantjes", L_.SDRF_MODE_HAANTJES, 0.5, 2)):
            crow, cord = graph.classical_order(ei, n)
            rate, done, status, lg = loop_rate(sdrf.SdrfState(crow, cord, max_additions=loops, mode=mode), loops, bnd, tu, uni)
            cpu_it = min(loops, 60)
            t0 = time.perf_counter()
            _, wl = sdrf_classical_oracle(ei, n, ct, cpu_it, True, bnd, tu, uni)
            dtc = time.perf_counter() - t0
            cl[ct] = {"iters_per_s": rate, "iterations": done, "status": status, "tau": tu, "removal_bound": bnd,
                      "cpu_baseline": {"value": len(wl) / dtc, "unit": "iterations/s", "cores": 1, "kind": "port",
                                       "sample": f"first {cpu_it} iterations, oracle/sdrf_classical.py — the statements of the "
                                                 "reference's own CPU loop rewiring/sdrf_no_cuda.py at Python speed"},
                      "prefix_matches_cpu": [tuple(int(v) for v in r) for r in lg[:len(wl)]] == tuples(wl),
                      "speedup_vs_cpu": rate / (len(wl) / dtc)}
        out["classical"] = cl
    except Exception as exc:
        out["classical"] = {"unavailable": repr(exc)[:300]}
    try:
        from dcr import lib as L_
        rng = np.random.default_rng(7)
        und = ei[:, ei[0] < ei[1]]
        both = rng.random(und.shape[1]) < 0.5                       # half of the edges keep both directions
        flip = rng.random(und.shape[1]) < 0.5
        one = np.where(flip, und[::-1], und)
        dei = np.concatenate([one, one[::-1][:, both]], axis=1)
        dei = dei[:, rng.permutation(dei.shape[1])]
        dl, dtau, dbound = min(loops, 300), 20, 0.5
        duni = np.random.RandomState(9).random_sample(dl)
        s_rp, s_ord, p_rp, p_ord = graph.digraph_order(dei, n)
        rate, done, status, lg = loop_rate(sdrf.SdrfState(s_rp, s_ord, max_additions=dl, mode=L_.SDRF_MODE_BFC_DIRECTED,
                                                          in_rowptr=p_rp, in_order=p_ord), dl, dbound, dtau, duni)
        cpu_it = 4
        t0 = time.perf_counter()
        _, wl = sdrf_oracle(dei, n, cpu_it, True, dbound, dtau, duni, rounding="compiled", incremental_a2=False,
                            is_undirected=False)
        dtc = time.perf_counter() - t0
        out["directed"] = {"workload": f"cora-shaped graph with one direction dropped on half of the edges ({dei.shape[1]} "
                                       f"directed entries), is_undirected=False, {dl} iterations, tau={dtau}, bound={dbound}",
                           "iters_per_s": rate, "iterations": done, "status": status,
                           "cpu_baseline": {"value": len(wl) / dtc, "unit": "iterations/s", "cores": host_threads(),
                                            "kind": "port", "sample": f"first {cpu_it} iterations, dense numpy restatement "
                                                                      "(oracle/sdrf.py, is_undirected=False)"},
                           "prefix_matches_cpu": [tuple(int(v) for v in r) for r in lg[:len(wl)]] == tuples(wl),
                           "speedup_vs_cpu": rate / (len(wl) / dtc)}
    except Exception as exc:
        out["directed"] = {"unavailable": repr(exc)[:300]}
    # The reference's OWN numba kernels on this GPU (oracle/_ref PTX, built from /root/reference by oracle/build_ref.py,
    # loaded with the driver API) driven the reference's way: two A@A + an N^2 x N kernel per iteration, one .item()
    # per candidate.  A reported baseline ("the repo's numba bfc_cuda on the same B200"), present when oracle/_ref is.
    try:
        from oracle import ref_gpu
        if ref_gpu.available():
            budget = 6.0
            ref_gpu.sdrf_reference_gpu(ei, n, 2, True, bound, tau, uni)                       # JIT + warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, rlog = ref_gpu.sdrf_reference_gpu(ei, n, loops, True, bound, tau, uni, time_budget_s=budget)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            k = len(rlog)
            same_ref = [tuple(int(v) for v in r) for r in glog[:k]] == [
                (r["x"], r["y"], r["n_candidates"], r["k"], r["l"], r["choice"],
                 -1 if r["removed"] is None else r["removed"][0], -1 if r["removed"] is None else r["removed"][1])
                for r in rlog]
            from curvature.bfc_cuda import balanced_forman_curvature as ours_dense
            def timed(fn, reps):
                fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / reps
            dense = []          # balanced_forman_curvature(A) on dense A: configs 1-4 (SURVEY.md §8d baseline 3)
            for shape in ("cornell", "wisconsin", "cora", "squirrel"):
                gei, gn = named_graph(shape)
                A = torch.zeros(gn, gn, device="cuda")
                A[torch.from_numpy(gei[0]).cuda(), torch.from_numpy(gei[1]).cuda()] = 1
                big = gn > 4000
                r_ms = timed(lambda: ref_gpu.balanced_forman_curvature(A), 1 if big else 3)
                o_ms = timed(lambda: ours_dense(A), 10)
                same_bits = bool(torch.equal(ref_gpu.balanced_forman_curvature(A).view(torch.int32),
                                             ours_dense(A).view(torch.int32)))
                dense.append({"shape": shape, "n": gn, "reference_ms": r_ms, "ours_dropin_ms": o_ms,
                              "bit_identical": same_bits})
                del A
            # config 2: the WebKB shapes with the reference's own hyper-parameters, whole rewiring, both sides end to end
            from dcr.synth import SDRF_PARAMS
            config2 = []
            for shape in ("wisconsin", "texas"):
                gei, gn = named_graph(shape)
                lp, tu, bd = SDRF_PARAMS[shape]
                for t_ in (tu, float("inf")):
                    u2 = np.random.RandomState(11).random_sample(lp)
                    sdrf.sdrf(gei, gn, lp, True, bd, t_, uniforms=u2)                     # warm-up
                    t0 = time.perf_counter()
                    g_out, g_log = sdrf.sdrf(gei, gn, lp, True, bd, t_, uniforms=u2, return_log=True)
                    ours_s = time.perf_counter() - t0
                    t0 = time.perf_counter()
                    r_out, r_log = ref_gpu.sdrf_reference_gpu(gei, gn, lp, True, bd, t_, u2)
                    torch.cuda.synchronize()
                    ref_s = time.perf_counter() - t0
                    config2.append({"shape": shape, "loops": lp, "tau": "inf" if t_ == float("inf") else t_,
                                    "removal_bound": bd, "iterations": len(r_log), "ours_e2e_s": ours_s,
                                    "reference_numba_s": ref_s, "identical_edge_index": bool(np.array_equal(g_out, r_out))})
            ref_ms = [d["reference_ms"] for d in dense if d["shape"] == "cora"][0]
            our_ms = [d["ours_dropin_ms"] for d in dense if d["shape"] == "cora"][0]
            out["reference_numba_on_this_gpu"] = {
                "sdrf_iters_per_s": k / dt, "iterations": k, "wall_s": dt, "sequence_prefix_matches_ours": bool(same_ref),
                "dense_bfc_ms_reference": ref_ms, "dense_bfc_ms_ours_dropin": our_ms, "dense_bfc": dense, "sdrf_config2": config2,
                "what": "unmodified numba kernels of curvature/bfc_cuda.py (PTX via numba.cuda.compile_ptx, driver JIT to "
                        "sm_100) + the reference's host statements (oracle/ref_gpu.py); dense_bfc = "
                        "balanced_forman_curvature(A) on the same cora-shaped dense A, ours through the drop-in module"}
            if "iters_per_s" in out:
                out["speedup_vs_reference_numba"] = out["iters_per_s"] / (k / dt)
    except Exception as exc:                     # a reported baseline must never take the bench down
        out["reference_numba_on_this_gpu"] = {"unavailable": repr(exc)[:200]}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libdcr has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # NCCL prints its version banner on stdout; stdout carries one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    from dcr import bfc
    from dcr import lib as L
    from dcr.dist import HostShardedPaperBFC, ShardedPaperBFC
    L.load()

    ei, n, rowptr, col, esrc, edst = build_graph(args.workload)
    E = int(esrc.size)
    per_edge_bytes, b_compulsory = algorithmic_bytes(rowptr, col, esrc, edst)
    b_gather_total = int(per_edge_bytes.sum())
    peak, peak_src = load_peaks()

    dev = torch.device("cuda", local)
    csr = bfc.DeviceCSR.from_host(rowptr, col, device=dev)
    csr._edges = (torch.from_numpy(esrc).to(dev), torch.from_numpy(edst).to(dev), None)
    sh = ShardedPaperBFC(csr, mode=args.exchange)
    if sh.mode == "peer":
        b_gather_rank = int(per_edge_bytes[sh.lo:sh.hi].sum())
        my_edges = sh.hi - sh.lo
    else:
        b_gather_rank = int(per_edge_bytes[rank::world].sum())
        my_edges = sh.count
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(x):
        if world == 1:
            return [list(x)]
        out = [None] * world
        dist.all_gather_object(out, [float(v) for v in x])
        return out

    def new_events(k):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        for a, b in evs:
            a.record()
            b.record()      # materialise the cudaEvent handles (the edge-kernel pair is recorded by the library)
        return evs

    # ---- device-resident throughput -------------------------------------------------------------------------
    # All K steps are ENQUEUED without a host sync in between (per-step CUDA events on the stream, L2 flush between
    # steps outside the events): the GPU never waits for the host, so host-side hiccups (e.g. the NVML sampler
    # thread) cannot leak into the device times.
    sampler = ClockSampler(local)
    if rank == 0 and not args.no_clocks:
        sampler.start()
    settle = 5 if world > 1 else 0
    for _ in range(args.warmup + settle):
        flush.zero_()
        sh.run()
    step_ev, edge_ev = new_events(args.steps), new_events(args.steps)
    barrier()
    wall0 = time.perf_counter()
    res = None
    for k in range(args.steps):
        flush.zero_()
        step_ev[k][0].record()
        res = sh.run(events=edge_ev[k])
        step_ev[k][1].record()
        if world == 1 and not args.no_clocks and k % max(1, args.steps // 8) == 0:
            sampler.probe()         # runs on a side stream while this step's kernels execute
    barrier()
    wall = time.perf_counter() - wall0
    sh.check()
    step_ms = [a.elapsed_time(b) for a, b in step_ev]
    edge_ms = [a.elapsed_time(b) for a, b in edge_ev]
    # where a step's time goes on this rank: planning (step begin -> first edge kernel), the edge kernels + closing
    # kernel (which is also the all-gather on the peer route), and what follows (waiting for the peers' results /
    # NCCL all-gather + re-interleave)
    plan_ms = [s0.elapsed_time(e0) for (s0, _), (e0, _) in zip(step_ev, edge_ev)]
    tail_ms = [e1.elapsed_time(s1) for (_, s1), (_, e1) in zip(step_ev, edge_ev)]

    # what the last timed step computed, copied before the untimed passes below reuse the result buffers
    last = {k: v.clone() for k, v in res.items()} if (args.dump_outputs and rank == 0) else None

    def untimed_step():
        flush.zero_()
        sh.run()
        if world > 1 and rank == 0 and not args.no_clocks:
            sampler.probe()         # N > 1: SM-clock probes ride on the untimed batch of the same steps

    if world > 1:
        sampler.probe_where = ("during an untimed batch of the same steps run right after the timed region (at N > 1 the "
                               "probe is kept out of the timed steps: it would be the only rank-asymmetric work in them)")
        n_untimed = max(args.steps, 16)              # every rank runs the same untimed batch (hand-shakes inside)
        if rank == 0 and not args.no_clocks:
            sampler.under_load(untimed_step, n_untimed, exact=True)
        else:
            for _ in range(n_untimed):
                untimed_step()
        barrier()
        clocks = sampler.result() if (rank == 0 and not args.no_clocks) else None
    else:
        clocks = None
        if not args.no_clocks:
            sampler.under_load(untimed_step, args.steps)
            clocks = sampler.result()
    total_ms = max_over_ranks(float(np.sum(step_ms)))
    ms_per_step = total_ms / args.steps
    value = E / (ms_per_step * 1e-3)
    edge_ms_avg = float(np.mean(edge_ms))
    all_step_ms = gather_floats(step_ms)
    per_step_max = np.max(np.array(all_step_ms), axis=0)            # slowest rank of every step
    all_edge_ms = gather_floats([edge_ms_avg, float(np.mean(plan_ms)), float(np.mean(tail_ms)), float(my_edges)])

    # parity spot check of what was just timed (full check lives in tests/): first 2000 edges vs the C oracle
    checked = None
    if rank == 0:
        from oracle.c_port import bfc_paper_c
        k = min(E, 2000)
        ref = bfc_paper_c(rowptr, col, esrc[:k], edst[:k], 1)
        checked = all(np.array_equal(res[key][:k].cpu().numpy(), ref[key]) for key in ("tri", "sq_i", "sq_j", "gamma", "bfc"))
    sh.close()

    # ---- end to end: host CSR in (pinned), host results out, copies inside the timed region -------------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_in = (pin(rowptr.astype(np.int32)), pin(col))          # the edge list is derived from the CSR on the device
    hs = HostShardedPaperBFC(n, int(col.size), E, csr.max_degree)
    for _ in range(min(args.warmup, 3)):
        hs.run(*h_in)
    e2e_ev = new_events(args.steps)
    barrier()
    for k in range(args.steps):
        flush.zero_()
        e2e_ev[k][0].record()
        hs.run(*h_in)
        e2e_ev[k][1].record()
    barrier()
    e2e_total = max_over_ranks(float(np.sum([a.elapsed_time(b) for a, b in e2e_ev])))
    e2e_value = E / (e2e_total / args.steps * 1e-3)
    h2d, d2h = hs.bytes_per_pass()
    e2e_checked = None
    if rank == 0:
        hv = hs.host_views()
        k = min(E, 2000)
        e2e_checked = all(np.array_equal(hv[key][:k].numpy(), ref[key]) for key in ("tri", "sq_i", "sq_j", "gamma", "bfc"))
    if world > 1:
        io = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
        dist.all_reduce(io)
        h2d, d2h = int(io[0]), int(io[1])
    hs.close()

    # kernels of one pass (dense mode, n <= 262144): node_s, classify, plan_groups, order; paper_group_kernel +
    # paper_light_warp_kernel; the closing kernel (value + exchange); at N > 1 the ready / wait hand-shake kernels
    launches_per_step = 4 + 2 + 1 + (2 if world > 1 else 0)
    prof = load_profile_summary() if (world == 1 and args.workload == "arxiv") else None
    clock_hz = (clocks["sm_mhz"] if clocks and clocks.get("sm_mhz") else 1965.0) * 1e6
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    roof = {
        "bound": "hbm", "kernel": "paper_group_kernel + paper_light_warp_kernel (the two edge kernels of one step, concurrent)",
        "achieved": b_gather_rank / (edge_ms_avg * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
        "frac": b_gather_rank / (edge_ms_avg * 1e-3) / 1e9 / peak, "peak_source": peak_src,
        "traffic": prof["dram_bytes_per_pass"] if prof else None,
        "traffic_source": prof["source"] if prof else None,
        "edge_kernels_ms": edge_ms_avg, "algorithmic_bytes": b_gather_rank,
        "algorithmic_bytes_model": "model_upper_bound: SURVEY.md §8d B_gather of this rank's edges — BOTH endpoints' 2-hop "
                                   "lists once per edge, no cross-edge reuse; the kernel streams only the cheaper side, out "
                                   "of L2, so frac > 1 is expected and is not a DRAM claim",
        "b_gather_total": b_gather_total, "b_compulsory": b_compulsory,
    }
    if prof:
        # what actually bounds the kernels: instruction issue.  issue_slots_ms = executed warp instructions / (SMs x 4
        # schedulers x SM clock) = the time the pass needs if every scheduler issued every cycle.
        issue_ms = prof["warp_instructions_per_pass"] / (sms * 4 * clock_hz) * 1e3
        roof.update({
            "streamed_bytes": 4 * prof["streamed_entries_per_pass"],
            "streamed_frac_of_hbm_peak": 4 * prof["streamed_entries_per_pass"] / (edge_ms_avg * 1e-3) / 1e9 / peak,
            "dram_frac_of_hbm_peak": prof["dram_bytes_per_pass"] / (edge_ms_avg * 1e-3) / 1e9 / peak,
            "warp_instructions": prof["warp_instructions_per_pass"], "issue_slots_ms": issue_ms,
            "frac_issue": issue_ms / edge_ms_avg,
            "note": "the pass is issue / latency bound, not DRAM bound: CSR and bitmaps are L2 / shared-memory resident "
                    "(dram_frac_of_hbm_peak), frac_issue = share of the issue slots of 148 SMs x 4 schedulers the "
                    "executed warp instructions fill during the edge kernels"})
    cfg = base_config(args.workload, n, E, world)
    line = {
        "metric": "bfc_edges_per_sec", "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32 counts + f64 value", "data": "synthetic",
        "config": cfg,
        "exchange": sh.mode, "wall_s_timed_region": wall, "parity_spot_check_vs_c_oracle": checked,
        "e2e_parity_spot_check_vs_c_oracle": e2e_checked,
        "step_ms": [round(x, 3) for x in per_step_max.tolist()],
        "step_ms_mean_over_median": round(float(np.mean(per_step_max) / np.median(per_step_max)), 4),
        "extra_untimed_steps_after_warmup": settle,
        "phase_ms_rank0": {"plan": round(float(np.mean(plan_ms)), 4), "edge_kernels_and_closing": round(edge_ms_avg, 4),
                           "wait_for_peers" if sh.mode == "peer" else "gather_unshard": round(float(np.mean(tail_ms)), 4)},
        "per_rank": [{"edge_kernels_ms": round(r[0], 4), "plan_ms": round(r[1], 4), "tail_ms": round(r[2], 4),
                      "edges": int(r[3])} for r in all_edge_ms],
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_total / args.steps,
                "what": "dcr.dist.HostShardedPaperBFC.run: pinned host CSR -> every rank uploads the graph, derives the "
                        "undirected edge list from it on the device, finds its work-balanced range, computes it and copies "
                        "its slice of the results into one host block shared by the ranks (bytes = sum over ranks)"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof,
    }
    if rank == 0 and world == 1 and not args.no_cpu:
        thr = host_threads()
        rate, m, dt = cpu_bfc_rate(rowptr, col, esrc, edst, thr, args.cpu_budget)
        line["cpu_baseline"] = {"value": rate, "unit": "edges/s", "cores": thr, "kind": "port",
                                "sample": f"oracle C port of curvature/bfc_naive.py (oracle/c/bfc_paper_csr.c), {thr} "
                                          f"pthreads, seeded uniform sample of {m} of {E} edges, {dt:.1f} s"}
        py_rate, py_m, py_dt = python_speed_rate(ei, n, esrc, edst, 6.0)
        line["python_speed_baseline"] = {
            "value": py_rate, "unit": "edges/s", "cores": 1, "kind": "port",
            "sample": f"oracle/paper_flavour.py — the set arithmetic of bfc_naive.bfc_edge at Python speed, the stand-in for "
                      f"the reference's own bfc_naive.bfc loop (the checkout is not on the GPU box); {py_m} sampled edges, "
                      f"{py_dt:.1f} s"}
    if rank == 0 and world == 1 and not args.no_dense:
        try:
            line["dense"] = dense_bench(args, torch)
            del line["dense"]["outputs"]
        except Exception as exc:
            line["dense"] = {"unavailable": repr(exc)[:300]}
    if args.workload == "arxiv" and not args.no_cuda_flavour:
        if world > 1 and sh.mode != "peer":
            # the sharded cuda flavour exchanges through peer memory only; every rank took the same (NCCL) route above
            cf = {"unavailable": "peer-memory exchange unavailable on this box (the paper-flavour pass fell back to NCCL)"}
        else:
            try:
                cf = cuda_flavour_bench(args, torch, dist, csr, esrc, edst, rowptr, world, rank, dev, flush)
            except Exception as exc:
                if world > 1:
                    raise
                cf = {"unavailable": repr(exc)[:300]}
        if rank == 0:
            line["cuda_flavour"] = cf
    if rank == 0 and not args.no_sdrf:
        line["sdrf"] = sdrf_bench(args, torch)
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cuda_flavour_bench(args, torch, dist, csr, esrc_np, edst_np, rowptr, world, rank, dev, flush):
    """Full-graph CUDA-flavour BFC (balanced_forman_curvature of curvature/bfc_cuda.py:51-65 at the arxiv shape): one work
    item per undirected edge, at N > 1 edge-range sharded with the all-gather of the supports fused between the two passes
    (SURVEY.md §8e row 2).  Every rank takes part; returns the object on rank 0."""
    from dcr import bfc
    from dcr.dist import ShardedCudaBFC
    E = int(esrc_np.size)
    steps, warmup = args.steps, 3
    sc = ShardedCudaBFC(csr)
    for _ in range(warmup + (3 if world > 1 else 0)):
        flush.zero_()
        sc.run()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        out = sc.run()
        ev[k][1].record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sc.check()
    ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor(ms, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total = float(t.sum().item())
    # parity: the per-entry kernels (the round-1 route) on a sample of entries of this rank's full arrays
    ref = bfc.cuda_flavour(csr, want_fields=False, tri=bfc.support(csr))
    entry = csr.undirected_edges()[2]
    if entry is None:
        deg = np.diff(rowptr.astype(np.int64))
        rows = np.repeat(np.arange(deg.size), deg)
        entry = torch.from_numpy(np.flatnonzero(rows < csr.colidx.cpu().numpy())).to(dev)
    same = bool(torch.equal(out["c32"].view(torch.int32), ref["c32"][entry].view(torch.int32))) and \
        bool(torch.equal(out["tri"], ref["tri"][entry]))
    flag = torch.tensor([1 if same else 0], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    deg = np.diff(rowptr.astype(np.int64))
    b_alg = int((16 + 4 * (deg[esrc_np] + deg[edst_np]) + 24).sum()) + 8 * int(out["tri"].sum().item())
    peak, peak_src = load_peaks()
    res = {"workload": "arxiv-shaped synthetic graph: full-graph CUDA-flavour BFC (curvature/bfc_cuda.py) per undirected edge "
                       "(tri, sharp, lambda, fp64 + fp32 value), supports all-gathered between the two passes at N > 1",
           "value": E / (total / steps * 1e-3), "unit": "edges/s", "ms_per_step": total / steps, "steps": steps, "n_gpus": world,
           "ranges": [int(b) for b in sc.bounds],
           "all_ranks_bit_identical_to_per_entry_kernels": bool(flag.item()),
           "roofline": {"bound": "hbm", "kernel": "edges_support_kernel + edges_closing_kernel (light + hub launches)",
                        "algorithmic_bytes": b_alg, "achieved": b_alg / world / (total / steps * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": b_alg / world / (total / steps * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                        "model": "SURVEY.md §8d: 16 + 4(d_i+d_j) + 8 tri + 24 bytes per edge, per rank = total / N"}}
    sc.close()
    return res if rank == 0 else None


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly one JSON line: anything libraries print to fd 1 (e.g. NCCL's version banner) goes to
    stderr instead; emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict):
    """`--dump-outputs DIR`: one DIR/<name>.npy per output array of the timed path's last step, so that two builds can
    be compared output for output on the same seeded inputs.  Integer fields are widened to float64, which holds them
    exactly."""
    host = {}
    for name, t in arrays.items():
        a = t.cpu().numpy()
        host[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def dense_bench(args, torch) -> dict:
    """Config 4: the dense-regime tensor path on the squirrel-shaped graph (1 GPU): supports A2[i,j] on the edges via the
    hand-written tcgen05 int8 A·A kernel, the full cuda-flavour pass through it, and the sorted-list route beside it."""
    from dcr import bfc
    ei, n, rowptr, col, esrc, edst = build_graph("squirrel")
    E = int(esrc.size)
    csr = bfc.DeviceCSR.from_host(rowptr, col)
    n_pad = (n + 127) // 128 * 128
    ws = torch.empty(int(bfc.L.load().dcr_bfc_support_tc_workspace_bytes(n, csr.nnz)), dtype=torch.uint8, device="cuda")
    tri = torch.empty(csr.nnz, dtype=torch.int32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    steps, warmup = args.steps, 3
    last = {}

    def timed(fn):
        for _ in range(warmup):
            fn()
        out = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last["out"] = fn()
            e1.record()
            e1.synchronize()
            out.append(e0.elapsed_time(e1))
        return float(np.mean(out))

    ms_tc = timed(lambda: bfc.support_tc(csr, out=tri, workspace=ws))
    ws2 = torch.empty(int(bfc.L.load().dcr_bfc_cuda_flavour_tc_workspace_bytes(n, csr.nnz)), dtype=torch.uint8,
                      device="cuda")
    ms_full = timed(lambda: bfc.cuda_flavour_tc(csr, want_fields=False, workspace=ws2))
    outputs = {k: last["out"][k] for k in ("tri", "c32")}        # per directed CSR entry
    ms_sparse = timed(lambda: bfc.support(csr, out=tri))
    ms_full_sparse = timed(lambda: bfc.cuda_flavour(csr, want_fields=False, tri=bfc.support(csr, out=tri)))
    same = bool(torch.equal(bfc.support_tc(csr), bfc.support(csr)))
    c_tc = bfc.cuda_flavour_tc(csr, want_fields=False)["c32"]
    c_sp = bfc.cuda_flavour(csr, want_fields=False)["c32"]
    same = same and bool(torch.equal(c_tc.view(torch.int32), c_sp.view(torch.int32)))
    ops = 2.0 * n_pad ** 3
    peak_i8, peak_src = int8_peak(torch)
    return {
        "workload": DENSE_WORKLOAD, "nodes": n, "undirected_edges": E, "n_pad": n_pad,
        "value": E / (ms_full * 1e-3), "unit": "edges/s", "ms_per_step": ms_full, "steps": steps,
        "dtype": "int8 x int8 -> int32 (tcgen05 kind::i8), f64 closing formula",
        "outputs_bit_identical_to_sparse_path": same,
        "roofline": {"bound": "tensor", "kernel": "tc_support_kernel (+ the operand fill and the mirror pass of the same call); achieved = the FULL product's "
                               "2*N_pad^3 ops / time — A*A is symmetric, the kernel issues the upper-triangular half of the MMAs",
                     "achieved": ops / (ms_tc * 1e-3) / 1e12, "peak": peak_i8, "unit": "TOP/s (int8)",
                     "frac": ops / (ms_tc * 1e-3) / 1e12 / peak_i8, "peak_source": peak_src,
                     "traffic": None, "support_tc_ms": ms_tc, "ops": ops},
        "sparse_path": {"support_ms": ms_sparse, "full_ms": ms_full_sparse,
                        "note": "sorted-list intersection kernels on the same CSR (dcr_bfc_support + dcr_bfc_cuda_flavour)"},
        "outputs": outputs,
    }


def int8_peak(torch):
    """Dense int8 tensor peak to hold the tcgen05 path against: measured on this GPU with the library's own
    resident-tile tcgen05 kind::i8 loop when it exports one, else the nominal figure (labelled)."""
    from dcr import lib as L
    lib = L.load()
    if hasattr(lib, "dcr_tc_int8_peak"):
        import ctypes as C
        out = torch.zeros(1, dtype=torch.float64, device="cuda")
        fn = lib.dcr_tc_int8_peak
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.c_void_p]
        best = 0.0
        for _ in range(3):
            if fn(out.data_ptr(), L.current_stream()) != 0:
                best = 0.0
                break
            torch.cuda.synchronize()
            best = max(best, float(out.item()))
        if best > 0:
            return best, "measured: resident-tile tcgen05 kind::i8 loop of libdcr (dcr_tc_int8_peak), best of 3"
    return 4500.0, "nominal dense int8 (no measured int8 peak in MEASURED_PEAKS.json)"


def run_dense(args):
    """`--workload squirrel-dense`: config 4 as a line of its own."""
    import torch

    import __graft_entry__
    __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    d = dense_bench(args, torch)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d["outputs"])
    line = {
        "metric": "bfc_edges_per_sec", "value": d["value"], "unit": "edges/s", "n_gpus": 1,
        "steps": d["steps"], "warmup": 3, "ms_per_step": d["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": d["dtype"], "data": "synthetic",
        "config": {"workload": DENSE_WORKLOAD, "nodes": d["nodes"], "undirected_edges": d["undirected_edges"],
                   "n_pad": d["n_pad"], "l2": "256 MiB memset between steps"},
        "outputs_bit_identical_to_sparse_path": d["outputs_bit_identical_to_sparse_path"],
        "gpu_launches": 5 * d["steps"], "roofline": d["roofline"], "sparse_path": d["sparse_path"],
    }
    emit(line)


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="arxiv", choices=sorted(WORKLOADS) + ["squirrel-dense"])
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--sdrf-loops", type=int, default=1000)
    ap.add_argument("--sdrf-cpu-iters", type=int, default=20)
    ap.add_argument("--sdrf-squirrel-loops", type=int, default=200)
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU exchange: fused peer-memory closing kernel (default) or NCCL all-gather")
    ap.add_argument("--no-dense", action="store_true")
    ap.add_argument("--no-cuda-flavour", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sdrf", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="debug: do not sample clocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the timed path computed in its last step to DIR/<name>.npy (float32/float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to our arm: the reference arm times seeded edge samples, not the full outputs")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "squirrel-dense":
        if args.impl == "reference":
            args.workload = "squirrel"
            run_reference(args)
        else:
            run_dense(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
