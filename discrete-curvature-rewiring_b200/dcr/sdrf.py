"""Host driver of the device-resident SDRF loop (``dcr_sdrf_*`` in include/dcr.h).

Mirrors the control flow of ``rewiring/sdrf_cuda_bfc.py:14-93`` of the reference: set the graph up on the host
(once), run all iterations inside one persistent kernel, come back to the host only when the kernel asks for a
host-side decision (a uniform within ``guard`` of a softmax CDF boundary, SURVEY.md App. E.3) or reports one of the
reference's exceptions.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import graph as G
from . import lib as L

# numpy's own messages for the ValueErrors np.random.choice raises (sdrf_cuda_bfc.py:64-68)
_MSG_NAN = "probabilities contain NaN"
_MSG_SUM = "probabilities do not sum to 1"
# the fields of dcr_sdrf_result that the host reads, in record order
_RESULT_KEYS = ("status", "iterations_done", "draws_used", "stopped", "pending_n", "pending_x", "pending_y")


def host_choice(improvements: np.ndarray, tau, u: float) -> int:
    """The reference's host-side selection for one iteration: ``utils.softmax.softmax`` + the algorithm of
    ``np.random.choice(range(n), p=p)`` for the uniform ``u`` it would draw (App. E.3)."""
    a = np.asarray(improvements, dtype=np.float64)
    if tau == float("inf"):
        p = np.zeros(len(a))
        p[np.argmax(a)] = 1
    else:
        e = np.exp(a * tau)
        p = e / e.sum()
    if np.isnan(p).any():
        raise ValueError(_MSG_NAN)
    if abs(p.sum() - 1.0) > np.sqrt(np.finfo(np.float64).eps):
        raise ValueError(_MSG_SUM)
    cdf = p.cumsum()
    cdf /= cdf[-1]
    return int(cdf.searchsorted(u, side="right"))


class SdrfState:
    """Owns one ``dcr_sdrf`` handle (device-resident dynamic adjacency + incremental curvature)."""

    def __init__(self, rowptr_order: np.ndarray, order: np.ndarray, max_additions: int, mode: int = L.SDRF_MODE_BFC,
                 in_rowptr: np.ndarray | None = None, in_order: np.ndarray | None = None):
        """``mode``: one of ``L.SDRF_MODE_*``.  The directed mode takes the successor lists as ``rowptr_order/order`` and
        the predecessor lists as ``in_rowptr/in_order`` (all in networkx insertion order)."""
        L.require_cuda()
        self.lib = L.load()
        self.mode = int(mode)
        self.n = int(len(rowptr_order) - 1)
        rp = np.ascontiguousarray(rowptr_order, dtype=np.int32)
        od = np.ascontiguousarray(order, dtype=np.int32)
        handle = C.c_void_p()
        if self.mode == L.SDRF_MODE_BFC_DIRECTED:
            irp = np.ascontiguousarray(in_rowptr, dtype=np.int32)
            iod = np.ascontiguousarray(in_order, dtype=np.int32)
        else:
            irp = iod = None
        self._keep = (rp, od, irp, iod)
        rows = np.repeat(np.arange(self.n, dtype=np.int64), np.diff(rp.astype(np.int64)))
        self.n_self = int(np.count_nonzero(od[: rows.size] == rows))      # nodes that list themselves (self-loops of G)
        L.check(self.lib.dcr_sdrf_create_mode(self.n, self.mode, rp.ctypes.data, od.ctypes.data if od.size else 0,
                                              irp.ctypes.data if irp is not None else 0,
                                              iod.ctypes.data if iod is not None and iod.size else 0,
                                              int(max_additions), C.byref(handle)), "dcr_sdrf_create_mode")
        self.handle = handle
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._result = torch.zeros(8, dtype=torch.int32, device=self.device)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dcr_sdrf_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, loops: int, remove_edges: bool, removal_bound: float, tau, uniforms: torch.Tensor,
            forced_choice: int = -1, guard: float = 1e-9, log: torch.Tensor | None = None):
        """One kernel launch, up to ``loops`` iterations.  Returns ``(result dict, log int32[iters, 8])`` (device log
        sliced after one D2H of the 32-byte result)."""
        if log is None:
            log = torch.empty((max(loops, 1), L.SDRF_LOG_INTS), dtype=torch.int32, device=self.device)
        L.check(self.lib.dcr_sdrf_run(self.handle, int(loops), int(bool(remove_edges)), float(removal_bound),
                                      float(tau), uniforms.data_ptr(), int(uniforms.numel()), int(forced_choice),
                                      float(guard), log.data_ptr(), self._result.data_ptr(), L.current_stream()),
                "dcr_sdrf_run")
        res = dict(zip(_RESULT_KEYS, self._result.cpu().tolist()))
        return res, log[: res["iterations_done"]]

    def pending_improvements(self, n: int) -> np.ndarray:
        out = torch.empty(max(n, 1), dtype=torch.float64, device=self.device)
        L.check(self.lib.dcr_sdrf_pending_improvements(self.handle, out.data_ptr(), int(n), L.current_stream()),
                "dcr_sdrf_pending_improvements")
        return out[:n].cpu().numpy()

    def nnz(self) -> int:
        return int(self.lib.dcr_sdrf_nnz(self.handle))

    def export(self, with_curvature: bool = False):
        """Current graph: ``(rowptr, order)`` numpy (networkx order); with curvature also sorted col / c32 / tri."""
        nnz = self.nnz()
        dev = self.device
        rowptr = torch.empty(self.n + 1, dtype=torch.int32, device=dev)
        if self.n_self and not with_curvature:
            # nodes that list themselves (self-loops of G): the insertion-order rows are longer than the adjacency rows
            order = torch.empty(max(nnz + self.n_self, 1), dtype=torch.int32, device=dev)
            L.check(self.lib.dcr_sdrf_export_order(self.handle, rowptr.data_ptr(), order.data_ptr(), L.current_stream()),
                    "dcr_sdrf_export_order")
            rp = rowptr.cpu().numpy()
            return rp, order[: int(rp[-1])].cpu().numpy()
        order = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        col = c32 = tri = None
        if with_curvature:
            col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
            c32 = torch.empty(max(nnz, 1), dtype=torch.float32, device=dev)
            tri = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        L.check(self.lib.dcr_sdrf_export(self.handle, rowptr.data_ptr(), 0 if self.n_self else order.data_ptr(), L.ptr(col),
                                         L.ptr(c32), L.ptr(tri), L.current_stream()), "dcr_sdrf_export")
        out = (rowptr.cpu().numpy(), order[:nnz].cpu().numpy() if not self.n_self else None)
        if with_curvature:
            out += (col[:nnz].cpu().numpy(), c32[:nnz].cpu().numpy(), tri[:nnz].cpu().numpy())
        return out


def _raise_for_status(status: int):
    if status == L.SDRF_PROB_NAN:
        raise ValueError(_MSG_NAN)
    if status == L.SDRF_PROB_SUM:
        raise ValueError(_MSG_SUM)
    if status == L.SDRF_REMOVE_NONEDGE:
        try:
            import networkx as nx
            raise nx.NetworkXError("The edge 0-0 is not in the graph")
        except ImportError:
            raise KeyError("The edge 0-0 is not in the graph")
    if status == L.SDRF_NO_UNIFORM:
        raise L.DcrError("ran out of uniforms (one is consumed per iteration that has candidates)")
    if status == L.SDRF_ARENA_FULL:
        raise L.DcrError("SDRF adjacency arena exhausted")
    if status == L.SDRF_EMPTY_GRAPH:
        raise ValueError("min() arg is an empty sequence")      # sdrf_no_cuda.py:26 on a graph without edges
    if status == L.SDRF_TOO_MANY_CANDIDATES:
        raise L.DcrError("candidate matrix (deg x + 1)(deg y + 1) exceeds the scratch of the SDRF state")
    raise L.DcrError(f"unexpected SDRF status {status}")


CLASSICAL_MODES = {"1d": L.SDRF_MODE_1D, "augmented": L.SDRF_MODE_AUGMENTED, "haantjes": L.SDRF_MODE_HAANTJES}


def _loop_mode(curv_type: str, is_undirected: bool):
    """``(L.SDRF_MODE_*, order)`` of the loop that runs ``curv_type``: ``order(edge_index, num_nodes)`` lists the input
    in the insertion order that loop starts from (``_new_state`` takes its result)."""
    if curv_type == "bfc":
        if is_undirected:    # G keeps self-loops (sdrf_cuda_bfc.py:31), A does not (:29)
            return L.SDRF_MODE_BFC, lambda ei, n: G.networkx_order(ei, n, keep_self_loops=True)
        return L.SDRF_MODE_BFC_DIRECTED, lambda ei, n: G.digraph_order(ei, n, keep_self_loops=True)
    if curv_type in CLASSICAL_MODES:
        return CLASSICAL_MODES[curv_type], lambda ei, n: G.classical_order(ei, n, keep_self_loops=True)
    raise Exception(f"Method {curv_type} not available.")    # classical_curvatures.py:27-28


def _new_state(mode: int, order: tuple, loops: int) -> SdrfState:
    """State of one run from its ``order`` (``_loop_mode``); the directed order also carries the predecessor lists."""
    return SdrfState(order[0], order[1], max(int(loops), 0), mode, *order[2:])


def _pad_uniforms(uniforms, loops: int):
    """``uniforms`` as fp64, padded with NaN ("not supplied") to ``loops`` values, and the number supplied."""
    u = np.ascontiguousarray(uniforms, dtype=np.float64)
    if u.size < loops:
        u = np.concatenate([u, np.full(loops - u.size, np.nan)])
    return u, int(np.count_nonzero(~np.isnan(u)))


def sdrf(edge_index, num_nodes: int, loops: int, remove_edges: bool, removal_bound: float, tau,
         uniforms: np.ndarray | None = None, guard: float = 1e-9, return_log: bool = False,
         state_out: list | None = None, is_undirected: bool = True, curv_type: str = "bfc"):
    """SDRF on the GPU.  Returns ``edge_index`` (int64 numpy) in the column order ``from_networkx`` produces, and with
    ``return_log`` the int32 ``[iters, 8]`` per-iteration log.

    ``curv_type='bfc'``: ``sdrf_cuda_bfc`` (rewiring/sdrf_cuda_bfc.py:14-93), undirected or — ``is_undirected=False`` —
    on the ``DiGraph`` of the input with single directed entries added / removed (:47-49, :72-73, :87-88).
    ``curv_type`` in ``'1d' | 'augmented' | 'haantjes'``: ``sdrf_no_cuda`` (rewiring/sdrf_no_cuda.py:9-68).

    ``uniforms``: the doubles ``np.random`` would produce (one per iteration that has candidates).  When omitted
    they are taken from numpy's global legacy generator exactly as the reference consumes it: the global state
    ends up advanced by the number of draws actually used.
    """
    L.require_cuda()
    mode, order = _loop_mode(curv_type, is_undirected)
    directed = mode == L.SDRF_MODE_BFC_DIRECTED
    state = _new_state(mode, order(edge_index, num_nodes), loops)
    own_stream = uniforms is None
    if own_stream:
        rng_state = np.random.get_state()
        uniforms = np.random.random_sample(max(int(loops), 0))
    uniforms, n_supplied = _pad_uniforms(uniforms, max(loops, 0))
    u_dev = torch.from_numpy(uniforms).to(state.device)
    logs = []
    done = draws = 0
    forced = -1
    try:
        while done < loops:
            res, log = state.run(loops - done, remove_edges, removal_bound, tau, u_dev[draws:n_supplied] if n_supplied > draws
                                 else u_dev[:0], forced_choice=forced, guard=guard)
            forced = -1
            done += res["iterations_done"]
            draws += res["draws_used"]
            if res["iterations_done"]:
                logs.append(log.cpu().numpy())
            if res["status"] == L.SDRF_OK:
                break
            if res["status"] == L.SDRF_NEED_HOST:
                imp = state.pending_improvements(res["pending_n"])
                forced = host_choice(imp, tau, float(uniforms[draws]))
                continue
            _raise_for_status(res["status"])
        out_rowptr, out_order = state.export()
    finally:
        if own_stream:   # advance numpy's global generator by exactly the draws the reference would have made
            np.random.set_state(rng_state)
            if draws:
                np.random.random_sample(draws)
        if state_out is not None:
            state_out.append(state)
        else:
            state.close()
    edge_index_out = (G.from_digraph_order if directed else G.from_networkx_order)(out_rowptr, out_order)
    if return_log:
        return edge_index_out, (np.concatenate(logs) if logs else np.zeros((0, L.SDRF_LOG_INTS), dtype=np.int32))
    return edge_index_out


def batch_workspace(count: int, device) -> torch.Tensor:
    """Device workspace for ``run_batch`` over up to ``count`` runs (8-byte aligned)."""
    nbytes = int(L.load().dcr_sdrf_batch_workspace_bytes(int(count)))
    return torch.empty(max(nbytes // 8, 1), dtype=torch.int64, device=device)


def run_batch(states, loops, removal_bounds, taus, uniforms, forced, logs, remove_edges: bool, guard: float,
              results: torch.Tensor, workspace: torch.Tensor):
    """One ``dcr_sdrf_run_batch`` launch: run ``b`` continues ``states[b]`` for up to ``loops[b]`` iterations, drawing
    from the device fp64 tensor ``uniforms[b]`` and logging into the device int32 tensor ``logs[b]`` (``[loops[b], 8]``,
    may be ``None`` when ``loops[b] == 0``).  ``results`` is a device int32 ``[>= B, 8]`` tensor.  Returns the B result
    dicts of ``SdrfState.run`` after ONE device-to-host copy."""
    b = len(states)
    runs = (L.SdrfBatchRun * b)()
    for i, s in enumerate(states):
        runs[i] = L.SdrfBatchRun(s.handle, int(loops[i]), int(forced[i]), float(removal_bounds[i]), float(taus[i]),
                                 uniforms[i].data_ptr(), int(uniforms[i].numel()), L.ptr(logs[i]),
                                 results[i].data_ptr())
    L.check(L.load().dcr_sdrf_run_batch(runs, b, int(bool(remove_edges)), float(guard), workspace.data_ptr(),
                                        workspace.numel() * workspace.element_size(), L.current_stream()),
            "dcr_sdrf_run_batch")
    return [dict(zip(_RESULT_KEYS, r)) for r in results[:b].cpu().tolist()]


def _per_run(name: str, value, count: int) -> list:
    is_seq = isinstance(value, (list, tuple)) or (isinstance(value, (np.ndarray, torch.Tensor)) and value.ndim > 0)
    if not is_seq:
        return [value] * count
    out = list(value)
    if len(out) != count:
        raise ValueError(f"{name}: {len(out)} values for a batch of {count} runs")
    return out


def sdrf_batch(edge_indices, num_nodes, loops, remove_edges: bool, removal_bound, tau, *, uniforms,
               guard: float = 1e-9, return_log: bool = False, is_undirected: bool = True, curv_type: str = "bfc",
               return_exceptions: bool = False):
    """B independent SDRF runs in one kernel launch, one CTA per run.  Run ``r`` computes exactly what
    ``sdrf(edge_indices[r], num_nodes[r], loops[r], remove_edges, removal_bound[r], tau[r], uniforms=uniforms[r],
    guard=guard, is_undirected=is_undirected, curv_type=curv_type)`` computes.

    ``edge_indices``: a list / tuple of B inputs, or ONE input (array or tensor) shared by every run (its networkx
    order is computed once).  ``num_nodes``, ``loops``, ``removal_bound``, ``tau``: scalars or length-B sequences.
    ``uniforms``: a ``[B, loops]`` array or a list of B 1-d arrays; it fixes B.  The batch never reads numpy's global
    generator (the draws of concurrent runs cannot be interleaved the way sequential calls would consume them).

    Runs that need a host-side decision (``guard``) re-enter together in the next launch; a failing run does not stop
    the others.  Returns a list of B ``edge_index`` arrays (and, with ``return_log``, a list of B logs).  A failed run
    raises after the batch — the lowest-index one, with the type and message ``sdrf`` raises — or, with
    ``return_exceptions``, leaves its exception in its ``edge_index`` slot (its log slot holds the iterations it
    completed)."""
    if isinstance(uniforms, np.ndarray) and uniforms.ndim != 2:
        raise ValueError("uniforms: a [B, loops] array or a list of B 1-d arrays")
    uni = [np.ascontiguousarray(u, dtype=np.float64) for u in uniforms]
    count = len(uni)
    if count < 1:
        raise ValueError("sdrf_batch: an empty batch")
    if any(u.ndim != 1 for u in uni):
        raise ValueError("uniforms: a [B, loops] array or a list of B 1-d arrays")
    shared_input = not isinstance(edge_indices, (list, tuple))
    inputs = [edge_indices] * count if shared_input else _per_run("edge_indices", edge_indices, count)
    nodes = [int(v) for v in _per_run("num_nodes", num_nodes, count)]
    iters = [max(int(v), 0) for v in _per_run("loops", loops, count)]
    bounds = [float(v) for v in _per_run("removal_bound", removal_bound, count)]
    taus = _per_run("tau", tau, count)
    mode, order = _loop_mode(curv_type, is_undirected)
    directed = mode == L.SDRF_MODE_BFC_DIRECTED
    L.require_cuda()

    orders = {}     # a shared input is put in order once per node count
    states = []
    try:
        for r in range(count):
            key = nodes[r] if shared_input else r
            if key not in orders:
                orders[key] = order(inputs[r], nodes[r])
            states.append(_new_state(mode, orders[key], iters[r]))
        dev = states[0].device
        padded, supplied = zip(*(_pad_uniforms(u, iters[r]) for r, u in enumerate(uni)))
        u_dev = [torch.from_numpy(u).to(dev) for u in padded]
        logs = [torch.empty((max(iters[r], 1), L.SDRF_LOG_INTS), dtype=torch.int32, device=dev) for r in range(count)]
        results = torch.zeros((count, 8), dtype=torch.int32, device=dev)
        workspace = batch_workspace(count, dev)
        done, draws, forced = [0] * count, [0] * count, [-1] * count
        errors = [None] * count
        active = [r for r in range(count) if iters[r] > 0]
        while active:
            res = run_batch([states[r] for r in active], [iters[r] - done[r] for r in active],
                            [bounds[r] for r in active], [taus[r] for r in active],
                            [u_dev[r][draws[r]:supplied[r]] if supplied[r] > draws[r] else u_dev[r][:0] for r in active],
                            [forced[r] for r in active], [logs[r][done[r]:] for r in active], remove_edges, guard,
                            results, workspace)
            again = []
            for r, rr in zip(active, res):
                forced[r] = -1
                done[r] += rr["iterations_done"]
                draws[r] += rr["draws_used"]
                try:
                    if rr["status"] == L.SDRF_NEED_HOST:
                        imp = states[r].pending_improvements(rr["pending_n"])
                        forced[r] = host_choice(imp, taus[r], float(padded[r][draws[r]]))
                        again.append(r)
                    elif rr["status"] != L.SDRF_OK:
                        _raise_for_status(rr["status"])
                except Exception as e:      # this run is over; the others go on
                    errors[r] = e
            active = again
        outs, out_logs = [], []
        for r in range(count):
            out_logs.append(logs[r][: done[r]].cpu().numpy())
            if errors[r] is not None:
                outs.append(errors[r])
                continue
            rp, od = states[r].export()
            outs.append((G.from_digraph_order if directed else G.from_networkx_order)(rp, od))
    finally:
        for s in states:
            s.close()
    if not return_exceptions:
        first = next((e for e in errors if e is not None), None)
        if first is not None:
            raise first
    return (outs, out_logs) if return_log else outs
