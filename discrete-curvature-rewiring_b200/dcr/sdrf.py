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
# the pairs each loop mode scores (dcr_sdrf_score_sizes), for the message of a rejected query
_QUERY_RULE = {
    L.SDRF_MODE_BFC: "node ids must lie in [0, n)",
    L.SDRF_MODE_BFC_DIRECTED: "node ids must lie in [0, n)",
    L.SDRF_MODE_1D: "not an edge of the graph (nor (u, u) of a node with a self-loop)",
    L.SDRF_MODE_AUGMENTED: "not an edge of the graph (nor (u, u) of a node with a self-loop)",
    L.SDRF_MODE_HAANTJES: "not an edge of the graph (nor (u, u) of a node with a self-loop)",
    L.SDRF_MODE_BFC_PAPER: "not an edge of the graph",
}


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

    @classmethod
    def _from_handle(cls, handle: C.c_void_p, like: "SdrfState") -> "SdrfState":
        """A state that owns ``handle``, a copy of ``like`` made by ``dcr_sdrf_fork``."""
        return cls._adopt(handle, like.lib, like.mode, like.n, like.n_self, like.device)

    @classmethod
    def _adopt(cls, handle: C.c_void_p, lib, mode: int, n: int, n_self: int, device) -> "SdrfState":
        self = cls.__new__(cls)
        self.lib, self.mode, self.n, self.n_self, self.device = lib, mode, n, n_self, device
        self._keep = None
        self.handle = handle
        self._result = torch.zeros(8, dtype=torch.int32, device=self.device)
        return self

    @classmethod
    def create_batch(cls, mode: int, num_nodes, rowptr: np.ndarray, order: np.ndarray, max_additions,
                     in_rowptr: np.ndarray | None = None, in_order: np.ndarray | None = None) -> list:
        """B states from one concatenated input with one ``dcr_sdrf_create_batch``: graph ``g`` has ``num_nodes[g]``
        rows of the int64 offsets ``rowptr`` (over all graphs' nodes, from 0) into ``order``, which lists LOCAL ids in
        insertion order (the directed mode: also the predecessor lists ``in_rowptr`` / ``in_order``), and the budget
        ``max_additions[g]``.  State ``g`` equals ``SdrfState`` of graph ``g`` alone; all share one device pool."""
        L.require_cuda()
        lib = L.load()
        nn = np.ascontiguousarray(num_nodes, dtype=np.int32)
        count = int(nn.size)
        rp = np.ascontiguousarray(rowptr, dtype=np.int64)
        od = np.ascontiguousarray(order, dtype=np.int32)
        ma = np.ascontiguousarray(max_additions, dtype=np.int64)
        if mode == L.SDRF_MODE_BFC_DIRECTED:
            irp = np.ascontiguousarray(in_rowptr, dtype=np.int64)
            iod = np.ascontiguousarray(in_order, dtype=np.int32)
        else:
            irp = iod = None
        handles = (C.c_void_p * max(count, 1))()
        L.check(lib.dcr_sdrf_create_batch(count, int(mode), nn.ctypes.data, rp.ctypes.data, od.ctypes.data if od.size else 0,
                                          irp.ctypes.data if irp is not None else 0,
                                          iod.ctypes.data if iod is not None and iod.size else 0, ma.ctypes.data, handles),
                "dcr_sdrf_create_batch")
        # nodes that list themselves, per graph (the neighbour / successor rows)
        graph_of_node = np.repeat(np.arange(count), nn)
        local = np.arange(nn.sum(), dtype=np.int64) - np.repeat(np.cumsum(nn, dtype=np.int64) - nn, nn)
        counts = np.diff(rp)
        is_self = od == np.repeat(local, counts)
        n_self = np.bincount(np.repeat(graph_of_node, counts)[is_self], minlength=count)
        device = torch.device("cuda", torch.cuda.current_device())
        return [cls._adopt(C.c_void_p(h), lib, int(mode), int(nn[g]), int(n_self[g]), device)
                for g, h in enumerate(handles[:count])]

    def fork(self, count: int) -> list:
        """``count`` independent copies of this state (graph, insertion order, curvature, budget) after one
        ``dcr_sdrf_fork``: device-to-device copies enqueued on the current stream, no host set-up."""
        count = int(count)
        handles = (C.c_void_p * max(count, 1))()
        L.check(self.lib.dcr_sdrf_fork(self.handle, count, handles, L.current_stream()), "dcr_sdrf_fork")
        return [SdrfState._from_handle(C.c_void_p(h), self) for h in handles[:count]]

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

    def edit(self, edits) -> dict:
        """Apply ``edits`` (``[m, 3]`` array or tensor of ``(op, u, v)``, op 1 = ``G.add_edge(u, v)``, 0 =
        ``G.remove_edge(u, v)``) in order with one launch, refreshing the curvature they change (``dcr_sdrf_edit``).
        Returns the result dict after one device-to-host copy: ``iterations_done`` is the number of edits applied;
        a status other than ``SDRF_OK`` names the edit it stopped before in ``pending_x`` / ``pending_y``."""
        e = edit_tensor(edits).to(self.device).contiguous()
        L.check(self.lib.dcr_sdrf_edit(self.handle, L.ptr(e) if e.numel() else 0, int(e.shape[0]),
                                       self._result.data_ptr(), L.current_stream()), "dcr_sdrf_edit")
        return dict(zip(_RESULT_KEYS, self._result.cpu().tolist()))

    def score(self, pairs: torch.Tensor, max_cells: int | None = None) -> dict:
        """Candidate scores of the Q >= 1 pairs ``(x, y)`` of the device int32 ``[Q, 2]`` tensor ``pairs``
        (``dcr_sdrf_score_sizes``, one read of the totals, ``dcr_sdrf_score``).  Returns device tensors:
        ``sizes`` int32 ``[Q, 2]`` ``(n_i, n_j)``; ``cand_offsets`` / ``cell_offsets`` int64 ``[Q + 1]``; ``cand`` int32
        (query q: its ``n_i`` row ids, then its ``n_j`` column ids); ``imp`` fp64 cells, row-major per query, a masked cell
        with all bits set; ``best`` int64 ``[Q, 4]``, the ``dcr_sdrf_score_best`` records.  Raises ``ValueError`` for the
        first pair this mode's loop cannot score, or when the cells exceed ``max_cells``, before the scoring launch."""
        q = int(pairs.shape[0])
        dev = self.device
        sizes = torch.empty((q, 2), dtype=torch.int32, device=dev)
        status = torch.empty(q, dtype=torch.int32, device=dev)
        L.check(self.lib.dcr_sdrf_score_sizes(self.handle, pairs.data_ptr(), q, sizes.data_ptr(), status.data_ptr(),
                                              L.current_stream()), "dcr_sdrf_score_sizes")
        s64 = sizes.to(torch.int64)
        cell_offsets = torch.zeros(q + 1, dtype=torch.int64, device=dev)
        cand_offsets = torch.zeros(q + 1, dtype=torch.int64, device=dev)
        torch.cumsum(s64[:, 0] * s64[:, 1], 0, out=cell_offsets[1:])
        torch.cumsum(s64.sum(1), 0, out=cand_offsets[1:])
        bad = status != L.SDRF_OK
        first_bad = torch.where(bad.any(), torch.argmax(bad.to(torch.int32)), -1)
        cells, cands, first_bad = torch.stack([cell_offsets[-1], cand_offsets[-1], first_bad]).cpu().tolist()
        if first_bad >= 0:
            st, (x, y) = int(status[first_bad]), pairs[first_bad].tolist()
            if st != L.SDRF_BAD_QUERY:
                _raise_for_status(st)
            raise ValueError(f"pairs[{first_bad}] = ({x}, {y}): {_QUERY_RULE[self.mode]}")
        if max_cells is not None and cells > max_cells:
            raise ValueError(f"the {q} queries have {cells} candidate cells, more than max_cells = {max_cells} "
                             f"({8 * cells + 4 * cands} bytes of output)")
        cand = torch.empty(max(cands, 1), dtype=torch.int32, device=dev)
        imp = torch.empty(max(cells, 1), dtype=torch.float64, device=dev)
        best = torch.empty((q, 4), dtype=torch.int64, device=dev)
        nbytes = int(self.lib.dcr_sdrf_score_workspace_bytes(self.handle, q))
        workspace = torch.empty(max(nbytes // 4, 1), dtype=torch.int32, device=dev)
        L.check(self.lib.dcr_sdrf_score(self.handle, pairs.data_ptr(), q, cell_offsets.data_ptr(), cand_offsets.data_ptr(),
                                        cand.data_ptr(), imp.data_ptr(), best.data_ptr(), workspace.data_ptr(), nbytes,
                                        L.current_stream()), "dcr_sdrf_score")
        return {"sizes": sizes, "cand_offsets": cand_offsets, "cell_offsets": cell_offsets, "cand": cand[:cands],
                "imp": imp[:cells], "best": best}

    def pending_improvements(self, n: int) -> np.ndarray:
        out = torch.empty(max(n, 1), dtype=torch.float64, device=self.device)
        L.check(self.lib.dcr_sdrf_pending_improvements(self.handle, out.data_ptr(), int(n), L.current_stream()),
                "dcr_sdrf_pending_improvements")
        return out[:n].cpu().numpy()

    def nnz(self) -> int:
        return int(self.lib.dcr_sdrf_nnz(self.handle))

    def export(self, with_curvature: bool = False):
        """Current graph: ``(rowptr, order)`` numpy (networkx order); with curvature also sorted col / c32 / tri.  The
        paper-flavour mode (``L.SDRF_MODE_BFC_PAPER``) keeps no fp32 curvature and no supports: its curvature is the fp64
        ``bfc_edge`` value of every entry (sorted order) and ``tri`` is ``None``."""
        nnz = self.nnz()
        dev = self.device
        rowptr = torch.empty(self.n + 1, dtype=torch.int32, device=dev)
        if with_curvature and self.mode == L.SDRF_MODE_BFC_PAPER:
            order = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
            col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
            c64 = torch.empty(max(nnz, 1), dtype=torch.float64, device=dev)
            L.check(self.lib.dcr_sdrf_export(self.handle, rowptr.data_ptr(), order.data_ptr(), col.data_ptr(), 0, 0,
                                             L.current_stream()), "dcr_sdrf_export")
            L.check(self.lib.dcr_sdrf_export_c64(self.handle, rowptr.data_ptr(), c64.data_ptr(), L.current_stream()),
                    "dcr_sdrf_export_c64")
            return (rowptr.cpu().numpy(), order[:nnz].cpu().numpy(), col[:nnz].cpu().numpy(), c64[:nnz].cpu().numpy(),
                    None)
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

    def edge_index(self) -> torch.Tensor:
        """The current graph as the int64 ``[2, E]`` device tensor ``from_networkx(G).edge_index`` gives, in the column
        order ``sdrf()`` returns (``dcr_sdrf_export_edge_index``)."""
        cap = self.nnz() + self.n_self
        rowptr = torch.empty(self.n + 1, dtype=torch.int32, device=self.device)
        out = torch.empty((2, max(cap, 1)), dtype=torch.int64, device=self.device)
        L.check(self.lib.dcr_sdrf_export_edge_index(self.handle, rowptr.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                                                    cap, L.current_stream()), "dcr_sdrf_export_edge_index")
        return out[:, : int(rowptr[-1])]


def export_edge_index_batch(states, node_offsets, capacity: int):
    """``SdrfState.edge_index`` of every state into one output with ``dcr_sdrf_export_edge_index_batch``: state ``b``'s
    columns follow state ``b-1``'s with node ids shifted by ``node_offsets[b]``.  Returns the device int64 ``[2, capacity]``
    output and the device int64 ``edge_ptr[B + 1]``; the columns are ``[:, :edge_ptr[B]]`` (``capacity`` bounds it)."""
    count = len(states)
    lib = L.load()
    dev = states[0].device
    handles = (C.c_void_p * count)(*[s.handle.value for s in states])
    offs = np.ascontiguousarray(node_offsets, dtype=np.int64)
    out = torch.empty((2, max(int(capacity), 1)), dtype=torch.int64, device=dev)
    edge_ptr = torch.empty(count + 1, dtype=torch.int64, device=dev)
    nbytes = int(lib.dcr_sdrf_export_edge_index_batch_workspace_bytes(handles, count))
    workspace = torch.empty(max(nbytes // 8, 1), dtype=torch.int64, device=dev)
    L.check(lib.dcr_sdrf_export_edge_index_batch(handles, count, offs.ctypes.data, out[0].data_ptr(), out[1].data_ptr(),
                                                 int(capacity), edge_ptr.data_ptr(), workspace.data_ptr(), nbytes,
                                                 L.current_stream()), "dcr_sdrf_export_edge_index_batch")
    return out, edge_ptr


def edit_tensor(edits) -> torch.Tensor:
    """``edits`` (array or tensor) as the int32 ``[m, 3]`` tensor ``dcr_sdrf_edit`` reads; ``ValueError`` for another
    shape, a non-integer type or a value int32 cannot hold (the cast would wrap it into another id)."""
    e = torch.as_tensor(edits)
    if e.numel() == 0:
        e = e.reshape(0, 3).to(torch.int32)
    if e.ndim != 2 or e.shape[1] != 3:
        raise ValueError(f"edits: an [m, 3] array of (op, u, v), got shape {tuple(e.shape)}")
    if e.is_floating_point() or e.is_complex() or e.dtype == torch.bool:
        raise ValueError(f"edits: integer (op, u, v) expected, got {e.dtype}")
    if e.numel() and e.dtype != torch.int32 and (int(e.min()) < -2**31 or int(e.max()) > 2**31 - 1):
        raise ValueError("edits: a value does not fit int32")
    return e.to(torch.int32)


def _raise_for_status(status: int, pair=(0, 0)):
    """Raise what the reference raises for a loop status; ``pair`` is the edge a failed removal or edit named."""
    if status == L.SDRF_PROB_NAN:
        raise ValueError(_MSG_NAN)
    if status == L.SDRF_PROB_SUM:
        raise ValueError(_MSG_SUM)
    if status == L.SDRF_REMOVE_NONEDGE:
        try:
            import networkx as nx
            raise nx.NetworkXError(f"The edge {pair[0]}-{pair[1]} is not in the graph")
        except ImportError:
            raise KeyError(f"The edge {pair[0]}-{pair[1]} is not in the graph")
    if status == L.SDRF_NO_UNIFORM:
        raise L.DcrError("ran out of uniforms (one is consumed per iteration that has candidates)")
    if status == L.SDRF_ARENA_FULL:
        raise L.DcrError("SDRF adjacency arena exhausted")
    if status == L.SDRF_EMPTY_GRAPH:
        raise ValueError("min() arg is an empty sequence")      # sdrf_no_cuda.py:26 on a graph without edges
    if status == L.SDRF_TOO_MANY_CANDIDATES:
        raise L.DcrError("candidate matrix (deg x + 1)(deg y + 1) exceeds the scratch of the SDRF state")
    if status == L.SDRF_BAD_EDIT:
        raise ValueError(f"edit ({pair[0]}, {pair[1]}): a self-loop or a node id out of range")
    raise L.DcrError(f"unexpected SDRF status {status}")


CLASSICAL_MODES = {"1d": L.SDRF_MODE_1D, "augmented": L.SDRF_MODE_AUGMENTED, "haantjes": L.SDRF_MODE_HAANTJES}


def _paper_order(edge_index, num_nodes: int):
    """``classical_order`` for ``curv_type='bfc_paper'``: bfc_naive.bfc_edge counts a node's degree and neighbours the
    networkx way, which gives a self-loop no meaning in the curvature, so an input with one is refused."""
    rowptr, order = G.classical_order(edge_index, num_nodes, keep_self_loops=True)
    rows = np.repeat(np.arange(rowptr.size - 1), np.diff(rowptr.astype(np.int64)))
    if np.any(order == rows):
        raise NotImplementedError("curv_type='bfc_paper' does not take graphs with self-loops")
    return rowptr, order


def _loop_mode(curv_type: str, is_undirected: bool):
    """``(L.SDRF_MODE_*, order)`` of the loop that runs ``curv_type``: ``order(edge_index, num_nodes)`` lists the input
    in the insertion order that loop starts from (``_new_state`` takes its result)."""
    if curv_type == "bfc":
        if is_undirected:    # G keeps self-loops (sdrf_cuda_bfc.py:31), A does not (:29)
            return L.SDRF_MODE_BFC, lambda ei, n: G.networkx_order(ei, n, keep_self_loops=True)
        return L.SDRF_MODE_BFC_DIRECTED, lambda ei, n: G.digraph_order(ei, n, keep_self_loops=True)
    if curv_type in CLASSICAL_MODES:
        return CLASSICAL_MODES[curv_type], lambda ei, n: G.classical_order(ei, n, keep_self_loops=True)
    if curv_type == "bfc_paper":
        if not is_undirected:
            raise NotImplementedError("curv_type='bfc_paper' runs on undirected graphs only")
        return L.SDRF_MODE_BFC_PAPER, _paper_order
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
    ``curv_type='bfc_paper'``: ``sdrf_no_cuda``'s loop with the paper-flavour curvature ``bfc_naive.bfc_edge``
    (curvature/bfc_naive.py:7-40) in fp64; undirected inputs without self-loops (``NotImplementedError`` otherwise).

    ``uniforms``: the doubles ``np.random`` would produce (one per iteration that has candidates).  When omitted
    they are taken from numpy's global legacy generator exactly as the reference consumes it: the global state
    ends up advanced by the number of draws actually used.
    """
    L.require_cuda()
    mode, order = _loop_mode(curv_type, is_undirected)
    directed = mode == L.SDRF_MODE_BFC_DIRECTED
    state = _new_state(mode, order(edge_index, num_nodes), loops)
    try:
        log = _run_state(state, loops, remove_edges, removal_bound, tau, uniforms, guard)
        out_rowptr, out_order = state.export()
    finally:
        if state_out is not None:
            state_out.append(state)
        else:
            state.close()
    edge_index_out = (G.from_digraph_order if directed else G.from_networkx_order)(out_rowptr, out_order)
    if return_log:
        return edge_index_out, log
    return edge_index_out


def _run_state(state: SdrfState, loops: int, remove_edges: bool, removal_bound: float, tau, uniforms, guard: float):
    """Up to ``loops`` iterations of the loop on ``state`` with ``sdrf``'s host protocol: launches until the loop is
    done, re-deciding on the host every draw the kernel hands back (``NEED_HOST``) and raising the reference's
    exception for a failed one.  ``uniforms=None`` draws from numpy's global legacy generator and leaves it advanced
    by exactly the draws used, also when this raises.  Returns the int32 ``[iters, 8]`` log."""
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
    finally:
        if own_stream:   # advance numpy's global generator by exactly the draws the reference would have made
            np.random.set_state(rng_state)
            if draws:
                np.random.random_sample(draws)
    return np.concatenate(logs) if logs else np.zeros((0, L.SDRF_LOG_INTS), dtype=np.int32)


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


def edit_batch_states(states, edits) -> list:
    """One ``dcr_sdrf_edit_batch`` launch: ``states[b]`` applies ``edits[b]`` (an ``[m, 3]`` array of ``(op, u, v)``, see
    ``SdrfState.edit``).  Returns the B result dicts of ``SdrfState.edit`` after ONE device-to-host copy."""
    b = len(states)
    dev = states[0].device
    host = [edit_tensor(e).cpu() for e in edits]
    counts = [int(e.shape[0]) for e in host]
    offsets = np.concatenate([[0], np.cumsum(counts)]).tolist()
    flat = torch.cat(host).to(dev)            # every edit list in one host-to-device copy
    results = torch.zeros((b, 8), dtype=torch.int32, device=dev)
    nbytes = int(L.load().dcr_sdrf_edit_batch_workspace_bytes(b))
    workspace = torch.empty(max(nbytes // 8, 1), dtype=torch.int64, device=dev)
    runs = (L.SdrfEditRun * b)()
    for i, s in enumerate(states):
        ptr = flat.data_ptr() + 3 * 4 * offsets[i] if counts[i] else 0
        runs[i] = L.SdrfEditRun(s.handle, ptr, counts[i], results[i].data_ptr())
    L.check(L.load().dcr_sdrf_edit_batch(runs, b, workspace.data_ptr(), workspace.numel() * workspace.element_size(),
                                         L.current_stream()), "dcr_sdrf_edit_batch")
    return [dict(zip(_RESULT_KEYS, r)) for r in results.cpu().tolist()]


def _batch_uniforms(uniforms, caller: str) -> list:
    """``uniforms`` of a batch (a ``[B, loops]`` array or a list of B 1-d arrays) as B fp64 arrays; B >= 1.  ``caller``
    names the public function in the errors."""
    if isinstance(uniforms, np.ndarray) and uniforms.ndim != 2:
        raise ValueError("uniforms: a [B, loops] array or a list of B 1-d arrays")
    uni = [np.ascontiguousarray(u, dtype=np.float64) for u in uniforms]
    if len(uni) < 1:
        raise ValueError(f"{caller}: an empty batch")
    if any(u.ndim != 1 for u in uni):
        raise ValueError("uniforms: a [B, loops] array or a list of B 1-d arrays")
    return uni


def _run_batch_states(states, iters, bounds, taus, uni, remove_edges: bool, guard: float):
    """Run ``r`` continues ``states[r]`` for up to ``iters[r]`` iterations with the uniforms ``uni[r]``, all runs in
    one ``dcr_sdrf_run_batch`` launch; runs that need a host-side decision re-enter together in the next launch, and a
    failing run does not stop the others.  Returns ``(logs, done, errors)``: the device logs, the iterations each run
    completed and, per run, ``None`` or the exception ``sdrf`` raises for it."""
    count = len(states)
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
    return logs, done, errors


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
    uni = _batch_uniforms(uniforms, "sdrf_batch")
    count = len(uni)
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
        logs, done, errors = _run_batch_states(states, iters, bounds, taus, uni, remove_edges, guard)
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
    return _batch_return(outs, out_logs, errors, return_log, return_exceptions)


def _batch_return(outs, out_logs, errors, return_log: bool, return_exceptions: bool):
    """A batch's return value: the lowest-index failure is raised unless ``return_exceptions`` (then it stays in its
    run's slot of ``outs``)."""
    if not return_exceptions:
        first = next((e for e in errors if e is not None), None)
        if first is not None:
            raise first
    return (outs, out_logs) if return_log else outs


# log fields that hold node ids (dcr.h: {x, y, n_candidates, k, l, choice, removed_x, removed_y}; -1 = none)
_LOG_NODE_FIELDS = [0, 1, 3, 4, 6, 7]


def dataset_ptr(ptr, count: int) -> np.ndarray:
    """``ptr`` of a batched dataset (PyG ``Batch.ptr``: graph ``g`` owns the nodes ``ptr[g] .. ptr[g+1] - 1``) as int64
    numpy, checked against ``count`` graphs; ``ValueError`` naming the graph for a non-monotone ``ptr`` or an empty
    graph."""
    p = ptr.detach().cpu().numpy() if hasattr(ptr, "detach") else np.asarray(ptr)
    if p.ndim != 1 or p.size < 2 or p.dtype.kind not in "iu":
        raise ValueError("ptr: a 1-d integer array of B + 1 node offsets")
    p = p.astype(np.int64)
    if p.size - 1 != count:
        raise ValueError(f"ptr describes {p.size - 1} graphs, the batch has {count} runs")
    if p[0] != 0:
        raise ValueError(f"ptr[0] = {p[0]}: the node offsets start at 0")
    d = np.diff(p)
    if (d < 0).any():
        g = int(np.flatnonzero(d < 0)[0])
        raise ValueError(f"graph {g}: ptr is not monotone (ptr[{g}] = {p[g]} > ptr[{g + 1}] = {p[g + 1]})")
    if (d == 0).any():
        g = int(np.flatnonzero(d == 0)[0])
        raise ValueError(f"graph {g} has no nodes (ptr[{g}] = ptr[{g + 1}] = {p[g]})")
    if d.max() > 2**31 - 1:
        g = int(np.argmax(d))
        raise ValueError(f"graph {g} has {d[g]} nodes, more than int32 ids can name")
    return p


def _column_graphs(ei: np.ndarray, p: np.ndarray) -> np.ndarray:
    """The graph of every column of the global ``edge_index`` ``ei``; ``ValueError`` naming the column and graph for an
    endpoint outside ``[0, ptr[B])`` or a column joining two graphs."""
    total = int(p[-1])
    outside = (ei < 0) | (ei >= total)
    if outside.any():
        t = int(np.flatnonzero(outside.any(0))[0])
        u, v = (int(x) for x in ei[:, t])
        inside = v if outside[0, t] else u
        where = (f"; its other endpoint lies in graph {int(np.searchsorted(p, inside, side='right')) - 1}"
                 if not outside[:, t].all() else "")
        raise ValueError(f"edge_index column {t} = ({u}, {v}) has a node outside [0, {total}){where}")
    gu = np.searchsorted(p, ei[0], side="right") - 1
    gv = np.searchsorted(p, ei[1], side="right") - 1
    if (gu != gv).any():
        t = int(np.flatnonzero(gu != gv)[0])
        raise ValueError(f"edge_index column {t} = ({ei[0, t]}, {ei[1, t]}) joins graph {gu[t]} and graph {gv[t]}")
    return gu


def _dataset_order(order, mode: int, ei: np.ndarray, p: np.ndarray, gid: np.ndarray) -> list:
    """``order`` (``_loop_mode``) computed ONCE on the disjoint union of the graphs, as ``create_batch`` takes it: int64
    row offsets over all nodes and LOCAL ids.  The order functions rank a column only against columns of the same source
    (or pair), all of one graph, and keep their relative order, so the union's rows are each graph's own rows.  A mode's
    input error names the graph it comes from."""
    try:
        lists = order(ei, int(p[-1]))
    except NotImplementedError as e:
        if mode == L.SDRF_MODE_BFC_PAPER:
            t = int(np.flatnonzero(ei[0] == ei[1])[0])             # a self-loop
        else:                                                      # a repeated directed pair
            _, first = np.unique(ei[0] * int(p[-1]) + ei[1], return_index=True)
            repeat = np.ones(ei.shape[1], dtype=bool)
            repeat[first] = False
            t = int(np.flatnonzero(repeat)[0])
        raise NotImplementedError(f"graph {gid[t]}: {e}") from None
    node_base = np.repeat(p[:-1], np.diff(p))                     # first node of the graph of every node
    out = []
    for rowptr, od in zip(lists[0::2], lists[1::2]):
        rowptr = np.asarray(rowptr, dtype=np.int64)
        out += [rowptr, (od - np.repeat(node_base, np.diff(rowptr))).astype(np.int32)]
    return out


def sdrf_dataset(edge_index, ptr, loops, remove_edges: bool, removal_bound, tau, *, uniforms, guard: float = 1e-9,
                 return_log: bool = False, is_undirected: bool = True, curv_type: str = "bfc",
                 return_exceptions: bool = False):
    """SDRF on every graph of a batched dataset (PyG layout: ``edge_index`` in global node ids, graph ``g`` owns the
    nodes ``ptr[g] .. ptr[g+1] - 1``), one CTA per graph in one launch.  Graph ``g``'s result is what
    ``sdrf(ei_g - ptr[g], ptr[g+1] - ptr[g], loops[g], remove_edges, removal_bound[g], tau[g], uniforms=uniforms[g],
    guard=guard, is_undirected=is_undirected, curv_type=curv_type)`` computes on its columns ``ei_g`` alone, shifted back
    by ``ptr[g]`` (in the edge_index and in the node ids of the log).

    ``loops``, ``removal_bound``, ``tau``: scalars or per-graph sequences; ``uniforms``: a ``[B, loops]`` array or a list
    of B 1-d arrays.  The insertion order is computed once on the whole input, all states are set up by one
    ``dcr_sdrf_create_batch`` and exported by one ``dcr_sdrf_export_edge_index_batch``.

    Returns ``(edge_index, edge_ptr)``: the device int64 ``[2, E']`` rewired dataset, graph ``g`` in the columns
    ``edge_ptr[g] .. edge_ptr[g+1] - 1`` of the device int64 ``edge_ptr[B + 1]``; with ``return_log`` also the list of
    B logs.  A failing graph does not stop the others; the lowest-index failure is raised afterwards with ``sdrf``'s
    type and message, or, with ``return_exceptions``, the graph is left empty in ``edge_ptr`` and the list of B
    exceptions (``None`` for a graph that succeeded) is appended to the return value.  The input is checked before
    anything is allocated: ``ValueError`` naming the graph for a column between two graphs or outside ``[0, ptr[B])``,
    a non-monotone ``ptr`` or a graph without nodes."""
    uni = _batch_uniforms(uniforms, "sdrf_dataset")
    count = len(uni)
    p = dataset_ptr(ptr, count)
    ei = G._as_numpy_edge_index(edge_index)
    gid = _column_graphs(ei, p)
    iters = [max(int(v), 0) for v in _per_run("loops", loops, count)]
    bounds = [float(v) for v in _per_run("removal_bound", removal_bound, count)]
    taus = _per_run("tau", tau, count)
    mode, order = _loop_mode(curv_type, is_undirected)
    lists = _dataset_order(order, mode, ei, p, gid)
    L.require_cuda()
    states = SdrfState.create_batch(mode, np.diff(p), lists[0], lists[1], iters, *lists[2:])
    try:
        logs, done, errors = _run_batch_states(states, iters, bounds, taus, uni, remove_edges, guard)
        first = next((e for e in errors if e is not None), None)
        if first is not None and not return_exceptions:
            raise first
        ok = [g for g in range(count) if errors[g] is None]
        dev = states[0].device
        if ok:
            entries = lists[0][p[1:]] - lists[0][p[:-1]]          # insertion-order entries at set-up, per graph
            cap = sum(int(entries[g]) + 2 * done[g] for g in ok)   # an iteration adds at most two
            out, ok_ptr = export_edge_index_batch([states[g] for g in ok], p[ok], cap)
        else:
            out, ok_ptr = torch.zeros((2, 0), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
        # a failed graph repeats the offset before it
        idx = torch.from_numpy(np.concatenate([[0], np.cumsum([e is None for e in errors])])).to(dev)
        edge_ptr = ok_ptr[idx]
        edge_index_out = out[:, : int(edge_ptr[-1])]
        result = [edge_index_out, edge_ptr]
        if return_log:
            flat = torch.cat([logs[g][: done[g]] for g in range(count)]).cpu().numpy()
            node = flat[:, _LOG_NODE_FIELDS]
            shift = np.repeat(p[:-1], done)[:, None]
            flat[:, _LOG_NODE_FIELDS] = np.where(node >= 0, node + shift, node)
            result.append(np.split(flat, np.cumsum(done)[:-1]))
        if return_exceptions:
            result.append(errors)
        return tuple(result)
    finally:
        for s in states:
            s.close()
