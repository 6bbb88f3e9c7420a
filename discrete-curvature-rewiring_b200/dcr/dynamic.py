"""Curvature of a device-resident graph under caller edits, and SDRF resumed from the edited graph.

``DynamicCurvature`` keeps one SDRF loop state (``dcr.sdrf.SdrfState``): the dynamic adjacency in networkx insertion
order plus the exact curvature of every edge, for any ``curv_type`` / ``is_undirected`` that ``sdrf()`` takes.  Edits
are applied on the device by ``dcr_sdrf_edit`` with the loop's own toggle, so the graph keeps exactly the insertion
order the same ``G.add_edge`` / ``G.remove_edge`` calls give the reference's ``G``, and only the curvature of the edges
an edit can change is recomputed.  ``rewire`` continues SDRF from the current graph (DESIGN §4.10).
"""
from __future__ import annotations

import copy

import numpy as np
import torch

from . import lib as L
from .sdrf import (CLASSICAL_MODES, _batch_return, _batch_uniforms, _loop_mode, _new_state, _per_run, _raise_for_status,
                   _run_batch_states, _run_state, edit_batch_states)

_INT32_MAX = 2**31 - 1
_MASKED64 = np.uint64(0xFFFFFFFFFFFFFFFF)      # a masked cell of dcr_sdrf_score


def align_to_columns(rowptr: np.ndarray, col: np.ndarray, values: np.ndarray, edge_index: np.ndarray,
                     loop_values: np.ndarray | None = None) -> np.ndarray:
    """``values`` of the sorted entries (row ``r``, ``col[p]``) of the CSR ``rowptr / col`` at every column ``(u, v)`` of
    ``edge_index``; a loop column ``(u, u)``, which the CSR does not hold, takes ``loop_values[u]`` (0 when omitted)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    n = rowptr.size - 1
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rowptr))
    keys = rows * n + col                                       # ascending: rows in order, each row sorted
    u, v = np.asarray(edge_index, dtype=np.int64)
    loop = u == v
    want = u * n + v
    pos = np.minimum(np.searchsorted(keys, want), max(keys.size - 1, 0))
    if keys.size:
        found = keys[pos] == want
    else:
        found = np.zeros(want.size, dtype=bool)
    if np.any(~found & ~loop):
        raise ValueError("align_to_columns: a column of edge_index is not an entry of the CSR")
    values = np.asarray(values)
    out = values[pos] if values.size else np.zeros(want.size, dtype=values.dtype)
    out = out.copy()
    if loop.any():
        out[loop] = 0 if loop_values is None else np.asarray(loop_values)[u[loop]]
    return out


def classical_loop_values(degrees: np.ndarray, curv_type: str) -> np.ndarray:
    """``compute_curvature_edge(G, (u, u))`` of a loop edge at a node with ``degrees[u]`` other neighbours: networkx
    counts the loop twice in the degree (d + 2) and the node is its own neighbour (d + 1 common neighbours)."""
    d = np.asarray(degrees, dtype=np.int64)
    if curv_type == "1d":
        return 4 - 2 * (d + 2)
    if curv_type == "augmented":
        return 4 - 2 * (d + 2) + 3 * (d + 1)
    return d + 1                                                # 'haantjes'


def edit_array(ops) -> np.ndarray:
    """``ops`` as an int64 ``[m, 3]`` array of ``(op, u, v)``; raises ``ValueError`` for another shape or an op other
    than 1 (add) / 0 (remove).  Node ids are checked on the device, in order (see :meth:`DynamicCurvature.edit`)."""
    e = ops.detach().cpu().numpy() if isinstance(ops, torch.Tensor) else np.asarray(ops)
    if e.size == 0:
        e = e.reshape(0, 3).astype(np.int64)
    if e.ndim != 2 or e.shape[1] != 3:
        raise ValueError(f"edits: an [m, 3] array of (op, u, v), got shape {e.shape}")
    if not np.issubdtype(e.dtype, np.integer):
        raise ValueError(f"edits: integer (op, u, v) expected, got {e.dtype}")
    e = e.astype(np.int64)
    if not np.isin(e[:, 0], (0, 1)).all():
        raise ValueError("edits: op must be 1 (add) or 0 (remove)")
    return e


def pair_array(pairs) -> np.ndarray:
    p = pairs.detach().cpu().numpy() if isinstance(pairs, torch.Tensor) else np.asarray(pairs)
    if p.size == 0:
        p = p.reshape(0, 2).astype(np.int64)
    if p.ndim != 2 or p.shape[1] != 2:
        raise ValueError(f"pairs: an [m, 2] array of (u, v), got shape {p.shape}")
    return p


class DynamicCurvature:
    """A graph on the device whose curvature stays current under edits.

    ``DynamicCurvature(edge_index, num_nodes, curv_type, is_undirected, capacity)`` sets the graph up exactly as
    ``sdrf(edge_index, num_nodes, ..., is_undirected=is_undirected, curv_type=curv_type)`` does (same modes, same
    input errors).  ``capacity`` is the additions budget: every add edit counts against it, also one that finds the edge
    present (add, remove, add of one pair counts 2), and so does every edge ``rewire`` adds.
    """

    def __init__(self, edge_index, num_nodes: int, curv_type: str = "bfc", is_undirected: bool = True,
                 capacity: int = 1024):
        L.require_cuda()
        mode, order = _loop_mode(curv_type, is_undirected)
        if int(capacity) < 0:
            raise ValueError(f"capacity must be >= 0, got {capacity}")
        self.curv_type = curv_type
        self.mode = mode
        self.directed = mode == L.SDRF_MODE_BFC_DIRECTED
        self.capacity = int(capacity)
        self._state = _new_state(mode, order(edge_index, num_nodes), self.capacity)
        self.n = self._state.n
        self._edit_adds = 0      # add edits applied (the state's own count)
        self._loop_adds = 0      # edges added by rewire()

    # ---- life cycle ---------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_state", None) is not None:
            self._state.close()
            self._state = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def fork(self, count: int = 1) -> list:
        """``count`` independent copies of this object (graph, insertion order, curvature, budget) made on the device
        with one ``dcr_sdrf_fork``; each is closed on its own."""
        out = []
        for st in self._state.fork(count):
            dc = copy.copy(self)
            dc._state = st
            out.append(dc)
        return out

    @property
    def remaining(self) -> int:
        """Additions left in the budget."""
        return self.capacity - self._edit_adds - self._loop_adds

    # ---- edits --------------------------------------------------------------------------------------------------
    def edit(self, ops) -> int:
        """Apply ``ops`` (``[m, 3]``: ``(1, u, v)`` = ``G.add_edge(u, v)``, ``(0, u, v)`` = ``G.remove_edge(u, v)``) in
        order in one launch and return how many were applied (all of them, or it raises).  A failing edit stops the
        batch before it, the edits before it stay applied and the object stays usable: ``networkx.NetworkXError`` for
        removing a non-edge, ``ValueError`` for a self-loop or an id outside ``[0, n)``, ``DcrError`` for an add beyond
        the budget."""
        e, stop, dev = self._prepare_edits(ops)
        return self._finish_edits(e, stop, self._state.edit(dev))

    def _prepare_edits(self, ops):
        """``(e, stop, dev)``: ``ops`` checked (:func:`edit_array`), the index of the first add beyond the budget (or
        ``m``) and the edits before it as the device takes them."""
        e = edit_array(ops)
        is_add = e[:, 0] == 1
        over = np.flatnonzero(is_add & (np.cumsum(is_add) > self.remaining))
        stop = int(over[0]) if over.size else e.shape[0]
        # the state counts its add edits against `capacity`, not the edges rewire() added: those are charged here by
        # ending the batch before the first add beyond the budget
        dev = e[:stop].copy()
        ids = dev[:, 1:]
        ids[(ids < 0) | (ids > _INT32_MAX)] = -1        # an id int32 cannot hold: out of range for the device as well
        return e, stop, dev

    def _finish_edits(self, e, stop: int, res: dict) -> int:
        """Count the add edits the device applied (``res``) and raise for the edit it stopped before, or for the first
        add beyond the budget; returns the number applied."""
        applied = res["iterations_done"]
        self._edit_adds += int(np.count_nonzero(e[:applied, 0] == 1))
        if res["status"] != L.SDRF_OK:                  # it stopped before edit `applied`: name that edit as given
            _raise_for_status(res["status"], tuple(int(x) for x in e[applied, 1:]))
        if stop < e.shape[0]:
            _, u, v = (int(x) for x in e[stop])
            if u == v or not (0 <= u < self.n and 0 <= v < self.n):
                _raise_for_status(L.SDRF_BAD_EDIT, (u, v))
            raise L.DcrError(f"edit {stop}: add ({u}, {v}) exceeds the additions budget (capacity {self.capacity})")
        return applied

    def add_edges(self, pairs) -> int:
        """``G.add_edge(u, v)`` for every row of the ``[m, 2]`` array ``pairs``, in order (see :meth:`edit`)."""
        p = pair_array(pairs)
        return self.edit(np.concatenate([np.ones((p.shape[0], 1), dtype=np.int64), p.astype(np.int64)], axis=1))

    def remove_edges(self, pairs) -> int:
        """``G.remove_edge(u, v)`` for every row of the ``[m, 2]`` array ``pairs``, in order (see :meth:`edit`)."""
        p = pair_array(pairs)
        return self.edit(np.concatenate([np.zeros((p.shape[0], 1), dtype=np.int64), p.astype(np.int64)], axis=1))

    # ---- reads --------------------------------------------------------------------------------------------------
    def insertion_order(self):
        """``(rowptr, order)`` numpy: the neighbours (directed mode: the successors) of every node in networkx insertion
        order, a node with a self-loop listing itself."""
        return self._state.export()

    def edge_index(self) -> np.ndarray:
        """int64 ``[2, nnz]`` in the column order ``sdrf()`` returns (``from_networkx(G).edge_index``), exported on the
        device."""
        return self._state.edge_index().cpu().numpy()

    def curvature(self) -> np.ndarray:
        """One value per column of :meth:`edge_index`: fp32 ``C[i,j]`` for ``'bfc'``, the integer curvature for
        ``'1d'`` / ``'augmented'`` / ``'haantjes'``, fp64 ``bfc_edge`` for ``'bfc_paper'``.  A self-loop column gets
        ``C[i,i] = 0`` in the BFC modes and ``compute_curvature_edge(G, (u, u))`` in the classical ones."""
        ei = self.edge_index()
        rp, _, col, val, _ = self._state.export(with_curvature=True)
        loop_values = None
        if self.curv_type in CLASSICAL_MODES:
            val = val.astype(np.int64)                          # small integers, exact in the fp32 store
            loop_values = classical_loop_values(np.diff(rp.astype(np.int64)), self.curv_type)
        return align_to_columns(rp, col, val, ei, loop_values)

    # ---- candidate scoring ----------------------------------------------------------------------------------------
    def _score(self, pairs, max_cells: int):
        """``dcr.sdrf.SdrfState.score`` of ``pairs``, ``None`` for no pairs.  Ids outside ``[0, n)`` raise here, the pairs
        the mode's loop cannot score on the device; both before the scoring launch."""
        device = self._state.device
        p = pair_array(pairs)
        if not np.issubdtype(p.dtype, np.integer):
            raise ValueError(f"pairs: integer (x, y) expected, got {p.dtype}")
        out_of_range = np.flatnonzero(((p < 0) | (p >= self.n)).any(axis=1))
        if out_of_range.size:       # (checked here: the device takes int32 ids)
            q = int(out_of_range[0])
            raise ValueError(f"pairs[{q}] = ({int(p[q, 0])}, {int(p[q, 1])}): node ids must lie in [0, {self.n})")
        if p.shape[0] == 0:
            return None
        return self._state.score(torch.from_numpy(p.astype(np.int32)).to(device), int(max_cells))

    def improvements(self, pairs, *, max_cells: int = 1 << 27) -> list:
        """For every pair ``(x, y)`` of the ``[Q, 2]`` array ``pairs``: ``(candidates, improvements)``, the int64 ``[m, 2]``
        candidate edges ``(i, j)`` and the fp64 ``[m]`` improvement of the curvature of ``(x, y)`` if ``(i, j)`` is
        added — exactly the candidates and the ``improvements`` array ``sdrf()`` draws from when its loop picks ``(x, y)``,
        in its order (``i`` from ``x``'s list, ``j`` from ``y``'s; the classical and paper loops log the chosen pair
        sorted).  The values: fp32 ``D - C[x,y]`` for ``'bfc'``, the integer improvement for ``'1d'`` / ``'augmented'`` /
        ``'haantjes'``, the fp64 difference for ``'bfc_paper'``.
        Valid pairs are those the loop can pick: ``'bfc'`` any nodes (a non-edge and ``x == y`` included, with
        ``C[x,y] = 0``; directed: ``x``'s successors times ``y``'s predecessors); the classical modes an edge in either
        orientation or ``(u, u)`` of a node with a self-loop; ``'bfc_paper'`` an edge.  Another pair raises ``ValueError``
        naming its index, and so do queries whose candidate cells exceed ``max_cells`` (8 bytes of device output each);
        both before the scoring launch.  One launch for all pairs, one CTA per pair; the object is left unchanged and no
        budget is charged."""
        out = self._score(pairs, max_cells)
        if out is None:
            return []
        sizes = out["sizes"].cpu().numpy().astype(np.int64)
        cand_off = out["cand_offsets"].cpu().numpy()
        cell_off = out["cell_offsets"].cpu().numpy()
        cand = out["cand"].cpu().numpy().astype(np.int64)
        imp = out["imp"].cpu().numpy()
        res = []
        for q, (n_i, n_j) in enumerate(sizes.tolist()):
            rows = cand[cand_off[q]: cand_off[q] + n_i]
            cols = cand[cand_off[q] + n_i: cand_off[q + 1]]
            cells = imp[cell_off[q]: cell_off[q + 1]]
            flat = np.flatnonzero(cells.view(np.uint64) != _MASKED64)
            res.append((np.stack([rows[flat // n_j], cols[flat % n_j]], axis=1), cells[flat]))
        return res

    def best_additions(self, pairs, *, max_cells: int = 1 << 27):
        """The greedy (``tau = inf``) choice of the loop for every pair of ``pairs`` (see :meth:`improvements`):
        ``(additions [Q, 2] int64, improvement [Q] fp64, n_candidates [Q] int64)``, the first candidate of maximal
        improvement in the loop's order; ``(-1, -1)`` and NaN for a pair without candidates.  Only the Q best records are
        copied to the host."""
        out = self._score(pairs, max_cells)
        if out is None:
            return np.zeros((0, 2), dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.int64)
        rec = out["best"].cpu().numpy()
        ij = np.ascontiguousarray(rec[:, 2]).view(np.int32).reshape(-1, 2).astype(np.int64)
        return ij, np.ascontiguousarray(rec[:, 3]).view(np.float64), rec[:, 0].copy()

    # ---- SDRF ---------------------------------------------------------------------------------------------------
    def rewire(self, loops: int, remove_edges: bool, removal_bound: float, tau, *, uniforms=None,
               return_log: bool = False):
        """Continue SDRF on the current graph for up to ``loops`` iterations with ``sdrf()``'s host protocol (host
        re-decisions near a CDF boundary; numpy's global generator when ``uniforms`` is omitted).  Returns the new
        ``edge_index`` (and with ``return_log`` the int32 ``[iters, 8]`` log).  Raises ``ValueError`` before any launch
        when ``loops`` exceeds :attr:`remaining`."""
        loops = int(loops)
        if loops > self.remaining:
            raise ValueError(f"rewire: {loops} iterations exceed the remaining additions budget ({self.remaining})")
        try:
            log = _run_state(self._state, loops, remove_edges, removal_bound, tau, uniforms, 1e-9)
        except BaseException:
            self._loop_adds += max(loops, 0)      # how many iterations added an edge is unknown: charge them all
            raise
        self._loop_adds += int(np.count_nonzero(log[:, 3] >= 0))
        ei = self.edge_index()
        return (ei, log) if return_log else ei

    def rewire_batch(self, loops, remove_edges: bool, removal_bound, tau, *, uniforms, guard: float = 1e-9,
                     return_log: bool = False, return_exceptions: bool = False):
        """B continuations of SDRF from the current graph in one launch, one CTA per run, on B forks of this object.
        Run ``r`` computes exactly what ``self.fork()[0].rewire(loops[r], remove_edges, removal_bound[r], tau[r],
        uniforms=uniforms[r])`` computes; ``self`` is left unchanged.

        ``uniforms``: a ``[B, loops]`` array or a list of B 1-d arrays; it fixes B.  ``loops``, ``removal_bound``,
        ``tau``: scalars or length-B sequences.  Raises ``ValueError`` before any launch when a run's ``loops`` exceeds
        :attr:`remaining`.  Returns and raises what ``sdrf_batch`` does: a list of B ``edge_index`` arrays (and with
        ``return_log`` a list of B logs); a failed run raises after the batch (the lowest-index one) or, with
        ``return_exceptions``, leaves its exception in its slot."""
        uni = _batch_uniforms(uniforms, "rewire_batch")
        count = len(uni)
        iters = [max(int(v), 0) for v in _per_run("loops", loops, count)]
        bounds = [float(v) for v in _per_run("removal_bound", removal_bound, count)]
        taus = _per_run("tau", tau, count)
        over = [r for r in range(count) if iters[r] > self.remaining]
        if over:
            raise ValueError(f"rewire_batch: run {over[0]}: {iters[over[0]]} iterations exceed the remaining additions "
                             f"budget ({self.remaining})")
        forks = self._state.fork(count)
        try:
            logs, done, errors = _run_batch_states(forks, iters, bounds, taus, uni, remove_edges, guard)
            outs, out_logs = [], []
            for r in range(count):
                out_logs.append(logs[r][: done[r]].cpu().numpy())
                outs.append(errors[r] if errors[r] is not None else forks[r].edge_index().cpu().numpy())
        finally:
            for f in forks:
                f.close()
        return _batch_return(outs, out_logs, errors, return_log, return_exceptions)


def edit_batch(objects, ops_list, *, return_exceptions: bool = False) -> list:
    """Apply ``ops_list[b]`` to ``objects[b]`` for every b in ONE launch, one CTA per object, and return the number of
    edits each applied.  Every object ends exactly as ``objects[b].edit(ops_list[b])`` would leave it (same budget rule,
    same stop).  A failed object raises after the batch (the lowest-index one, with the type and message ``edit``
    raises) or, with ``return_exceptions``, leaves its exception in its slot; the others are applied either way.
    Objects of different modes, or one object twice, raise ``ValueError`` before any launch."""
    objects, ops_list = list(objects), list(ops_list)
    if not objects:
        raise ValueError("edit_batch: an empty batch")
    if len(ops_list) != len(objects):
        raise ValueError(f"edit_batch: {len(ops_list)} edit lists for {len(objects)} objects")
    if len({id(o) for o in objects}) != len(objects):
        raise ValueError("edit_batch: the same object appears twice (each edit list needs its own object)")
    if any(o.mode != objects[0].mode for o in objects):
        raise ValueError("edit_batch: objects of different modes (one mode per call)")
    if any(o._state is None for o in objects):
        raise ValueError("edit_batch: a closed object")
    prepared = [o._prepare_edits(ops) for o, ops in zip(objects, ops_list)]
    results = edit_batch_states([o._state for o in objects], [dev for _, _, dev in prepared])
    counts, errors = [], []
    for o, (e, stop, _), res in zip(objects, prepared, results):
        try:
            counts.append(o._finish_edits(e, stop, res))
            errors.append(None)
        except Exception as ex:      # this object stopped; the others are applied
            counts.append(ex)
            errors.append(ex)
    return _batch_return(counts, None, errors, False, return_exceptions)
