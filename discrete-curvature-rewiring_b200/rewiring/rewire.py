"""Drop-in for the reference's ``rewiring/rewire.py`` (rewiring/rewire.py:7-14): curvature-type dispatch.

``rewire(dt, curv_type, max_iterations, removal_bound, tau) -> edge_index``

* ``'bfc'``                              -> the device-resident BFC loop (``rewiring.sdrf_cuda_bfc``), undirected
* ``'1d'`` / ``'augmented'`` / ``'haantjes'`` -> the classical-curvature loop on the same device kernel
  (``rewiring.sdrf_no_cuda``)
* ``'bfc_paper'``                        -> the same loop with the paper-flavour curvature ``bfc_naive.bfc_edge``
  (``rewiring.sdrf_no_cuda``; no self-loops)
* ``None``                               -> no rewiring: the input's ``edge_index`` comes back unchanged

Every flavour removes edges (``remove_edges=True``), as the reference's dispatcher does.

``rewire_batch`` runs many such rewirings — one per seed, per graph or per hyper-parameter setting — in one kernel launch
(``dcr.sdrf.sdrf_batch``, one CTA per run).  ``rewire_dataset`` rewires every graph of a dataset in the PyG batch layout
(``edge_index`` + ``ptr``) and returns it in that layout (``dcr.sdrf.sdrf_dataset``).
"""
import numpy as np
import torch

from dcr import sdrf as _sdrf
from rewiring.sdrf_cuda_bfc import sdrf_cuda_bfc
from rewiring.sdrf_no_cuda import sdrf_no_cuda


def rewire(dt, curv_type, max_iterations, removal_bound, tau):
    if curv_type is None:
        return dt.edge_index
    common = dict(loops=max_iterations, remove_edges=True, removal_bound=removal_bound, tau=tau)
    if curv_type == 'bfc':
        rewired = sdrf_cuda_bfc(dt, is_undirected=True, **common)
    else:
        rewired = sdrf_no_cuda(dt, curv_type, **common)
    return rewired.edge_index


def rewire_batch(datasets, curv_type, max_iterations, removal_bound, tau, *, seeds=None, uniforms=None,
                 return_exceptions=False):
    """Many independent ``rewire`` calls in one launch.  ``datasets``: one ``Data`` (shared by every run) or a sequence;
    ``max_iterations``, ``removal_bound``, ``tau``: scalars or per-run sequences.  Exactly one of

    * ``seeds``: run ``r`` draws ``np.random.RandomState(seeds[r]).random_sample(max_iterations[r])``, the stream the
      reference consumes after ``np.random.seed(seeds[r])``, so ``rewire_batch(d, c, m, b, t, seeds=S)[r]`` equals
      ``np.random.seed(S[r]); rewire(d, c, m, b, t)``;
    * ``uniforms``: those doubles given explicitly (a ``[B, loops]`` array or a list of B 1-d arrays).

    numpy's global generator is neither read nor advanced.  Returns a list of int64 ``edge_index`` tensors; with
    ``return_exceptions`` a failed run's slot holds its exception instead (see ``dcr.sdrf.sdrf_batch``)."""
    if (seeds is None) == (uniforms is None):
        raise TypeError("rewire_batch: pass exactly one of seeds= or uniforms=")
    one = not isinstance(datasets, (list, tuple))
    if uniforms is None:
        count = len(seeds)
        iters = _sdrf._per_run("max_iterations", max_iterations, count)
        uniforms = [np.random.RandomState(s).random_sample(max(int(m), 0)) for s, m in zip(seeds, iters)]
    count = len(uniforms)
    data = [datasets] * count if one else _sdrf._per_run("datasets", datasets, count)
    if curv_type is None:
        return [d.edge_index for d in data]
    inputs = datasets.edge_index if one else [d.edge_index for d in data]
    nodes = int(datasets.num_nodes) if one else [int(d.num_nodes) for d in data]
    outs = _sdrf.sdrf_batch(inputs, nodes, max_iterations, True, removal_bound, tau, uniforms=uniforms,
                            curv_type=curv_type, return_exceptions=return_exceptions)
    return [o if isinstance(o, BaseException) else torch.from_numpy(o).to(torch.long) for o in outs]


def _dataset_layout(data):
    """``(edge_index, ptr)`` of a ``Batch``-like object (its own) or of a sequence of ``Data`` (concatenated, graph ``g``
    owning ``max(num_nodes, max id + 1)`` nodes, the node count ``rewire`` uses)."""
    if not isinstance(data, (list, tuple)):
        return torch.as_tensor(data.edge_index), torch.as_tensor(data.ptr)
    if not data:
        raise ValueError("rewire_dataset: an empty dataset")
    eis = [torch.as_tensor(d.edge_index, dtype=torch.long).cpu().reshape(2, -1) for d in data]
    sizes = [max(int(d.num_nodes), int(e.max()) + 1 if e.numel() else 0) for d, e in zip(data, eis)]
    ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)])).to(torch.long)
    return torch.cat([e + int(o) for e, o in zip(eis, ptr[:-1])], dim=1), ptr


def rewire_dataset(data, curv_type, max_iterations, removal_bound, tau, *, seeds=None, uniforms=None,
                   return_exceptions=False):
    """``rewire`` on every graph of a dataset in one launch (``dcr.sdrf.sdrf_dataset``).  ``data``: a ``Batch``-like object
    with ``edge_index`` (global node ids) and ``ptr``, or a list of ``Data``, which is concatenated.  ``max_iterations``,
    ``removal_bound``, ``tau``: scalars or per-graph sequences.  Exactly one of ``seeds`` / ``uniforms``, as in
    ``rewire_batch``: graph ``g`` equals ``np.random.seed(seeds[g]); rewire(data_g, ...)`` with its node ids shifted by
    ``ptr[g]``.

    Returns ``(edge_index, edge_ptr)``: graph ``g`` in the columns ``edge_ptr[g] .. edge_ptr[g+1] - 1``; with
    ``return_exceptions`` also the list of B exceptions (``None`` where a graph succeeded; a failed graph is empty).
    ``curv_type=None`` returns the input's ``edge_index`` and the offsets of its per-graph columns (a ``Batch`` lists
    each graph's columns together)."""
    if (seeds is None) == (uniforms is None):
        raise TypeError("rewire_dataset: pass exactly one of seeds= or uniforms=")
    edge_index, ptr = _dataset_layout(data)
    count = int(ptr.numel()) - 1
    if uniforms is None:
        if len(seeds) != count:
            raise ValueError(f"seeds: {len(seeds)} values for a dataset of {count} graphs")
        iters = _sdrf._per_run("max_iterations", max_iterations, count)
        uniforms = [np.random.RandomState(s).random_sample(max(int(m), 0)) for s, m in zip(seeds, iters)]
    if curv_type is None:
        p = _sdrf.dataset_ptr(ptr, count)
        graphs = np.searchsorted(p, edge_index[0].cpu().numpy(), side="right") - 1
        edge_ptr = np.concatenate([[0], np.cumsum(np.bincount(graphs, minlength=count))])
        out = (edge_index, torch.from_numpy(edge_ptr).to(torch.long))
        return out + ([None] * count,) if return_exceptions else out
    return _sdrf.sdrf_dataset(edge_index, ptr, max_iterations, True, removal_bound, tau, uniforms=uniforms,
                              curv_type=curv_type, return_exceptions=return_exceptions)
