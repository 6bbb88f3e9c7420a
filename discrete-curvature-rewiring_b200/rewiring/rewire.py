"""Drop-in for the reference's ``rewiring/rewire.py`` (rewiring/rewire.py:7-14): curvature-type dispatch.

``rewire(dt, curv_type, max_iterations, removal_bound, tau) -> edge_index``

* ``'bfc'``                              -> the device-resident BFC loop (``rewiring.sdrf_cuda_bfc``), undirected
* ``'1d'`` / ``'augmented'`` / ``'haantjes'`` -> the classical-curvature loop on the same device kernel
  (``rewiring.sdrf_no_cuda``)
* ``None``                               -> no rewiring: the input's ``edge_index`` comes back unchanged

Every flavour removes edges (``remove_edges=True``), as the reference's dispatcher does.

``rewire_batch`` runs many such rewirings — one per seed, per graph or per hyper-parameter setting — in one kernel launch
(``dcr.sdrf.sdrf_batch``, one CTA per run).
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
