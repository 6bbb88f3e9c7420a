"""Drop-in for the reference's ``rewiring/sdrf_no_cuda.py`` (rewiring/sdrf_no_cuda.py:9-68).

Same signature and return type.  The reference recomputes every edge's curvature in Python each iteration
(``compute_curvature_graph``, curvature/classical_curvatures.py:31-46) and scores each candidate by adding and removing it
on the networkx graph (:40-45).  Here the loop runs inside the same persistent sm_100a kernel as the BFC loop
(csrc/dcr_sdrf.cu, ``LOOP_CLASSICAL``): degrees and common-neighbour counts are maintained incrementally, the three
curvatures ('1d', 'augmented', 'haantjes') are integer functions of them, ``min`` / ``max`` over ``G.edges`` keep the
reference's first-in-iteration-order tie-break, and the candidate improvements come in closed form.

``curv_type='bfc_paper'`` (an extension: the reference raises ``Method … not available.``) runs the same loop with
``curvature.bfc_naive.bfc_edge``, the paper-flavour Balanced Forman curvature, as ``compute_curvature_edge`` — the SDRF of
the paper.  Values, improvements and the removal comparison are fp64; inputs with self-loops raise ``NotImplementedError``.
"""
import torch

from dcr import compat as _compat
from dcr import sdrf as _sdrf

_compat.ensure_torch_geometric()
from torch_geometric.data import Data  # noqa: E402


def sdrf_no_cuda(data, curv_type, loops, remove_edges, removal_bound, tau, *, uniforms=None, return_log=False):
    """
    Perform SDRF graph rewiring using the given classical discrete curvature type.
    :param data: data to be rewired (undirected by default in this work).
    :param curv_type: type of discrete curvature used for the rewiring ('1d', 'augmented', 'haantjes' or 'bfc_paper').
    :param loops: number of edge addition/deletion iterations.
    :param remove_edges: whether to delete highly curved edges each iteration to compensate for the addition.
    :param removal_bound: curvature lower bound of deleting edges (delete edges only with higher curvature).
    :param tau: parameter specifying the randomness of choosing candidate edge to add; if infinite, max value is chosen.
    :return: rewired data.
    """
    num_nodes = int(data.num_nodes)
    res = _sdrf.sdrf(data.edge_index, num_nodes, int(loops), bool(remove_edges), float(removal_bound), tau,
                     uniforms=uniforms, return_log=return_log, curv_type=curv_type)
    ei, log = res if return_log else (res, None)
    out = Data(edge_index=torch.from_numpy(ei).to(torch.long))
    x = getattr(data, "x", None)
    if x is not None:
        out.x = x          # from_networkx(G) re-collects the node attribute 'x' (:19, :68)
    out.num_nodes = max(num_nodes, int(ei.max()) + 1 if ei.size else 0)
    if return_log:
        out.sdrf_log = log
    return out
