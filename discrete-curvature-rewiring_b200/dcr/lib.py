"""ctypes binding of ``libdcr.so`` — one Python callable per symbol declared in ``include/dcr.h``."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DCR_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "libdcr.so")   # override: experiments


class DcrError(RuntimeError):
    pass


class SdrfBatchRun(C.Structure):
    """``dcr_sdrf_batch_run``: one run of ``dcr_sdrf_run_batch`` (pointers are device pointers)."""
    _fields_ = [("state", C.c_void_p), ("loops", C.c_int32), ("forced_choice", C.c_int32),
                ("removal_bound", C.c_double), ("tau", C.c_double), ("uniforms", C.c_void_p),
                ("n_uniforms", C.c_int64), ("log", C.c_void_p), ("result", C.c_void_p)]


# status codes of include/dcr.h
SDRF_OK, SDRF_NEED_HOST, SDRF_PROB_NAN, SDRF_PROB_SUM, SDRF_REMOVE_NONEDGE, SDRF_NO_UNIFORM, SDRF_ARENA_FULL, \
    SDRF_TOO_MANY_CANDIDATES, SDRF_EMPTY_GRAPH = range(9)
SDRF_MODE_BFC, SDRF_MODE_BFC_DIRECTED, SDRF_MODE_1D, SDRF_MODE_AUGMENTED, SDRF_MODE_HAANTJES = range(5)
SDRF_LOG_INTS = 8

_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_D = C.c_double

# symbol -> (restype, argtypes); the single source of truth for tests/test_abi.py as well
SIGNATURES = {
    "dcr_last_error": (C.c_char_p, []),
    "dcr_version": (_I, []),
    "dcr_sm_clock_probe": (_I, [_P, _P]),
    "dcr_dense_count": (_I, [_P, _I, _P, _P, _P]),
    "dcr_dense_fill": (_I, [_P, _I, _P, _P, _P]),
    "dcr_scatter_dense": (_I, [_P, _P, _I, _P, _P, _P]),
    "dcr_csr_upper_count": (_I, [_P, _P, _I, _P, _P]),
    "dcr_csr_upper_fill": (_I, [_P, _P, _I, _P, _P, _P, _P]),
    "dcr_bfc_support": (_I, [_P, _P, _I, _P, _L, _L, _P]),
    "dcr_bfc_cuda_flavour": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _L, _L, _P]),
    "dcr_bfc_cuda_flavour_directed": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _L, _L, _P]),
    "dcr_bfc_support_tc_workspace_bytes": (_L, [_I, _L]),
    "dcr_bfc_support_tc": (_I, [_P, _P, _I, _L, _P, _P, _L, _P]),
    "dcr_tc_int8_peak": (_I, [_P, _P]),
    "dcr_bfc_cuda_flavour_tc_workspace_bytes": (_L, [_I, _L]),
    "dcr_bfc_cuda_flavour_tc": (_I, [_P, _P, _I, _L, _P, _P, _P, _P, _P, _P, _L, _P]),
    "dcr_bfc_cuda_dense_small_workspace_bytes": (_L, [_I]),
    "dcr_bfc_cuda_dense_small": (_I, [_P, _I, _P, _P, _P, _L, _P]),
    "dcr_bfc_paper_scratch_bytes": (_L, [_I, _I, _L]),
    "dcr_bfc_paper": (_I, [_P, _P, _I, _I, _P, _P, _L, _L, _L, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P]),
    "dcr_bfc_paper_unshard": (_I, [_P, _I, _L, _L, _P, _P, _P, _P, _P, _P]),
    "dcr_bfc_paper_set_mode": (_I, [_I]),
    "dcr_bfc_paper_edge_cost": (_I, [_P, _P, _I, _P, _P, _L, _P, _P, _P]),
    "dcr_comm_create": (_I, [_I, _I, _L, C.POINTER(_P)]),
    "dcr_comm_handle": (_I, [_P, _P]),
    "dcr_comm_connect": (_I, [_P, _P]),
    "dcr_comm_buffer": (_P, [_P]),
    "dcr_comm_chunk": (_L, [_P]),
    "dcr_comm_error": (_I, [_P]),
    "dcr_comm_destroy": (_I, [_P]),
    "dcr_bfc_paper_sharded": (_I, [_P, _P, _I, _I, _P, _P, _L, _L, _P, _P, _L, _P, _P, _P]),
    "dcr_bfc_cuda_edges_aux_ints": (_L, [_L, _L]),
    "dcr_bfc_cuda_edges_prepare": (_I, [_P, _P, _I, _P, _P, _L, _L, _P, _P]),
    "dcr_bfc_cuda_edges": (_I, [_P, _P, _I, _P, _P, _L, _P, _L, _L, _P, _P, _P, _P, _P, _I, _P]),
    "dcr_bfc_cuda_sharded": (_I, [_P, _P, _I, _P, _P, _L, _P, _L, _L, _P, _P]),
    "dcr_post_delta_workspace_bytes": (_L, [_I, _I, _I]),
    "dcr_post_delta": (_I, [_P, _P, _I, _P, _I, _I, _P, _I, _P, _I, _P, _P, _L, _P]),
    "dcr_post_delta_directed": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _I, _P, _I, _P, _P, _L, _P]),
    "dcr_sdrf_create": (_I, [_I, _P, _P, _L, C.POINTER(_P)]),
    "dcr_sdrf_create_mode": (_I, [_I, _I, _P, _P, _P, _P, _L, C.POINTER(_P)]),
    "dcr_sdrf_destroy": (None, [_P]),
    "dcr_sdrf_run": (_I, [_P, _I, _I, _D, _D, _P, _L, _I, _D, _P, _P, _P]),
    "dcr_sdrf_batch_workspace_bytes": (_L, [_I]),
    "dcr_sdrf_run_batch": (_I, [_P, _I, _I, _D, _P, _L, _P]),
    "dcr_sdrf_pending_improvements": (_I, [_P, _P, _L, _P]),
    "dcr_sdrf_nnz": (_L, [_P]),
    "dcr_sdrf_export": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "dcr_sdrf_export_order": (_I, [_P, _P, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load (once) and return the library; raises :class:`DcrError` when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DcrError(f"{LIB_PATH} is missing: build it with discrete-curvature-rewiring_b200/csrc/build.sh "
                       "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().dcr_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise DcrError(f"{what or 'libdcr'} failed ({rc}): {last_error()}")


def ptr(t) -> int:
    """Device (or host) address of a torch tensor / numpy array, or 0 for None."""
    if t is None:
        return 0
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise DcrError("a CUDA device is required: libdcr has no CPU fallback")
