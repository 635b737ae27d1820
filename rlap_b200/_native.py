"""ctypes binding of the C ABI in include/rlap_b200.h. There is no CPU fallback: if the CUDA
library is missing or no GPU is visible, every compute entry point raises."""
import ctypes
import os

from . import _build

_lib = None

RLAP_OK = 0
RLAP_ERR_POOL_OVERFLOW = 5
OV = {"random": 0, "degree": 1, "coarsen": 2}
ON = {"asc": 0, "desc": 1, "random": 2}
FLAG_FULL_CLIQUE = 1
FLAG_SHARED_ORDER = 2
FLAG_NO_VALIDATE = 4
FLAG_CHECK_LIVE = 8
FLAG_KEEP = 16
RLAP_ERR_STAR_TOO_LARGE = 6

EXPORTS = [
    "rlap_status_string", "rlap_last_cuda_error", "rlap_version", "rlap_ingest_workspace_bytes", "rlap_ingest",
    "rlap_schur_workspace_bytes", "rlap_schur_eliminate", "rlap_schur_emit", "rlap_approximate_cholesky_host",
    "rlap_free_host", "rlap_schur_colptr", "rlap_expand_cols_host", "rlap_schur_release", "rlap_schur_relabel", "rlap_schur_emit_ids",
    "rlap_schur_eliminate_keep",
]


class RlapError(RuntimeError):
    def __init__(self, status, where=""):
        self.status = status
        msg = lib().rlap_status_string(status).decode()
        if status == 8:
            msg += " [" + lib().rlap_last_cuda_error().decode() + "]"
        super().__init__(f"rlap_b200: {where}: {msg} (status {status})")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            f"rlap_b200: native CUDA library not found at {path}; build it with "
            "`python -m rlap_b200._build` (nvcc, sm_100a). There is no CPU fallback.")
    L = ctypes.CDLL(path)
    P, i64, u64, sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint64, ctypes.c_size_t
    L.rlap_status_string.argtypes = [ctypes.c_int]
    L.rlap_status_string.restype = ctypes.c_char_p
    L.rlap_last_cuda_error.restype = ctypes.c_char_p
    L.rlap_version.restype = ctypes.c_int
    L.rlap_ingest_workspace_bytes.argtypes = [i64, i64, ctypes.POINTER(sz)]
    L.rlap_ingest.argtypes = [P, P, P, i64, i64, P, P, P, ctypes.POINTER(i64), ctypes.c_int, P, sz, P]
    L.rlap_schur_workspace_bytes.argtypes = [i64, i64, i64, i64, i64, i64, ctypes.c_int, ctypes.POINTER(sz)]
    L.rlap_schur_eliminate.argtypes = [i64, i64, P, P, P, i64, P, P, ctypes.c_int, ctypes.c_int, u64, i64, i64,
                                       ctypes.c_int, i64, i64, P, sz, P, P, P]
    L.rlap_schur_eliminate_keep.argtypes = L.rlap_schur_eliminate.argtypes[:-1] + [P, P]
    L.rlap_schur_emit.argtypes = [i64, i64, P, P, P, i64, P, sz, P, P, P, P, P]
    L.rlap_approximate_cholesky_host.argtypes = [P, i64, i64, i64, ctypes.c_char_p, ctypes.c_char_p, u64,
                                                 ctypes.POINTER(ctypes.POINTER(ctypes.c_double)),
                                                 ctypes.POINTER(i64)]
    L.rlap_schur_colptr.argtypes = [i64, i64, i64, P, sz, P, P]
    L.rlap_expand_cols_host.argtypes = [P, i64, i64, P, P, ctypes.c_int]
    L.rlap_schur_release.argtypes = [P]
    L.rlap_schur_relabel.argtypes = [i64, i64, i64, P, sz, P, P, P]
    L.rlap_schur_emit_ids.argtypes = [i64, i64, P, P, P, i64, P, sz, P, P, P, P, P, P]
    L.rlap_free_host.argtypes = [P]
    L.rlap_free_host.restype = None
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def check(status, where):
    if status != RLAP_OK:
        raise RlapError(status, where)
