"""ctypes access to oracle/_build/liboracle.so (oracle/rlap_oracle.cc), the in-repo CPU
restatement. TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline leg - never from rlap_b200/.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_OVERRIDE = os.environ.get("RLAP_ORACLE_LIB")   # experiments with an older build: loaded as it is, never built
_LIB_PATH = _OVERRIDE or os.path.join(_HERE, "_build", "liboracle.so")
_lib = None

OV = {"random": 0, "degree": 1, "coarsen": 2}
ON = {"asc": 0, "desc": 1, "random": 2}
FLAG_FULL_CLIQUE = 1
FLAG_SHARED_ORDER = 2


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])


def lib():
    global _lib
    if _lib is None:
        if not _OVERRIDE:
            build()   # a no-op when the library is newer than rlap_oracle.cc; a stale one is rebuilt, never loaded
        L = ctypes.CDLL(_LIB_PATH)
        P = ctypes.c_void_p
        L.oracle_ref_approximate_cholesky.argtypes = [
            P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_char_p, ctypes.c_char_p,
            ctypes.c_uint64, ctypes.c_uint64, ctypes.POINTER(ctypes.POINTER(ctypes.c_double)), P,
            ctypes.POINTER(ctypes.c_int)]
        L.oracle_ref_approximate_cholesky.restype = ctypes.c_int64
        L.oracle_free.argtypes = [P]
        L.oracle_philox4x32_10.argtypes = [ctypes.c_uint32] * 6 + [P]
        L.oracle_ingest.argtypes = [P, P, P, ctypes.c_int64, ctypes.c_int64, P, P, P, ctypes.POINTER(ctypes.c_int)]
        L.oracle_ingest.restype = ctypes.c_int64
        L.oracle_keyed_schur.argtypes = [
            ctypes.c_int64, P, P, P, ctypes.c_int64, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_uint64,
            ctypes.c_uint32, ctypes.c_int, P, P, P, ctypes.c_int64, P, P, P]
        L.oracle_keyed_schur.restype = ctypes.c_int64
        L.oracle_ref_random_order.argtypes = [ctypes.c_int64, ctypes.c_uint64, P]
        L.oracle_rank_perm.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, P]
        if hasattr(L, "oracle_star_order"):
            L.oracle_star_order.argtypes = [P, ctypes.c_int32, ctypes.c_int, P]
        _lib = L
    return _lib


def ref_approximate_cholesky(edge_info, num_nodes, num_remove, o_v, o_n, sample_seed=5489, rd_seed=0,
                             return_counters=False):
    """ref mode: bit-for-bit restatement of the reference given the injected seeds."""
    ei = np.ascontiguousarray(edge_info, dtype=np.float64)
    out = ctypes.POINTER(ctypes.c_double)()
    cnt = np.zeros(3, dtype=np.int64)
    st = ctypes.c_int(0)
    rows = lib().oracle_ref_approximate_cholesky(ei.ctypes.data, ei.shape[0], num_nodes, num_remove, o_v.encode(),
                                                 o_n.encode(), sample_seed, rd_seed, ctypes.byref(out),
                                                 cnt.ctypes.data, ctypes.byref(st))
    res = np.ctypeslib.as_array(out, shape=(max(rows, 1), 3))[:rows].copy()
    lib().oracle_free(out)
    if st.value != 0:
        raise ValueError("adjacency matrix is not symmetric")
    return (res, cnt) if return_counters else res


def philox(k0, k1, c0, c1, c2, c3):
    out = np.zeros(4, dtype=np.uint32)
    lib().oracle_philox4x32_10(k0, k1, c0, c1, c2, c3, out.ctypes.data)
    return out


def rank_perm(seed, graph, view, n_g):
    out = np.zeros(n_g, dtype=np.uint32)
    lib().oracle_rank_perm(seed, graph, view, n_g, out.ctypes.data)
    return out


def star_order(q, o_n):
    """o_n order (ids) of a star whose merged neighbours 0..n-1 carry the fixed-point weights q"""
    q = np.ascontiguousarray(q, dtype=np.uint64)
    out = np.zeros(q.shape[0], dtype=np.int32)
    lib().oracle_star_order(q.ctypes.data, q.shape[0], ON[o_n], out.ctypes.data)
    return out


def ref_random_order(n, rd_seed):
    """elimination (pop) order of the reference's random queue for the injected random_device stream"""
    out = np.zeros(n, dtype=np.int64)
    lib().oracle_ref_random_order(n, rd_seed, out.ctypes.data)
    return out


def ingest(edge_index, weights, n):
    src = np.ascontiguousarray(edge_index[0], dtype=np.int64)
    dst = np.ascontiguousarray(edge_index[1], dtype=np.int64)
    E = src.shape[0]
    w = None if weights is None else np.ascontiguousarray(np.asarray(weights).reshape(-1), dtype=np.float32)
    ptr = np.zeros(n + 1, dtype=np.int64)
    col = np.zeros(max(E, 1), dtype=np.int32)
    wo = np.zeros(max(E, 1), dtype=np.float32)
    st = ctypes.c_int(0)
    nnz = lib().oracle_ingest(src.ctypes.data, dst.ctypes.data, None if w is None else w.ctypes.data, E, n,
                              ptr.ctypes.data, col.ctypes.data, wo.ctypes.data, ctypes.byref(st))
    if st.value == 2:
        raise ValueError("node id out of range")
    if st.value == 3:
        raise ValueError("self loop")
    return ptr, col[:nnz].copy(), wo[:nnz].copy()


def keyed_schur(ptr, col, w, num_remove, o_v, o_n, seed=0, view=0, graph_ptr=None, flags=0, return_stats=False,
                return_order=False, keep=None):
    """keyed mode on a coalesced CSR: returns (row, col, w) sorted by (col,row), then the stats and the elimination
    order if asked for. keep (n entries, nonzero = protected; None = no mask): DESIGN.md §3.7."""
    n = ptr.shape[0] - 1
    if keep is not None:
        keep = np.asarray(keep)
        if keep.shape != (n,):
            raise ValueError(f"keep must have one entry per vertex ({n}), got shape {keep.shape}")
        keep = np.ascontiguousarray(keep != 0, dtype=np.uint8)
    if graph_ptr is None:
        graph_ptr = np.array([0, n], dtype=np.int64)
    graph_ptr = np.ascontiguousarray(graph_ptr, dtype=np.int64)
    G = graph_ptr.shape[0] - 1
    t = np.ascontiguousarray(np.broadcast_to(np.asarray(num_remove, dtype=np.int64), (G,)))
    ptr = np.ascontiguousarray(ptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    w = np.ascontiguousarray(w, dtype=np.float32)
    cap = max(int(col.shape[0]), 1)
    stats = np.zeros(5, dtype=np.int64)
    order = np.zeros(max(n, 1), dtype=np.int32)
    while True:
        orow = np.zeros(cap, dtype=np.int32)
        ocol = np.zeros(cap, dtype=np.int32)
        ow = np.zeros(cap, dtype=np.float32)
        rows = lib().oracle_keyed_schur(n, ptr.ctypes.data, col.ctypes.data, w.ctypes.data, G, graph_ptr.ctypes.data,
                                        t.ctypes.data, OV[o_v], ON[o_n], seed, view, flags, orow.ctypes.data,
                                        ocol.ctypes.data, ow.ctypes.data, cap, stats.ctypes.data, order.ctypes.data,
                                        None if keep is None else keep.ctypes.data)
        if rows <= cap:
            break
        cap = rows
    res = [orow[:rows].copy(), ocol[:rows].copy(), ow[:rows].copy()]
    if return_stats:
        res.append(dict(D=int(stats[0]), F=int(stats[1]), maxlen=int(stats[2]), rounds=int(stats[3]), Draw=int(stats[4])))
    if return_order:
        res.append(order[:n].copy())
    return tuple(res)
