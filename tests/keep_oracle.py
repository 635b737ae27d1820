"""ctypes access to tests/native/keep_oracle.cc: the keyed oracle's driver restated with a keep mask (DESIGN.md §3.7).
TEST INFRASTRUCTURE ONLY. The library is compiled with g++ on first use into a fresh temporary directory (the checkout
may be read-only); the rest of the keyed oracle (ingest, rank permutation) is used through oracle.port."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import port

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "keep_oracle.cc")
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="rlap_keep_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libkeep_oracle.so")
        subprocess.check_call(["g++", "-O3", "-std=c++17", "-shared", "-fPIC", "-w", "-o", so, _SRC])
        L = ctypes.CDLL(so)
        P = ctypes.c_void_p
        L.oracle_keyed_schur_keep.argtypes = [
            ctypes.c_int64, P, P, P, ctypes.c_int64, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_uint64,
            ctypes.c_uint32, ctypes.c_int, P, P, P, ctypes.c_int64, P, P, P]
        L.oracle_keyed_schur_keep.restype = ctypes.c_int64
        _lib = L
    return _lib


def keyed_schur(ptr, col, w, num_remove, o_v, o_n, seed=0, view=0, graph_ptr=None, flags=0, return_stats=False,
                return_order=False, keep=None):
    """port.keyed_schur with a keep mask (n entries, nonzero = protected; None = no mask): (row, col, w) sorted by
    (col, row), then the stats and the elimination order if asked for"""
    n = ptr.shape[0] - 1
    if keep is not None:
        keep = np.ascontiguousarray(np.asarray(keep) != 0, dtype=np.uint8)
        assert keep.shape == (n,), "keep must have one entry per vertex"
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
        rows = lib().oracle_keyed_schur_keep(n, ptr.ctypes.data, col.ctypes.data, w.ctypes.data, G,
                                             graph_ptr.ctypes.data, t.ctypes.data, port.OV[o_v], port.ON[o_n], seed,
                                             view, flags, orow.ctypes.data, ocol.ctypes.data, ow.ctypes.data, cap,
                                             stats.ctypes.data, order.ctypes.data,
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
