"""C-ABI side of the keep mask that needs no GPU: the workspace query accounts for the mask under RLAP_FLAG_KEEP
only, and a mask given with a workspace sized without that flag is refused before any device work."""
import ctypes

import numpy as np


def test_keep_workspace_accounting_and_refusal():
    from rlap_b200 import _native
    L = _native.lib()
    n, nnz = 1000, 5000
    sizes = {}
    for flags in (0, _native.FLAG_FULL_CLIQUE, _native.FLAG_KEEP, _native.FLAG_FULL_CLIQUE | _native.FLAG_KEEP):
        b = ctypes.c_size_t(0)
        assert L.rlap_schur_workspace_bytes(n, nnz, 1, 4, 0, 0, flags, ctypes.byref(b)) == 0
        sizes[flags] = b.value
    # the mask needs two int arrays over the vertices (flags, then their prefix count)
    assert sizes[_native.FLAG_KEEP] >= sizes[0] + 8 * n + 4
    assert sizes[_native.FLAG_KEEP | _native.FLAG_FULL_CLIQUE] - sizes[_native.FLAG_FULL_CLIQUE] == \
        sizes[_native.FLAG_KEEP] - sizes[0]
    # keep != NULL with a workspace sized without RLAP_FLAG_KEEP: RLAP_ERR_WORKSPACE, checked before any device call
    gp = np.array([0, n], dtype=np.int64)
    nr = np.array([n // 2], dtype=np.int64)
    rows = np.zeros(4, dtype=np.int64)
    fake = 256    # never dereferenced: the call returns before it touches device memory
    st = L.rlap_schur_eliminate_keep(n, nnz, fake, fake, fake, 1, gp.ctypes.data, nr.ctypes.data, 1, 0, 0, 0, 4, 0, 0,
                                     0, fake, sizes[0], rows.ctypes.data, None, fake, None)
    assert st == 7
