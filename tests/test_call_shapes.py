"""Call shapes without a GPU (tests/shapes.py): every class of view-group cut is reached by a case in every o_v where
it applies, the C ABI refuses calls beyond its limits before it touches the device, and the oracle side of the
degenerate batch follows DESIGN.md §3.7."""
import ctypes

import numpy as np
import pytest

from tests import shapes

RLAP_ERR_INVALID_ARG, RLAP_ERR_WORKSPACE = 1, 7


def test_every_shape_class_is_reached():
    """for the B200's 148 SMs; removing a case that is the only one to reach a class fails here"""
    assert shapes.unreached() == []


@pytest.mark.parametrize("sms", [1, 37, 148, 160])
def test_launch_shape_is_a_partition(sms):
    """the groups tile the views and the blocks in order, none empty; K and the grid stay inside the launch table"""
    for c in shapes.ALL_CASES:
        for o_v, o_n in c.modes:
            s = shapes.launch_shape(c.n, c.V, o_v, o_n, c.full, sms)
            assert 1 <= s.K <= min(shapes.TAB_GROUPS, c.V, s.blocks) and s.blocks <= shapes.TAB_BLOCKS
            assert s.groups[0][0] == 0 and s.groups[-1][1] == c.V
            assert s.groups[0][2] == 0 and s.groups[-1][3] == s.blocks
            for (v0, v1, b0, b1), nxt in zip(s.groups, s.groups[1:] + ((c.V, None, s.blocks, None),)):
                assert v0 < v1 == nxt[0] and b0 < b1 == nxt[2]


def _fake_call(L, n, V, view_base, ws_bytes):
    """rlap_schur_eliminate_keep on pointers that are never dereferenced: the call must return before any device work"""
    gp = np.array([0, n], dtype=np.int64)
    nr = np.array([n // 2], dtype=np.int64)
    rows = np.zeros(V, dtype=np.int64)
    fake = 256
    return L.rlap_schur_eliminate_keep(n, 4 * n, fake, fake, fake, 1, gp.ctypes.data, nr.ctypes.data, 1, 0, 0,
                                       view_base, V, 0, 0, 0, fake, ws_bytes, rows.ctypes.data, None, None, None)


def test_view_ids_must_stay_below_2_32():
    """view ids are 32-bit words of the Philox counter. A call whose last id is 2^32 - 1 passes the argument checks
    (and meets the workspace check, one byte short here); one more view, or a view_base at or above 2^32, would wrap
    onto view (id mod 2^32) and is refused as an invalid argument"""
    from rlap_b200 import _native
    L = _native.lib()
    n = 100
    for V in (1, 3, 65):
        b = ctypes.c_size_t(0)
        assert L.rlap_schur_workspace_bytes(n, 4 * n, 1, V, 0, 0, 0, ctypes.byref(b)) == 0
        short = b.value - 1
        assert _fake_call(L, n, V, 0, short) == RLAP_ERR_WORKSPACE
        assert _fake_call(L, n, V, shapes.VIEW_IDS - V, short) == RLAP_ERR_WORKSPACE
        assert _fake_call(L, n, V, shapes.VIEW_IDS - V + 1, short) == RLAP_ERR_INVALID_ARG
        assert _fake_call(L, n, V, shapes.VIEW_IDS + 5, short) == RLAP_ERR_INVALID_ARG
        assert _fake_call(L, n, V, -1, short) == RLAP_ERR_INVALID_ARG


def test_workspace_query_takes_vn_below_2_30():
    """n_views * n < 2^30: 7 161 * 149 943 = 2^30 - 1 and 1 * (2^30 - 1) are answered, 2^15 * 2^15 is refused"""
    from rlap_b200 import _native
    L = _native.lib()
    b = ctypes.c_size_t(0)
    assert 7161 * 149943 == shapes.VN_LIMIT - 1
    for V, n, ok in ((7161, 149943, True), (1, shapes.VN_LIMIT - 1, True), (1 << 15, 1 << 15, False),
                     (1, shapes.VN_LIMIT, False), (7161, 149944, False)):
        st = L.rlap_schur_workspace_bytes(n, 1000, 1, V, 0, 0, 0, ctypes.byref(b))
        assert st == (0 if ok else RLAP_ERR_INVALID_ARG), (V, n)


@pytest.mark.parametrize("masked", [False, True], ids=["no_mask", "keep"])
def test_degenerate_batch_caps_follow_the_spec(oracle_port, masked):
    """empty graphs, singletons, pairs and small BA graphs with num_remove negative, 0, 1, n_g - 1 and 10^9: the oracle
    removes exactly t_g vertices of every graph (DESIGN.md §3.7), in every mode, views 0 and 7"""
    from tests import util
    ei, gp, nr = shapes.degenerate_batch()
    n = int(gp[-1])
    sizes = np.diff(gp)
    assert {0, 1, 2} <= set(sizes.tolist()) and n == shapes.GRAPH_N["degenerate"]
    keep = shapes.degenerate_keep(gp) if masked else None
    unprot = None if keep is None else [int((~keep[gp[g]:gp[g + 1]]).sum()) for g in range(sizes.shape[0])]
    want = shapes.expected_removals(sizes.tolist(), nr.tolist(), unprot)
    if masked:
        assert 0 in unprot and 1 in unprot
    ptr, col, w = oracle_port.ingest(ei, util.sym_weights(ei), n)
    for o_v, o_n in shapes.MODES:
        for view in (0, 7):
            *_, order = oracle_port.keyed_schur(ptr, col, w, nr, o_v, o_n, seed=3, view=view, graph_ptr=gp, keep=keep,
                                                return_order=True)
            got = [int((order[gp[g]:gp[g + 1]] >= 0).sum()) for g in range(sizes.shape[0])]
            assert got == want, (o_v, o_n, view)


def test_one_vertex_per_graph_returns_the_coalesced_input(oracle_port):
    """G = n: every graph is a single vertex, nothing can go, whatever num_remove says"""
    spec = shapes.graph("singletons")
    ptr, col, w = oracle_port.ingest(spec.ei, spec.w, spec.n)
    want = shapes.coalesced(ptr, col, w)
    for o_v, o_n in shapes.MODES:
        for keep in (None, np.arange(spec.n) % 3 == 0):
            r, c, wt = oracle_port.keyed_schur(ptr, col, w, spec.num_remove, o_v, o_n, seed=3, graph_ptr=spec.gptr,
                                               keep=keep)
            assert np.array_equal(r, want[0]) and np.array_equal(c, want[1]), (o_v, o_n)
            assert np.array_equal(wt.view(np.uint32), want[2].view(np.uint32)), (o_v, o_n)
