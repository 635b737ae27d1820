"""Call shapes on the GPU (tests/shapes.py): every case is one call, compared bit for bit (rows, columns, fp32 weights)
with the keyed oracle view by view, together with the stats the view groups fold, and compared by per-view digests with
the same views from calls that are split differently (V = 1 calls at the group boundaries, chunks that do not divide
the groups): a view must not depend on the group it lands in (DESIGN.md §6)."""
import functools
import hashlib
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from tests import shapes

pytestmark = pytest.mark.gpu

SEED = 20261
SLOW = ("ba20000", "c3", "c4")


@functools.lru_cache(maxsize=None)
def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


@functools.lru_cache(maxsize=None)
def _host_graph(key, port):
    spec = shapes.graph(key)
    return port.ingest(spec.ei, spec.w, spec.n)


@functools.lru_cache(maxsize=None)
def _device_graph(key):
    import rlap_b200
    spec = shapes.graph(key)
    g = rlap_b200.prepare(torch.from_numpy(spec.ei).cuda(), None if spec.w is None else torch.from_numpy(spec.w).cuda(),
                          spec.n, graph_ptr=spec.gptr)
    assert g.n == shapes.GRAPH_N[key]
    return g


def _call(case, o_v, o_n, view_base, V, **kw):
    import rlap_b200
    spec = shapes.graph(case.graph)
    out, vp, st = rlap_b200.schur_views(_device_graph(case.graph), spec.num_remove, o_v, o_n, num_views=V, seed=SEED,
                                        view_base=view_base, dtype=None, keep=spec.keep, full_clique=case.full,
                                        shared_order=case.shared, pool_cap=case.pool_cap, return_stats=True, **kw)
    return out, vp.numpy(), st


def _rows(case, o_v, o_n, view_base, V):
    (row, col, w), vp, st = _call(case, o_v, o_n, view_base, V)
    return row.cpu().numpy(), col.cpu().numpy(), w.cpu().numpy(), vp, st


def _digests(row, col, w, vp):
    return [hashlib.sha256(row[a:b].tobytes() + col[a:b].tobytes() + w[a:b].tobytes()).hexdigest()
            for a, b in zip(vp[:-1], vp[1:])]


def _oracle(port, case, o_v, o_n, views):
    """{view: (row, col, w, stats)} from the keyed oracle, on a thread pool (the ctypes call drops the GIL)"""
    spec = shapes.graph(case.graph)
    ptr, col, w = _host_graph(case.graph, port)
    flags = (port.FLAG_FULL_CLIQUE if case.full else 0) | (port.FLAG_SHARED_ORDER if case.shared else 0)

    def one(v):
        return port.keyed_schur(ptr, col, w, spec.num_remove, o_v, o_n, seed=SEED, view=case.view_base + v,
                                graph_ptr=spec.gptr, flags=flags, keep=spec.keep, return_stats=True)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        return dict(zip(views, ex.map(one, views)))


def _chunk(s):
    """a chunk size below V that divides no group's view count (0: there is none)"""
    c = s.V // 3 + 1
    while c < s.V and any(k % c == 0 for k in s.views_per_group()):
        c += 1
    return c if c < s.V else 0


def _check(port, case, o_v, o_n):
    """one call of the case in one mode: the oracle (every view of a cheap graph, else the first and last view of every
    group), the folded stats where every view was checked, and shape independence; returns the call's rows"""
    spec = shapes.graph(case.graph)
    s = shapes.launch_shape(spec.n, case.V, o_v, o_n, case.full, _sms())
    row, col, w, vp, st = _rows(case, o_v, o_n, case.view_base, case.V)
    what = (case.name, o_v, o_n)
    assert vp.shape[0] == case.V + 1 and st["rows"] == vp[-1], what
    views = list(range(case.V)) if spec.cheap else s.boundary_views()
    want = _oracle(port, case, o_v, o_n, views)
    for v in views:
        a, b = vp[v], vp[v + 1]
        r0, c0, w0, _ = want[v]
        assert b - a == r0.shape[0], what + (v, b - a, r0.shape[0])
        assert np.array_equal(row[a:b], r0) and np.array_equal(col[a:b], c0), what + (v,)
        assert np.array_equal(w[a:b].view(np.uint32), w0.view(np.uint32)), what + (v,)
    if spec.cheap:
        so = [want[v][3] for v in views]
        got = dict(fills=st["fills"], raw=st["raw_entries_read"], max_star=st["max_star"])
        exp = dict(fills=sum(x["F"] for x in so), raw=sum(x["D"] for x in so), max_star=max(x["maxlen"] for x in so))
        if o_v != "random":
            got["rounds"], exp["rounds"] = st["rounds"], max(x["rounds"] for x in so)
        assert got == exp, what + (got, exp)
    if case.V > 1:
        dig = _digests(row, col, w, vp)
        for v in s.boundary_views():
            assert _digests(*_rows(case, o_v, o_n, case.view_base + v, 1)[:4]) == [dig[v]], what + ("V=1", v)
        c = _chunk(s)
        for v0 in range(0, case.V, c) if c else ():
            m = min(c, case.V - v0)
            assert _digests(*_rows(case, o_v, o_n, case.view_base + v0, m)[:4]) == dig[v0:v0 + m], what + ("chunk", v0)
    return row, col, w, vp, st


def test_device_reaches_every_shape_class():
    """the cases were chosen for 148 SMs; on this device's SM count every class must still be reached"""
    assert shapes.unreached(_sms()) == [], _sms()


def _params():
    out = []
    for c in shapes.CASES:
        marks = [pytest.mark.timeout(600)] if c.graph in SLOW else []
        out.append(pytest.param(c.name, marks=marks, id=c.name))
    return out


@pytest.mark.parametrize("name", _params())
def test_call_shape_matches_oracle(oracle_port, name):
    case = next(c for c in shapes.CASES if c.name == name)
    for o_v, o_n in case.modes:
        row, col, w, vp, st = _check(oracle_port, case, o_v, o_n)
        if case.graph == "singletons":
            ptr, c, wt = _host_graph(case.graph, oracle_port)
            r0, c0, w0 = shapes.coalesced(ptr, c, wt)
            for v in range(case.V):
                a, b = vp[v], vp[v + 1]
                assert np.array_equal(row[a:b], r0) and np.array_equal(col[a:b], c0)
                assert np.array_equal(w[a:b].view(np.uint32), w0.view(np.uint32))


@pytest.mark.timeout(600)
def test_more_views_than_grid_y(oracle_port):
    """70 000 views of a 24-vertex graph (contrastive augmentation of molecule-sized graphs): more views than a grid's y
    dimension holds. From a pool of 32 entries per view, which every view outgrows (25 fills or more, two entries
    each), so the overflow retry runs too. Then the separate launches of the packed outputs: relabel=True with
    weights=False, and colptr=True"""
    from rlap_b200 import ops
    case = shapes.MANY_VIEWS
    assert case.V > shapes.MAX_GRID_Y
    for o_v, o_n in case.modes:
        row, col, w, vp, st = _check(oracle_port, case, o_v, o_n)
        assert st["pool_cap"] > case.pool_cap
    V, n = case.V, case.n
    ((r2, c2, w2), newid), vp2, _ = _call(case, o_v, o_n, case.view_base, V, relabel=True, weights=False)
    assert w2 is None and np.array_equal(vp2, vp)
    vid = np.repeat(np.arange(V), np.diff(vp))
    present = np.zeros((V, n), dtype=bool)
    present[vid, row] = True
    present[vid, col] = True
    want = np.where(present, np.cumsum(present, axis=1) - 1, -1).astype(np.int32)
    assert np.array_equal(newid.cpu().numpy(), want)
    assert np.array_equal(r2.cpu().numpy(), want[vid, row]) and np.array_equal(c2.cpu().numpy(), want[vid, col])
    (r3, cp, w3), vp3, _ = _call(case, o_v, o_n, case.view_base, V, colptr=True)
    assert np.array_equal(vp3, vp) and tuple(cp.shape) == (V, n + 1)
    assert np.array_equal(ops.expand_cols(cp.cpu(), torch.from_numpy(vp3)).numpy(), col)
    assert np.array_equal(r3.cpu().numpy(), row) and np.array_equal(w3.cpu().numpy().view(np.uint32), w.view(np.uint32))


def test_view_ids_up_to_2_32(oracle_port):
    """the last 65 view ids there are, 2^32 - 65 .. 2^32 - 1, over 26 groups: every view is the oracle's view of that
    id (a call one view longer is refused, tests/test_call_shapes.py)"""
    case = shapes.TOP_VIEWS
    assert case.view_base + case.V == shapes.VIEW_IDS
    for o_v, o_n in case.modes:
        _check(oracle_port, case, o_v, o_n)
