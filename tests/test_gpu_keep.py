"""Views onto a caller-chosen vertex set (keep mask, DESIGN.md §3.7) on the GPU: bit-exact against the keyed oracle
with the same mask (rows, columns, fp32 weights), the exact Kron reduction of full-clique mode, and an all-false mask
that changes nothing."""
import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu


def _gpu_graph(ei, w, n, gptr):
    import rlap_b200
    return rlap_b200.prepare(torch.from_numpy(ei).cuda(), None if w is None else torch.from_numpy(w).cuda(), n,
                             graph_ptr=gptr)


def _mask_cases():
    """(name, edge_index, n, graph_ptr or None, [num_remove], [(mask name, keep)])"""
    from rlap_b200 import graphs
    rng = np.random.default_rng(17)
    cases = []
    n = 300
    ei = graphs.barabasi_albert(n, 3, seed=2)
    masks = [(f"rand{int(f * 100)}", rng.random(n) < f) for f in (0.1, 0.5, 0.9)]
    cases.append(("ba300", ei, n, None, [150, n], masks))
    ei, gp = graphs.proteins_like_batch(40, seed=3)
    n = int(gp[-1])
    masks = [("rand50", rng.random(n) < 0.5)] + util.batch_masks(gp)
    cases.append(("proteins40", ei, n, gp, [np.diff(gp) // 2, np.diff(gp)], masks))
    return cases


def _check_views(oracle_port, optr, ocol, ow, row, col, wt, vp, t, o_v, o_n, seed, view_base, gptr, keep, flags=0,
                 what=""):
    for v in range(vp.shape[0] - 1):
        r0, c0, w0 = oracle_port.keyed_schur(optr, ocol, ow, t, o_v, o_n, seed=seed, view=view_base + v,
                                             graph_ptr=gptr, flags=flags, keep=keep)
        s, e = vp[v], vp[v + 1]
        assert e - s == r0.shape[0], (what, v, e - s, r0.shape[0])
        assert np.array_equal(row[s:e], r0) and np.array_equal(col[s:e], c0), (what, v)
        assert np.array_equal(wt[s:e].view(np.uint32), w0.view(np.uint32)), (what, v)


@pytest.mark.parametrize("o_v,o_n", util.COMBOS)
@pytest.mark.parametrize("weighted", [False, True])
def test_keep_views_match_oracle_bit_exact(oracle_port, o_v, o_n, weighted):
    import rlap_b200
    for name, ei, n, gptr, ts, masks in _mask_cases():
        w = util.sym_weights(ei) if weighted else None
        optr, ocol, ow = oracle_port.ingest(ei, w, n)
        g = _gpu_graph(ei, w, n, gptr)
        for t in ts:
            for mname, keep in masks:
                what = (name, mname, int(np.asarray(t).sum()))
                (row, col, wt), vp = rlap_b200.schur_views(g, t, o_v, o_n, num_views=4, seed=77, view_base=5,
                                                           dtype=None, keep=torch.from_numpy(keep).cuda())
                row, col, wt, vp = row.cpu().numpy(), col.cpu().numpy(), wt.cpu().numpy(), vp.numpy()
                _check_views(oracle_port, optr, ocol, ow, row, col, wt, vp, t, o_v, o_n, 77, 5, gptr, keep, what=what)
                # the same four views sharded over two calls by view_base (mask as a host array this time)
                for half in range(2):
                    (r2, c2, w2), vp2 = rlap_b200.schur_views(g, t, o_v, o_n, num_views=2, seed=77,
                                                              view_base=5 + 2 * half, dtype=None, keep=keep)
                    s, e = vp[2 * half], vp[2 * half + 2]
                    assert np.array_equal(r2.cpu().numpy(), row[s:e]) and np.array_equal(c2.cpu().numpy(), col[s:e])
                    assert np.array_equal(w2.cpu().numpy().view(np.uint32), wt[s:e].view(np.uint32)), what


@pytest.mark.parametrize("o_v", ["random", "degree", "coarsen"])
def test_keep_with_relabel_and_colptr(oracle_port, o_v):
    import rlap_b200
    from rlap_b200 import ops
    name, ei, n, gptr, ts, masks = _mask_cases()[1]
    optr, ocol, ow = oracle_port.ingest(ei, None, n)
    g = _gpu_graph(ei, None, n, gptr)
    t = ts[1]
    for mname, keep in masks:
        kt = torch.from_numpy(keep.astype(np.int64))            # a 0/1 integer tensor on the host
        (row, cp, wt), vp = rlap_b200.schur_views(g, t, o_v, "asc", num_views=3, seed=4, dtype=None, colptr=True,
                                                  keep=kt)
        col = ops.expand_cols(cp.cpu(), vp).numpy()
        _check_views(oracle_port, optr, ocol, ow, row.cpu().numpy(), col, wt.cpu().numpy(), vp.numpy(), t, o_v, "asc",
                     4, 0, gptr, keep, what=(mname, "colptr"))
        ((r2, c2, w2), newid), vp2 = rlap_b200.schur_views(g, t, o_v, "asc", num_views=3, seed=4, dtype=None,
                                                           relabel=True, keep=kt)
        assert torch.equal(vp, vp2) and torch.equal(wt, w2)
        newid = newid.cpu().numpy()
        r2, c2 = r2.cpu().numpy(), c2.cpu().numpy()
        row = row.cpu().numpy()
        for v in range(3):
            s, e = int(vp[v]), int(vp[v + 1])
            nodes = np.unique(np.concatenate([row[s:e], col[s:e]]))
            want = np.full(n, -1, dtype=np.int32)
            want[nodes] = np.arange(nodes.shape[0])
            assert np.array_equal(newid[v], want), (mname, v)
            assert np.array_equal(r2[s:e], want[row[s:e]]) and np.array_equal(c2[s:e], want[col[s:e]]), (mname, v)


def _kron(L, keep_idx):
    iso = np.where(np.diag(L) == 0)[0]
    idx = np.union1d(keep_idx, iso)
    S = util.exact_schur(L, idx)
    pos = np.searchsorted(idx, keep_idx)
    return S[np.ix_(pos, pos)]


@pytest.mark.parametrize("o_v", ["random", "degree"])
def test_full_clique_kron_reduction(oracle_port, o_v):
    """full_clique with every unprotected vertex removed: the exact Schur complement onto the protected set (1e-5),
    and bit-exact against the oracle's full-clique mode with the same mask"""
    import rlap_b200
    from rlap_b200 import graphs
    rng = np.random.default_rng(5)
    for ei, n in ((graphs.barabasi_albert(100, 3, seed=1), 100), (graphs.sbm(300, 3, 1200, seed=4), 300)):
        w = util.sym_weights(ei)
        g = _gpu_graph(ei, w, n, None)
        optr, ocol, ow = oracle_port.ingest(ei, w, n)
        L0 = util.laplacian(ei[0], ei[1], w, n)
        for f in (0.1, 0.3, 0.7):
            keep = rng.random(n) < f
            (row, col, wt), vp = rlap_b200.schur_views(g, n, o_v, "asc", seed=7, full_clique=True, dtype=None, keep=keep)
            row, col, wt = row.cpu().numpy(), col.cpu().numpy(), wt.cpu().numpy()
            k = np.where(keep)[0]
            Ls = util.laplacian(row, col, wt, n)[np.ix_(k, k)]
            ex = _kron(L0, k)
            assert np.linalg.norm(Ls - ex) / np.linalg.norm(ex) < 1e-5, (n, f)
            _check_views(oracle_port, optr, ocol, ow, row, col, wt, vp.numpy(), n, o_v, "asc", 7, 0, None, keep,
                         flags=oracle_port.FLAG_FULL_CLIQUE, what=(n, f))


@pytest.mark.parametrize("o_v", ["random", "degree"])
def test_arxiv_shape_half_protected_matches_oracle(oracle_port, o_v):
    """arxiv-shaped BA (n = 169,343, m = 7), 50 % of the vertices protected, every unprotected vertex removed"""
    import rlap_b200
    from rlap_b200 import graphs
    n = 169343
    ei = graphs.barabasi_albert(n, 7, seed=0)
    keep = np.random.default_rng(1).random(n) < 0.5
    optr, ocol, ow = oracle_port.ingest(ei, None, n)
    g = rlap_b200.prepare(torch.from_numpy(ei).cuda(), None, n)
    (row, col, wt), vp = rlap_b200.schur_views(g, n, o_v, "asc", num_views=1, seed=13, dtype=None, keep=keep)
    row, col, wt = row.cpu().numpy(), col.cpu().numpy(), wt.cpu().numpy()
    r0, c0, w0 = oracle_port.keyed_schur(optr, ocol, ow, n, o_v, "asc", seed=13, keep=keep)
    assert np.array_equal(row, r0) and np.array_equal(col, c0)
    assert np.array_equal(wt.view(np.uint32), w0.view(np.uint32))
    assert keep[row].all() and keep[col].all()                  # only protected vertices are left


@pytest.mark.parametrize("o_v,o_n", util.COMBOS)
def test_all_false_mask_is_bit_identical_to_no_mask(o_v, o_n):
    import rlap_b200
    for name, ei, n, gptr, t in util.small_cases():
        g = _gpu_graph(ei, util.sym_weights(ei), n, gptr)
        (a_r, a_c, a_w), a_vp = rlap_b200.schur_views(g, t, o_v, o_n, num_views=2, seed=21, dtype=None)
        (b_r, b_c, b_w), b_vp = rlap_b200.schur_views(g, t, o_v, o_n, num_views=2, seed=21, dtype=None,
                                                      keep=torch.zeros(n, dtype=torch.bool, device="cuda"))
        assert torch.equal(a_vp, b_vp) and torch.equal(a_r, b_r) and torch.equal(a_c, b_c), (name, o_v, o_n)
        assert torch.equal(a_w.view(torch.int32), b_w.view(torch.int32)), (name, o_v, o_n)


def test_bad_masks_raise():
    import rlap_b200
    from rlap_b200 import graphs
    n = 100
    ei = graphs.barabasi_albert(n, 3, seed=1)
    g = _gpu_graph(ei, None, n, None)
    for bad in (np.zeros(n - 1, dtype=bool), np.zeros(n + 1, dtype=bool), torch.zeros(n, dtype=torch.float32),
                np.zeros(n, dtype=np.float64), np.zeros((2, n // 2), dtype=bool), np.full(n, 2, dtype=np.int64),
                torch.full((n,), -1, dtype=torch.int32, device="cuda"), ["a"] * n):
        with pytest.raises(ValueError):
            rlap_b200.schur_views(g, 10, "degree", "asc", keep=bad)
    # accepted forms: bool / 0-1 integer tensors on any device, arrays, sequences
    want, _ = rlap_b200.schur_views(g, 50, "random", "asc", seed=3, keep=np.arange(n) % 3 == 0)
    for ok in ((np.arange(n) % 3 == 0).astype(np.uint8), [int(i % 3 == 0) for i in range(n)],
               torch.from_numpy(np.arange(n) % 3 == 0).cuda(), torch.from_numpy((np.arange(n) % 3 == 0).astype(np.int32))):
        got, _ = rlap_b200.schur_views(g, 50, "random", "asc", seed=3, keep=ok)
        assert torch.equal(got, want)
    out = rlap_b200.ops.approximate_cholesky(torch.from_numpy(ei), None, n, n, "degree", "asc", seed=3,
                                             keep=np.arange(n) < 10)
    assert set(np.unique(out[:, :2].numpy()).astype(int).tolist()) <= set(range(10))
