"""The keyed specification with a keep mask (DESIGN.md §3.7): protected vertices are never eliminated. The sequential
form is the keyed oracle's `keep` argument. An all-false mask (and no mask) gives the oracle's unmasked output; the
invariants, the cap, the degree bucket over unprotected vertices and the exact Kron reduction of full-clique mode."""
import numpy as np
import pytest

from rlap_b200 import graphs
from tests import util


def _t_eff(num_remove, n_g, m_g):
    return min(max(num_remove, 0), m_g if m_g < n_g else n_g - 1)


@pytest.mark.parametrize("case", util.small_cases(), ids=lambda c: c[0])
def test_all_false_mask_is_no_mask(oracle_port, case):
    """keep=None and an all-false mask both give the keyed oracle's unmasked output, bit for bit, with the same stats
    and elimination order"""
    name, ei, n, gp, t = case
    ptr, col, w = oracle_port.ingest(ei, None, n)
    for o_v, o_n in util.COMBOS:
        a = oracle_port.keyed_schur(ptr, col, w, t, o_v, o_n, seed=5, graph_ptr=gp, return_stats=True,
                                    return_order=True)
        for keep in (None, np.zeros(n, dtype=bool)):
            b = oracle_port.keyed_schur(ptr, col, w, t, o_v, o_n, seed=5, graph_ptr=gp, return_stats=True,
                                        return_order=True, keep=keep)
            for x, y in zip(a[:3], b[:3]):
                assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), (name, o_v, o_n)
            assert a[3] == b[3] and np.array_equal(a[4], b[4]), (name, o_v, o_n)


def _check_invariants(oracle_port, ptr, col, w, n, gp, t, o_v, o_n, keep, seed):
    r, c, wt, order = oracle_port.keyed_schur(ptr, col, w, t, o_v, o_n, seed=seed, graph_ptr=gp, return_order=True,
                                              keep=keep)
    gp = np.array([0, n]) if gp is None else gp
    tt = np.broadcast_to(np.asarray(t), (gp.shape[0] - 1,))
    elim = order >= 0
    assert not elim[keep].any()                                           # every protected vertex survives
    for g in range(gp.shape[0] - 1):
        lo, hi = gp[g], gp[g + 1]
        m_g = int((~keep[lo:hi]).sum())
        assert int(elim[lo:hi].sum()) == _t_eff(int(tt[g]), hi - lo, m_g), (g, o_v, o_n)
    assert not elim[r].any() and not elim[c].any()                         # no row names an eliminated vertex
    A = np.zeros((n, n))
    A[r, c] = wt
    # symmetric: the pattern exactly, the weights to fp32 rounding (each end merges a multi-edge on its own star's
    # fixed-point scale, DESIGN.md §3.3; the same holds without a mask once most vertices are eliminated)
    assert np.array_equal(A != 0, A.T != 0)
    assert np.abs(A - A.T).max() <= 2 ** -23 * np.abs(A).max()
    assert (wt > 0).all()
    return r, c, wt, order


@pytest.mark.parametrize("o_v,o_n", util.COMBOS)
def test_keep_invariants(oracle_port, o_v, o_n):
    rng = np.random.default_rng(7)
    n = 300
    ei = graphs.barabasi_albert(n, 4, seed=11)
    ptr, col, w = oracle_port.ingest(ei, util.sym_weights(ei), n)
    for frac in (0.1, 0.5, 0.9):
        keep = rng.random(n) < frac
        for t in (120, n):                                                 # n: every unprotected vertex goes
            _check_invariants(oracle_port, ptr, col, w, n, None, t, o_v, o_n, keep, seed=3)
    # a batch: per-graph caps, a graph without protected vertices keeps its n_g - 1 rule
    ei, gp = graphs.proteins_like_batch(30, seed=5)
    n = int(gp[-1])
    ptr, col, w = oracle_port.ingest(ei, None, n)
    keep = rng.random(n) < 0.3
    keep[gp[2]:gp[3]] = False
    for t in (np.diff(gp) // 2, np.diff(gp)):
        _check_invariants(oracle_port, ptr, col, w, n, gp, t, o_v, o_n, keep, seed=9)


@pytest.mark.parametrize("o_v", ["random", "degree", "coarsen"])
def test_fully_protected_graph_returns_its_input(oracle_port, o_v):
    ei, gp = graphs.proteins_like_batch(12, seed=2)
    n = int(gp[-1])
    w = util.sym_weights(ei)
    ptr, col, ww = oracle_port.ingest(ei, w, n)
    owner = np.repeat(np.arange(n), np.diff(ptr))
    r, c, wt = oracle_port.keyed_schur(ptr, col, ww, n, o_v, "asc", seed=1, keep=np.ones(n, dtype=bool))
    assert np.array_equal(r, col) and np.array_equal(c, owner) and np.array_equal(wt, ww)
    # one whole graph of a batch protected, the others reduced to one vertex: that graph's rows are its input
    keep = np.zeros(n, dtype=bool)
    keep[gp[4]:gp[5]] = True
    r, c, wt = oracle_port.keyed_schur(ptr, col, ww, n, o_v, "asc", seed=1, graph_ptr=gp, keep=keep)
    sel = (owner >= gp[4]) & (owner < gp[5])
    mine = (c >= gp[4]) & (c < gp[5])
    assert np.array_equal(r[mine], col[sel]) and np.array_equal(c[mine], owner[sel]) and np.array_equal(wt[mine], ww[sel])
    assert not ((c < gp[4]) | (c >= gp[5])).any()                          # every other graph: one vertex, no edge


def _kron(L, keep_idx):
    """exact Schur complement onto keep_idx; vertices without an edge are dropped from the eliminated set (they do
    not change the result, and their zero rows would make the solve singular)"""
    iso = np.where(np.diag(L) == 0)[0]
    idx = np.union1d(keep_idx, iso)
    S = util.exact_schur(L, idx)
    pos = np.searchsorted(idx, keep_idx)
    return S[np.ix_(pos, pos)]


def kron_cases():
    return [("ba100", graphs.barabasi_albert(100, 3, seed=1), 100), ("sbm300", graphs.sbm(300, 3, 1200, seed=4), 300)]


@pytest.mark.parametrize("o_v", ["random", "degree"])
@pytest.mark.parametrize("case", kron_cases(), ids=lambda c: c[0])
def test_full_clique_is_kron_reduction(oracle_port, case, o_v):
    name, ei, n = case
    w = util.sym_weights(ei)
    ptr, col, ww = oracle_port.ingest(ei, w, n)
    L0 = util.laplacian(ei[0], ei[1], w, n)
    rng = np.random.default_rng(3)
    masks = [rng.random(n) < f for f in (0.1, 0.3, 0.7)] + [np.arange(n) % 17 == 0]
    for keep in masks:
        r, c, wt = oracle_port.keyed_schur(ptr, col, ww, n, o_v, "asc", seed=7, flags=oracle_port.FLAG_FULL_CLIQUE,
                                           keep=keep)
        k = np.where(keep)[0]
        Ls = util.laplacian(r, c, wt, n)[np.ix_(k, k)]
        ex = _kron(L0, k)
        assert np.linalg.norm(Ls - ex) / np.linalg.norm(ex) < 1e-5, (name, o_v, keep.sum())


@pytest.mark.parametrize("o_v", ["degree", "coarsen"])
def test_degree_bucket_ignores_protected_vertices(oracle_port, o_v):
    n = 300
    ei = graphs.barabasi_albert(n, 3, seed=8)
    ptr, col, w = oracle_port.ingest(ei, None, n)
    deg = np.diff(ptr)
    rng = np.random.default_rng(1)
    for trial in range(5):
        keep = rng.random(n) < 0.4
        keep[np.where(deg == deg.min())[0][-1]] = True        # the vertex an unmasked run would take first
        free = np.where(~keep)[0]
        m = deg[free].min()
        want = free[deg[free] == m][-1]                        # highest id among the unprotected of minimum degree
        _, _, _, order = oracle_port.keyed_schur(ptr, col, w, 1, o_v, "asc", seed=trial, keep=keep, return_order=True)
        assert np.where(order >= 0)[0].tolist() == [want]


def test_random_order_ranks_the_unprotected_vertices(oracle_port):
    """o_v = random: the vertices eliminated are the t lowest ranks of the keyed permutation over the m_g unprotected
    vertices (numbered by ascending id), in rank order"""
    n, t = 200, 40
    ei = graphs.barabasi_albert(n, 3, seed=5)
    ptr, col, w = oracle_port.ingest(ei, None, n)
    keep = np.random.default_rng(2).random(n) < 0.5
    free = np.where(~keep)[0]
    for view in (0, 3):
        _, _, _, order = oracle_port.keyed_schur(ptr, col, w, t, "random", "asc", seed=11, view=view, keep=keep,
                                                 return_order=True)
        rank = oracle_port.rank_perm(11, 0, view, free.shape[0])
        by_rank = free[np.argsort(rank)]
        assert np.array_equal(order[by_rank[:t]], np.arange(t))
        assert (order[by_rank[t:]] == -1).all()
