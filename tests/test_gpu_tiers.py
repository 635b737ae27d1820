"""Every tier of the CUDA path, steered (tests/tiers.py): each case runs in the modes where its tier exists and is
compared bit for bit (rows, columns, fp32 weights) with the keyed oracle under the same keep mask, together with the
run's stats; then the padded, multi-view, batched and packed-output variants, the scratch-slot retry, the exact
rank-one Schur complement of a full-clique star, and the ingest rows of every tier."""
import functools

import numpy as np
import pytest
import torch

from tests import tiers

pytestmark = pytest.mark.gpu


@functools.lru_cache(maxsize=None)
def _cases():
    return tiers.cases()


def _graph(ei, w, n, gptr=None):
    import rlap_b200
    return rlap_b200.prepare(torch.from_numpy(ei).cuda(), None if w is None else torch.from_numpy(w).cuda(), n,
                             graph_ptr=gptr)


def _oracle(port, ptr, col, w, case, o_v, o_n, seed, view=0, keep=None, gptr=None, t=None, stats=False):
    return port.keyed_schur(ptr, col, w, case.num_remove if t is None else t, o_v, o_n, seed=seed, view=view,
                            graph_ptr=gptr, keep=case.keep if keep is None else keep, return_stats=stats,
                            flags=port.FLAG_FULL_CLIQUE if case.full else 0)


def _same(got, want, what):
    row, col, wt = got
    r0, c0, w0 = want
    assert row.shape[0] == r0.shape[0], (what, row.shape[0], r0.shape[0])
    assert np.array_equal(row, r0) and np.array_equal(col, c0), what
    assert np.array_equal(wt.view(np.uint32), w0.view(np.uint32)), what


def _views(case, g, o_v, o_n, seed, **kw):
    import rlap_b200
    (row, col, wt), vp, st = rlap_b200.schur_views(g, case.num_remove, o_v, o_n, seed=seed, dtype=None,
                                                   keep=case.keep, full_clique=case.full, return_stats=True, **kw)
    return row.cpu().numpy(), col.cpu().numpy(), wt.cpu().numpy(), vp.numpy(), st


@pytest.mark.parametrize("name", [c.name for c in tiers.cases()])
def test_tier_case_matches_oracle(oracle_port, name):
    """(a) the compact graph in every mode and weight kind of the case, with the stats of the single view:
    max_star = maxlen, fills = F, raw_entries_read = D, and rounds = rounds under degree / coarsen"""
    case = next(c for c in _cases() if c.name == name)
    for wk in case.wkinds:
        w = tiers.weights(case.ei, wk)
        ptr, col, ow = oracle_port.ingest(case.ei, w, case.n)
        g = _graph(case.ei, w, case.n)
        for o_v, o_n in case.modes:
            seed = case.seeds[o_v]
            row, c, wt, vp, st = _views(case, g, o_v, o_n, seed)
            r0, c0, w0, s0 = _oracle(oracle_port, ptr, col, ow, case, o_v, o_n, seed, stats=True)
            what = (name, wk, o_v, o_n)
            _same((row, c, wt), (r0, c0, w0), what)
            got = dict(max_star=st["max_star"], fills=st["fills"], raw=st["raw_entries_read"])
            want = dict(max_star=s0["maxlen"], fills=s0["F"], raw=s0["D"])
            assert got == want, (what, got, want, s0)
            if o_v != "random":
                assert st["rounds"] == s0["rounds"], (what, st["rounds"], s0["rounds"])


@pytest.mark.parametrize("o_v,o_n", [("random", "random"), ("degree", "asc"), ("coarsen", "desc")])
def test_tier_cases_padded(oracle_port, o_v, o_n):
    """(b) padded with protected isolated vertices to 40 000 (a view group spans many blocks, the scratch-owning blocks
    are distinct), one view at view 0: the protected padding leaves the unprotected count and the steering seed alone,
    so every case still runs its steered tier"""
    import rlap_b200
    for case in _cases():
        if (o_v, o_n) not in case.modes:
            continue
        wk = case.wkinds[-1]
        n = max(case.n, 40000)
        keep = np.ones(n, dtype=bool)
        keep[:case.n] = case.keep
        w = tiers.weights(case.ei, wk)
        ptr, col, ow = oracle_port.ingest(case.ei, w, n)
        g = _graph(case.ei, w, n)
        seed = case.seeds[o_v]
        (row, c, wt), vp, st = rlap_b200.schur_views(g, case.num_remove, o_v, o_n, seed=seed, dtype=None, keep=keep,
                                                     full_clique=case.full, return_stats=True)
        r0, c0, w0, s0 = _oracle(oracle_port, ptr, col, ow, case, o_v, o_n, seed, keep=keep, stats=True)
        _same((row.cpu().numpy(), c.cpu().numpy(), wt.cpu().numpy()), (r0, c0, w0), (case.name, o_v, o_n))
        assert st["max_star"] == s0["maxlen"], (case.name, st["max_star"], s0["maxlen"])
        if not case.protected:
            assert st["max_star"] == case.claims[o_v]["L"], (case.name, st["max_star"])


@pytest.mark.parametrize("o_v,o_n", [("random", "random"), ("degree", "asc"), ("coarsen", "desc")])
def test_tier_cases_multi_view(oracle_port, o_v, o_n):
    """(c) three views from view_base 5, each checked; under o_v = random the seed is steered for view 5 (the rank
    permutation depends on the view), so at least that view runs the case's tier"""
    import rlap_b200
    for case in _cases():
        if (o_v, o_n) not in case.modes:
            continue
        wk = case.wkinds[-1]
        w = tiers.weights(case.ei, wk)
        ptr, col, ow = oracle_port.ingest(case.ei, w, case.n)
        g = _graph(case.ei, w, case.n)
        seed = case.seeds[o_v]
        if o_v == "random" and not case.protected:
            seed = tiers.steer_seed(case.keep, case.centre, 5, seed)
        (row, c, wt), vp = rlap_b200.schur_views(g, case.num_remove, o_v, o_n, num_views=3, seed=seed, view_base=5,
                                                 dtype=None, keep=case.keep, full_clique=case.full)
        row, c, wt, vp = row.cpu().numpy(), c.cpu().numpy(), wt.cpu().numpy(), vp.numpy()
        for v in range(3):
            want = _oracle(oracle_port, ptr, col, ow, case, o_v, o_n, seed, view=5 + v)
            s, e = vp[v], vp[v + 1]
            _same((row[s:e], c[s:e], wt[s:e]), want, (case.name, o_v, o_n, v))


@pytest.mark.parametrize("name", [c.name for c in tiers.unmasked_cases()])
def test_unmasked_random_first_star_matches_oracle(oracle_port, name):
    """(f) o_v = random without a keep mask (the ranking spans all n vertices, num_remove is capped at n - 1): the
    centre has rank 0, so num_remove = 1 eliminates exactly its star, in each o_n; then half the graph is removed,
    unsteered. Bit for bit against the oracle without a mask, with the stats of the first star"""
    import rlap_b200
    case = next(c for c in tiers.unmasked_cases() if c.name == name)
    seed = case.seeds["random"]
    q = case.claims["random"]
    for wk in case.wkinds:
        w = tiers.weights(case.ei, wk)
        ptr, col, ow = oracle_port.ingest(case.ei, w, case.n)
        g = _graph(case.ei, w, case.n)
        for o_n in ("asc", "desc", "random"):
            (row, c, wt), _, st = rlap_b200.schur_views(g, 1, "random", o_n, seed=seed, dtype=None, return_stats=True)
            r0, c0, w0, s0 = oracle_port.keyed_schur(ptr, col, ow, 1, "random", o_n, seed=seed, return_stats=True)
            _same((row.cpu().numpy(), c.cpu().numpy(), wt.cpu().numpy()), (r0, c0, w0), (name, wk, o_n))
            assert (st["max_star"], st["raw_entries_read"]) == (s0["maxlen"], s0["D"]) == (q["L"], q["lv"]), (name, st)
            assert st["fills"] == s0["F"], (name, wk, o_n, st["fills"], s0["F"])
            (row, c, wt), _ = rlap_b200.schur_views(g, case.n // 2, "random", o_n, seed=seed, dtype=None)
            want = oracle_port.keyed_schur(ptr, col, ow, case.n // 2, "random", o_n, seed=seed)
            _same((row.cpu().numpy(), c.cpu().numpy(), wt.cpu().numpy()), want, (name, wk, o_n, "half"))


@pytest.mark.parametrize("o_v,o_n", [("degree", "asc"), ("degree", "desc"), ("coarsen", "random")])
def test_tier_cases_batched_in_one_call(oracle_port, o_v, o_n):
    """(d) one graph per elimination tier in one batched call (graph_ptr): lane, tile, warp, block and scratch stars
    in the same rounds (degree / coarsen: every graph's centre goes in its own last round)"""
    names = ["lane_L8_D40", "lane_multi_L5_dup2", "tile_L17_dup4", "warp_L60_dup30_clean20", "warp_dead_L4_dead120",
             "block_L600_dup100_clean100", "scratch_L1100_dup1500", "merge_class_lv513", "fsort_warp_nb41"]
    cs = [c for c in _cases() if c.name in names]
    off, eis, keeps, ts, gp = 0, [], [], [], [0]
    for c in cs:
        eis.append(c.ei + off)
        keeps.append(c.keep)
        ts.append(c.num_remove)
        off += c.n
        gp.append(off)
    ei, keep, gp = np.concatenate(eis, axis=1), np.concatenate(keeps), np.array(gp, dtype=np.int64)
    w = tiers.weights(ei, "two")
    ptr, col, ow = oracle_port.ingest(ei, w, off)
    import rlap_b200
    g = _graph(ei, w, off, gp)
    (row, c, wt), vp = rlap_b200.schur_views(g, np.array(ts), o_v, o_n, seed=11, dtype=None, keep=keep)
    want = oracle_port.keyed_schur(ptr, col, ow, np.array(ts), o_v, o_n, seed=11, graph_ptr=gp, keep=keep)
    _same((row.cpu().numpy(), c.cpu().numpy(), wt.cpu().numpy()), want, (o_v, o_n))


@pytest.mark.parametrize("o_v", ["random", "degree", "coarsen"])
def test_emission_cases_packed_outputs(oracle_port, o_v):
    """(e) colptr=True, relabel=True and weights=False on the emission cases, against the packed rows"""
    import rlap_b200
    from rlap_b200 import ops
    for case in _cases():
        if not case.protected:
            continue
        w = tiers.weights(case.ei, "wide")
        ptr, col, ow = oracle_port.ingest(case.ei, w, case.n)
        g = _graph(case.ei, w, case.n)
        seed = case.seeds[o_v]
        r0, c0, w0 = _oracle(oracle_port, ptr, col, ow, case, o_v, "random", seed)
        (row, cp, wt), vp = rlap_b200.schur_views(g, case.num_remove, o_v, "random", seed=seed, dtype=None,
                                                  colptr=True, keep=case.keep)
        cc = ops.expand_cols(cp.cpu(), vp).numpy()
        _same((row.cpu().numpy(), cc, wt.cpu().numpy()), (r0, c0, w0), (case.name, "colptr"))
        ((r2, c2, w2), newid), _ = rlap_b200.schur_views(g, case.num_remove, o_v, "random", seed=seed, dtype=None,
                                                         relabel=True, weights=False, keep=case.keep)
        assert w2 is None
        nodes = np.unique(np.concatenate([r0, c0]))
        want = np.full(case.n, -1, dtype=np.int32)
        want[nodes] = np.arange(nodes.shape[0])
        assert np.array_equal(newid.cpu().numpy()[0], want), case.name
        assert np.array_equal(r2.cpu().numpy(), want[r0]) and np.array_equal(c2.cpu().numpy(), want[c0]), case.name


@pytest.mark.parametrize("o_n", ["asc", "desc", "random"])
def test_scratch_cap_retry_matches_oracle(oracle_port, o_n):
    """an explicit scratch_cap of 4096 with a 6 000-star and a 13 000-entry surviving hub: the call meets
    RLAP_ERR_STAR_TOO_LARGE, retries with a slot of nnz + 1 entries and returns the oracle's result"""
    for case in tiers.retry_cases():
        for wk in case.wkinds:
            w = tiers.weights(case.ei, wk)
            ptr, col, ow = oracle_port.ingest(case.ei, w, case.n)
            g = _graph(case.ei, w, case.n)
            for o_v in ("random", "degree"):
                seed = case.seeds[o_v]
                row, c, wt, vp, st = _views(case, g, o_v, o_n, seed, scratch_cap=case.scratch_cap)
                _same((row, c, wt), _oracle(oracle_port, ptr, col, ow, case, o_v, o_n, seed), (case.name, wk, o_v))


@pytest.mark.parametrize("which", [0, 1], ids=["elim_star_6000", "emit_segment_13000"])
def test_scratch_cap_too_small_is_a_status(which):
    """the library itself reports the oversized elimination star (scratch slot of k_eliminate) and the oversized
    surviving segment (scratch branch of the emission sort, above CAP_BIG) as RLAP_ERR_STAR_TOO_LARGE (status 6), not
    a fault: the status the retry of schur_views answers"""
    import ctypes
    from rlap_b200 import _native
    case = tiers.retry_cases()[which]
    g = _graph(case.ei, None, case.n)
    L = _native.lib()
    keep = torch.from_numpy(case.keep.astype(np.uint8)).cuda()
    flags = _native.FLAG_KEEP
    wsb = ctypes.c_size_t(0)
    gp = np.array([0, case.n], dtype=np.int64)
    nr = np.array([case.num_remove], dtype=np.int64)
    _native.check(L.rlap_schur_workspace_bytes(g.n, g.nnz, 1, 1, 0, 4096, flags, ctypes.byref(wsb)), "ws")
    ws = torch.empty(wsb.value, dtype=torch.uint8, device="cuda")
    rows, stats = np.zeros(1, dtype=np.int64), np.zeros(16, dtype=np.int64)
    st = L.rlap_schur_eliminate_keep(g.n, g.nnz, g.ptr.data_ptr(), g.col.data_ptr(), g.w.data_ptr(), 1, gp.ctypes.data,
                                     nr.ctypes.data, 1, 0, 11, 0, 1, flags, 0, 4096, ws.data_ptr(), wsb.value,
                                     rows.ctypes.data, stats.ctypes.data, keep.data_ptr(),
                                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    L.rlap_schur_release(ws.data_ptr())
    assert st == _native.RLAP_ERR_STAR_TOO_LARGE


@pytest.mark.parametrize("o_v", ["random", "degree", "coarsen"])
def test_full_clique_star_is_the_exact_rank_one_update(oracle_port, o_v):
    """single-centre full-clique elimination: L_KK - b b^T / L_cc in float64, to 1e-5 relative"""
    import rlap_b200
    from tests import util
    for case in _cases():
        if not case.full or case.claims[o_v]["L"] > 2500:
            continue
        w = tiers.weights(case.ei, "wide")
        g = _graph(case.ei, w, case.n)
        (row, col, wt), _ = rlap_b200.schur_views(g, case.num_remove, o_v, "asc", seed=case.seeds[o_v], dtype=None,
                                                  keep=case.keep, full_clique=True)
        k = np.nonzero(case.keep)[0]
        Lg = util.laplacian(row.cpu().numpy(), col.cpu().numpy(), wt.cpu().numpy(), case.n)[np.ix_(k, k)]
        L0 = util.laplacian(case.ei[0], case.ei[1], np.ones(case.ei.shape[1]) if w is None else w, case.n)
        c = case.centre
        b = L0[k, c]
        ex = L0[np.ix_(k, k)] - np.outer(b, b) / L0[c, c]
        assert np.linalg.norm(Lg - ex) / np.linalg.norm(ex) < 1e-5, (case.name, o_v)


def test_ingest_rows_of_every_tier_match_oracle(oracle_port):
    """owner rows of 128 (warp), 129 and 2048 (block), 2049 and 5000 (scratch) raw entries with order-sensitive
    duplicate runs and zero weights, in shuffled input order: the fp32 sums in input order, bit for bit"""
    import rlap_b200
    ei, w, n = tiers.ingest_rows()
    ptr, col, wo = oracle_port.ingest(ei, w, n)
    g = rlap_b200.prepare(torch.from_numpy(ei).cuda(), torch.from_numpy(w).cuda(), n, validate=False)
    assert g.nnz == col.shape[0]
    assert np.array_equal(g.ptr.cpu().numpy(), ptr)
    assert np.array_equal(g.col.cpu().numpy()[:g.nnz], col)
    assert np.array_equal(g.w.cpu().numpy()[:g.nnz].view(np.uint32), wo.view(np.uint32))


def test_ingest_row_above_the_scratch_cap_is_a_status(oracle_port):
    """the scratch cap of the ingest is pow2(max(min(max(n, 4096), e), 2049)): 4096 for n = 100 and e > 4096. A row
    of exactly 4096 raw entries is ingested like the oracle does, one of 4097 raises RLAP_ERR_STAR_TOO_LARGE"""
    import rlap_b200
    from rlap_b200 import _native
    for k, ok in ((4096, True), (4097, False)):
        ei, w, n = tiers.ingest_rows((k,), n=100, seed=3)
        assert ei.shape[1] > 4096
        if ok:
            ptr, col, wo = oracle_port.ingest(ei, w, n)
            g = rlap_b200.prepare(torch.from_numpy(ei).cuda(), torch.from_numpy(w).cuda(), n, validate=False)
            assert np.array_equal(g.col.cpu().numpy()[:g.nnz], col)
            assert np.array_equal(g.w.cpu().numpy()[:g.nnz].view(np.uint32), wo.view(np.uint32))
        else:
            with pytest.raises(_native.RlapError) as e:
                rlap_b200.prepare(torch.from_numpy(ei).cuda(), torch.from_numpy(w).cuda(), n, validate=False)
            assert e.value.status == _native.RLAP_ERR_STAR_TOO_LARGE
