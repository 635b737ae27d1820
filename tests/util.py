"""Shared helpers for the test-suite (graphs, dense Laplacians, exact Schur complements)."""
import hashlib

import numpy as np

from rlap_b200 import graphs

COMBOS = [(ov, on) for ov in ("random", "degree", "coarsen") for on in ("asc", "desc", "random")]

# injected seeds of the comparison with the reference build on the larger graphs (non-default sampling seed)
REF_BUILD_SEEDS = dict(sample_seed=77, rd_seed=5)


def sym_weights(ei: np.ndarray, lo=0.5, hi=1.5) -> np.ndarray:
    """deterministic symmetric weights in [lo, hi): a hash of the unordered pair"""
    a, b = np.minimum(ei[0], ei[1]), np.maximum(ei[0], ei[1])
    h = (a * 7919 + b * 104729) % 1000
    return (lo + (hi - lo) * h / 1000.0).astype(np.float32)


def edge_info(ei: np.ndarray, w=None) -> np.ndarray:
    E = ei.shape[1]
    w = np.ones(E) if w is None else np.asarray(w, dtype=np.float64)
    return np.concatenate([ei.T.astype(np.float64), w.reshape(-1, 1)], axis=1)


def laplacian(rows, cols, w, n) -> np.ndarray:
    A = np.zeros((n, n))
    np.add.at(A, (np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64)), np.asarray(w, dtype=np.float64))
    return np.diag(A.sum(0)) - A


def exact_schur(L: np.ndarray, keep: np.ndarray) -> np.ndarray:
    n = L.shape[0]
    F = np.setdiff1d(np.arange(n), keep)
    if F.size == 0:
        return L[np.ix_(keep, keep)]
    return L[np.ix_(keep, keep)] - L[np.ix_(keep, F)] @ np.linalg.solve(L[np.ix_(F, F)], L[np.ix_(F, keep)])


def small_cases():
    """(name, edge_index, n, graph_ptr or None, num_remove) for the parity tests"""
    cases = []
    cases.append(("ba100_m50", graphs.barabasi_albert(100, 50, seed=1), 100, None, 50))
    cases.append(("ba300_m3", graphs.barabasi_albert(300, 3, seed=2), 300, None, 150))
    cases.append(("sbm_cora", graphs.sbm(2708, 7, 5278, seed=0), 2708, None, 812))
    ei, ptr = graphs.proteins_like_batch(40, seed=3)
    cases.append(("proteins40_union", ei, int(ptr[-1]), None, int(ptr[-1]) // 2))
    cases.append(("proteins40_pergraph", ei, int(ptr[-1]), ptr, (np.diff(ptr) // 2)))
    return cases


def reference_build_cases():
    """(name, edge_index, weights or None, n, num_remove) compared with the reference build at REF_BUILD_SEEDS: the
    Cora-shaped SBM and BA(500, 4), each with unit weights ("sbm2708", "ba500") and with sym_weights (name + "w")"""
    cases = []
    for name, ei, n, t in (("sbm2708", graphs.sbm(2708, 7, 5278, seed=0), 2708, 812),
                           ("ba500", graphs.barabasi_albert(500, 4, seed=9), 500, 250)):
        cases.append((name, ei, None, n, t))
        cases.append((name + "w", ei, sym_weights(ei).astype(np.float64), n, t))
    return cases


def output_digest(out: np.ndarray) -> np.ndarray:
    """SHA-256 of an [E',3] float64 output as uint8 [32]: equal digests = bit-identical outputs"""
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(out, dtype=np.float64).tobytes()).digest(), dtype=np.uint8)


def batch_masks(gp: np.ndarray):
    """[(name, keep)] of a batch: one whole graph protected, and a single unprotected vertex per graph"""
    n = int(gp[-1])
    whole = np.zeros(n, dtype=bool)
    whole[gp[3]:gp[4]] = True
    single = np.ones(n, dtype=bool)
    for g in range(gp.shape[0] - 1):
        single[gp[g] + g % (gp[g + 1] - gp[g])] = False
    return [("whole_graph", whole), ("single_free", single)]


def keyed_pin_runs(port):
    """(id, ptr, col, w, keyword arguments of port.keyed_schur) of the keyed-mode runs pinned by stored digests
    (tests/golden/keyed/cases.npz): small_cases() x unit / sym_weights x masks (none, random 10 % and 50 %, and for the
    proteins batch batch_masks) x num_remove (the case's own, n) x COMBOS; then a non-zero view, FLAG_SHARED_ORDER and
    FLAG_FULL_CLIQUE with masks"""
    from rlap_b200 import graphs
    _, gp40 = graphs.proteins_like_batch(40, seed=3)
    for name, ei, n, gp, t in small_cases():
        rng = np.random.default_rng(17)
        masks = [("none", None), ("rand10", rng.random(n) < 0.1), ("rand50", rng.random(n) < 0.5)]
        if name.startswith("proteins40"):
            masks += batch_masks(gp40)
        for wname, wts in (("unit", None), ("sym", sym_weights(ei))):
            ptr, col, w = port.ingest(ei, wts, n)
            for mname, keep in masks:
                for tname, tt in (("own", t), ("all", n)):
                    for o_v, o_n in COMBOS:
                        yield (f"{name}/{wname}/{mname}/t_{tname}/{o_v}/{o_n}", ptr, col, w,
                               dict(num_remove=tt, o_v=o_v, o_n=o_n, seed=5, graph_ptr=gp, keep=keep))
    n = 300
    ei = graphs.barabasi_albert(n, 3, seed=2)
    ptr, col, w = port.ingest(ei, None, n)
    keep = np.random.default_rng(3).random(n) < 0.5
    for mname, k in (("none", None), ("rand50", keep)):
        for o_v, o_n in COMBOS:
            yield (f"ba300_m3/unit/{mname}/view7/{o_v}/{o_n}", ptr, col, w,
                   dict(num_remove=150, o_v=o_v, o_n=o_n, seed=9, view=7, keep=k))
        for o_n in ("asc", "desc", "random"):
            yield (f"ba300_m3/unit/{mname}/view7_shared_order/random/{o_n}", ptr, col, w,
                   dict(num_remove=150, o_v="random", o_n=o_n, seed=9, view=7, flags=port.FLAG_SHARED_ORDER, keep=k))
    n = 100
    ei = graphs.barabasi_albert(n, 3, seed=1)
    ptr, col, w = port.ingest(ei, sym_weights(ei), n)
    rng = np.random.default_rng(4)
    masks = [("none", None), ("rand10", rng.random(n) < 0.1), ("rand50", rng.random(n) < 0.5)]
    for mname, k in masks:
        for o_v in ("random", "degree"):
            yield (f"ba100_m3/sym/{mname}/full_clique/{o_v}/asc", ptr, col, w,
                   dict(num_remove=n, o_v=o_v, o_n="asc", seed=7, flags=port.FLAG_FULL_CLIQUE, keep=k))


def keyed_digest(port, ptr, col, w, kw) -> np.ndarray:
    """SHA-256 (uint8 [32]) of one keyed-mode run: row, col and fp32 weight bytes, the five stats, the elimination order"""
    r, c, wt, st, order = port.keyed_schur(ptr, col, w, return_stats=True, return_order=True, **kw)
    h = hashlib.sha256()
    for a in (r.astype(np.int32), c.astype(np.int32), wt.astype(np.float32),
              np.array([st[k] for k in ("D", "F", "maxlen", "rounds", "Draw")], dtype=np.int64), order.astype(np.int32)):
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)
