"""The steered cases of tests/tiers.py do what they claim, proven on the keyed oracle (CPU): the intended elimination
order, the tier quantities of the centre, a case for every row of the tier table in every mode where that tier
exists, the 32-bit shuffle-key tie, and order-sensitive ingest runs."""
import functools

import numpy as np
import pytest

from tests import tiers


@functools.lru_cache(maxsize=None)
def _cases():
    return tiers.cases() + tiers.retry_cases()


def _oracle_graph(port, case, wkind="unit"):
    return port.ingest(case.ei, tiers.weights(case.ei, wkind), case.n)


def _run(port, g, case, keep, t, o_v, o_n="asc"):
    ptr, col, w = g
    return port.keyed_schur(ptr, col, w, t, o_v, o_n, seed=case.seeds.get(o_v, 11), keep=keep, return_stats=True,
                            return_order=True, flags=port.FLAG_FULL_CLIQUE if case.full else 0)


def _measured(port, case, o_v):
    """the centre's quantities recomputed from the oracle: lv = its raw live entries (D of its elimination), fl = raw
    entries read (Draw) minus its CSR row, L = its merged star (maxlen); a protected centre is measured on the same
    graph with the centre unprotected, under degree (every quantity of an emission case is order independent)"""
    g = _oracle_graph(port, case)
    ptr = g[0]
    c = case.centre
    keep = case.keep.copy()
    if case.protected:
        keep[c] = False
        o_v = "degree"
    m = int((~keep).sum())
    *_, s1, _ = _run(port, g, case, keep, m - 1, o_v)
    *_, s2, order = _run(port, g, case, keep, m, o_v)
    nb = int(ptr[c + 1] - ptr[c])
    return dict(lv=s2["D"] - s1["D"], nb=nb, fl=s2["Draw"] - s1["Draw"] - nb, L=s2["maxlen"]), order


@pytest.mark.parametrize("name", [c.name for c in _cases()])
def test_elimination_order_is_the_steered_one(oracle_port, name):
    case = next(c for c in _cases() if c.name == name)
    g = _oracle_graph(oracle_port, case)
    c = case.centre
    for o_v in sorted(case.seeds):
        *_, st, order = _run(oracle_port, g, case, case.keep, case.num_remove, o_v)
        un = ~case.keep
        assert (order[un] >= 0).all(), (name, o_v)             # every unprotected vertex goes
        assert (order[case.keep] == -1).all(), (name, o_v)     # no protected one does
        if case.protected:
            continue
        others = order[un & (np.arange(case.n) != c)]
        assert (others < order[c]).all(), (name, o_v)           # the centre goes last, alone


@pytest.mark.parametrize("name", [c.name for c in _cases()])
def test_claimed_quantities_are_the_oracles(oracle_port, name):
    case = next(c for c in _cases() if c.name == name)
    for o_v in sorted(case.seeds):
        claim = case.claims[o_v]
        if case.name.startswith("write_overflow"):
            # 32 survivors 0..31, each with 16 fills and no live base entry: its merged row is its 16 fills
            r, cc, _ = oracle_port.keyed_schur(*_oracle_graph(oracle_port, case), case.num_remove, o_v, "asc",
                                              seed=case.seeds[o_v], keep=case.keep)
            counts = np.bincount(cc, minlength=case.n)[:32]
            assert (counts == claim["fills"]).all() and claim["warp_fills"] == counts.sum(), (name, o_v)
            continue
        got, _ = _measured(oracle_port, case, o_v)
        want = {k: claim[k] for k in ("lv", "nb", "fl", "L")}
        if case.protected:
            want["fl"] = claim["fills"]              # a surviving centre: live fills only, no dead entry
        assert got == want, (name, o_v, got, want)
        assert (claim["lv"] > claim["L"]) == (claim["multi"] != "none"), (name, o_v)


def test_every_tier_is_reached_in_every_mode_where_it_exists():
    cs = _cases()
    missing = []
    for group, tier, where, pred, modes in tiers.TIERS:
        for o_v, o_n, full in modes:
            hit = [c.name for c in cs if c.full == full and (o_v, o_n) in c.modes
                   and pred(tiers.quantities(c, o_v, o_n))]
            if not hit:
                missing.append((tier, o_v, o_n, full))
    assert not missing, missing


def test_shuffle_key_tie_pair(oracle_port):
    """the stored pair ties in the top 32 bits of its shuffle key and differs in 64 (oracle Philox), and a search
    finds it again"""
    u1, u2 = tiers.TIE_PAIR
    a = oracle_port.philox(tiers.TIE_SEED, 0, 0, u1, 0, tiers.TAG_STAR)
    b = oracle_port.philox(tiers.TIE_SEED, 0, 0, u2, 0, tiers.TAG_STAR)
    assert a[2] == b[2] and a[3] > b[3]          # equal in 32 bits, and the 64-bit order is not the id order
    z, k = tiers.shuffle_keys(tiers.TIE_SEED, 0, [u1, u2], 0)
    assert z[0] == a[2] and z[1] == b[2] and k[0] != k[1]
    assert tiers.TIE_PAIR in tiers.find_key_tie(tiers.TIE_SEED, 0, 0, 1 << 17)
    for c in _cases():
        if any(q["tie"] for q in c.claims.values()):
            assert all(s == tiers.TIE_SEED for s in c.seeds.values()), c.name


def test_numpy_philox_matches_oracle(oracle_port):
    rng = np.random.default_rng(0)
    for _ in range(20):
        k0, k1, *ctr = (int(x) for x in rng.integers(0, 1 << 32, 6, dtype=np.uint64))
        want = oracle_port.philox(k0, k1, *ctr)
        got = np.array([x[()] for x in tiers.philox_np(k0, k1, *ctr)], dtype=np.uint32)
        assert np.array_equal(got, want)


def test_ingest_rows_are_order_sensitive(oracle_port):
    """the raw owner rows have the asked lengths, and the oracle's in-order fp32 sum differs from the reversed sum
    in every row: a kernel that summed a run in another order would not match it"""
    lengths = (128, 129, 2048, 2049, 5000)
    ei, w, n = tiers.ingest_rows(lengths)
    nz = w != 0
    assert np.array_equal(np.bincount(ei[1][nz], minlength=n)[:len(lengths)], lengths)
    ptr, col, wo = oracle_port.ingest(ei, w, n)
    for o in range(len(lengths)):
        sel = np.nonzero((ei[1] == o) & nz)[0]                 # input order
        diff = 0
        for j, u in enumerate(col[ptr[o]:ptr[o + 1]]):
            run = w[sel[ei[0][sel] == u]]
            fwd, rev = np.float32(0), np.float32(0)
            for x in run:
                fwd = np.float32(fwd + x)
            for x in run[::-1]:
                rev = np.float32(rev + x)
            assert fwd == wo[ptr[o] + j]
            diff += int(fwd != rev)
        assert diff > 0, o


@pytest.mark.parametrize("name", [c.name for c in tiers.unmasked_cases()])
def test_unmasked_random_centre_goes_first_alone(oracle_port, name):
    """without a keep mask: the centre is rank 0 of the permutation over all n vertices, so num_remove = 1 eliminates
    it alone, with its whole CSR row as the star (D = Draw = maxlen = L, L - 1 fills)"""
    case = next(c for c in tiers.unmasked_cases() if c.name == name)
    ptr, col, w = _oracle_graph(oracle_port, case)
    q = case.claims["random"]
    assert oracle_port.rank_perm(case.seeds["random"], 0, 0, case.n)[case.centre] == 0
    assert ptr[case.centre + 1] - ptr[case.centre] == q["nb"]
    for o_n in ("asc", "desc", "random"):
        *_, st, order = oracle_port.keyed_schur(ptr, col, w, 1, "random", o_n, seed=case.seeds["random"],
                                                return_stats=True, return_order=True)
        assert order[case.centre] == 0 and (np.delete(order, case.centre) == -1).all(), (name, o_n)
        assert (st["D"], st["Draw"], st["maxlen"], st["F"]) == (q["lv"], q["nb"], q["L"], q["L"] - 1), (name, st)


def test_unmasked_cases_reach_every_elimination_tier():
    want = ["lane", "lane_lv16", "tile", "tile_lv17", "warp_smem", "block", "scratch", "scratch_lv1025"]
    rows = {t[1]: t for t in tiers.TIERS}
    for tier in want:
        for o_n in ("asc", "desc", "random"):
            assert any(rows[tier][3](tiers.quantities(c, "random", o_n)) for c in tiers.unmasked_cases()), (tier, o_n)
