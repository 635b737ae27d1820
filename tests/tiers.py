"""Steered stars: graphs whose elimination order, and therefore the kernel tier every interesting star, survivor and
ingest row takes, is known in advance (tests/test_oracle_tiers.py proves it on the oracle, tests/test_gpu_tiers.py runs
them on the GPU bit for bit against it).

A steered star has a centre c (vertex 0) and, around it,
  * L leaves: protected, joined in a ring, adjacent to c;
  * D pendants: unprotected, adjacent to c only; they go first and leave dead entries in c's CSR row;
  * F_dup feeders: unprotected, adjacent to c and to leaf i; the fill (c, leaf i) is a multi-edge at c;
  * F_clean feeders: unprotected, adjacent to c and to a protected z_i not adjacent to c; the fill (c, z_i) is new;
  * F_pair feeder pairs: two feeders sharing one protected z_i: two fills (c, z_i), a multi-edge between fills;
  * F_dead feeders f_i with partners y_i (y_i < f_i, y_i adjacent to f_i and to a leaf): when f_i goes before y_i its
    fill (c, y_i) dies with y_i, whose own star {leaf, c} adds the live fill (c, leaf).
Unprotected c goes last (num_remove = every unprotected vertex): the case drives one elimination tier. Protected c
survives: the case drives one emission tier.

Under degree / coarsen every feeder and partner has key <= 2 (pendants 1) and c more, so c goes alone in the last round;
a partner waits for its feeder because it has the lower id and the same key. Under o_v = random the seed is searched
so that c has the last rank among the unprotected vertices (`steer_seed`); the partners that happen to rank before their
feeder give a live fill instead of a dead one, and `claims` counts them from the same permutation.
"""
from dataclasses import dataclass, field

import numpy as np

LCAP, LANE_NB_MAX = 16, 48               # schur.cu eliminate_star_lane
TILE_MAX, FCAP = 32, 16                  # schur.cu run_warp_items: register tiles (eliminate_star_regs)
CAP_WARP, STAGE_CAP, HUB_DEG = 128, 128, 64   # schur.cuh
ELIM_CAP_CTA = 1024                      # schur.cuh: CAP_WARP x 8 warps of the elimination block
FS_LANE, FS_NB_MAX, FSORT_MAX = 16, 40, 32    # emit.cu k_emit_fsort
CAP_REGS, CAP_CTA, CAP_BIG = 512, 2048, 12288  # emit.cu size classes
WF_CAP = 448                             # emit.cu k_emit_write
INGEST_WARP, INGEST_CTA = 128, 2048      # ingest.cu

TAG_STAR = 2
# two neighbours of centre 0 whose 32-bit shuffle keys (x.z of Philox(c, u, view, TAG_STAR) under key (5, 0)) are equal
# while the 64-bit keys (z, w) differ, the lower id having the larger key: a sort on 32 bits that kept the id order
# would get them the wrong way round. Found by `find_key_tie(5, 0, 0, 1 << 17)`
TIE_SEED, TIE_PAIR = 5, (122190, 124857)

MODES = [(ov, on) for ov in ("random", "degree", "coarsen") for on in ("asc", "desc", "random")]


# ------------------------------------------------------------------------------------------------ Philox (numpy)
def philox_np(k0, k1, c0, c1, c2, c3):
    """Philox4x32-10 over uint32 arrays (the oracle's and the kernels' generator), vectorised"""
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    c = [np.asarray(x, dtype=np.uint64) & np.uint64(0xFFFFFFFF) for x in np.broadcast_arrays(c0, c1, c2, c3)]
    a, b = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        h0, l0, h1, l1 = p0 >> np.uint64(32), p0 & m32, p1 >> np.uint64(32), p1 & m32
        c = [h1 ^ c[1] ^ a, l1, h0 ^ c[3] ^ b, l0]
        a, b = (a + np.uint64(0x9E3779B9)) & m32, (b + np.uint64(0xBB67AE85)) & m32
    return [x.astype(np.uint32) for x in c]


def shuffle_keys(seed, centre, nbrs, view):
    """(32-bit x.z, 64-bit (z, w)) shuffle keys of the neighbours `nbrs` in the star of `centre`"""
    _, _, z, w = philox_np(seed & 0xFFFFFFFF, seed >> 32, centre, np.asarray(nbrs), view, TAG_STAR)
    return z, (z.astype(np.uint64) << np.uint64(32)) | w.astype(np.uint64)


def find_key_tie(seed, centre, view, limit):
    """pairs (u1 < u2 < limit, neither = centre) with equal 32-bit and different 64-bit shuffle keys"""
    u = np.arange(1, limit, dtype=np.int64)
    u = u[u != centre]
    z, k = shuffle_keys(seed, centre, u, view)
    o = np.argsort(z, kind="stable")
    zs = z[o]
    hit = np.nonzero(zs[1:] == zs[:-1])[0]
    return [tuple(sorted((int(u[o[i]]), int(u[o[i + 1]])))) for i in hit if k[o[i]] != k[o[i + 1]]]


# ------------------------------------------------------------------------------------------------ weights
def weights(ei, kind):
    """symmetric fp32 weights of the unordered pairs: 'unit'; 'two' (1 and 3, long runs of ties); 'wide' (log-uniform
    over about 2^-40 .. 2^10, so that light entries quantise to 0 inside a star)"""
    if kind == "unit":
        return None
    a, b = np.minimum(ei[0], ei[1]).astype(np.uint64), np.maximum(ei[0], ei[1]).astype(np.uint64)
    h = (a * np.uint64(0x9E3779B1) + b * np.uint64(0x85EBCA77)) & np.uint64(0xFFFFFFFF)
    h = (h ^ (h >> np.uint64(15))) * np.uint64(0x2C1B3C6D) & np.uint64(0xFFFFFFFF)
    h = (h ^ (h >> np.uint64(12))) & np.uint64(0xFFFFFF)
    if kind == "two":
        return np.where(h % np.uint64(3) == 0, 3.0, 1.0).astype(np.float32)
    assert kind == "wide"
    return np.exp2(-40.0 + 50.0 * h.astype(np.float64) / float(1 << 24)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ generator
@dataclass
class Case:
    name: str
    ei: np.ndarray            # [2, E] int64, both directions
    n: int
    keep: np.ndarray          # bool [n]
    num_remove: int           # every unprotected vertex
    centre: int
    protected: bool           # the centre survives (an emission case)
    full: bool
    claims: dict              # tier quantities of the centre, per o_v ('random' may differ from degree / coarsen)
    modes: list               # (o_v, o_n) this case is run in
    seeds: dict = field(default_factory=dict)   # o_v -> seed of the view (view_base 0)
    wkinds: tuple = ("unit",)


def _edges(pairs):
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    return np.concatenate([p.T, p[:, ::-1].T], axis=1)


def steered_star(name, L, D=0, F_dup=0, F_clean=0, F_pair=0, F_dead=0, protected=False, full=False, leaves=None,
                 modes=None, wkinds=("unit",), pad_to=0, seed=11, view=0):
    """a steered star (module docstring). leaves: explicit leaf ids (default 1..L). pad_to: add protected isolated
    vertices up to this many."""
    c = 0
    leaves = list(range(1, L + 1)) if leaves is None else sorted(leaves)
    assert len(leaves) == L and L >= 3 and c not in leaves
    nxt = max(leaves) + 1
    pairs, prot = [], set(leaves)
    for i in range(L):
        pairs += [(c, leaves[i]), (leaves[i], leaves[(i + 1) % L])]
    if L == 3:           # the ring of three has each edge once
        pairs = [(c, u) for u in leaves] + [(leaves[0], leaves[1]), (leaves[1], leaves[2]), (leaves[2], leaves[0])]
    unprot = []

    def new(k):
        nonlocal nxt
        ids = list(range(nxt, nxt + k))
        nxt += k
        return ids

    for p in new(D):
        pairs.append((c, p)); unprot.append(p)
    for i, f in enumerate(new(F_dup)):
        pairs += [(c, f), (f, leaves[i % L])]; unprot.append(f)
    for f in new(F_clean):
        z = new(1)[0]
        pairs += [(c, f), (f, z)]; unprot.append(f); prot.add(z)
    for _ in range(F_pair):
        f1, f2, z = new(3)
        pairs += [(c, f1), (f1, z), (c, f2), (f2, z)]; unprot += [f1, f2]; prot.add(z)
    dead = []
    for i in range(F_dead):
        y, f = new(2)           # y < f: under degree / coarsen the partner waits for its feeder
        pairs += [(c, f), (f, y), (y, leaves[(i * 7 + 3) % L])]; unprot += [f, y]; dead.append((f, y))
    n = max(nxt, pad_to)
    keep = np.zeros(n, dtype=bool)
    keep[:] = True
    keep[unprot] = False
    keep[c] = protected
    m = int((~keep).sum())
    ei = _edges(pairs)
    modes = list(MODES) if modes is None else list(modes)
    seeds = {}
    for ov in {ov for ov, _ in modes}:
        seeds[ov] = seed if ov != "random" or protected else steer_seed(keep, c, view, seed)
    claims = {}
    base_nb = L + D + F_dup + F_clean + 2 * F_pair + F_dead
    fills = F_dup + F_clean + 2 * F_pair + F_dead
    for ov in seeds:
        a = F_dead
        if ov == "random" and F_dead:
            rank = _ranks(keep, seeds[ov], view)
            a = sum(int(rank[f] < rank[y]) for f, y in dead)
        claims[ov] = dict(lv=L + fills, nb=base_nb, fl=fills + a, L=L + F_clean + F_pair, fills=fills, dead=a,
                          multi=("fill_base" if F_dup or F_dead else "fill_fill" if F_pair else "none"),
                          tie=bool(set(TIE_PAIR) <= set(leaves)))
    return Case(name, ei, n, keep, m, c, protected, full, claims, modes, seeds, tuple(wkinds))


def _ranks(keep, seed, view):
    """rank of every unprotected vertex under o_v = random (graph 0); -1 for protected ones"""
    from oracle import port
    un = np.nonzero(~keep)[0]
    r = port.rank_perm(seed, 0, view, un.shape[0])
    out = np.full(keep.shape[0], -1, dtype=np.int64)
    out[un] = r
    return out


def steer_seed(keep, c, view, start=11):
    """the first seed >= start under which the unprotected vertex c has the last rank (o_v = random)"""
    from oracle import port
    un = np.nonzero(~keep)[0]
    m = un.shape[0]
    i = int(np.searchsorted(un, c))
    for s in range(start, start + 200 * m + 1000):
        if port.rank_perm(s, 0, view, m)[i] == m - 1:
            return s
    raise AssertionError("no steering seed")


def write_overflow_case(k=32, fills=16):
    """k protected survivors with consecutive ids 0..k-1 (one warp of k_emit_write), each with `fills` clean fills and
    no base entry left: k * fills staged fills for the warp (512 > WF_CAP = 448 for the defaults)"""
    pairs, unprot = [], []
    nxt = k
    for c in range(k):
        for _ in range(fills):
            f, z = nxt, nxt + 1
            nxt += 2
            pairs += [(c, f), (f, z)]
            unprot.append(f)
    n = nxt
    keep = np.ones(n, dtype=bool)
    keep[unprot] = False
    claims = {ov: dict(lv=fills, nb=fills, fl=fills, L=fills, fills=fills, dead=0, multi="none", tie=False,
                       warp_fills=k * fills) for ov in ("random", "degree", "coarsen")}
    return Case(f"write_overflow_{k}x{fills}", _edges(pairs), n, keep, len(unprot), 0, True, False, claims,
                list(MODES), {ov: 11 for ov in ("random", "degree", "coarsen")})


# ------------------------------------------------------------------------------------------------ tier table
def _lane(q):
    return not q["full"] and q["lv"] <= LCAP and q["nb"] <= LANE_NB_MAX


def _tile(q):
    return (not _lane(q) and q["lv"] <= TILE_MAX and q["nb"] <= TILE_MAX and q["fl"] <= FCAP
            and q["nb"] + q["fl"] <= TILE_MAX)


def _warp_smem(q):
    return q["lv"] <= CAP_WARP and not _lane(q) and not _tile(q)


def _shuffle(q):
    return q["o_v"] == "coarsen" or q["o_n"] == "random"


def _fsort_clean(q):
    return q["multi"] == "none" and 1 <= q["fills"] <= FSORT_MAX


# (group, name, code location, predicate over the centre's quantities, modes where the tier exists)
_NOT_FULL = [(ov, on, False) for ov, on in MODES]
_ALL = _NOT_FULL + [(ov, "asc", True) for ov in ("random", "degree", "coarsen")]
_SHUF = [(ov, on, False) for ov, on in MODES if ov == "coarsen" or on == "random"]
TIERS = [
    ("elim", "lane", "schur.cu run_warp_items K_LANE / eliminate_star_lane",
     lambda q: not q["prot"] and _lane(q) and q["multi"] == "none" and not q["tie"], _NOT_FULL),
    ("elim", "lane_to_smem_multi", "schur.cu eliminate_star_lane: dup -> return false",
     lambda q: not q["prot"] and _lane(q) and q["multi"] != "none", _NOT_FULL),
    ("elim", "lane_to_smem_key_tie", "schur.cu eliminate_star_lane: tie |= ky == kx",
     lambda q: not q["prot"] and _lane(q) and q["tie"] and _shuffle(q), _SHUF),
    ("elim", "tile", "schur.cu run_warp_items K_TILE / eliminate_star_regs",
     lambda q: not q["prot"] and _tile(q), _ALL),
    ("elim", "tile_key_tie", "schur.cu eliminate_star_regs with a 32-bit shuffle-key tie",
     lambda q: not q["prot"] and _tile(q) and q["tie"] and _shuffle(q), _SHUF),
    ("elim", "warp_smem", "schur.cu run_warp_items K_SMEM / run_smem_items",
     lambda q: not q["prot"] and _warp_smem(q), _ALL),
    ("elim", "warp_smem_key_tie", "schur.cu eliminate_star<false> with a 32-bit shuffle-key tie",
     lambda q: not q["prot"] and _warp_smem(q) and q["tie"] and _shuffle(q), _SHUF),
    ("elim", "warp_smem_long_fill_list", "schur.cu StagedList rest walk (fill list > STAGE_CAP)",
     lambda q: not q["prot"] and _warp_smem(q) and q["fl"] > STAGE_CAP and q["dead"] > 0, _NOT_FULL),
    ("elim", "warp_smem_random_hub", "schur.cu run_smem_items: hub fill lists (nb >= HUB_DEG, o_v = random)",
     lambda q: not q["prot"] and _warp_smem(q) and q["nb"] >= HUB_DEG and q["fills"] > 0 and q["o_v"] == "random",
     [(ov, on, False) for ov, on in MODES if ov == "random"]),
    ("elim", "lane_lv16", "schur.cu run_warp_items: the largest lane star, lv = LCAP",
     lambda q: not q["prot"] and _lane(q) and q["lv"] == LCAP and q["multi"] == "none", _NOT_FULL),
    ("elim", "tile_lv17", "schur.cu eliminate_star_regs: the smallest tile after the lane stars, lv = LCAP + 1",
     lambda q: not q["prot"] and _tile(q) and q["lv"] == LCAP + 1, _NOT_FULL),
    ("elim", "block", "schur.cu run_block_items, lv <= ELIM_CAP_CTA",
     lambda q: not q["prot"] and CAP_WARP < q["lv"] <= ELIM_CAP_CTA, _ALL),
    ("elim", "block_multi", "schur.cu run_block_items with multi-edges",
     lambda q: not q["prot"] and CAP_WARP < q["lv"] <= ELIM_CAP_CTA and q["multi"] != "none", _NOT_FULL),
    ("elim", "scratch", "star.cuh scratch slot, lv > ELIM_CAP_CTA",
     lambda q: not q["prot"] and q["lv"] > ELIM_CAP_CTA, _ALL),
    ("elim", "scratch_lv1025", "star.cuh scratch slot: the smallest star above ELIM_CAP_CTA",
     lambda q: not q["prot"] and q["lv"] == ELIM_CAP_CTA + 1, _NOT_FULL),
    ("elim", "scratch_key_copy_3000", "star_tie_order at the 3000 size",
     lambda q: not q["prot"] and q["lv"] == 3000 and not q["full"], _NOT_FULL),
    ("elim", "scratch_in_place_6000", "star_tie_order at the 6000 size",
     lambda q: not q["prot"] and q["lv"] == 6000 and not q["full"], _NOT_FULL),
    ("elim", "scratch_multi", "scratch slot with multi-edges",
     lambda q: not q["prot"] and q["lv"] > ELIM_CAP_CTA and q["multi"] != "none", _NOT_FULL),
    ("elim", "scratch_overflow_retry", "ops.schur_views RLAP_ERR_STAR_TOO_LARGE retry",
     lambda q: not q["prot"] and q["lv"] > q.get("scratch_cap", 1 << 62), _NOT_FULL),
    ("emit", "fsort_lane", "emit.cu k_emit_fsort lane path",
     lambda q: q["prot"] and _fsort_clean(q) and q["fills"] <= FS_LANE and q["nb"] <= FS_NB_MAX, _NOT_FULL),
    ("emit", "fsort_warp", "emit.cu k_emit_fsort warp path",
     lambda q: q["prot"] and _fsort_clean(q) and (q["fills"] > FS_LANE or q["nb"] > FS_NB_MAX), _NOT_FULL),
    ("emit", "fsort_warp_nb41", "emit.cu k_emit_fsort: 16 fills, nb = 41",
     lambda q: q["prot"] and _fsort_clean(q) and q["fills"] == FS_LANE and q["nb"] == FS_NB_MAX + 1, _NOT_FULL),
    ("emit", "merge_many_fills", "emit.cu k_emit_fsort: > 32 fills -> merge path",
     lambda q: q["prot"] and q["multi"] == "none" and q["fills"] > FSORT_MAX, _NOT_FULL),
    ("emit", "merge_fill_fill_lane", "emit.cu k_emit_fsort lane: two fills to one neighbour",
     lambda q: q["prot"] and q["multi"] == "fill_fill" and q["fills"] <= FS_LANE and q["nb"] <= FS_NB_MAX, _NOT_FULL),
    ("emit", "merge_fill_fill_warp", "emit.cu k_emit_fsort warp: two fills to one neighbour",
     lambda q: q["prot"] and q["multi"] == "fill_fill" and FS_LANE < q["fills"] <= FSORT_MAX, _NOT_FULL),
    ("emit", "merge_fill_base_lane", "emit.cu k_emit_fsort lane: a fill parallel to a base edge",
     lambda q: q["prot"] and q["multi"] == "fill_base" and q["fills"] <= FS_LANE and q["nb"] <= FS_NB_MAX, _NOT_FULL),
    ("emit", "merge_fill_base_warp", "emit.cu k_emit_fsort warp: a fill parallel to a base edge",
     lambda q: q["prot"] and q["multi"] == "fill_base" and FS_LANE < q["fills"] <= FSORT_MAX, _NOT_FULL),
] + [
    ("emit", f"merge_class_{lv}", "emit.cu size_class / k_emit_sort_mid<R>, k_emit_sort_block, k_emit_sort_big",
     (lambda lv: lambda q: q["prot"] and q["multi"] != "none" and q["lv"] == lv)(lv), _NOT_FULL)
    for lv in (32, 33, 64, 65, 128, 129, 256, 257, 512, 513, 2048, 2049, 12288, 12289)
] + [
    ("emit", "merge_scratch_overflow_retry", "emit.cu emit_sort_staged lraw > cap -> retry",
     lambda q: q["prot"] and q["lv"] > q.get("scratch_cap", 1 << 62), _NOT_FULL),
    ("emit", "write_overflow", "emit.cu k_emit_write: > WF_CAP staged fills in one warp",
     lambda q: q["prot"] and q.get("warp_fills", 0) > WF_CAP, _NOT_FULL),
]


def quantities(case, o_v, o_n, claims=None):
    q = dict(case.claims[o_v] if claims is None else claims)
    q.update(o_v=o_v, o_n=o_n, full=case.full, prot=case.protected)
    if getattr(case, "scratch_cap", 0):
        q["scratch_cap"] = case.scratch_cap
    return q


def tiers_of(case, o_v, o_n):
    q = quantities(case, o_v, o_n)
    return [t[1] for t in TIERS if t[3](q)]


# ------------------------------------------------------------------------------------------------ the cases
def _tie_leaves(L):
    return list(TIE_PAIR) + list(range(1, L - 1))


def cases():
    """every steered case: elimination (unprotected centre) and emission (protected centre)"""
    ALLW = ("unit", "two", "wide")
    out = [
        steered_star("lane_L5", 5, wkinds=ALLW),
        steered_star("lane_L8_D40", 8, D=40, wkinds=ALLW),                          # nb = 48: longest lane row
        steered_star("lane_L16", 16, wkinds=ALLW),                                  # lv = 16: largest lane star
        steered_star("tile_L17", 17, wkinds=ALLW),                                  # lv = 17: smallest tile
        steered_star("lane_multi_L5_dup2", 5, F_dup=2, wkinds=ALLW),
        steered_star("lane_multi_L6_clean3_dup1", 6, F_dup=1, F_clean=3, D=4, wkinds=ALLW),
        steered_star("tile_L20", 20, wkinds=ALLW),
        steered_star("tile_L17_dup4", 17, F_dup=4, wkinds=ALLW),
        steered_star("tile_L12_clean8", 12, F_clean=8, wkinds=ALLW),
        steered_star("warp_L8_D41", 8, D=41, wkinds=ALLW),                          # nb = 49 > LANE_NB_MAX
        steered_star("warp_L100", 100, wkinds=ALLW),
        steered_star("warp_L60_dup30_clean20", 60, F_dup=30, F_clean=20, D=5, wkinds=ALLW),
        steered_star("warp_dead_L4_dead120", 4, F_dead=120, wkinds=("unit", "wide")),
        steered_star("warp_hub_L8_D64_clean20", 8, D=64, F_clean=20, wkinds=ALLW,
                     modes=[m for m in MODES if m[0] == "random"]),
        steered_star("block_L200", 200, wkinds=ALLW),
        steered_star("block_L1000_dup24", 1000, F_dup=24, wkinds=ALLW),            # lv = 1024
        steered_star("block_L600_dup100_clean100", 600, F_dup=100, F_clean=100, D=50, wkinds=ALLW),
        steered_star("scratch_L1000_dup25", 1000, F_dup=25, wkinds=ALLW),          # lv = 1025
        steered_star("scratch_L3000", 3000, wkinds=ALLW),
        steered_star("scratch_L6000", 6000, wkinds=("unit", "two")),
        steered_star("scratch_L1100_dup1500", 1100, F_dup=1500, wkinds=("unit", "wide")),
    ]
    # 32-bit shuffle-key ties: only o_n = random and coarsen compare shuffle keys
    shuf = [m for m in MODES if m[0] == "coarsen" or m[1] == "random"]
    for nm, L in (("lane_tie_L6", 6), ("tile_tie_L20", 20), ("warp_tie_L100", 100)):
        out.append(steered_star(nm, L, leaves=_tie_leaves(L), modes=shuf, seed=TIE_SEED, wkinds=("unit", "two")))
    # full clique: single-centre elimination, all three o_v
    full_modes = [(ov, "asc") for ov in ("random", "degree", "coarsen")]
    for L in (5, 20, 100, 600, 1100, 2500):
        out.append(steered_star(f"full_L{L}", L, full=True, modes=full_modes, wkinds=("unit", "wide")))
    # emission: protected centre
    E = dict(protected=True, wkinds=ALLW)
    out += [
        steered_star("fsort_lane_clean10", 5, F_clean=10, **E),
        steered_star("fsort_warp_clean20", 3, F_clean=20, **E),
        steered_star("fsort_warp_nb41", 25, F_clean=16, **E),
        steered_star("merge_clean40", 4, F_clean=40, **E),
        steered_star("merge_fillfill_lane", 5, F_pair=1, F_clean=2, **E),
        steered_star("merge_fillfill_warp", 5, F_pair=2, F_clean=16, **E),
        steered_star("merge_fillbase_lane", 5, F_dup=1, F_clean=3, **E),
        steered_star("merge_fillbase_warp", 5, F_dup=10, F_clean=10, **E),
    ]
    for lv in (32, 33, 64, 65, 128, 129, 256, 257, 512, 513, 2048, 2049, 12288, 12289):
        kinds = ("unit", "wide") if lv > 2049 else ALLW
        out.append(steered_star(f"merge_class_lv{lv}", lv - 3, F_dup=2, F_pair=0, F_clean=1, protected=True,
                                wkinds=kinds))
    out.append(write_overflow_case())
    return out


def unmasked_star(name, L, seed=11, view=0, wkinds=("unit", "two", "wide")):
    """o_v = random without a keep mask: every vertex is ranked, over all n of the graph. The centre of a star with L
    ring leaves (n = L + 1) is placed on the vertex of rank 0, so with num_remove = 1 it goes first and alone, its star
    being its whole CSR row: lv = nb = L, no fill"""
    from oracle import port
    n = L + 1
    c = int(np.argmin(port.rank_perm(seed, 0, view, n)))
    leaves = [u for u in range(n) if u != c]
    pairs = [(c, u) for u in leaves] + [(leaves[i], leaves[(i + 1) % L]) for i in range(L)]
    claims = {"random": dict(lv=L, nb=L, fl=0, L=L, fills=0, dead=0, multi="none", tie=False)}
    return Case(name, _edges(pairs), n, None, 1, c, False, False, claims,
                [m for m in MODES if m[0] == "random"], {"random": seed}, tuple(wkinds))


def unmasked_cases():
    """the unmasked path, one steered first star per elimination tier (lane, its last size, tile, warp, block, the
    first scratch size, scratch)"""
    return [unmasked_star(f"unmasked_L{L}", L) for L in (5, 16, 17, 30, 100, 600, 1025, 3000)]


def retry_cases():
    """stars and surviving hubs larger than an explicit scratch_cap of 4096: RLAP_ERR_STAR_TOO_LARGE, then the retry"""
    a = steered_star("retry_elim_L6000", 6000, wkinds=("unit",))
    b = steered_star("retry_emit_lv13000", 12998, F_dup=2, protected=True, wkinds=("unit", "wide"))
    for c in (a, b):
        c.scratch_cap = 4096
    return [a, b]


def ingest_rows(lengths=(128, 129, 2048, 2049, 5000), n=6000, seed=0):
    """(edge_index, weights, n) whose owner rows 0, 1, ... (the entries with dst = owner) have the given raw lengths:
    non-zero entries, duplicates included, plus zero weights the ingest drops. Duplicate runs are order sensitive in
    fp32 (1.0 before or after several 2^-24) and the input order is shuffled. The twin direction has one unit entry per
    distinct neighbour: the graph is not symmetric (ingest it with validate=False)."""
    rng = np.random.default_rng(seed)
    src, dst, w = [], [], []
    for owner, k in enumerate(lengths):
        cnt = 0
        while cnt < k:
            u = int(rng.integers(len(lengths), n))
            run = int(min(k - cnt, rng.integers(1, 7)))
            vals = [1.0] + [2.0 ** -24] * (run - 1) + ([0.0] if rng.random() < 0.3 else [])
            rng.shuffle(vals)
            for x in vals:
                src.append(u); dst.append(owner); w.append(x)
            cnt += run
    src, dst, w = np.array(src), np.array(dst), np.array(w, dtype=np.float32)
    perm = rng.permutation(src.shape[0])
    src, dst, w = src[perm], dst[perm], w[perm]
    twin = np.unique(np.stack([dst, src]), axis=1)
    ei = np.concatenate([np.stack([src, dst]), twin], axis=1).astype(np.int64)
    wt = np.concatenate([w, np.ones(twin.shape[1], dtype=np.float32)])
    return ei, wt, n
