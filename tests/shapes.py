"""Call shapes: how `rlap_schur_eliminate_keep` cuts one call into view groups, restated, and the cases that put every
kind of cut under test (tests/test_call_shapes.py checks the table and the oracle side on the CPU,
tests/test_gpu_call_shapes.py runs the cases bit for bit against the keyed oracle).

One call is ONE cooperative launch of k_eliminate. Its blocks are split into K view groups; group g owns a range of
views, a range of blocks, its own list regions, counters, scratch slots and barrier (api.cu, DESIGN.md §4). The
emission then runs over all V views. A view must come out the same whatever group it lands in, at whatever offset,
beside however many other views.
"""
import functools
from dataclasses import dataclass

import numpy as np

SMS = 148                                 # B200: the device the coverage table is computed for
CTAS_PER_SM, CTAS_PER_SM_KEYS = 4, 3      # schur.cu mode_ctas: 3 for the modes with 32-bit shuffle keys
TAB_BLOCKS = 1280                         # schur.cu TAB_BLOCKS = api.cu MAX_SCRATCH_SLOTS: blocks of one launch
TAB_GROUPS = 64                           # schur.cu TAB_GROUPS = api.cu MAX_GROUPS: view groups of one launch
VIEW_VERTS_PER_BLOCK = 256                # api.cu rlap_schur_eliminate_keep: want = ceil(V n / 256) blocks
SEL_BLOCK = 1024                          # schur.cuh: ids per block of the truncation search
ELIM_CAP_CTA = 1024                       # schur.cuh: larger stars go to a scratch slot
MAX_GRID_Y = 65535                        # CUDA: gridDim.y limit (emit.cu k_emit_scatter walks the views past it)
VIEW_IDS = 1 << 32                        # view ids are 32-bit Philox counter words (api.cu, include/rlap_b200.h)
VN_LIMIT = 1 << 30                        # api.cu check_dims: V n < 2^30, work-list positions are 32-bit

O_V = ("random", "degree", "coarsen")
MODES = [(ov, on) for ov in O_V for on in ("asc", "desc", "random")]


# ------------------------------------------------------------------------------------------------ the partition
@dataclass(frozen=True)
class Shape:
    n: int
    V: int
    blocks: int
    K: int
    groups: tuple         # per group (v0, v1, b0, b1): views [v0, v1), blocks [b0, b1)

    def views_per_group(self):
        return [v1 - v0 for v0, v1, _, _ in self.groups]

    def blocks_per_group(self):
        return [b1 - b0 for _, _, b0, b1 in self.groups]

    def boundary_views(self):
        """the first and the last view of every group"""
        return sorted({v for v0, v1, _, _ in self.groups for v in (v0, v1 - 1)})


def ctas_per_sm(o_v, o_n, full=False):
    """schur.cu mode_ctas / mode_ctas_of: o_n = random and coarsen keep 32-bit shuffle keys (full clique never does;
    coarsen with full clique runs the degree kernel)"""
    return CTAS_PER_SM_KEYS if not full and (o_v == "coarsen" or o_n == "random") else CTAS_PER_SM


def launch_shape(n, V, o_v, o_n, full=False, sms=SMS):
    """api.cu rlap_schur_eliminate_keep: the grid and its view groups"""
    blocks = min(sms * ctas_per_sm(o_v, o_n, full), TAB_BLOCKS)
    blocks = min(blocks, max(1, -(-V * n // VIEW_VERTS_PER_BLOCK)))
    K = max(1, min(V, TAB_GROUPS, blocks))
    groups = tuple((V * g // K, V * (g + 1) // K, blocks * g // K, blocks * (g + 1) // K) for g in range(K))
    return Shape(n, V, blocks, K, groups)


# ------------------------------------------------------------------------------------------------ graphs
@dataclass
class GraphSpec:
    ei: np.ndarray                # [2, E] int64, both directions
    w: object                     # fp32 [E] or None (unit)
    n: int
    gptr: object                  # int64 [G + 1] or None
    num_remove: object            # int or int64 [G]
    keep: object = None           # bool [n] or None
    cheap: bool = True            # an oracle call costs well under a millisecond: every view is checked


def degenerate_sizes():
    """graph sizes and num_remove of the degenerate batch: empty graphs, singletons, pairs and small BA graphs
    interleaved (a cycle of 9 sizes), num_remove cycling through negative, 0, 1, the cap n_g - 1 and 10^9 (a cycle of
    5): every size meets every value once"""
    sizes = [0, 1, 2, 12, 0, 1, 30, 2, 7] * 5
    nr = [[-2, 0, 1, max(s - 1, 0), 10 ** 9][g % 5] for g, s in enumerate(sizes)]
    return sizes, nr


def degenerate_keep(gptr):
    """the first 30-vertex graph wholly protected, every vertex but one of the first 12-vertex graph protected"""
    sizes = np.diff(gptr)
    keep = np.zeros(int(gptr[-1]), dtype=bool)
    g30 = int(np.nonzero(sizes == 30)[0][0])
    g12 = int(np.nonzero(sizes == 12)[0][0])
    keep[gptr[g30]:gptr[g30 + 1]] = True
    keep[gptr[g12]:gptr[g12 + 1]] = True
    keep[gptr[g12] + 5] = False
    return keep


def degenerate_batch():
    from rlap_b200 import graphs
    sizes, nr = degenerate_sizes()
    eis, off = [], 0
    for g, s in enumerate(sizes):
        if s == 2:
            eis.append(np.array([[off, off + 1], [off + 1, off]], dtype=np.int64))
        elif s > 2:
            eis.append(graphs.barabasi_albert(s, min(3, s - 1), seed=g) + off)
        off += s
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return np.concatenate(eis, axis=1), gptr, np.array(nr, dtype=np.int64)


@functools.lru_cache(maxsize=None)
def graph(key):
    """the graphs of the cases, by key"""
    from rlap_b200 import graphs
    from tests import tiers, util
    if key == "ba100":                    # C1
        ei = graphs.barabasi_albert(100, 50, seed=0)
        return GraphSpec(ei, util.sym_weights(ei), 100, None, 50)
    if key == "sbm2708":                  # C2
        ei = graphs.sbm(2708, 7, 5278, seed=0)
        return GraphSpec(ei, util.sym_weights(ei), 2708, None, 812)
    if key == "ba20000":
        ei = graphs.barabasi_albert(20000, 7, seed=1)
        return GraphSpec(ei, None, 20000, None, 10000, cheap=False)
    if key == "c3":                       # C3: 1 113 PROTEINS-sized graphs
        ei, gp = graphs.proteins_like_batch(1113, seed=0)
        return GraphSpec(ei, None, int(gp[-1]), gp, np.diff(gp) // 2, cheap=False)
    if key == "c4":                       # C4: arxiv-shaped
        ei = graphs.barabasi_albert(169343, 7, seed=0)
        return GraphSpec(ei, None, 169343, None, 169343 // 2, cheap=False)
    if key == "star6000":                 # the steered 6 000-star of tests/tiers.py: a scratch-slot star in every view
        c = tiers.steered_star("scratch_L6000", 6000, modes=[m for m in MODES if m[0] != "random"])
        return GraphSpec(c.ei, None, c.n, None, c.num_remove, keep=c.keep)
    if key == "ba24":                     # molecule-sized: many views of one small graph
        ei = graphs.barabasi_albert(24, 3, seed=0)
        return GraphSpec(ei, util.sym_weights(ei), 24, None, 12)
    if key in ("degenerate", "degenerate_keep"):
        ei, gp, nr = degenerate_batch()
        keep = degenerate_keep(gp) if key == "degenerate_keep" else None
        return GraphSpec(ei, util.sym_weights(ei), int(gp[-1]), gp, nr, keep=keep)
    if key == "singletons":               # G = n: nothing can go, the output is the coalesced input
        ei = graphs.barabasi_albert(60, 3, seed=4)
        return GraphSpec(ei, util.sym_weights(ei), 60, np.arange(61, dtype=np.int64), 10 ** 9)
    raise KeyError(key)


# vertex counts, so that the coverage table needs no graph built
GRAPH_N = dict(ba100=100, sbm2708=2708, ba20000=20000, c3=42923, c4=169343, star6000=6001, ba24=24, degenerate=275,
               degenerate_keep=275, singletons=60)


# ------------------------------------------------------------------------------------------------ the cases
@dataclass(frozen=True)
class Case:
    name: str
    graph: str
    V: int
    modes: tuple
    view_base: int = 0
    full: bool = False
    shared: bool = False
    pool_cap: int = 0

    @property
    def n(self):
        return GRAPH_N[self.graph]


ONE_PER_O_V = (("random", "random"), ("degree", "asc"), ("coarsen", "desc"))
FULL = tuple((ov, "asc") for ov in O_V)


def _cases():
    out = []
    for V in (1, 3, 64, 65, 256):
        out.append(Case(f"ba100_V{V}", "ba100", V, tuple(MODES)))
    for V in (65, 129, 256):
        out.append(Case(f"sbm2708_V{V}", "sbm2708", V, tuple(MODES)))
    for V in (1, 48, 65, 128):
        out.append(Case(f"ba20000_V{V}", "ba20000", V, ONE_PER_O_V))
    for V in (16, 65):
        out.append(Case(f"c3_V{V}", "c3", V, tuple(MODES)))
    out.append(Case("c4_V128", "c4", 128, (("degree", "asc"), ("random", "asc"), ("coarsen", "asc"))))
    for V in (65, 128):
        out.append(Case(f"star6000_V{V}", "star6000", V, (("degree", "asc"), ("coarsen", "random"))))
    # full clique in the two multi-view classes. On the SBM, o_v = random eliminates hubs late: 1.9 M fills a view,
    # 60 MB of pool each, so it runs in the orders that keep the cliques small
    out.append(Case("ba100_V64_full", "ba100", 64, FULL, full=True))
    out.append(Case("sbm2708_V256_full", "sbm2708", 256, FULL[1:], full=True))
    # one order for every view, ids from 1000: the shared order is keyed on view 0, not on a group's first view
    out.append(Case("sbm2708_V65_shared_base1000", "sbm2708", 65, tuple((ov, on) for ov, on in MODES if ov == "random"),
                    view_base=1000, shared=True))
    out.append(Case("degenerate_V3", "degenerate", 3, tuple(MODES)))
    out.append(Case("degenerate_keep_V3", "degenerate_keep", 3, tuple(MODES)))
    out.append(Case("singletons_V2", "singletons", 2, ONE_PER_O_V))
    return out


CASES = _cases()
# their own tests (tests/test_gpu_call_shapes.py): more views than a grid's y dimension, an explicit small pool (the
# overflow retry), and the last view ids there are
MANY_VIEWS = Case("ba24_V70000", "ba24", 70000, (("random", "asc"), ("degree", "desc"), ("coarsen", "random")),
                  pool_cap=32)
TOP_VIEWS = Case("ba100_V65_ids_to_2^32", "ba100", 65, ONE_PER_O_V, view_base=VIEW_IDS - 65)
ALL_CASES = CASES + [MANY_VIEWS, TOP_VIEWS]


# ------------------------------------------------------------------------------------------------ shape classes
def _off_sel_block(s, c):
    return any((v0 * s.n) % SEL_BLOCK for v0, _, _, _ in s.groups[1:])


# (class, condition, predicate over (Shape, Case), o_v where it applies)
SHAPES = [
    ("one_block_one_view", "a single small view",
     lambda s, c: s.blocks == 1 and s.V == 1, O_V),
    ("one_block_several_views", "groups of one block holding several views",
     lambda s, c: s.K > 1 and max(s.blocks_per_group()) == 1 and max(s.views_per_group()) > 1, O_V),
    ("several_blocks_one_view", "several groups, each one view over several blocks",
     lambda s, c: s.K > 1 and min(s.blocks_per_group()) > 1 and max(s.views_per_group()) == 1, O_V),
    ("several_blocks_several_views", "several groups, each several views over several blocks",
     lambda s, c: s.K > 1 and min(s.blocks_per_group()) > 1 and min(s.views_per_group()) > 1, O_V),
    ("one_group_whole_grid", "one view group over every block of the launch",
     lambda s, c: s.K == 1 and s.blocks > 1, O_V),
    ("uneven_views", "groups with different view counts",
     lambda s, c: len(set(s.views_per_group())) > 1, O_V),
    ("uneven_blocks", "groups with different block counts",
     lambda s, c: len(set(s.blocks_per_group())) > 1, O_V),
    ("group_off_sel_block", "a group's first vertex-view v0 n is not a multiple of SEL_BLOCK (its blockcnt region)",
     _off_sel_block, O_V),
    ("scratch_star_every_group", "a star above ELIM_CAP_CTA in every view of every group",
     lambda s, c: c.graph == "star6000" and s.K == TAB_GROUPS, ("degree", "coarsen")),
    ("views_beyond_grid_y", "more views than gridDim.y allows",
     lambda s, c: s.V > MAX_GRID_Y, O_V),
    ("view_ids_end_at_2^32", "the last view id of the call is 2^32 - 1",
     lambda s, c: c.view_base + s.V == VIEW_IDS and s.K > 1, O_V),
]


def reached(sms=SMS):
    """{(class, o_v): [(case, o_v, o_n)]}: the cases whose shape on `sms` SMs falls into each class"""
    out = {(name, ov): [] for name, _, _, ovs in SHAPES for ov in ovs}
    for c in ALL_CASES:
        for o_v, o_n in c.modes:
            s = launch_shape(c.n, c.V, o_v, o_n, c.full, sms)
            for name, _, pred, ovs in SHAPES:
                if o_v in ovs and pred(s, c):
                    out[(name, o_v)].append((c.name, o_v, o_n))
    return out


def unreached(sms=SMS):
    return sorted(k for k, v in reached(sms).items() if not v)


# ------------------------------------------------------------------------------------------------ oracle side
def expected_removals(sizes, nr, keep_counts=None):
    """DESIGN.md §3.7: t_g = min(max(num_remove, 0), n_g - 1) for a graph without a protected vertex (never below 0),
    and min(max(num_remove, 0), m_g) for one with a protected vertex (m_g unprotected vertices)"""
    out = []
    for g, (s, t) in enumerate(zip(sizes, nr)):
        m = s if keep_counts is None else keep_counts[g]
        cap = m if m < s else s - 1
        out.append(max(0, min(max(t, 0), cap)))
    return out


def coalesced(ptr, col, w):
    """the coalesced input in output order (by column, then row): what a call that can remove nothing returns"""
    n = ptr.shape[0] - 1
    return col.astype(np.int32), np.repeat(np.arange(n, dtype=np.int32), np.diff(ptr)), w
