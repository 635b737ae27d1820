// schur.cu — ordering, elimination and emission kernels of the rLap randomized Schur complement.
//
// Replaces {Random,Priority,Coarsening}Preconditioner::getSchurComplement
// (rlap/csrc/preconditioner.cc:348-476, 713-825, 835-957) with a round-parallel design:
//   * the graph is an immutable coalesced CSR shared by all views; every view keeps only
//     per-vertex state, a head pointer per vertex and an append-only pool of fill entries
//     (lazy deletion: an entry dies when the vertex it points to is eliminated);
//   * one persistent cooperative kernel runs ALL rounds of the views of a view group (grid.sync between phases);
//     the groups of a call run as concurrent launches (api.cu);
//   * inside a round, vertices that are pairwise non-adjacent are eliminated concurrently, one warp
//     (or one thread block for big stars) per vertex: gather -> fixed-point quantise -> bitonic sort
//     by neighbour -> merge multi-edges -> o_n sort -> warp-shuffle prefix sums -> Philox-driven
//     binary-search sampling -> atomic append of the fill edges to both endpoints.
// The sequential specification this file implements bit for bit is oracle/rlap_oracle.cc (keyed mode)
// and DESIGN.md §3.
#include <stdio.h>
#include <mutex>
#include "rlap_device.cuh"
#include "schur.cuh"
#include "scan.cuh"
#include "star.cuh"

namespace rlap {

__device__ __forceinline__ int graph_of(const SchurParams& P, int v) { return P.gid ? __ldg(P.gid + v) : 0; }

// The kernel is compiled once per (vertex order, neighbour order, full-clique) combination: the members below hide
// the run-time fields of the same name, so every `P.o_v == 0` in the device code is decided at compile time and an
// instantiation carries only its own branch of the star arithmetic (half the register spills of the generic kernel,
// ptxas -v). Same layout as SchurParams: the host passes a plain SchurParams.
template <int OV, int ON, bool FULL>
struct ModeParams : SchurParams {
    static constexpr int o_v = OV;
    static constexpr int o_n = ON;
    static constexpr bool full = FULL;
};

// key of the degree bucket queue (preconditioner.cc:125-246 restated, DESIGN.md §3.4): number of live
// list entries, never below 1 once the vertex had an edge (DegreePQDec is a no-op at key 1), 0 for
// vertices that were isolated from the start; computed inline where it is needed as
// (state == 4) ? 0 : max(live, 1).
// state byte: 0 kept (o_v = random, not eligible; any order: protected by the keep mask), 1 pending, 2 eliminated,
// 4 pending and isolated from the start
// degree / coarsen: a vertex the minimum key, the bucket and the independent-set test see (pending, 1 or 4; not
// eliminated and not protected). Vertices that are not open may still be appended to a low list (the live-counter
// crossings of the elimination phase do not read the state byte); the readers of the list drop them.
__device__ __forceinline__ bool open_st(uint8_t st) { return (st & 5u) != 0; }

// ---------------------------------------------------------------------------------------------
// star staging
// ---------------------------------------------------------------------------------------------

// Gather the raw live entries of v into sb.A (unordered). Returns their count (group uniform);
// *wmaxb receives the bit pattern of the largest weight. Entries beyond sb.cap are counted, not stored.
// A fill list that a single lane has already walked (run_warp_items: the lists of all shared-memory stars of a chunk
// are walked side by side, one per lane): `n` raw entries in global memory, and the list position the walk stopped at.
struct StagedList {
    const uint64_t* e = nullptr;
    int n = 0;
    int rest = -1;        // continue the walk here (-1: the list was walked to its end)
    bool valid = false;   // false: nothing staged, start at the list head
};

template <bool CTA, class PT>
__device__ int star_gather(const PT& P, int view, int v, StarBuf sb, CtaScratch* cs, uint32_t* wmaxb_out,
                           const StagedList stl = StagedList()) {
    const size_t vb = (size_t)view * (size_t)P.n;
    const uint8_t* st = P.state + vb;
    const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const int b = __ldg(P.ptr + v), e = __ldg(P.ptr + v + 1);
    uint32_t wmaxb = 0;
    int cnt = 0;
    if (CTA) {
        if (threadIdx.x == 0) cs->icount = 0;
        __syncthreads();
    }
    // base CSR segment: coalesced
    const int stride = g_size<CTA>();
    for (int p0 = b; p0 < e; p0 += stride) {
        int p = p0 + g_rank<CTA>();
        bool ok = p < e;
        int u = 0;
        float w = 0.f;
        if (ok) {
            u = __ldg(P.col + p);
            ok = !is_dead(P, view, (unsigned)u);
        }
        if (ok) w = __ldg(P.w + p);
        unsigned m = __ballot_sync(RLAP_FULL_MASK, ok);
        int base;
        if (CTA) {
            base = 0;
            if (lane == 0 && m) base = atomicAdd(&cs->icount, __popc(m));
            base = __shfl_sync(RLAP_FULL_MASK, base, 0);
        } else {
            base = cnt;
            cnt += __popc(m);
        }
        if (ok) {
            int pos = base + __popc(m & lt);
            if (pos < sb.cap) sb.A[pos] = pack_a((uint32_t)u, w);
            wmaxb = max(wmaxb, __float_as_uint(w));
        }
    }
    // appended fill entries: a linked list, walked by one warp; 32 hops are collected before the
    // (dependent) state lookups so that those run in parallel
    int hub = -1;
    if (P.o_v == 0) hub = __ldg(P.hubidx + v);
    if (hub >= 0) {
        // a hub's fills: HUB_HEADS lists, one per lane of a warp
        if (!CTA || (threadIdx.x >> 5) == 0) {
            const int* heads = P.hubheads + ((size_t)view * (size_t)P.nhmax + (size_t)hub) * HUB_HEADS;
            int p = ldcg_i32(heads + lane);
            while (__any_sync(RLAP_FULL_MASK, p >= 0)) {
                const bool have = p >= 0;
                int4 en = make_int4(0, 0, -1, 0);
                if (have) { en = __ldcg(pool + p); p = en.z; }
                const bool ok = have && !is_dead(P, view, (unsigned)en.x);
                const unsigned m = __ballot_sync(RLAP_FULL_MASK, ok);
                int base;
                if (CTA) {
                    base = 0;
                    if (lane == 0 && m) base = atomicAdd(&cs->icount, __popc(m));
                    base = __shfl_sync(RLAP_FULL_MASK, base, 0);
                } else {
                    base = cnt;
                    cnt += __popc(m);
                }
                if (ok) {
                    const int pos = base + __popc(m & lt);
                    if (pos < sb.cap) sb.A[pos] = pack_a((uint32_t)en.x, __int_as_float(en.y));
                    wmaxb = max(wmaxb, (uint32_t)en.y);
                }
            }
        }
    } else if (!CTA || (threadIdx.x >> 5) == 0) {
        int p;
        if (!CTA && stl.valid) {
            // the staged part: 32 entries per step, coalesced
            for (int t0 = 0; t0 < stl.n; t0 += 32) {
                const int t = t0 + lane;
                const bool have = t < stl.n;
                const uint64_t a = have ? __ldcg(stl.e + t) : 0ull;
                const bool ok = have && !is_dead(P, view, a_nbr(a));
                const unsigned m = __ballot_sync(RLAP_FULL_MASK, ok);
                if (ok) {
                    const int pos = cnt + __popc(m & lt);
                    if (pos < sb.cap) sb.A[pos] = a;
                    wmaxb = max(wmaxb, (uint32_t)a);
                }
                cnt += __popc(m);
            }
            p = stl.rest;
        } else {
            p = ldcg_i32(head_p(P, vb + v));
        }
        while (p >= 0) {
            int4 mine = make_int4(0, 0, 0, 0);
            bool have = false;
            for (int k = 0; k < 32 && p >= 0; k++) {
                int4 en = __ldcg(pool + p);
                if (lane == k) { mine = en; have = true; }
                p = en.z;
            }
            bool ok = have && !is_dead(P, view, (unsigned)mine.x);
            unsigned m = __ballot_sync(RLAP_FULL_MASK, ok);
            int base;
            if (CTA) {
                base = 0;
                if (lane == 0 && m) base = atomicAdd(&cs->icount, __popc(m));
                base = __shfl_sync(RLAP_FULL_MASK, base, 0);
            } else {
                base = cnt;
                cnt += __popc(m);
            }
            if (ok) {
                int pos = base + __popc(m & lt);
                if (pos < sb.cap) sb.A[pos] = pack_a((uint32_t)mine.x, __int_as_float(mine.y));
                wmaxb = max(wmaxb, (uint32_t)mine.y);
            }
        }
    }
    if (CTA) {
        __syncthreads();
        cnt = cs->icount;
    }
    *wmaxb_out = g_max_u32<CTA>(wmaxb, cs);
    g_sync<CTA>();
    return cnt;
}

// degree / coarsen: appends to the next round's low list through a small per-warp shared buffer, so that the list
// tail is bumped once per few dozen entries. Every member is warp-collective.
constexpr int LOWBUF = 64;
struct LowAppender {
    unsigned int* buf = nullptr;   // [LOWBUF] shared memory, one per warp
    const SchurParams* P = nullptr;
    int par = -1;                  // parity of the list being written (-1: disabled, o_v = random)
    int fill = 0;
    __device__ __forceinline__ unsigned int* dst() const { return P->low + (size_t)par * (size_t)P->low_cap; }
    __device__ __forceinline__ int* tail() const { return P->ctr + CTR_LOW0 + par; }
    __device__ __forceinline__ int* ovf() const { return P->ctr + CTR_LOWOVF0 + par; }
    __device__ __forceinline__ void flush() {
        if (fill == 0) return;
        const int lane = threadIdx.x & 31;
        int pos0 = 0;
        if (lane == 0) pos0 = atomicAdd(tail(), fill);
        pos0 = __shfl_sync(RLAP_FULL_MASK, pos0, 0);
        __syncwarp();
        unsigned int* d = dst();
        for (int i = lane; i < fill; i += 32) {
            if ((long long)pos0 + i < P->low_cap) d[pos0 + i] = buf[i]; else *ovf() = 1;
        }
        __syncwarp();
        fill = 0;
    }
    __device__ __forceinline__ void push(bool pred, unsigned int val) {
        if (par < 0) return;
        const unsigned m = __ballot_sync(RLAP_FULL_MASK, pred);
        if (m == 0) return;
        if (fill + 32 > LOWBUF) flush();
        if (pred) buf[fill + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = val;
        fill += __popc(m);
    }
    // one entry from one lane, outside any warp-collective pattern (rare paths)
    __device__ __forceinline__ void push_single(unsigned int val) const {
        if (par < 0) return;
        const int pos = atomicAdd(tail(), 1);
        if ((long long)pos < P->low_cap) dst()[pos] = val; else *ovf() = 1;
    }
};

// Results that are still on their way back when a register tile finishes a star: the `next` fields of the two pool
// entries of its fill edge (from the list-head exchanges) and the old value of the live counter it decremented.
// Consuming them is deferred until the tile has issued the loads of its next star, so the warp does not wait for
// those round trips (degree / coarsen: a grid barrier separates the writers of a list from its readers; o_v =
// random flushes before its fence).
struct PendingPush {
    int4 e0, e1;
    int4* p0 = nullptr;
    int lo_old = 0, lo_lim = 0, lo_M = 0x7fffffff;   // crossing test: lo_M < lo_old <= lo_lim
    unsigned int lo_idx = 0;
    __device__ __forceinline__ void flush(LowAppender& la) {   // warp-collective
        if (p0) { p0[0] = e0; p0[1] = e1; p0 = nullptr; }
        la.push(lo_old > lo_M && lo_old <= lo_lim, lo_idx);
        lo_M = 0x7fffffff;
    }
};

// the list head a fill for vertex j in pool slot `slot` is linked into (o_v = random: hubs keep HUB_HEADS lists)
template <class PT>
__device__ __forceinline__ int* fill_head_p(const PT& P, int view, size_t vb, int j, int slot) {
    if (P.o_v == 0) {
        const int h = __ldg(P.hubidx + j);
        if (h >= 0) return P.hubheads + ((size_t)view * (size_t)P.nhmax + (size_t)h) * HUB_HEADS + ((slot >> 1) & (HUB_HEADS - 1));
    }
    return head_p(P, vb + j);
}

// fill edge (j,k,w): append to both endpoints; o_v = random also records the new dependency.
// LIVE: bump the live counters of both endpoints here (the register tiles apply net deltas instead).
// Returns false for an underflowed fill (weight 0: not created).
template <bool LIVE, class PT>
__device__ __forceinline__ bool push_fill(const PT& P, int view, size_t vb, int4* pool, int j, int k, float w,
                                          long long slot, PendingPush* pend = nullptr, int dep = -1) {
    if (!(w > 0.f)) {  // underflowed fill: leave two tombstones so that the pool can be read linearly
        pool[slot] = make_int4(-1, 0, -1, -1);
        pool[slot + 1] = make_int4(-1, 0, -1, -1);
        // the callers count a star's fills before they are sampled: take this one back (the stat counts fill edges,
        // as the lane path and the oracle do; the group's sum stays exact modulo 2^64)
        atomicAdd(P.stats + ST_FILLS, ~0ull);
        return false;
    }
    {   // both list heads are exchanged before either entry is written: the two round trips overlap
        const int s0 = (int)slot, s1 = (int)slot + 1;
        const int n0 = atomicExch(fill_head_p(P, view, vb, j, s0), s0);
        const int n1 = atomicExch(fill_head_p(P, view, vb, k, s0), s1);
        if (pend) {
            pend->e0 = make_int4(k, __float_as_int(w), n0, j);
            pend->e1 = make_int4(j, __float_as_int(w), n1, k);
            pend->p0 = pool + s0;
        } else {
            pool[s0] = make_int4(k, __float_as_int(w), n0, j);
            pool[s1] = make_int4(j, __float_as_int(w), n1, k);
        }
        if (LIVE) { atomicAdd(live_p(P, vb + j), 1); atomicAdd(live_p(P, vb + k), 1); }
    }
    if (P.o_v == 0) {
        // dep: what the caller already knows about the new dependency (-1 nothing, 0 none, 1 k waits for j, 2 j waits for k)
        if (dep < 0) {
            if (ldcg_u8(P.state + vb + j) == 1 && ldcg_u8(P.state + vb + k) == 1) {
                int rj = ldcg_i32(P.rank + vb + j), rk = ldcg_i32(P.rank + vb + k);
                if (rj < rk) atomicAdd(P.blk + vb + k, 1); else atomicAdd(P.blk + vb + j, 1);
            }
        } else if (dep == 1) {
            atomicAdd(P.blk + vb + k, 1);
        } else if (dep == 2) {
            atomicAdd(P.blk + vb + j, 1);
        }
    }
    return true;
}

// Eliminate vertex v of `view` (A.2 clique sampling / A.4 coarsening / full clique), DESIGN.md §3.3.
// one record per warp in shared memory, updated by one lane at a time (kept out of the registers of the persistent kernel)
struct LocalStats { unsigned long long fills, raw; int maxstar; unsigned nsm; };

template <bool CTA, class PT>
__device__ void eliminate_star(const PT& P, const RoundCtx& rc, int view, int v, StarBuf sb, CtaScratch* cs,
                               LocalStats* ls, LowAppender& la, const StagedList stl = StagedList(),
                               uint64_t* work = nullptr, int work_bytes = 0) {
    const size_t vb = (size_t)view * (size_t)P.n;
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    const uint32_t view_id = P.view_base + (uint32_t)view;
    int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
    uint32_t wmaxb;
    int lraw = star_gather<CTA>(P, view, v, sb, cs, &wmaxb, stl);
    if (lraw > sb.cap) {  // cannot happen for the smem tiers (callers check live); scratch tier: report
        if (r == 0) set_status(P, 6);
        lraw = 0;  // leave the vertex in place; the run is invalid anyway
        g_sync<CTA>();
        return;
    }
    int P2 = 0, L = 0;
    if (lraw > 0) {
        const int shift = star_shift(__uint_as_float(wmaxb), lraw);
        L = star_sort_merge<CTA>(sb, lraw, shift, cs, &P2);
        const bool full = P.full;
        const bool coarsen = (P.o_v == 2) && !full;
        const int on = coarsen ? 2 : P.o_n;
        if (!full && on != 2 && L > 16) {     // asc / desc: equal weights among more than 16 neighbours stand the way
            if (on == 1) star_tie_order<CTA, true>(sb, lraw, L, P2, work, work_bytes);    // std::sort leaves them
            else star_tie_order<CTA, false>(sb, lraw, L, P2, work, work_bytes);
        }
        if (!full && on == 2) {               // shuffle key
            for (int i = r; i < lraw; i += gs) {
                uint64_t a = sb.A[i];
                if (!a_dead(a)) {
                    uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(a), view_id, TAG_STAR);
                    sb.K[i] = ((uint64_t)x.z << 32) | (uint64_t)x.w;
                }
            }
            g_sync<CTA>();
        }
        if (full || on == 0) g_bitonic_sort<CTA, SORT_ASC>(sb, P2);
        else if (on == 1) g_bitonic_sort<CTA, SORT_DESC>(sb, P2);
        else g_bitonic_sort<CTA, SORT_KEY>(sb, P2);
        g_incl_scan_u64<CTA>(sb.Q, sb.K, L, cs);
        const unsigned long long S = sb.K[L - 1];
        // ---- fill edges
        long long nf = full ? (long long)L * (L - 1) / 2 : (long long)(L - 1);
        long long slot0 = 0;
        bool ovf = false;
        if (nf > 0) {
            if (CTA) {
                if (threadIdx.x == 0) cs->carry = atomicAdd(P.pool_cursor + view, (unsigned long long)(2 * nf));
                __syncthreads();
                slot0 = (long long)cs->carry;
            } else {
                unsigned long long s0 = 0;
                if (r == 0) s0 = atomicAdd(P.pool_cursor + view, (unsigned long long)(2 * nf));
                slot0 = (long long)__shfl_sync(RLAP_FULL_MASK, s0, 0);
            }
            ovf = slot0 + 2 * nf > P.pool_cap;
            if (ovf && r == 0) set_status(P, 5);
        }
        if (nf > 0 && !ovf) {
            if (full) {
                const double Sf = __dmul_rn(__ull2double_rn(S), pow2d(-shift));
                for (int a = 0; a < L - 1; a++) {
                    const uint64_t ea = sb.A[a];
                    const long long off = (long long)a * (2LL * L - a - 1) / 2;
                    for (int b2 = a + 1 + r; b2 < L; b2 += gs) {
                        const uint64_t eb = sb.A[b2];
                        float w = __double2float_rn(__ddiv_rn(__dmul_rn((double)a_w(ea), (double)a_w(eb)), Sf));
                        push_fill<true>(P, view, vb, pool, (int)a_nbr(ea), (int)a_nbr(eb), w, slot0 + 2 * (off + (b2 - a - 1)));
                    }
                }
            } else if (coarsen) {
                uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, 0xffffffffu, view_id, TAG_PICK);
                unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
                unsigned long long rr = __umul64hi(u, S);
                int koff = upper_bound_u64(sb.K, L, rr);
                if (koff >= L) koff = L - 1;
                const uint64_t ek = sb.A[koff];
                const double wk = (double)a_w(ek);
                for (int m = r; m < L; m += gs) {
                    if (m == koff) continue;
                    const uint64_t em = sb.A[m];
                    const double wm = (double)a_w(em);
                    float w = __double2float_rn(__ddiv_rn(__dmul_rn(wk, wm), __dadd_rn(wk, wm)));
                    int sl = m < koff ? m : m - 1;
                    push_fill<true>(P, view, vb, pool, (int)a_nbr(em), (int)a_nbr(ek), w, slot0 + 2LL * sl);
                }
            } else {
                for (int m = r; m < L - 1; m += gs) {
                    const uint64_t em = sb.A[m];
                    const unsigned long long Cm = sb.K[m];
                    const unsigned long long rem = S - Cm;
                    uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(em), view_id, TAG_STAR);
                    unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
                    unsigned long long rr = Cm + __umul64hi(u, rem);
                    int koff = upper_bound_u64(sb.K, L, rr);
                    if (koff >= L) koff = L - 1;
                    float w = __double2float_rn(
                        __ddiv_rn(__dmul_rn((double)a_w(em), __ull2double_rn(rem)), __ull2double_rn(S)));
                    push_fill<true>(P, view, vb, pool, (int)a_nbr(em), (int)a_nbr(sb.A[koff]), w, slot0 + 2LL * m);
                }
            }
        }
        // every push (and, for o_v = random, every dependency increment) is ordered before the
        // decrements below: a neighbour's counter can only reach zero once all its lower-ranked
        // eventual neighbours are gone (DESIGN.md §3.5)
        if (P.o_v == 0) __threadfence();
        g_sync<CTA>();
        // a neighbour whose live counter moves from above the segment's level to the level or below joins the
        // next round's low list (degree / coarsen)
        const int M = (P.o_v != 0) ? ldcg_i32(P.lvl + (size_t)view * P.G + graph_of(P, v)) : -1;
        for (int base = 0; base < P2; base += gs) {
            const int i = base + r;
            bool cross = false;
            int u = 0;
            if (i < P2) {
                const uint64_t a = sb.A[i];
                if (a != RLAP_PAD_A) {
                    u = (int)a_nbr(a);
                    const int old = atomicSub(live_p(P, vb + u), 1);
                    cross = old > M && old - 1 <= M;
                    if (P.o_v == 0 && ldcg_u8(P.state + vb + u) == 1) {
                        int oldb = atomicSub(P.blk + vb + u, 1);
                        if (oldb == 1) {
                            int pos = rc.wl_base + atomicAdd(P.ctr + rc.wslot, 1);
                            P.wl[pos] = (unsigned int)(vb + (size_t)u);
                        }
                    }
                }
            }
            la.push(cross, (unsigned int)(vb + (size_t)u));
        }
        if (r == 0) {
            ls->fills += (unsigned long long)(ovf ? 0 : nf);
            ls->maxstar = max(ls->maxstar, L);
            ls->raw += (unsigned long long)lraw;
        }
    }
    if (r == 0) { P.state[vb + v] = 2; *live_p(P, vb + v) = RLAP_LIVE_DEAD; mark_dead(P, view, (unsigned)v); }
    g_sync<CTA>();
}

// Register-resident elimination: the warp holds one star, one entry per lane. `idx` is the warp's work item, warp
// uniform and always a real star. The caller has already read the star's CSR bounds (b, nb) and walked its fill list
// into shared memory (`fills`, nfill entries), and guarantees nb + nfill <= 32: the raw list always fits, nothing is
// retried.
// `slot0` / `nslots`: pool slots reserved for this star by the caller (an upper bound, 2 per possible fill).
template <class PT>
__device__ void eliminate_star_regs(const PT& P, const RoundCtx& rc, unsigned int idx, int b, int nb,
                                    const uint64_t* fills, int nfill, long long slot0, int nslots, int M,
                                    LocalStats* ls, PendingPush& pend, LowAppender& la) {
    const int tl = threadIdx.x & 31;
    const int view = (int)(idx / (unsigned)P.n), v = (int)(idx % (unsigned)P.n);
    const size_t vb = (size_t)view * (size_t)P.n;
    const uint32_t view_id = P.view_base + (uint32_t)view;
    int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
    uint64_t a = RLAP_PAD_A;
    if (tl < nb) a = pack_a((uint32_t)__ldg(P.col + b + tl), __ldg(P.w + b + tl));
    else if (tl - nb < nfill) a = fills[tl - nb];
    bool dead = false;
    // dead test on the neighbour's (live, head) record: the sector is the one its live counter and list head are
    // updated in further down
    if (a != RLAP_PAD_A) dead = is_dead(P, view, a_nbr(a));
    // the previous star's pool entries: their `next` fields have arrived by now
    pend.flush(la);
    if (dead) a = RLAP_PAD_A;
    __syncwarp();
    a = warp_sort_u64(a);
    const bool rawvalid = a != RLAP_PAD_A;         // raw live entry (multi-edge duplicates included)
    const int rawnbr = (int)a_nbr(a);
    const int lraw = __popc(__ballot_sync(RLAP_FULL_MASK, rawvalid));
    unsigned long long q;
    int shift;
    int mult;
    const unsigned hmask = warp_merge_sorted(a, q, shift, mult);
    const int L = __popc(hmask);
    // live counters: a neighbour loses its entries to v (all `mult` of them) and gains one entry per fill it
    // receives. The extra multiplicity goes now, the rest is netted per merged neighbour after sampling.
    bool cross0 = false;
    if (((hmask >> tl) & 1u) && mult > 1) {
        const int old = atomicSub(live_p(P, vb + rawnbr), mult - 1);
        cross0 = old > M && old - (mult - 1) <= M;
    }
    const bool live = (hmask >> tl) & 1u;
    const bool full = P.full;
    const bool coarsen = (P.o_v == 2) && !full;
    const int on = coarsen ? 2 : P.o_n;
    uint64_t key = ~0ull, tie = 0;
    // asc / desc ties among more than 16 merged neighbours: position in the arrangement std::sort's partition loop
    // leaves (star.cuh). The warp's FCAP staged fills (128 bytes, read into `a` above) serve as its workspace.
    uint64_t tiepos = 0;
    if (!full && on != 2 && L > 16)
        tiepos = (on == 1) ? warp_tie_order<true>(q, hmask, (uint8_t*)const_cast<uint64_t*>(fills))
                           : warp_tie_order<false>(q, hmask, (uint8_t*)const_cast<uint64_t*>(fills));
    if (live) {
        uint64_t shuf = tiepos;
        if (!full && on == 2) {
            uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(a), view_id, TAG_STAR);
            shuf = ((uint64_t)x.z << 32) | (uint64_t)x.w;
        }
        if (full || on == 0) { key = q; tie = shuf; }
        else if (on == 1) { key = ~q; tie = shuf; }
        else key = shuf;
    } else {
        a = RLAP_PAD_A;
        q = 0;
        tie = ~0ull;   // padding sorts after every live entry, also after one whose key is ~0 (q = 0 under desc)
    }
    warp_sort_ktaq(key, tie, a, q);
    // o_v = random: the entry's neighbour still to be eliminated? and its rank, read here for all lanes at once instead
    // of by every push (a neighbour of the vertex being eliminated cannot change state inside this round)
    bool pend_mine = false;
    int rank_mine = 0;
    if (P.o_v == 0 && a != RLAP_PAD_A) {
        pend_mine = ldcg_u8(P.state + vb + a_nbr(a)) == 1;
        rank_mine = ldcg_i32(P.rank + vb + a_nbr(a));
    }
    const unsigned long long C = warp_incl_scan_u64(q);
    const unsigned long long S = __shfl_sync(RLAP_FULL_MASK, C, (L > 0 ? L - 1 : 0));
    const long long nf = (L < 1) ? 0 : (full ? (long long)L * (L - 1) / 2 : (long long)(L - 1));
    const bool ovf = nslots > 0 && slot0 + nslots > P.pool_cap;
    if (ovf && tl == 0) set_status(P, 5);
    const bool emit = nf > 0 && !ovf;
    // reserved but unused slots (multi-edges merged): tombstones, the pool is read linearly at emission
    if (!ovf)
        for (long long u = 2 * nf + tl; u < nslots; u += 32) pool[slot0 + u] = make_int4(-1, 0, -1, -1);
    int delta = -1;   // net change of live[neighbour] for the merged neighbour held by this lane
    if (full) {
        const double Sf = __dmul_rn(__ull2double_rn(S), pow2d(-shift));
        for (int b2 = 1; b2 < 32; b2++) {
            const uint64_t eb = __shfl_sync(RLAP_FULL_MASK, a, b2);
            bool done = false;
            if (emit && b2 < L && tl < b2) {
                float w = __double2float_rn(__ddiv_rn(__dmul_rn((double)a_w(a), (double)a_w(eb)), Sf));
                long long off = (long long)tl * (2LL * L - tl - 1) / 2;
                done = push_fill<false>(P, view, vb, pool, (int)a_nbr(a), (int)a_nbr(eb), w, slot0 + 2 * (off + (b2 - tl - 1)));
            }
            unsigned dm = __ballot_sync(RLAP_FULL_MASK, done);
            if (done) delta++;
            if (tl == b2) delta += __popc(dm);
        }
    } else if (coarsen) {
        uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, 0xffffffffu, view_id, TAG_PICK);
        unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
        int koff = warp_upper_bound(C, L, __umul64hi(u, S));
        if (koff >= L) koff = L - 1;
        if (koff < 0) koff = 0;
        const uint64_t ek = __shfl_sync(RLAP_FULL_MASK, a, koff);
        int dep = -1;
        if (P.o_v == 0) {
            const bool pk = __shfl_sync(RLAP_FULL_MASK, pend_mine, koff);
            const int rkk = __shfl_sync(RLAP_FULL_MASK, rank_mine, koff);
            dep = (pend_mine && pk) ? (rank_mine < rkk ? 1 : 2) : 0;
        }
        bool done = false;
        if (emit && tl < L && tl != koff) {
            const double wk = (double)a_w(ek), wm = (double)a_w(a);
            float w = __double2float_rn(__ddiv_rn(__dmul_rn(wk, wm), __dadd_rn(wk, wm)));
            int sl = tl < koff ? tl : tl - 1;
            done = push_fill<false>(P, view, vb, pool, (int)a_nbr(a), (int)a_nbr(ek), w, slot0 + 2LL * sl, &pend, dep);
        }
        unsigned dm = __ballot_sync(RLAP_FULL_MASK, done);
        if (done) delta++;
        if (tl == koff) delta += __popc(dm);
    } else {
        const bool act = tl < L - 1;
        unsigned long long rr = 0, rem = 0;
        if (act) {
            rem = S - C;
            uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(a), view_id, TAG_STAR);
            unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
            rr = C + __umul64hi(u, rem);
        }
        int koff = warp_upper_bound(C, L, rr);
        if (koff >= L) koff = L - 1;
        if (koff < 0) koff = 0;
        const uint64_t ek = __shfl_sync(RLAP_FULL_MASK, a, koff);
        int dep = -1;
        if (P.o_v == 0) {
            const bool pk = __shfl_sync(RLAP_FULL_MASK, pend_mine, koff);
            const int rkk = __shfl_sync(RLAP_FULL_MASK, rank_mine, koff);
            dep = (pend_mine && pk) ? (rank_mine < rkk ? 1 : 2) : 0;
        }
        if (emit && act) {
            float w = __double2float_rn(__ddiv_rn(__dmul_rn((double)a_w(a), __ull2double_rn(rem)), __ull2double_rn(S)));
            if (push_fill<false>(P, view, vb, pool, (int)a_nbr(a), (int)a_nbr(ek), w, slot0 + 2LL * tl, &pend, dep)) {
                delta++;
                atomicAdd(live_p(P, vb + (int)a_nbr(ek)), 1);
            }
        }
    }
    // o_v = random: pushes and dependency increments are ordered before the decrements (DESIGN.md §3.5);
    // the other orders separate rounds by grid barriers
    if (P.o_v == 0) { pend.flush(la); __threadfence(); }
    __syncwarp();
    // neighbours whose live counter crossed the segment's level downwards join the next round's low list; the test
    // on the value the atomic returns is left to the next flush of `pend`
    if (tl < L && delta != 0) {
        const int old = atomicAdd(live_p(P, vb + (int)a_nbr(a)), delta);
        if (delta < 0) { pend.lo_old = old; pend.lo_M = M; pend.lo_lim = M - delta; pend.lo_idx = (unsigned int)(vb + (size_t)a_nbr(a)); }
    }
    la.push(cross0, (unsigned int)(vb + (size_t)rawnbr));
    if (rawvalid) {
        if (P.o_v == 0 && ldcg_u8(P.state + vb + rawnbr) == 1) {
            int old = atomicSub(P.blk + vb + rawnbr, 1);
            if (old == 1) {
                int pos = rc.wl_base + atomicAdd(P.ctr + rc.wslot, 1);
                P.wl[pos] = (unsigned int)(vb + (size_t)rawnbr);
            }
        }
    }
    if (tl == 0) {
        ls->fills += (unsigned long long)(ovf ? 0 : nf);
        ls->maxstar = max(ls->maxstar, L);
        ls->raw += (unsigned long long)lraw;
        P.state[vb + v] = 2;
        *live_p(P, vb + v) = RLAP_LIVE_DEAD;
        mark_dead(P, view, (unsigned)v);
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// lane stars: one THREAD per star
// ---------------------------------------------------------------------------------------------
// A star with at most LCAP live entries and no multi-edge is gathered, ordered, sampled and pushed by a single lane
// out of its own shared-memory slot: a warp keeps 32 dependent chains of memory round trips in flight, and every lane
// runs a short insertion sort over an almost sorted list instead of a warp-wide sorting network (DESIGN.md §4, "Lane
// stars"). The arithmetic is the keyed specification's (DESIGN.md §3.3) to the bit: same fixed point, same tie rules
// (a star of at most 16 neighbours breaks asc / desc ties by neighbour id), same Philox counters, same IEEE double
// weight formula.
// Stars the lane cannot finish alone (a multi-edge, which needs the summed fixed-point weight of the run; two equal
// 32-bit shuffle keys, which need the full 64-bit key; more entries than announced) are handed to the cooperative
// path untouched: the lane returns false before it has modified anything.
constexpr int LCAP = 16;          // entries per lane slot
constexpr int LANE_NB_MAX = 48;   // longest base row a single lane scans
static_assert(HUB_DEG > LANE_NB_MAX && HUB_DEG > 32, "lane stars and register tiles read a single fill list: hubs must never reach them");

struct LaneSlot {                 // element e of this lane: A[e * 32], K[e * 32] (conflict free when the lanes of a
    uint64_t* A;                  // warp touch the same e)
    uint32_t* K;                  // 32-bit shuffle keys (o_n = random, coarsen), nullptr otherwise
    __device__ __forceinline__ uint64_t& a(int e) const { return A[e * 32]; }
    __device__ __forceinline__ uint32_t& k(int e) const { return K[e * 32]; }
};

// `cross` / `cross_idx`: the neighbour whose live counter this star moved to the segment's level or below (at most
// one per star: the last one in o_n order, or the contraction target); the caller appends it to the low list with
// one warp-collective push.
// first half: gather the live entries into the lane's slot (loads only: the pool reservation of the chunk is in flight
// meanwhile). Returns the entry count; *nbase_out = how many of them came from the (ascending) base row.
template <class PT>
__device__ int lane_star_gather(const PT& P, unsigned int idx, int b, int nb, LaneSlot sl, uint32_t* wmaxb_out,
                                int* nbase_out) {
    const int view = (int)(idx / (unsigned)P.n);
    const size_t vb = (size_t)view * (size_t)P.n;
    const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
    // base row four at a time (ids and weights, then the dead tests together), then the fill list with the next hop in
    // flight while the previous entry's neighbour is tested
    int p = ldcg_i32(head_p(P, idx));
    int cnt = 0;
    uint32_t wmaxb = 0;
    for (int p0 = 0; p0 < nb; p0 += 4) {
        int u4[4], l4[4];
        float w4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const bool in = p0 + k < nb;
            u4[k] = in ? __ldg(P.col + b + p0 + k) : -1;
            w4[k] = in ? __ldg(P.w + b + p0 + k) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) l4[k] = (u4[k] >= 0) ? (is_dead(P, view, (unsigned)u4[k]) ? -1 : 0) : -1;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (l4[k] >= 0) {
                if (cnt < LCAP) sl.a(cnt) = pack_a((uint32_t)u4[k], w4[k]);
                cnt++;
                wmaxb = max(wmaxb, __float_as_uint(w4[k]));
            }
        }
    }
    *nbase_out = cnt;
    {
        int4 pe = make_int4(-1, 0, -1, 0);
        while (true) {
            int4 en = make_int4(-1, 0, -1, 0);
            if (p >= 0) en = __ldcg(pool + p);
            if (pe.x >= 0 && !is_dead(P, view, (unsigned)pe.x)) {
                if (cnt < LCAP) sl.a(cnt) = pack_a((uint32_t)pe.x, __int_as_float(pe.y));
                cnt++;
                wmaxb = max(wmaxb, (uint32_t)pe.y);
            }
            if (p < 0) break;
            pe = en;
            p = en.z;
        }
    }
    *wmaxb_out = wmaxb;
    return cnt;
}

// second half: order, sample, push. `cross` / `cross_idx`: the neighbour whose live counter this star moved to the
// segment's level or below (at most one per star: the last one in o_n order, or the contraction target); the caller
// appends it to the low list with one warp-collective push.
template <class PT>
__device__ bool eliminate_star_lane(const PT& P, const RoundCtx& rc, unsigned int idx, int cnt, uint32_t wmaxb, int nbase,
                                    long long slot0, int nslots, int M, LaneSlot sl, int& made_out, int& len_out,
                                    const LowAppender& la, bool& cross, unsigned int& cross_idx) {
    const int view = (int)(idx / (unsigned)P.n), v = (int)(idx % (unsigned)P.n);
    const size_t vb = (size_t)view * (size_t)P.n;
    const uint32_t view_id = P.view_base + (uint32_t)view;
    int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
    if (cnt > LCAP || 2 * (cnt - 1) > nslots) return false;   // more live entries than the counter announced: not this path
    const int L = cnt;
    // ---- order by neighbour (the base entries are ascending already); a multi-edge sends the star to the cooperative path
    {
        bool dup = false;
        for (int i = (nbase > 1 ? nbase : 1); i < L; i++) {
            const uint64_t x = sl.a(i);
            int j = i - 1;
            while (j >= 0) {
                const uint64_t y = sl.a(j);
                if (a_nbr(y) <= a_nbr(x)) { dup |= a_nbr(y) == a_nbr(x); break; }
                sl.a(j + 1) = y;
                j--;
            }
            sl.a(j + 1) = x;
        }
        if (dup) return false;
    }
    const bool coarsen = P.o_v == 2;
    const int on = coarsen ? 2 : P.o_n;
    const int shift = L > 0 ? star_shift(__uint_as_float(wmaxb), L) : 0;
    // ---- o_n order: stable insertion sorts, so ties keep the neighbour-id order
    if (on == 2) {
        for (int e = 0; e < L; e++) {
            const uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(sl.a(e)), view_id, TAG_STAR);
            sl.k(e) = x.z;
        }
        bool tie = false;
        for (int i = 1; i < L; i++) {
            const uint64_t x = sl.a(i);
            const uint32_t kx = sl.k(i);
            int j = i - 1;
            while (j >= 0) {
                const uint32_t ky = sl.k(j);
                if (ky <= kx) { tie |= ky == kx; break; }
                sl.a(j + 1) = sl.a(j);
                sl.k(j + 1) = ky;
                j--;
            }
            sl.a(j + 1) = x;
            sl.k(j + 1) = kx;
        }
        if (tie) return false;   // the full key is (z, w) of the Philox block: let the cooperative path compare all 64 bits
    } else {
        for (int i = 1; i < L; i++) {
            const uint64_t x = sl.a(i);
            const unsigned long long qx = quantize(a_w(x), shift);
            int j = i - 1;
            while (j >= 0) {
                const uint64_t y = sl.a(j);
                if ((uint32_t)y == (uint32_t)x) break;   // equal weights: equal keys
                const unsigned long long qy = quantize(a_w(y), shift);
                if (on == 0 ? !(qx < qy) : !(qx > qy)) break;
                sl.a(j + 1) = y;
                j--;
            }
            sl.a(j + 1) = x;
        }
    }
    unsigned long long S = 0;
    for (int e = 0; e < L; e++) S += quantize(a_w(sl.a(e)), shift);
    const int nf = L > 0 ? L - 1 : 0;
    const bool ovf = nslots > 0 && slot0 + nslots > P.pool_cap;
    if (ovf) set_status(P, 5);
    cross = false;
    int made = 0;
    // one fill edge behind: the `next` fields of a fill's two pool entries (the values its list-head exchanges
    // return) are stored while the next fill is being sampled
    int4* pp = nullptr;
    int pj = 0, pk = 0, pn0 = 0, pn1 = 0, pw = 0;
    // o_v = random: which neighbours are still to be eliminated (state 1), read for all entries at once: a neighbour
    // of the vertex being eliminated cannot change state inside this round (DESIGN.md §3.5)
    unsigned pendm = 0;
    if (P.o_v == 0) {
#pragma unroll 4
        for (int e = 0; e < L; e++) pendm |= (ldcg_u8(P.state + vb + a_nbr(sl.a(e))) == 1 ? 1u : 0u) << e;
    }
    auto emit_fill = [&](int j, int k, float w, long long slot, int ej_pos, int ek_pos) -> bool {
        if (!(w > 0.f)) {   // underflowed fill: two tombstones, the pool is read linearly at emission
            pool[slot] = make_int4(-1, 0, -1, -1);
            pool[slot + 1] = make_int4(-1, 0, -1, -1);
            return false;
        }
        const int s0 = (int)slot, s1 = (int)slot + 1;
        const int n0 = atomicExch(fill_head_p(P, view, vb, j, s0), s0);
        const int n1 = atomicExch(fill_head_p(P, view, vb, k, s0), s1);
        if (P.o_v == 0 && ((pendm >> ej_pos) & (pendm >> ek_pos) & 1u)) {
            const int rj = ldcg_i32(P.rank + vb + j), rk = ldcg_i32(P.rank + vb + k);
            if (rj < rk) atomicAdd(P.blk + vb + k, 1); else atomicAdd(P.blk + vb + j, 1);
        }
        if (pp) { pp[0] = make_int4(pk, pw, pn0, pj); pp[1] = make_int4(pj, pw, pn1, pk); }
        pp = pool + s0; pj = j; pk = k; pn0 = n0; pn1 = n1; pw = __float_as_int(w);
        return true;
    };
    // a neighbour that lost its entry to v and got no fill in return
    auto lose_one = [&](int u) {
        const int old = atomicSub(live_p(P, vb + u), 1);
        if (old > M && old - 1 <= M) la.push_single((unsigned int)(vb + (size_t)u));
    };
    if (L > 0 && !ovf) {
        if (coarsen) {
            const uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, 0xffffffffu, view_id, TAG_PICK);
            const unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
            const unsigned long long rr = __umul64hi(u, S);
            int koff = L - 1;
            unsigned long long c = 0;
            for (int k = 0; k < L - 1; k++) {
                c += quantize(a_w(sl.a(k)), shift);
                if (c > rr) { koff = k; break; }
            }
            const uint64_t ek = sl.a(koff);
            const double wk = (double)a_w(ek);
            for (int m = 0; m < L; m++) {
                if (m == koff) continue;
                const uint64_t em = sl.a(m);
                const double wm = (double)a_w(em);
                const float w = __double2float_rn(__ddiv_rn(__dmul_rn(wk, wm), __dadd_rn(wk, wm)));
                if (emit_fill((int)a_nbr(em), (int)a_nbr(ek), w, slot0 + 2LL * (m < koff ? m : m - 1), m, koff)) made++;
                else lose_one((int)a_nbr(em));
            }
            // the contraction target loses its entry to v and gains one per fill
            if (made != 1) {
                const int old = atomicAdd(live_p(P, vb + (int)a_nbr(ek)), made - 1);
                if (made == 0) { cross = old > M && old - 1 <= M; cross_idx = (unsigned int)(vb + (size_t)a_nbr(ek)); }
            }
        } else {
            unsigned long long C = 0;
            const double Sd = __ull2double_rn(S);
            for (int j = 0; j < L - 1; j++) {
                const uint64_t ej = sl.a(j);
                C += quantize(a_w(ej), shift);
                const unsigned long long rem = S - C;
                const uint4 x = philox4x32_10(P.k0, P.k1, (uint32_t)v, a_nbr(ej), view_id, TAG_STAR);
                const unsigned long long u = ((unsigned long long)x.x << 32) | (unsigned long long)x.y;
                const unsigned long long rr = C + __umul64hi(u, rem);
                int koff = L - 1;
                unsigned long long c = C;
                for (int k = j + 1; k < L - 1; k++) {
                    c += quantize(a_w(sl.a(k)), shift);
                    if (c > rr) { koff = k; break; }
                }
                const int kn = (int)a_nbr(sl.a(koff));
                const float w = __double2float_rn(__ddiv_rn(__dmul_rn((double)a_w(ej), __ull2double_rn(rem)), Sd));
                if (emit_fill((int)a_nbr(ej), kn, w, slot0 + 2LL * j, j, koff)) { made++; atomicAdd(live_p(P, vb + kn), 1); }
                else lose_one((int)a_nbr(ej));
            }
            // the last neighbour only loses its entry
            const int ul = (int)a_nbr(sl.a(L - 1));
            const int old = atomicSub(live_p(P, vb + ul), 1);
            cross = old > M && old - 1 <= M;
            cross_idx = (unsigned int)(vb + (size_t)ul);
        }
        if (pp) { pp[0] = make_int4(pk, pw, pn0, pj); pp[1] = make_int4(pj, pw, pn1, pk); }
        // reserved but unused slots (cannot happen while the live counters are exact): tombstones
        for (int u = 2 * nf; u < nslots; u++) pool[slot0 + u] = make_int4(-1, 0, -1, -1);
    } else if (L > 0) {
        for (int e = 0; e < L; e++) atomicSub(live_p(P, vb + (int)a_nbr(sl.a(e))), 1);   // pool overflow: the run is invalid, keep it going
    }
    if (P.o_v == 0) {
        // pushes and dependency increments are ordered before the decrements (DESIGN.md §3.5)
        __threadfence();
        for (int e = 0; e < L; e++) {
            const int u = (int)a_nbr(sl.a(e));
            if ((pendm >> e) & 1u) {
                const int old = atomicSub(P.blk + vb + u, 1);
                if (old == 1) {
                    const int pos = rc.wl_base + atomicAdd(P.ctr + rc.wslot, 1);
                    P.wl[pos] = (unsigned int)(vb + (size_t)u);
                }
            }
        }
    }
    made_out = made;
    len_out = L;
    P.state[vb + v] = 2;
    *live_p(P, vb + v) = RLAP_LIVE_DEAD;
    mark_dead(P, view, (unsigned)v);
    return true;
}

// ---------------------------------------------------------------------------------------------
// the persistent elimination kernel
// ---------------------------------------------------------------------------------------------

constexpr int FCAP = 16;  // fill entries per item that the chunk prologue stages in shared memory (32 x FCAP words = the lane slots)
static_assert(FCAP * sizeof(uint64_t) >= 96, "warp_tie_order keeps 3 x 32 bytes in a tile's staged-fill slot");

// shared memory of the elimination phase, per warp: the lane slots (LCAP x 32 entries, plus 32-bit shuffle keys when
// the neighbour order is random), overlaid by the staging area of the register tiles and the star buffer of the
// shared-memory path, which run after the lane stars of a chunk
constexpr int LANE_A_WORDS = LCAP * 32;                       // uint64 per warp
__host__ __device__ __forceinline__ int warp_region_words(bool need_keys) {
    return LANE_A_WORDS + (need_keys ? LCAP * 32 / 2 : 0);    // uint64 words: 4 KB (+ 2 KB)
}
template <class PT>
__device__ __forceinline__ bool lane_keys_needed(const PT& P) { return !P.full && (P.o_v == 2 || P.o_n == 2); }
template <class PT>
__device__ __forceinline__ StarBuf warp_region_buf(const PT& P, uint64_t* smem) {
    uint64_t* base = smem + (size_t)(threadIdx.x >> 5) * warp_region_words(lane_keys_needed(P));
    StarBuf sb;
    sb.A = base;
    sb.Q = base + CAP_WARP;
    sb.K = base + 2 * CAP_WARP;
    sb.cap = CAP_WARP;
    return sb;
}

// process work-list items [start, end): a warp takes a chunk of up to 32 items, one per lane. Stars of at most LCAP
// live entries are eliminated by their lane alone (eliminate_star_lane); up to 32 raw entries by the warp as a
// register tile; up to CAP_WARP by the warp in shared memory; big stars go to the block phase.
template <class PT>
__device__ void run_warp_items(const PT& P, const RoundCtx& rc, uint64_t* smem, CtaScratch* cs, int start, int end,
                               LocalStats* ls, LowAppender& la) {
    const int nw = (int)((P.gblocks * blockDim.x) >> 5);
    const int lane = threadIdx.x & 31;
    StarBuf sb = warp_region_buf(P, smem);
    uint64_t* fbuf = sb.A;   // 32 x FCAP staged fill entries of the register tiles; the shared-memory path reuses the area
    LaneSlot slot;
    slot.A = sb.A + lane;
    slot.K = lane_keys_needed(P) ? (uint32_t*)(sb.A + LANE_A_WORDS) + lane : nullptr;
    const int count = end - start;
    if (count <= 0) return;
    // All warps of the launch (a view group) fetch chunks of the round's work list from one global cursor, with a
    // guided size: 1 / (2 x warps) of what is left, at least 8 and at most 32 items. A stale read of the cursor only
    // changes a chunk size.
    const bool full = P.full;
    enum { K_NONE = 0, K_LANE = 1, K_TILE = 2, K_SMEM = 3 };
    // pool slots are reserved once per chunk and tier: 2 per possible fill (L <= live), one atomic per view present in
    // the chunk instead of one per star. Issue and use are split: the atomic's round trip overlaps the gathers.
    struct Resv { unsigned long long b0; int first, incl; bool same; };
    auto reserve_issue = [&](int nslots, int view) -> Resv {
        Resv r;
        r.b0 = 0ull; r.first = 0; r.same = true;
        int incl = nslots;  // inclusive prefix over the lanes of the chunk
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(RLAP_FULL_MASK, incl, d);
            if (lane >= d) incl += t;
        }
        r.incl = incl;
        const unsigned need = __ballot_sync(RLAP_FULL_MASK, nslots > 0);
        if (need) {
            const int first = __ffs(need) - 1, last = 31 - __clz(need);
            const int v0 = __shfl_sync(RLAP_FULL_MASK, view, first);
            r.first = first;
            r.same = __all_sync(RLAP_FULL_MASK, nslots == 0 || view == v0);
            if (r.same) {
                const int total = __shfl_sync(RLAP_FULL_MASK, incl, last);
                if (lane == first) r.b0 = atomicAdd(P.pool_cursor + v0, (unsigned long long)total);
            } else if (nslots > 0) {
                r.b0 = atomicAdd(P.pool_cursor + view, (unsigned long long)nslots);
            }
        }
        return r;
    };
    auto reserve_finish = [&](const Resv& r, int nslots) -> long long {
        if (!r.same) return (long long)r.b0;
        const unsigned long long b0 = __shfl_sync(RLAP_FULL_MASK, r.b0, r.first);
        return (long long)b0 + r.incl - nslots;
    };
    // The claim of a chunk is one returning atomic on the group's cursor; it is issued one chunk ahead (the next chunk
    // is claimed before the current one is processed), so its round trip never sits on the warp's critical path. A
    // claim past the end of the list is harmless: the cursor is only read inside the round.
    // o_v = random: late rounds hold few, large stars (the shared-memory path takes them one after the other), so a
    // short list is dealt out star by star instead of eight at a time
    auto chunk_size = [&](int left) {
        if (P.o_v == 0) {   // a chunk costs a fixed chain of round trips (dependency counters, work-list pushes): one chunk per warp
            const int c1 = (left + nw - 1) / nw;
            return c1 < 1 ? 1 : (c1 > 32 ? 32 : c1);
        }
        int c = left / (2 * nw);
        c = (c + 7) & ~7;
        return c < 8 ? 8 : (c > 32 ? 32 : c);
    };
    int c0_next = 0, c_next = 0;
    if (lane == 0) {
        c_next = chunk_size(count);
        c0_next = start + atomicAdd(P.ctr + rc.sslot, c_next);
    }
    while (true) {
        const int c0 = __shfl_sync(RLAP_FULL_MASK, c0_next, 0);
        const int chunk_now = __shfl_sync(RLAP_FULL_MASK, c_next, 0);
        if (c0 >= end) break;
        if (lane == 0) {
            c_next = chunk_size(end - (c0 + chunk_now));
            c0_next = start + atomicAdd(P.ctr + rc.sslot, c_next);
        }
        const int it = c0 + lane;
        unsigned int idx = 0xffffffffu;
        int lv = -1, kind = K_NONE, b = 0, nb = 0, nfill = 0, M = -1, view = -1;
        __syncwarp();   // the previous chunk is done with the shared-memory region
        if (lane < chunk_now && it < end) {
            idx = __ldcg(P.wl + it);
            view = (int)(idx / (unsigned)P.n);
            const int v = (int)(idx % (unsigned)P.n);
            bool skip = false;
            if (P.o_v != 0) {  // truncated final round of a graph: only the highest ids go
                size_t seg = (size_t)view * P.G + graph_of(P, v);
                skip = ldcg_i32(P.ovfseg + seg) && idx < __ldcg(P.thresh + seg);
                M = ldcg_i32(P.lvl + seg);
            }
            if (!skip) {
                lv = ldcg_i32(live_p(P, idx));
                b = __ldg(P.ptr + v);
                nb = __ldg(P.ptr + v + 1) - b;
                if (lv > CAP_WARP) kind = K_NONE;          // deferred to the block phase below
                else if (!full && lv <= LCAP && nb <= LANE_NB_MAX) kind = K_LANE;
                else if (lv <= 32 && nb <= 32) kind = K_TILE;   // if its fill list is short enough, see below
                else kind = K_SMEM;
            } else {
                idx = 0xffffffffu;
            }
        }
        __syncwarp();
        if (lv > CAP_WARP) {
            int pos = rc.dl_base + atomicAdd(P.ctr + rc.dslot, 1);
            P.dl[pos] = idx;
        }
        // ---- lane stars
        if (__any_sync(RLAP_FULL_MASK, kind == K_LANE)) {
            const int nslots = (kind == K_LANE && lv >= 2) ? 2 * (lv - 1) : 0;
            const Resv rv = reserve_issue(nslots, view);
            bool cross = false;
            unsigned int cross_idx = 0;
            int made = 0, len = 0, cnt = 0, nbase = 0;
            uint32_t wmaxb = 0;
            if (kind == K_LANE) cnt = lane_star_gather(P, idx, b, nb, slot, &wmaxb, &nbase);
            const long long slot0 = reserve_finish(rv, nslots);
            if (kind == K_LANE) {
                if (eliminate_star_lane(P, rc, idx, cnt, wmaxb, nbase, slot0, nslots, M, slot, made, len, la, cross, cross_idx)) {
                    kind = K_NONE;
                } else {
                    // handed to the cooperative path, which reserves its own slots: these stay tombstones
                    for (int u = 0; u < nslots; u++) {
                        if (slot0 + u < P.pool_cap) (P.pool + (size_t)view * (size_t)P.pool_cap)[slot0 + u] = make_int4(-1, 0, -1, -1);
                    }
                    kind = K_SMEM;
                }
            }
            __syncwarp();
            la.push(cross, cross_idx);
            made = __reduce_add_sync(RLAP_FULL_MASK, made);
            const int lsum = __reduce_add_sync(RLAP_FULL_MASK, len), lmax = __reduce_max_sync(RLAP_FULL_MASK, len);
            if (lane == 0) {
                ls->fills += (unsigned long long)made;
                ls->raw += (unsigned long long)lsum;
                ls->maxstar = max(ls->maxstar, lmax);
            }
        }
        // ---- register tiles (17 .. 32 raw entries): every lane first walks the fill list of its own item (32 chains
        // in flight) into the staging buffer; with the CSR bounds this gives the exact raw length
        if (__any_sync(RLAP_FULL_MASK, kind == K_TILE)) {
            if (kind == K_TILE) {
                const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
                int p = ldcg_i32(head_p(P, idx));
                while (p >= 0 && nfill < FCAP) {
                    const int4 en = __ldcg(pool + p);
                    fbuf[lane * FCAP + nfill] = pack_a((uint32_t)en.x, __int_as_float(en.y));
                    nfill++;
                    p = en.z;
                }
                if (p >= 0 || nb + nfill > 32) kind = K_SMEM;   // the shared-memory path gathers it itself
            }
            __syncwarp();
            int nslots = 0;
            if (kind == K_TILE && lv >= 2) nslots = full ? lv * (lv - 1) : 2 * (lv - 1);
            const Resv rv = reserve_issue(nslots, view);
            const long long slot0 = reserve_finish(rv, nslots);
            // The & 31 changes no value (mt != 0). It steers ptxas, CUDA 12.9: without it k_eliminate<0, 0 or 1, false>
            // spill 128 / 104 bytes instead of 88 / 80.
            unsigned mt = __ballot_sync(RLAP_FULL_MASK, kind == K_TILE);
            PendingPush pend;
            while (mt) {
                const int k = (__ffs(mt) - 1) & 31;
                mt &= mt - 1;
                const unsigned int kidx = __shfl_sync(RLAP_FULL_MASK, idx, k);
                const int kb = __shfl_sync(RLAP_FULL_MASK, b, k), knb = __shfl_sync(RLAP_FULL_MASK, nb, k);
                const int knfill = __shfl_sync(RLAP_FULL_MASK, nfill, k);
                const long long kslot0 = __shfl_sync(RLAP_FULL_MASK, slot0, k);
                const int knslots = __shfl_sync(RLAP_FULL_MASK, nslots, k);
                const int kM = __shfl_sync(RLAP_FULL_MASK, M, k);
                eliminate_star_regs(P, rc, kidx, kb, knb, fbuf + k * FCAP, knfill, kslot0, knslots, kM, ls, pend, la);
            }
            pend.flush(la);
            __syncwarp();
        }
        // ---- shared-memory path
        unsigned msm = __ballot_sync(RLAP_FULL_MASK, kind == K_SMEM);
        if (msm == 0) continue;
        if (lane == 0) ls->nsm += (unsigned)__popc(msm);
        if (P.o_v == 0) {
            // o_v = random: the late rounds hold few and large stars, and a warp that took them one after the other
            // inside its chunk kept the whole group waiting at the round's barrier. They are listed instead and dealt
            // out again, star by star, after the barrier (run_smem_items), next to the block-sized ones.
            int pos0 = 0;
            if (lane == 0) pos0 = atomicAdd(P.ctr + rc.s2slot, __popc(msm));
            pos0 = __shfl_sync(RLAP_FULL_MASK, pos0, 0);
            if (kind == K_SMEM) P.dl[rc.sl_top - 1 - (pos0 + __popc(msm & ((1u << lane) - 1u)))] = idx;
            continue;
        }
        // The fill list of a star is a chain of dependent loads (an L2 round trip per entry); a warp that walked the
        // lists of its shared-memory stars one after the other spent most of its time there. Every lane walks the list
        // of its own star into a global staging row first (up to 32 chains in flight), the warp then reads the rows
        // 32 entries at a time.
        const bool staging = P.stage_cap > 0;
        uint64_t* const stage = staging ? P.stage + ((size_t)blockIdx.x * ELIM_WARPS + (threadIdx.x >> 5)) * 32 * (size_t)P.stage_cap : nullptr;
        int st_n = 0, st_rest = -1;
        if (staging && kind == K_SMEM) {
            const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
            uint64_t* row = stage + (size_t)lane * (size_t)P.stage_cap;
            int p = ldcg_i32(head_p(P, idx));
            while (p >= 0 && st_n < P.stage_cap) {
                const int4 en = __ldcg(pool + p);
                row[st_n++] = pack_a((uint32_t)en.x, __int_as_float(en.y));
                p = en.z;
            }
            st_rest = p;
        }
        __syncwarp();
        while (msm) {
            int k = __ffs(msm) - 1;
            msm &= msm - 1;
            unsigned int kidx = __shfl_sync(RLAP_FULL_MASK, idx, k);
            StagedList stl;
            stl.valid = staging;
            stl.e = stage + (size_t)k * (size_t)P.stage_cap;
            stl.n = __shfl_sync(RLAP_FULL_MASK, st_n, k);
            stl.rest = __shfl_sync(RLAP_FULL_MASK, st_rest, k);
            eliminate_star<false>(P, rc, (int)(kidx / (unsigned)P.n), (int)(kidx % (unsigned)P.n), sb, cs, ls, la, stl);
        }
    }
}

// dynamic shared memory every mode of k_eliminate has at least (phases A2 / B, eliminate_smem_bytes): what a star in the
// global scratch slot may use as workspace
constexpr int ELIM_SMEM_MIN_BYTES = (6 * 1024 + ELIM_WARPS * (224 + 160)) * (int)sizeof(int);

__device__ __forceinline__ StarBuf elim_cta_buf(uint64_t* smem) {
    StarBuf sb;
    sb.A = smem;
    sb.Q = smem + ELIM_CAP_CTA;
    sb.K = smem + 2 * ELIM_CAP_CTA;
    sb.cap = ELIM_CAP_CTA;
    return sb;
}

// o_v = random: the stars of the round that need the warp's shared-memory buffer (`count` of them, listed downwards
// from dl[sl_top - 1]). Warps fetch them with one cursor, few at a time when the list is short; the fill lists of a
// fetch are walked side by side, one per lane, into the warp's staging rows before the stars are taken in turn.
template <class PT>
__device__ void run_smem_items(const PT& P, const RoundCtx& rc, uint64_t* smem, CtaScratch* cs, int count,
                               LocalStats* ls, LowAppender& la) {
    const int nw = (int)((P.gblocks * blockDim.x) >> 5);
    const int lane = threadIdx.x & 31;
    StarBuf sb = warp_region_buf(P, smem);
    int c = (count + 2 * nw - 1) / (2 * nw);
    c = c < 1 ? 1 : (c > 32 ? 32 : c);
    const bool staging = P.stage_cap > 0;
    uint64_t* const stage = staging ? P.stage + ((size_t)blockIdx.x * ELIM_WARPS + (threadIdx.x >> 5)) * 32 * (size_t)P.stage_cap : nullptr;
    while (true) {
        int c0 = 0;
        if (lane == 0) c0 = atomicAdd(P.ctr + rc.c2slot, c);
        c0 = __shfl_sync(RLAP_FULL_MASK, c0, 0);
        if (c0 >= count) break;
        const int it = c0 + lane;
        unsigned int idx = 0xffffffffu;
        if (lane < c && it < count) idx = __ldcg(P.dl + (rc.sl_top - 1 - it));
        int st_n = 0, st_rest = -1;
        if (staging && idx != 0xffffffffu && __ldg(P.hubidx + (int)(idx % (unsigned)P.n)) < 0) {   // a hub's lists are walked by the warp
            const int4* pool = P.pool + (size_t)(idx / (unsigned)P.n) * (size_t)P.pool_cap;
            uint64_t* row = stage + (size_t)lane * (size_t)P.stage_cap;
            int p = ldcg_i32(head_p(P, idx));
            while (p >= 0 && st_n < P.stage_cap) {
                const int4 en = __ldcg(pool + p);
                row[st_n++] = pack_a((uint32_t)en.x, __int_as_float(en.y));
                p = en.z;
            }
            st_rest = p;
        }
        __syncwarp();
        unsigned m = __ballot_sync(RLAP_FULL_MASK, idx != 0xffffffffu);
        while (m) {
            const int k = __ffs(m) - 1;
            m &= m - 1;
            const unsigned int kidx = __shfl_sync(RLAP_FULL_MASK, idx, k);
            StagedList stl;
            stl.valid = staging;
            stl.e = stage + (size_t)k * (size_t)P.stage_cap;
            stl.n = __shfl_sync(RLAP_FULL_MASK, st_n, k);
            stl.rest = __shfl_sync(RLAP_FULL_MASK, st_rest, k);
            eliminate_star<false>(P, rc, (int)(kidx / (unsigned)P.n), (int)(kidx % (unsigned)P.n), sb, cs, ls, la, stl);
        }
        __syncwarp();
    }
}

// deferred items [start, end): one block per item in shared memory; stars beyond ELIM_CAP_CTA go to the
// NSLOT blocks that own a global scratch slot
template <class PT>
__device__ void run_block_items(const PT& P, const RoundCtx& rc, uint64_t* smem, CtaScratch* cs, int start,
                                int end, LocalStats* ls, LowAppender& la) {
    const int lb = (int)blockIdx.x - P.gblock0;   // block index inside the view group
    for (int it = start + lb; it < end; it += P.gblocks) {
        unsigned int idx = __ldcg(P.dl + it);
        int view = (int)(idx / (unsigned)P.n), v = (int)(idx % (unsigned)P.n);
        if (ldcg_i32(live_p(P, idx)) <= ELIM_CAP_CTA) eliminate_star<true>(P, rc, view, v, elim_cta_buf(smem), cs, ls, la);
        __syncthreads();
    }
    const int nslot = min(NSLOT, P.gblocks);   // a view group may run on fewer blocks than there are slots
    if (lb < nslot) {
        int j = 0;
        for (int it = start; it < end; it++) {
            unsigned int idx = __ldcg(P.dl + it);
            if (ldcg_i32(live_p(P, idx)) <= ELIM_CAP_CTA) continue;
            if ((j++ % nslot) != lb) continue;
            int view = (int)(idx / (unsigned)P.n), v = (int)(idx % (unsigned)P.n);
            eliminate_star<true>(P, rc, view, v, scratch_buf(P), cs, ls, la, StagedList(), smem, ELIM_SMEM_MIN_BYTES);
            __syncthreads();
        }
    }
}

// Barrier of one view group (the blocks [gblock0, gblock0 + gblocks) of a cooperative launch, all co-resident): a
// counter of arrivals and a generation word in the group's control block. A group of one block needs no global
// barrier at all: its phases are separated by __syncthreads alone.
__device__ __forceinline__ void group_sync(int* bar, int nblocks) {
    __syncthreads();
    if (nblocks > 1) {
        if (threadIdx.x == 0) {
            volatile int* gen_p = bar + 1;
            const int gen = *gen_p;
            __threadfence();
            if (atomicAdd(bar, 1) == nblocks - 1) {
                *(volatile int*)bar = 0;
                __threadfence();
                atomicAdd(bar + 1, 1);
            } else {
                while (*gen_p == gen) {}
            }
            __threadfence();
        }
        __syncthreads();
    }
}

// One cooperative launch serves every view group of a call: block b works on the parameter block tab.g[tab.bg[b]].
// The table travels as a kernel parameter (22 KB of the 32 KB parameter space), so every field of every group is a
// constant-bank operand; a table in global memory costs the persistent kernel 160 B more spill stores and 0.9 ms per
// 64 arxiv-shaped views (measured, profiles/README.md).
constexpr int TAB_GROUPS = 64;
constexpr int TAB_BLOCKS = 1280;   // 4 blocks per SM x 148 SMs and room for other block sizes
template <int OV, int ON, bool FULL>
struct GroupTable {
    ModeParams<OV, ON, FULL> g[TAB_GROUPS];
    unsigned short bg[TAB_BLOCKS];
};
struct GroupTableRaw {               // what the host fills: same layout
    SchurParams g[TAB_GROUPS];
    unsigned short bg[TAB_BLOCKS];
};

// Blocks per SM, per mode. The modes that keep 32-bit shuffle keys beside the lane slots (o_n = random, coarsen) need
// 48 KB of dynamic shared memory per block: four such blocks push the SM to its largest shared-memory carve-out, which
// leaves 23 KB of L1 for the kernel's global loads and register spills - ncu: three times the short-scoreboard stalls
// (shared-memory accesses queueing behind L1 misses), 5.74 ms against 3.91 ms per 64 arxiv views with room for a 56 KB
// L1 (profiles/README.md). Three blocks per SM (24 warps, 80 registers: half the spills) is the fast side for them.
__host__ __device__ constexpr int mode_ctas(int ov, int on, bool full) {
    return (ELIM_THREADS == 256 && !full && (ov == 2 || on == 2)) ? 3 : ELIM_CTAS_PER_SM;
}

template <int OV, int ON, bool FULL>
__global__ void __launch_bounds__(ELIM_THREADS, mode_ctas(OV, ON, FULL)) k_eliminate(const __grid_constant__ GroupTable<OV, ON, FULL> tab) {
    const ModeParams<OV, ON, FULL>& P = tab.g[tab.bg[blockIdx.x]];
    extern __shared__ __align__(16) uint64_t smem[];
    __shared__ CtaScratch cs;
    __shared__ int s_nsel;
    __shared__ unsigned int s_lowbuf[ELIM_WARPS][LOWBUF];
    __shared__ LocalStats s_stats[ELIM_WARPS];
    const long long tid = (long long)((int)blockIdx.x - P.gblock0) * blockDim.x + threadIdx.x;   // inside the view group
    const long long nthr = (long long)P.gblocks * blockDim.x;
    int* const bar = P.ctr + CTR_BAR;
    const int gblocks = P.gblocks;
    const long long VN = (long long)P.V * P.n;
    const long long VG = (long long)P.V * P.G;
    const bool random_order = (P.o_v == 0);

    if (random_order) {
        const long long rows = ldcg_i32(P.hubcount);
        for (long long i = tid; i < (long long)P.V * rows * HUB_HEADS; i += nthr) {
            const long long view = i / (rows * HUB_HEADS), r = i % (rows * HUB_HEADS);
            P.hubheads[(view * P.nhmax) * HUB_HEADS + r] = -1;
        }
    }
    // ---- init: per-vertex state (ordering kernel for o_v = random: keyed Feistel rank)
    for (long long idx = tid; idx < VN; idx += nthr) {
        int view = (int)(idx / P.n), v = (int)(idx % P.n);
        *live_p(P, idx) = __ldg(P.ptr + v + 1) - __ldg(P.ptr + v);
        *head_p(P, idx) = -1;
        // keep mask: protected vertices are state 0; o_v = random ranks c(v), the number of unprotected vertices of
        // the graph below v, over the graph's m_g unprotected vertices (without a mask c(v) = v - gb and m_g = n_g)
        const bool prot = P.ucount && __ldg(P.ucount + v + 1) == __ldg(P.ucount + v);
        if (random_order) {
            int g = graph_of(P, v);
            int gb = __ldg(P.gptr + g), ng = __ldg(P.gptr + g + 1) - gb;
            int c = v - gb, mg = ng;
            if (P.ucount) {
                const int u0 = __ldg(P.ucount + gb);
                c = __ldg(P.ucount + v) - u0;
                mg = __ldg(P.ucount + gb + ng) - u0;
            }
            int rk = 0x7fffffff;
            if (!prot) {
                RankPerm rp;
                uint32_t oview = (P.flags & 2) ? 0u : (P.view_base + (uint32_t)view);
                rp.init(P.k0, P.k1, (uint32_t)g, oview, (uint32_t)mg);
                rk = (int)rp.rank((uint32_t)c);
            }
            P.rank[idx] = rk;
            P.state[idx] = rk < __ldg(P.teff + g) ? 1 : 0;
        } else {
            P.state[idx] = prot ? 0 : (__ldg(P.ptr + v + 1) == __ldg(P.ptr + v)) ? 4 : 1;
            P.candround[idx] = -1;
            P.rank[idx] = -1;   // degree / coarsen: round stamp of the low list
            P.outoff[idx] = 0;  // (round, key) snapshot of phase A (rounds are stored + 1: 0 = never visited)
        }
    }
    if (!random_order) {
        for (long long s = tid; s < VG; s += nthr) {
            int g = (int)(s % P.G);
            P.rem[s] = __ldg(P.teff + g);
            P.lvl[s] = -1;
            P.minkey[s] = 0x7fffffff;
            P.minkey[VG + s] = 0x7fffffff;
            P.cntI[s] = 0;
            P.ovfseg[s] = 0;
        }
    }
    for (long long s = tid; s < P.V; s += nthr) P.pool_cursor[s] = 0ull;
    for (long long s = tid; s < (long long)P.V * P.nw32; s += nthr) P.deadbits[s] = 0u;
    group_sync(bar, gblocks);

    // phase timing (block 0, thread 0; nanoseconds between grid barriers, waits included)
    unsigned long long tmark = 0;
#ifdef RLAP_DEBUG
    unsigned int rt[6] = {0, 0, 0, 0, 0, 0};   // this round's phase times (ns), printed with flags & 512
#endif
    auto lap = [&](int slot) {
        if (tid == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (slot >= 0) P.stats[slot] += now - tmark;
#ifdef RLAP_DEBUG
            if (slot >= ST_T_INIT) rt[slot - ST_T_INIT] += (unsigned int)(now - tmark);
#endif
            tmark = now;
        }
    };
    lap(-1);
    // grid barrier that ends a phase; a -DRLAP_DEBUG build with flags & 128 also records how long every warp waited there
#ifdef RLAP_DEBUG
    const bool wait_timers = (P.flags & 128) != 0;
#endif
    auto gsync = [&](int slot) {
#ifdef RLAP_DEBUG
        unsigned long long t0 = 0;
        if (wait_timers && (threadIdx.x & 31) == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
#endif
        group_sync(bar, gblocks);
#ifdef RLAP_DEBUG
        if (wait_timers && (threadIdx.x & 31) == 0) {
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            atomicAdd(P.stats + ST_W_INIT + (slot - ST_T_INIT), t1 - t0);
        }
#endif
        lap(slot);
    };
    // -DRLAP_DEBUG with flags & 512: thread 0 of block 0 times the parts of phase B
#ifdef RLAP_DEBUG
    unsigned long long dmark = 0;
#endif
    auto dlap = [&](int slot) {
#ifdef RLAP_DEBUG
        if ((P.flags & 512) && tid == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (slot >= 0) P.stats[ST_DBG + slot] += now - dmark;
            dmark = now;
        }
#else
        (void)slot;
#endif
    };
    int wl_start = 0;   // first unconsumed work-list item
    int dl_start = 0;
    int sl_top = (int)((long long)P.V * P.n);   // o_v = random: top of the group's dl region (one slot of slack above)
    int rounds = 0;
    RoundCtx rc;
    LocalStats* ls = s_stats + (threadIdx.x >> 5);
    if ((threadIdx.x & 31) == 0) { ls->fills = 0; ls->raw = 0; ls->maxstar = 0; ls->nsm = 0; }
    __syncwarp();
    LowAppender la;
    la.buf = s_lowbuf[threadIdx.x >> 5];
    la.P = &P;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const unsigned uVN = (unsigned)VN, un = (unsigned)P.n;

    if (random_order) {
        // dependency counters: pending lower-ranked eligible neighbours; roots seed the work list
        // (they count as appended in round -1, i.e. on counter slot 2)
        for (unsigned base = (unsigned)(tid - lane); base < uVN; base += (unsigned)nthr) {
            unsigned idx = base + lane;
            bool elig = idx < uVN && ldcg_u8(P.state + idx) == 1;
            int view = 0, v = 0, rv = 0, b = 0, e = 0;
            if (elig) {
                view = (int)(idx / un); v = (int)(idx % un);
                rv = ldcg_i32(P.rank + idx);
                b = __ldg(P.ptr + v); e = __ldg(P.ptr + v + 1);
            }
            const bool longrow = elig && (e - b) > 64;
            int c = 0;
            if (elig && !longrow) {
                size_t vb = (size_t)view * P.n;
                for (int p = b; p < e; p++) {
                    int u = __ldg(P.col + p);
                    if (ldcg_u8(P.state + vb + u) == 1 && ldcg_i32(P.rank + vb + u) < rv) c++;
                }
            }
            unsigned todo = __ballot_sync(RLAP_FULL_MASK, longrow);
            while (todo) {  // hubs: the warp walks the row together
                int k = __ffs(todo) - 1;
                todo &= todo - 1;
                int kb = __shfl_sync(RLAP_FULL_MASK, b, k), ke = __shfl_sync(RLAP_FULL_MASK, e, k);
                int krv = __shfl_sync(RLAP_FULL_MASK, rv, k);
                size_t kvb = (size_t)__shfl_sync(RLAP_FULL_MASK, view, k) * P.n;
                int cc = 0;
                for (int p = kb + lane; p < ke; p += 32) {
                    int u = __ldg(P.col + p);
                    if (ldcg_u8(P.state + kvb + u) == 1 && ldcg_i32(P.rank + kvb + u) < krv) cc++;
                }
                cc = __reduce_add_sync(RLAP_FULL_MASK, cc);
                if (lane == k) c = cc;
            }
            if (elig) P.blk[idx] = c;
            bool root = elig && c == 0;
            unsigned rm = __ballot_sync(RLAP_FULL_MASK, root);
            if (rm) {
                int pos0 = 0;
                if (lane == 0) pos0 = atomicAdd(P.ctr + CTR_WCNT0 + 2, __popc(rm));
                pos0 = __shfl_sync(RLAP_FULL_MASK, pos0, 0);
                if (root) P.wl[pos0 + __popc(rm & lt)] = idx;
            }
        }
        gsync(ST_T_INIT);
        while (true) {
            // items to consume were appended in the previous round
            int wl_end = wl_start + ldcg_i32(P.ctr + CTR_WCNT0 + (rounds + 2) % 3);
            if (wl_end == wl_start) break;
            if (tid == 0) {
                P.ctr[CTR_WCNT0 + (rounds + 1) % 3] = 0; P.ctr[CTR_DCNT0 + (rounds + 1) % 3] = 0; P.ctr[CTR_STEAL0 + (rounds + 1) % 3] = 0;
                P.ctr[CTR_SCNT0 + (rounds + 1) % 3] = 0; P.ctr[CTR_SSTEAL0 + (rounds + 1) % 3] = 0;
            }
            rc.sslot = CTR_STEAL0 + rounds % 3;
            rc.wl_base = wl_end; rc.wslot = CTR_WCNT0 + rounds % 3;
            rc.dl_base = dl_start; rc.dslot = CTR_DCNT0 + rounds % 3;
            rc.sl_top = sl_top; rc.s2slot = CTR_SCNT0 + rounds % 3; rc.c2slot = CTR_SSTEAL0 + rounds % 3;
#ifdef RLAP_DEBUG
            const int items_dbg = wl_end - wl_start;
#endif
            run_warp_items(P, rc, smem, &cs, wl_start, wl_end, ls, la);
            wl_start = wl_end;
            gsync(ST_T_D1);
            // stars too large for a lane or a register tile: the block-sized ones first (a block per star), then every
            // warp fetches from the list of the warp-sized ones; blocks without a block-sized star start there at once
            const int dl_end = dl_start + ldcg_i32(P.ctr + rc.dslot);
            const int s_cnt = ldcg_i32(P.ctr + rc.s2slot);
#ifdef RLAP_DEBUG
            const int hubs_dbg = dl_end - dl_start;
#endif
            if (dl_end != dl_start || s_cnt > 0) {
                if (dl_end != dl_start) run_block_items(P, rc, smem, &cs, dl_start, dl_end, ls, la);
                if (s_cnt > 0) run_smem_items(P, rc, smem, &cs, s_cnt, ls, la);
                dl_start = dl_end;
                sl_top -= s_cnt;
                gsync(ST_T_D2);
            }
#ifdef RLAP_DEBUG
            if ((P.flags & 512) && tid == 0 && P.view_base == 0) {
                printf("round %d items %d warp-sized %d block-sized %d | D1 %u D2 %u ns\n", rounds, items_dbg, s_cnt, hubs_dbg, rt[4], rt[5]);
                for (int q = 0; q < 6; q++) rt[q] = 0;
            }
#endif
            rounds++;
        }
    } else {
        lap(ST_T_INIT);
        // degree / coarsen: rounds over the minimum-key bucket of every (view, graph) segment (DESIGN.md §3.4).
        // Full scans of the vertices are only made when a segment's level advances: lvl[seg] is the minimum key
        // the last full scan found, and every open vertex (alive, unprotected) whose key is <= lvl[seg] is on the round's low list
        // (bucket members that were blocked, listed vertices that were not in the bucket, and every vertex whose
        // live counter was seen crossing from above lvl to lvl or below by the elimination phase). While the low
        // list of a segment has an entry in play the bucket is taken from the list alone.
        constexpr int SEG_SM = 1024, WBUF = 224, MBUF = 160;
        const int INF = 0x7fffffff;
        // (round, key) snapshots written by phase A, read by the bucket test of phase B; the emission's row offsets
        // are not needed before the elimination is over
        unsigned long long* mark = (unsigned long long*)P.outoff;
        auto mark_of = [](int round, int key) { return ((unsigned long long)(unsigned)(round + 1) << 32) | (unsigned)key; };
        int* mkl = P.minkey;          // minimum over the low list
        int* mks = P.minkey + VG;     // minimum over a full scan
        const bool bsm = VG <= (long long)SEG_SM;
        while (true) {
            const int par = rounds & 1;
            const unsigned int* low_in = P.low + (size_t)par * (size_t)P.low_cap;
            la.par = par ^ 1;
            long long n_in = ldcg_i32(P.ctr + CTR_LOW0 + par);
            if (n_in > P.low_cap) n_in = P.low_cap;
            if (ldcg_i32(P.ctr + CTR_LOWOVF0 + par)) n_in = 0;   // entries were lost: every segment rescans
            rc.wl_base = wl_start; rc.wslot = CTR_WCNT0 + rounds % 3;
            rc.dl_base = dl_start; rc.dslot = CTR_DCNT0 + rounds % 3;
            rc.sslot = CTR_STEAL0 + rounds % 3;
            if (tid == 0) {
                P.ctr[CTR_ACTIVE0 + (par ^ 1)] = 0; P.ctr[CTR_OVF0 + (par ^ 1)] = 0;
                P.ctr[CTR_WCNT0 + (rounds + 1) % 3] = 0; P.ctr[CTR_DCNT0 + (rounds + 1) % 3] = 0;
                P.ctr[CTR_STEAL0 + (rounds + 1) % 3] = 0;
                P.ctr[CTR_LOW0 + (par ^ 1)] = 0; P.ctr[CTR_LOWOVF0 + (par ^ 1)] = 0;
            }
            for (long long s = tid; s < VG; s += nthr) { P.cntI[s] = 0; P.ovfseg[s] = 0; }
            // ---- phase A1: minimum key over the low-list entries in play
            {
                bool any = false;
                for (long long i0 = tid - lane; i0 < n_in; i0 += nthr) {
                    const long long i = i0 + lane;
                    bool valid = false;
                    int seg = 0, key = INF;
                    if (i < n_in) {
                        const unsigned idx = __ldcg(low_in + i);
                        const uint8_t st = ldcg_u8(P.state + idx);
                        if (open_st(st)) {
                            seg = (int)(idx / un) * P.G + graph_of(P, (int)(idx % un));
                            key = (st == 4) ? 0 : max(ldcg_i32(live_p(P, idx)), 1);
                            valid = ldcg_i32(P.rem + seg) > 0 && key <= ldcg_i32(P.lvl + seg);
                            if (valid) mark[idx] = mark_of(rounds, key);
                        }
                    }
                    const unsigned vm = __ballot_sync(RLAP_FULL_MASK, valid);
                    if (vm == 0) continue;
                    any = true;
                    const int leader = __ffs(vm) - 1;
                    const int seg0 = __shfl_sync(RLAP_FULL_MASK, seg, leader);
                    if (__all_sync(RLAP_FULL_MASK, !valid || seg == seg0)) {
                        const int k = __reduce_min_sync(RLAP_FULL_MASK, valid ? key : INF);
                        if (lane == leader) atomicMin(mkl + seg0, k);
                    } else if (valid) {
                        atomicMin(mkl + seg, key);
                    }
                }
                if (any && lane == 0) P.ctr[CTR_ACTIVE0 + par] = 1;
            }
            gsync(ST_T_A);
#ifdef RLAP_DEBUG
            if ((P.flags & 512) && tid == 0) {   // debug: list size and number of rescanning segments per round
                int ns = 0, mn = INF;
                for (long long q = 0; q < VG; q++) {
                    if (ldcg_i32(P.rem + q) > 0 && ldcg_i32(mkl + q) == INF) ns++;
                    mn = min(mn, ldcg_i32(mkl + q));
                }
                printf("round %d: low list %lld entries, %d of %lld segments rescan, min list key %d, lvl[0] %d rem[0] %d\n",
                       rounds, n_in, ns, VG, mn, P.lvl[0], P.rem[0]);
            }
#endif
            // ---- phase A2: segments with nothing in play on the list scan all their vertices for the minimum key
            {
                int* smin = (int*)smem;         // [VG] block-level minima
                int* sneed = smin + SEG_SM;     // [VG] 1 = the segment rescans
                int* sviews = sneed + SEG_SM;   // views with a rescanning segment (the scan visits only their vertices)
                int* sflag = sviews + SEG_SM;
                unsigned nsel = (unsigned)P.V;
                if (bsm) {
                    for (int q = threadIdx.x; q < P.V; q += blockDim.x) sflag[q] = 0;
                    if (threadIdx.x == 0) s_nsel = 0;
                    __syncthreads();
                    for (int q = threadIdx.x; q < (int)VG; q += blockDim.x) {
                        smin[q] = INF;
                        const int need = (ldcg_i32(P.rem + q) > 0 && ldcg_i32(mkl + q) == INF) ? 1 : 0;
                        sneed[q] = need;
                        if (need) sflag[q / P.G] = 1;
                    }
                    __syncthreads();
                    // ascending view order: every block must enumerate the selected vertices identically
                    for (int q = threadIdx.x; q < P.V; q += blockDim.x) {
                        if (sflag[q]) {
                            int pos = 0;
                            for (int j = 0; j < q; j++) pos += sflag[j];
                            sviews[pos] = q;
                            atomicAdd(&s_nsel, 1);
                        }
                    }
                    __syncthreads();
                    nsel = (unsigned)s_nsel;
                }
                bool any = false;
                // four independent elements per thread and iteration; every load is issued before the first use;
                // (selected view, vertex) of the running index are advanced incrementally: no division in the loop
                const unsigned total = nsel * un;
                const unsigned step_q = (unsigned)nthr / un, step_r = (unsigned)nthr % un;
                unsigned cview = (unsigned)tid / un, cv = (unsigned)tid % un;
                for (unsigned base = (unsigned)(tid - lane); base < total; base += 4u * (unsigned)nthr) {
                    uint8_t st4[4];
                    int lv4[4], sg4[4];
                    unsigned ix4[4];
                    bool nd4[4];
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        const unsigned e = base + (unsigned)q4 * (unsigned)nthr + lane;
                        st4[q4] = 2; lv4[q4] = 0; sg4[q4] = 0; nd4[q4] = false;
                        const unsigned sv = cview;
                        const int v = (int)cv;
                        cview += step_q; cv += step_r;
                        if (cv >= un) { cv -= un; cview++; }
                        if (e < total) {
                            const int view = bsm ? sviews[sv] : (int)sv;
                            const unsigned idx = (unsigned)view * un + (unsigned)v;
                            ix4[q4] = idx;
                            sg4[q4] = view * P.G + graph_of(P, v);
                            nd4[q4] = bsm ? (sneed[sg4[q4]] != 0)
                                          : (ldcg_i32(P.rem + sg4[q4]) > 0 && ldcg_i32(mkl + sg4[q4]) == INF);
                            if (nd4[q4]) {
                                st4[q4] = ldcg_u8(P.state + idx);
                                lv4[q4] = ldcg_i32(live_p(P, idx));
                            }
                        }
                    }
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        const bool valid = nd4[q4] && open_st(st4[q4]);
                        const int seg = sg4[q4];
                        const int key = valid ? ((st4[q4] == 4) ? 0 : max(lv4[q4], 1)) : INF;
                        if (valid) mark[ix4[q4]] = mark_of(rounds, key);
                        const unsigned vm = __ballot_sync(RLAP_FULL_MASK, valid);
                        if (vm == 0) continue;
                        any = true;
                        const int leader = __ffs(vm) - 1;
                        const int seg0 = __shfl_sync(RLAP_FULL_MASK, seg, leader);
                        if (__all_sync(RLAP_FULL_MASK, !valid || seg == seg0)) {
                            const int k = __reduce_min_sync(RLAP_FULL_MASK, key);
                            if (lane == leader) { if (bsm) atomicMin(smin + seg0, k); else atomicMin(mks + seg0, k); }
                        } else if (valid) {
                            if (bsm) atomicMin(smin + seg, key); else atomicMin(mks + seg, key);
                        }
                    }
                }
                if (bsm) {
                    __syncthreads();
                    for (int q = threadIdx.x; q < (int)VG; q += blockDim.x) {
                        const int k = smin[q];
                        if (k != INF) atomicMin(mks + q, k);
                    }
                    __syncthreads();
                }
                if (any && lane == 0) P.ctr[CTR_ACTIVE0 + par] = 1;
            }
            gsync(ST_T_A);
            if (ldcg_i32(P.ctr + CTR_ACTIVE0 + par) == 0) break;
            if (rounds > P.n + 8) { if (tid == 0) set_status(P, 10); break; }   // every round removes a vertex of every active segment
            // ---- phase B: members of the minimum bucket with no bucket neighbour of higher id are selected, the
            // other members (and the listed vertices below the level that are not in the bucket) go to the next list.
            // Shared memory (the star buffers are idle): per-segment copies if there are few enough segments, a
            // candidate buffer per warp so that the work-list tail is bumped once per few hundred candidates.
            dlap(-1);
            int* srem = (int*)smem;                 // remaining removals (0: the segment is done)
            int* smk = srem + SEG_SM;               // bucket key of the round (INF: nothing to do)
            int* scnt = smk + SEG_SM;               // candidates selected by this block
            int* slv = scnt + SEG_SM;               // level; -1 marks a segment that rescans in this round
            int* sviews = slv + SEG_SM;             // views with a segment that rescans in this round
            int* sflag = sviews + SEG_SM;
            unsigned int* wbuf = (unsigned int*)((int*)smem + 6 * SEG_SM) + (size_t)(threadIdx.x >> 5) * WBUF;
            int wfill = 0;
            unsigned nselB = (unsigned)P.V;
            // per-segment view of the round: bucket key m, scan flag, level
            auto seg_round = [&](int seg, int& rm, int& m, bool& scan, int& lv) {
                if (bsm) {
                    rm = srem[seg]; m = smk[seg]; lv = slv[seg]; scan = lv < 0;
                } else {
                    rm = ldcg_i32(P.rem + seg);
                    const int ml = ldcg_i32(mkl + seg);
                    scan = ml == INF;
                    m = scan ? ldcg_i32(mks + seg) : ml;
                    lv = scan ? -1 : ldcg_i32(P.lvl + seg);
                }
            };
            if (bsm) {
                for (int q = threadIdx.x; q < P.V; q += blockDim.x) sflag[q] = 0;
                if (threadIdx.x == 0) s_nsel = 0;
                __syncthreads();
                for (int q = threadIdx.x; q < (int)VG; q += blockDim.x) {
                    const int ml = ldcg_i32(mkl + q);
                    const bool scan = ml == INF;
                    srem[q] = ldcg_i32(P.rem + q);
                    smk[q] = scan ? ldcg_i32(mks + q) : ml;
                    slv[q] = scan ? -1 : ldcg_i32(P.lvl + q);
                    scnt[q] = 0;
                    if (scan && srem[q] > 0 && smk[q] != INF) sflag[q / P.G] = 1;
                }
                __syncthreads();
                for (int q = threadIdx.x; q < P.V; q += blockDim.x) {   // ascending view order, identical in every block
                    if (sflag[q]) {
                        int pos = 0;
                        for (int j = 0; j < q; j++) pos += sflag[j];
                        sviews[pos] = q;
                        atomicAdd(&s_nsel, 1);
                    }
                }
                __syncthreads();
                nselB = (unsigned)s_nsel;
            }
            auto flush = [&]() {
                if (wfill == 0) return;
                int pos0 = 0;
                if (lane == 0) pos0 = atomicAdd(P.ctr + rc.wslot, wfill);
                pos0 = __shfl_sync(RLAP_FULL_MASK, pos0, 0);
                __syncwarp();
                for (int i = lane; i < wfill; i += 32) P.wl[rc.wl_base + pos0 + i] = wbuf[i];
                __syncwarp();
                wfill = 0;
            };
            // bucket member v of `view` (key m): true if no alive neighbour of higher id has key m. Phase A left the
            // (round, key) snapshot of every vertex it visited in `mark`: all alive vertices of a rescanning segment,
            // all vertices in play otherwise, i.e. every alive vertex whose key can equal m. One 8-byte load per
            // neighbour answers "alive bucket member?" (an eliminated or unvisited neighbour carries an older round).
            auto member_free = [&](unsigned idx, int view, int v, int m) -> bool {
                const size_t vb = (size_t)view * P.n;
                const unsigned long long want = mark_of(rounds, m);
                bool ok = true;
                // base neighbours, four at a time: ids first, then their snapshots together
                const int pb = __ldg(P.ptr + v), pe = __ldg(P.ptr + v + 1);
                for (int p = pb; p < pe && ok; p += 4) {
                    int u4[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) u4[k] = (p + k < pe) ? __ldg(P.col + p + k) : -1;
                    unsigned long long k4[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) k4[k] = (u4[k] > v) ? __ldcg(mark + vb + u4[k]) : 0ull;
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        if (u4[k] > v && k4[k] == want) ok = false;
                }
                const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
                for (int p = ldcg_i32(head_p(P, idx)); p >= 0 && ok;) {
                    int4 en = __ldcg(pool + p);
                    if (en.x > v && __ldcg(mark + vb + en.x) == want) ok = false;
                    p = en.z;
                }
                return ok;
            };
            // warp-collective: record the selected members (`cand`) of one pass over 32 vertices
            auto select = [&](bool cand, unsigned idx, int seg, int rm) {
                const unsigned cm = __ballot_sync(RLAP_FULL_MASK, cand);
                if (cm == 0) return;
                if (wfill + 32 > WBUF) flush();
                if (cand) {
                    P.candround[idx] = rounds;
                    wbuf[wfill + __popc(cm & lt)] = idx;
                    if (bsm) {
                        atomicAdd(scnt + seg, 1);
                    } else {
                        int c = atomicAdd(P.cntI + seg, 1);
                        if (c + 1 > rm) P.ctr[CTR_OVF0 + par] = 1;
                    }
                }
                wfill += __popc(cm);
            };
            // member buffer of the scan part: up to 32 left over + 128 new per iteration
            unsigned int* mbuf = (unsigned int*)((int*)smem + 6 * SEG_SM + ELIM_WARPS * WBUF) + (size_t)(threadIdx.x >> 5) * MBUF;
            int mfill = 0;
            auto test_members = [&](int first, int count) {      // warp-collective: lane i tests member first + i
                bool cand = false, keep = false;
                unsigned idx = 0;
                int seg = 0, rm = 0;
                if (lane < count) {
                    idx = mbuf[first + lane];
                    const int view = (int)(idx / un), v = (int)(idx % un);
                    seg = view * P.G + graph_of(P, v);
                    int m, lvq;
                    bool scan;
                    seg_round(seg, rm, m, scan, lvq);
                    if (member_free(idx, view, v, m)) cand = true; else keep = true;
                }
                __syncwarp();
                select(cand, idx, seg, rm);
                la.push(keep, idx);
            };
            dlap(0);
            // B1: the low list (segments that do not rescan)
            for (long long i0 = tid - lane; i0 < n_in; i0 += nthr) {
                const long long i = i0 + lane;
                bool cand = false, keep = false;
                unsigned idx = 0;
                int seg = 0, rm = 0;
                if (i < n_in) {
                    idx = __ldcg(low_in + i);
                    const uint8_t st = ldcg_u8(P.state + idx);
                    if (open_st(st)) {
                        const int view = (int)(idx / un), v = (int)(idx % un);
                        seg = view * P.G + graph_of(P, v);
                        int m, lv;
                        bool scan;
                        seg_round(seg, rm, m, scan, lv);
                        const int key = (st == 4) ? 0 : max(ldcg_i32(live_p(P, idx)), 1);
                        // in play, and the first copy of this vertex on the list (P.rank holds the round stamp)
                        if (rm > 0 && !scan && key <= lv && atomicExch(P.rank + idx, rounds) != rounds) {
                            if (key == m && member_free(idx, view, v, m)) cand = true; else keep = true;
                        }
                    }
                }
                select(cand, idx, seg, rm);
                la.push(keep, idx);
            }
            dlap(1);
            // B2: full scan of the segments that rescan; their level becomes the bucket key the scan found
            for (long long q = tid; q < VG; q += nthr) {
                if (ldcg_i32(mkl + q) == INF) { const int m2 = ldcg_i32(mks + q); if (m2 != INF) P.lvl[q] = m2; }
            }
            {
                const unsigned total = nselB * un;
                const unsigned step_q = (unsigned)nthr / un, step_r = (unsigned)nthr % un;
                unsigned cview = (unsigned)tid / un, cv = (unsigned)tid % un;
                for (unsigned base = (unsigned)(tid - lane); base < total; base += 4u * (unsigned)nthr) {
                    uint8_t st4[4];
                    int lv4[4], rm4[4], sg4[4], mk4[4], vw4[4], vx4[4];
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        const unsigned e = base + (unsigned)q4 * (unsigned)nthr + lane;
                        st4[q4] = 2; lv4[q4] = 0; rm4[q4] = 0; sg4[q4] = 0; mk4[q4] = -1;
                        const unsigned sv = cview;
                        const int v = (int)cv;
                        vw4[q4] = 0; vx4[q4] = v;
                        cview += step_q; cv += step_r;
                        if (cv >= un) { cv -= un; cview++; }
                        if (e < total) {
                            const int view = bsm ? sviews[sv] : (int)sv;
                            vw4[q4] = view;
                            const unsigned idx = (unsigned)view * un + (unsigned)v;
                            sg4[q4] = view * P.G + graph_of(P, v);
                            int lvq;
                            bool scan;
                            seg_round(sg4[q4], rm4[q4], mk4[q4], scan, lvq);
                            if (scan && rm4[q4] > 0 && mk4[q4] != INF) {
                                st4[q4] = ldcg_u8(P.state + idx);
                                lv4[q4] = ldcg_i32(live_p(P, idx));
                            } else {
                                mk4[q4] = -1;
                            }
                        }
                    }
                    // the bucket members among these 128 vertices go to the warp's member buffer; the tests run on full
                    // batches of 32 members, one per lane (testing in place left three quarters of the lanes idle while
                    // the warp waited for the longest list of each of the four passes)
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        const unsigned idx = (unsigned)vw4[q4] * un + (unsigned)vx4[q4];
                        const int m = mk4[q4];
                        const int key = (st4[q4] == 4) ? 0 : max(lv4[q4], 1);
                        const bool alive = m >= 0 && open_st(st4[q4]);
                        const bool member = alive && key == m;
                        const unsigned mm = __ballot_sync(RLAP_FULL_MASK, member);
                        if (member) mbuf[mfill + __popc(mm & lt)] = idx;
                        mfill += __popc(mm);
                    }
                    __syncwarp();
                    while (mfill >= 32) { mfill -= 32; test_members(mfill, 32); }
                }
                if (mfill > 0) { test_members(0, mfill); mfill = 0; }
            }
            dlap(2);
            flush();
            la.flush();
            dlap(3);
            if (bsm) {
                __syncthreads();
                for (int q = threadIdx.x; q < (int)VG; q += blockDim.x) {
                    int c = scnt[q];
                    if (c > 0) {
                        int c0 = atomicAdd(P.cntI + q, c);
                        if (c0 + c > srem[q]) P.ctr[CTR_OVF0 + par] = 1;
                    }
                }
            }
            __syncthreads();   // the shared copies are star buffers again from here on
            dlap(4);
            gsync(ST_T_B);
            dlap(5);
            // phase C: a graph that selected more than it may still remove keeps its highest ids
            if (ldcg_i32(P.ctr + CTR_OVF0 + par)) {
                const int gw = (int)(tid >> 5), nw = (int)(nthr >> 5), lane = threadIdx.x & 31;
                const long long nblk = (VN + SEL_BLOCK - 1) / SEL_BLOCK;
                for (long long bk = gw; bk < nblk; bk += nw) {
                    int c = 0;
                    for (int j = 0; j < SEL_BLOCK / 32; j++) {
                        long long idx = bk * SEL_BLOCK + j * 32 + lane;
                        bool f = idx < VN && ldcg_i32(P.candround + idx) == rounds;
                        c += __popc(__ballot_sync(RLAP_FULL_MASK, f));
                    }
                    if (lane == 0) P.blockcnt[bk] = c;
                }
                group_sync(bar, gblocks);
                for (long long s = gw; s < VG; s += nw) {
                    int need = ldcg_i32(P.rem + s);
                    if (ldcg_i32(P.cntI + s) <= need) continue;
                    int view = (int)(s / P.G), g = (int)(s % P.G);
                    long long lo = (long long)view * P.n + __ldg(P.gptr + g);
                    long long hi = (long long)view * P.n + __ldg(P.gptr + g + 1);  // exclusive
                    // walk down from hi in SEL_BLOCK-aligned pieces until `need` candidates are covered
                    long long cur = hi;
                    int acc = 0;
                    long long T = lo;
                    while (cur > lo) {
                        long long pb = ((cur - 1) / SEL_BLOCK) * SEL_BLOCK;  // aligned block holding cur-1
                        long long pstart = pb > lo ? pb : lo;
                        bool whole = (pstart == pb) && (cur == pb + SEL_BLOCK);
                        int c;
                        if (whole) {
                            c = ldcg_i32(P.blockcnt + pb / SEL_BLOCK);
                        } else {
                            c = 0;
                            for (long long q0 = pstart; q0 < cur; q0 += 32) {
                                long long q = q0 + lane;
                                bool f = q < cur && ldcg_i32(P.candround + q) == rounds;
                                c += __popc(__ballot_sync(RLAP_FULL_MASK, f));
                            }
                        }
                        if (acc + c >= need) {
                            // the threshold lies inside [pstart, cur): scan it from the top, 32 ids at a time
                            long long q1 = cur;
                            while (q1 > pstart) {
                                long long q0 = q1 - 32 > pstart ? q1 - 32 : pstart;
                                long long q = q0 + lane;
                                bool f = q < q1 && ldcg_i32(P.candround + q) == rounds;
                                unsigned mb = __ballot_sync(RLAP_FULL_MASK, f);
                                int cc = __popc(mb);
                                if (acc + cc >= need) {
                                    int want = need - acc;  // keep the `want` highest set bits of mb
                                    int bit = 31;
                                    for (;; bit--) {
                                        if (mb & (1u << bit)) { want--; if (want == 0) break; }
                                    }
                                    T = q0 + bit;
                                    acc = need;
                                    break;
                                }
                                acc += cc;
                                q1 = q0;
                            }
                            break;
                        }
                        acc += c;
                        cur = pstart;
                    }
                    if (lane == 0) { P.thresh[s] = (unsigned int)T; P.ovfseg[s] = 1; }
                }
                gsync(ST_T_C);
            }
            // the truncated count is what phase D will eliminate; the per-round minima are reset for the next round
            for (long long q = tid; q < VG; q += nthr) {
                int rm = ldcg_i32(P.rem + q), c = ldcg_i32(P.cntI + q);
                if (c > 0) P.rem[q] = rm - min(rm, c);
                mkl[q] = INF; mks[q] = INF;
            }
            // phase D: eliminate
            int wl_end = wl_start + ldcg_i32(P.ctr + rc.wslot);
#ifdef RLAP_DEBUG
            const int items_dbg = wl_end - wl_start;
#endif
            run_warp_items(P, rc, smem, &cs, wl_start, wl_end, ls, la);
            wl_start = wl_end;
            la.flush();
            gsync(ST_T_D1);
            int dl_end = dl_start + ldcg_i32(P.ctr + rc.dslot);
            if (dl_end != dl_start) {
                run_block_items(P, rc, smem, &cs, dl_start, dl_end, ls, la);
                dl_start = dl_end;
                la.flush();
                gsync(ST_T_D2);
            }
#ifdef RLAP_DEBUG
            if ((P.flags & 512) && tid == 0 && P.view_base == 0) {
                printf("round %d items %d low_in %lld | A %u B %u C %u D1 %u D2 %u ns\n", rounds, items_dbg, n_in, rt[1], rt[2], rt[3], rt[4], rt[5]);
                for (int q = 0; q < 6; q++) rt[q] = 0;
            }
#endif
            rounds++;
        }
    }
    if (tid == 0) P.ctr[CTR_ROUNDS] = rounds;
    __syncwarp();
    if ((threadIdx.x & 31) == 0 && (ls->raw | ls->fills)) {
        atomicAdd(P.stats + ST_FILLS, ls->fills);
        atomicAdd(P.stats + ST_RAW, ls->raw);
        atomicMax(P.stats + ST_MAXSTAR, (unsigned long long)ls->maxstar);
        if (ls->nsm) atomicAdd(P.stats + ST_DEFERRED, (unsigned long long)ls->nsm);
    }
}

// gid[v] = graph of vertex v, teff[g] = min(max(num_remove, 0), n_g - 1); with a keep mask (ucount, see SchurParams)
// a graph with a protected vertex may lose all its m_g unprotected vertices: teff[g] = min(max(num_remove, 0), m_g)
__global__ void k_setup_graphs(int n, int G, const int* gptr, const long long* num_remove, const int* ucount, int* gid,
                               int* teff) {
    long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid < G) {
        long long ng = gptr[tid + 1] - gptr[tid];
        long long mg = ucount ? ucount[gptr[tid + 1]] - ucount[gptr[tid]] : ng;
        long long t = num_remove[tid];
        if (t < 0) t = 0;
        if (t > (mg < ng ? mg : ng - 1)) t = mg < ng ? mg : ng - 1;
        if (t < 0) t = 0;
        teff[tid] = (int)t;
    }
    if (gid && tid < n) {
        int lo = 0, hi = G;  // last g with gptr[g] <= v
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (gptr[mid] <= (int)tid) lo = mid; else hi = mid;
        }
        gid[tid] = lo;
    }
}

// ---------------------------------------------------------------------------------------------
// host-side launchers (called from api.cu)
// ---------------------------------------------------------------------------------------------
// dynamic shared memory of k_eliminate: the block-level star buffer (3 x CAP_CTA words) or the per-warp regions of the
// elimination phase, whichever is larger
static size_t eliminate_smem_bytes(bool need_keys) {
    const size_t cta = (size_t)3 * ELIM_CAP_CTA * sizeof(uint64_t);
    const size_t warps = (size_t)ELIM_WARPS * (size_t)warp_region_words(need_keys) * sizeof(uint64_t);
    // phases A2 / B: six per-segment arrays of 1 024 ints + the candidate and member buffers of every warp (224 + 160 ints)
    const size_t phases = (size_t)ELIM_SMEM_MIN_BYTES;
    size_t m = cta > warps ? cta : warps;
    return m > phases ? m : phases;
}

// o_v = random: rows of the hub head table (vertices of at least HUB_DEG input entries), in no particular order
__global__ void k_hub_index(int n, const int* __restrict__ ptr, int* __restrict__ hubidx, int* __restrict__ count) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    int h = -1;
    if (ptr[v + 1] - ptr[v] >= HUB_DEG) h = atomicAdd(count, 1);
    hubidx[v] = h;
}

cudaError_t launch_hub_index(int n, const int* ptr, int* hubidx, int* count, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(count, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    k_hub_index<<<(n + 255) / 256, 256, 0, stream>>>(n, ptr, hubidx, count);
    return cudaGetLastError();
}

cudaError_t launch_setup_graphs(int n, int G, const int* gptr, const long long* num_remove, const int* ucount, int* gid,
                                int* teff, cudaStream_t stream) {
    long long work = n > G ? n : G;
    int blocks = (int)((work + 255) / 256);
    if (blocks < 1) blocks = 1;
    k_setup_graphs<<<blocks, 256, 0, stream>>>(n, G, gptr, num_remove, ucount, gid, teff);
    return cudaGetLastError();
}

__global__ void k_unprotected(int n, const uint8_t* __restrict__ keep, int* __restrict__ flag) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) flag[v] = keep[v] ? 0 : 1;
}

// keep mask -> ucount[n + 1]: exclusive prefix count of the unprotected vertices (flag: n ints of scratch)
cudaError_t launch_count_unprotected(int n, const uint8_t* keep, int* flag, int* ucount, long long* blocksum,
                                     cudaStream_t stream) {
    k_unprotected<<<(n + 255) / 256, 256, 0, stream>>>(n, keep, flag);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_exclusive_scan<int>(flag, n, ucount, blocksum, nullptr, stream);
}

// One instantiation of k_eliminate per mode. Coarsening fixes the neighbour order (shuffle, preconditioner.cc:831) and
// the full-clique test mode ignores it, so nine kernels cover every (o_v, o_n, flags) combination.
constexpr int N_MODES = 9;
static int mode_index(int o_v, int o_n, bool full) {
    if (full) return o_v == 0 ? 7 : 8;
    if (o_v == 2) return 6;
    return o_v * 3 + o_n;
}
static bool mode_needs_keys(int m) { return m == 2 || m == 5 || m == 6; }
static const void* mode_kernel(int m) {
    switch (m) {
        case 0: return (const void*)k_eliminate<0, 0, false>;
        case 1: return (const void*)k_eliminate<0, 1, false>;
        case 2: return (const void*)k_eliminate<0, 2, false>;
        case 3: return (const void*)k_eliminate<1, 0, false>;
        case 4: return (const void*)k_eliminate<1, 1, false>;
        case 5: return (const void*)k_eliminate<1, 2, false>;
        case 6: return (const void*)k_eliminate<2, 2, false>;
        case 7: return (const void*)k_eliminate<0, 0, true>;
        default: return (const void*)k_eliminate<1, 0, true>;
    }
}

static int mode_ctas_of(int m) {
    switch (m) {
        case 2: return mode_ctas(0, 2, false);
        case 5: return mode_ctas(1, 2, false);
        case 6: return mode_ctas(2, 2, false);
        default: return mode_ctas(1, 0, false);
    }
}

// Function attributes and occupancy are per device: one cached record per device ordinal, filled under a lock.
constexpr int MAX_DEVICES = 64;
struct DeviceInfo { bool ready = false; int blocks[N_MODES] = {0}; int sms = 0; };
static DeviceInfo g_dev[MAX_DEVICES];
static std::mutex g_dev_mutex;

// largest cooperative grid of the mode's kernel on the current device
cudaError_t eliminate_grid(int* blocks_out, int o_v, int o_n, int flags) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= MAX_DEVICES) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lk(g_dev_mutex);
    DeviceInfo& d = g_dev[dev];
    if (!d.ready) {
        cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev);
        for (int m = 0; m < N_MODES; m++) {
            const size_t smem = eliminate_smem_bytes(mode_needs_keys(m));
            e = cudaFuncSetAttribute(mode_kernel(m), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            int occ = 0;
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mode_kernel(m), ELIM_THREADS, smem);
            if (e != cudaSuccess) return e;
            if (occ > mode_ctas_of(m)) occ = mode_ctas_of(m);
            if (occ < 1) return cudaErrorLaunchOutOfResources;
            d.blocks[m] = d.sms * occ;
        }
        d.ready = true;
    }
    *blocks_out = d.blocks[mode_index(o_v, o_n, (flags & 1) != 0)];
    return cudaSuccess;
}

int eliminate_max_groups() { return TAB_GROUPS; }
int eliminate_max_blocks() { return TAB_BLOCKS; }

cudaError_t launch_eliminate(const SchurParams* groups_host, int K, int blocks, int o_v, int o_n, int flags,
                             cudaStream_t stream) {
    if (K < 1 || K > TAB_GROUPS || blocks < 1 || blocks > TAB_BLOCKS) return cudaErrorInvalidValue;
    static thread_local GroupTableRaw tab;     // copied into the launch's parameter buffer by the launch call
    for (int g = 0; g < K; g++) tab.g[g] = groups_host[g];
    for (int g = 0; g < K; g++)
        for (int b = 0; b < groups_host[g].gblocks; b++) tab.bg[groups_host[g].gblock0 + b] = (unsigned short)g;
    void* args[] = {(void*)&tab};
    const int m = mode_index(o_v, o_n, (flags & 1) != 0);
    return cudaLaunchCooperativeKernel(mode_kernel(m), dim3(blocks), dim3(ELIM_THREADS), args,
                                       eliminate_smem_bytes(mode_needs_keys(m)), stream);
}

// fold the control blocks of the view groups into the caller-visible one: first error, largest round count,
// summed counters, longest phase times
__global__ void k_combine_groups(int K, const int* gctr, const unsigned long long* gstats, int* ctr,
                                 unsigned long long* stats) {
    const int t = threadIdx.x;
    if (t == 0) {
        int status = 0, rounds = 0;
        for (int g = 0; g < K; g++) {
            const int* c = gctr + (size_t)g * CTR_COUNT;
            if (status == 0) status = c[CTR_STATUS];
            rounds = max(rounds, c[CTR_ROUNDS]);
        }
        ctr[CTR_STATUS] = status;
        ctr[CTR_ROUNDS] = rounds;
    }
    if (t < ST_COUNT) {
        unsigned long long acc = 0;
        for (int g = 0; g < K; g++) {
            const unsigned long long v = gstats[(size_t)g * ST_COUNT + t];
            if (t == ST_MAXSTAR || t >= ST_T_INIT) acc = v > acc ? v : acc; else acc += v;
        }
        stats[t] = acc;
    }
}

cudaError_t launch_combine_groups(int K, const int* gctr, const unsigned long long* gstats, int* ctr,
                                  unsigned long long* stats, cudaStream_t stream) {
    k_combine_groups<<<1, 32, 0, stream>>>(K, gctr, gstats, ctr, stats);
    return cudaGetLastError();
}

}  // namespace rlap
