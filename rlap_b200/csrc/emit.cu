// emit.cu — emission (A.5): surviving vertices, multi-edges merged, rows sorted by (col, row).
// Replaces the output assembly of the reference (rlap/csrc/preconditioner.cc:435-457 / 789-810 /
// 916-934: pop every remaining vertex, walk its list, sort, merge, push rows).
//
// No list walking here: the exact live count of every surviving vertex is known (the `live`
// counters the elimination maintains), so every survivor owns a staging segment of `live` slots:
//   k_emit_prep     live counts of survivors            -> scan -> rawoff
//   k_emit_scatter  streams the fill pool: entries with two alive endpoints go to the TAIL of their owner's segment
//   k_emit_fsort    per survivor with at most 32 fill entries: sorts them in place and looks for a multi-edge (two
//                   fills to the same neighbour, or a fill parallel to a base edge). Without one - 99 % of the
//                   survivors - the row count is the live count and nothing else is staged: "clean".
//   the rest (a multi-edge, or more than 32 fills: the hubs) take the merge path: k_emit_base stages their alive
//   base entries at the front of the segment, k_emit_sort_* sort the segment by neighbour and merge multi-edges
//   with the fixed-point rule, in place                  -> scan -> outoff
//   k_emit_write    clean survivors: the alive base entries (streamed from the CSR, ascending) and the sorted fills
//                   are merged by rank straight into the caller's buffers; the others are copied from staging
#include <stdlib.h>
#include <mutex>
#include "rlap_device.cuh"
#include "schur.cuh"
#include "scan.cuh"
#include "star.cuh"

namespace rlap {

// rawcnt / cursor reuse two per-vertex arrays that are dead once the elimination kernel has returned
__device__ __forceinline__ int* rawcnt_of(const SchurParams& P) { return P.blk; }
__device__ __forceinline__ int* cursor_of(const SchurParams& P) { return P.candround; }

// a failed elimination (pool overflow, scratch overflow) leaves reserved-but-unwritten pool slots and inconsistent
// counters behind: the emission kernels do nothing then, the caller only reads the status
__device__ __forceinline__ bool run_failed(const SchurParams& P) { return ldcg_i32(P.ctr + CTR_STATUS) != 0; }

__global__ void k_emit_prep(SchurParams P) {
    const long long VN = (long long)P.V * P.n;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= VN) return;
    if (run_failed(P)) { rawcnt_of(P)[idx] = 0; cursor_of(P)[idx] = 0; P.outcnt[idx] = 0; return; }
    int c = (P.state[idx] != 2) ? *live_p(P, idx) : 0;
    rawcnt_of(P)[idx] = c;
    cursor_of(P)[idx] = 0;
}

// Merge-path segments are listed by size class in dense lists (the low-list buffers of the elimination are free by
// now): a hub-heavy stretch of vertex ids (the old vertices of a preferential-attachment graph) would otherwise hand
// all its big segments to the few warps that own that stretch.
constexpr int CAP_REGS = 512;   // largest segment sorted in registers
constexpr int N_CLASS = 7;
// classes 6, 0..3: at most 32 / 64 / 128 / 256 / 512 entries (register sort, k_emit_sort_mid), 4: at most CAP_CTA
// (k_emit_sort_block), 5: above (k_emit_sort_big, or a scratch slot in k_emit_sort_block)
__host__ __device__ constexpr int size_class(int lv) {
    return lv <= 32 ? 6 : lv <= 64 ? 0 : lv <= 128 ? 1 : lv <= 256 ? 2 : lv <= CAP_REGS ? 3 : lv <= CAP_CTA ? 4 : 5;
}
__device__ __forceinline__ unsigned int* class_list(const SchurParams& P, int c) {
    const size_t VN = (size_t)P.V * (size_t)P.n;
    if (c == 0) return P.wl;
    if (c == 1) return P.wl + VN;
    if (c == 5) return P.dl;
    if (c == 6) return P.low + (size_t)3 * (VN + 16);
    return P.low + (size_t)(c - 2) * (VN + 16);
}
__device__ __forceinline__ int* class_tail(const SchurParams& P, int c) { return P.ctr + CTR_EMIT_C0 + c; }

// Base entries of the survivors on the merge path (cursor == MERGE_PATH): a warp per vertex walks its
// (neighbour-ascending) CSR row and writes the entries whose neighbour is alive to the front of the vertex's staging
// segment, in order and without atomics. The vertices come from the size-class lists k_emit_fsort built (one virtual
// list: the classes back to back) - about 1 % of the survivors, mostly hubs; a sweep over every vertex of every view
// spent 197 M warp instructions (0.35 ms per 64 arxiv views) finding them.
constexpr int MERGE_PATH = -1;
__global__ void __launch_bounds__(256) k_emit_base(SchurParams P) {
    if (run_failed(P)) return;
    const int gw = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nw = (int)(((long long)gridDim.x * blockDim.x) >> 5);
    const int lane = threadIdx.x & 31;
    int tails[N_CLASS], total = 0;
#pragma unroll
    for (int c = 0; c < N_CLASS; c++) { tails[c] = P.ctr[CTR_EMIT_C0 + c]; total += tails[c]; }
    for (int it = gw; it < total; it += nw) {
        int c = 0, r = it;
#pragma unroll
        for (int k = 0; k < N_CLASS - 1; k++) {
            if (c == k && r >= tails[k]) { r -= tails[k]; c = k + 1; }
        }
        const unsigned int idx = class_list(P, c)[r];
        const int v = (int)(idx % (unsigned)P.n);
        const size_t vb = (size_t)idx - (size_t)v;
        const int b = __ldg(P.ptr + v), nb = __ldg(P.ptr + v + 1) - b;
        const long long off = P.rawoff[idx];
        int cnt = 0;
        for (int p0 = 0; p0 < nb; p0 += 32) {
            const int p = p0 + lane;
            int u = 0;
            bool ok = p < nb;
            if (ok) { u = __ldg(P.col + b + p); ok = P.state[vb + u] != 2; }
            const unsigned m = __ballot_sync(RLAP_FULL_MASK, ok);
            if (ok) P.raw[off + cnt + __popc(m & ((1u << lane) - 1u))] = pack_a((uint32_t)u, __ldg(P.w + b + p));
            cnt += __popc(m);
        }
    }
}

// Fill entries: grid-stride over the view's pool (blockIdx.y walks the views), one thread per fill edge = the two
// entries (j <- k), (k <- j) it left in adjacent slots (reservations are even, so pairs never straddle); if both
// endpoints are alive each entry goes to the tail of its owner's staging segment, filled from the end backwards (the
// front is where the alive base entries of a merge-path vertex go; cursor[v] counts the fills of v)
constexpr long long MAX_GRID_Y = 65535;   // CUDA's limit on gridDim.y: a call may have more views
__global__ void __launch_bounds__(256) k_emit_scatter(SchurParams P) {
    if (run_failed(P)) return;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, nt = (long long)gridDim.x * blockDim.x;
    for (int view = blockIdx.y; view < P.V; view += gridDim.y) {
        const size_t vb = (size_t)view * (size_t)P.n;
        long long used = (long long)P.pool_cursor[view];
        if (used > P.pool_cap) used = P.pool_cap;
        const int4* pool = P.pool + (size_t)view * (size_t)P.pool_cap;
        for (long long e = 2 * t0; e + 1 < used; e += 2 * nt) {
            const int4 e0 = __ldcs(pool + e);        // {k, w, next, j}
            if (e0.w < 0) continue;                  // tombstones come in pairs as well
            const int j = e0.w, k = e0.x;
            if (P.state[vb + j] == 2 || P.state[vb + k] == 2) continue;
            const long long p0 = P.rawoff[vb + j + 1] - 1 - atomicAdd(cursor_of(P) + vb + j, 1);
            const long long p1 = P.rawoff[vb + k + 1] - 1 - atomicAdd(cursor_of(P) + vb + k, 1);
            if (p0 >= 0 && p1 >= 0 && p0 < P.raw_cap && p1 < P.raw_cap) {
                P.raw[p0] = ((uint64_t)(uint32_t)k << 32) | (uint64_t)(uint32_t)e0.y;
                P.raw[p1] = ((uint64_t)(uint32_t)j << 32) | (uint64_t)(uint32_t)e0.y;
            } else {
                set_status(P, 6);
            }
        }
    }
}

// sort + merge a staged star (shared memory or scratch) with the whole thread block and write the merged entries back
// to the start of the vertex's raw segment, neighbours ascending
__device__ void emit_sort_staged(const SchurParams& P, size_t idx, StarBuf sb, CtaScratch* cs) {
    const int gs = (int)blockDim.x, r = (int)threadIdx.x, lane = threadIdx.x & 31;
    const int lraw = rawcnt_of(P)[idx];
    const long long off = P.rawoff[idx];
    if (lraw > sb.cap) {
        if (r == 0) { set_status(P, 6); P.outcnt[idx] = 0; }
        __syncthreads();
        return;
    }
    uint32_t wmaxb = 0;
    const int P2 = next_pow2(lraw);
    for (int i = r; i < P2; i += gs) {
        uint64_t a = (i < lraw) ? P.raw[off + i] : RLAP_PAD_A;
        sb.A[i] = a;
        if (i < lraw) wmaxb = max(wmaxb, (uint32_t)a);
    }
    __syncthreads();
    g_bitonic_sort_keys<true>(sb.A, P2);
    // multi-edges are rare among survivors: look for one before paying for the fixed-point merge
    int dup = 0;
    for (int i = r + 1; i < lraw; i += gs) dup |= (a_nbr(sb.A[i]) == a_nbr(sb.A[i - 1]));
    dup = __syncthreads_or(dup);
    int L = lraw;
    if (dup) {
        wmaxb = g_max_u32<true>(wmaxb, cs);
        __syncthreads();
        const int shift = star_shift(__uint_as_float(wmaxb), lraw);
        L = star_merge_sorted<true>(sb, lraw, shift, cs);
    }
    int carry = 0;
    for (int base = 0; base < lraw; base += gs) {
        int i = base + r;
        uint64_t a = (i < lraw) ? sb.A[i] : RLAP_PAD_A;
        bool keep = (i < lraw) && !a_dead(a);
        unsigned m = __ballot_sync(RLAP_FULL_MASK, keep);
        int pos = __popc(m & ((1u << lane) - 1u));
        const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
        __syncthreads();
        if (lane == 0) cs->wsum[w] = (unsigned long long)__popc(m);
        __syncthreads();
        int add = 0, tot = 0;
        for (int k = 0; k < nw; k++) { int c = (int)cs->wsum[k]; if (k < w) add += c; tot += c; }
        pos += add + carry;
        carry += tot;
        if (keep) P.raw[off + pos] = a;
    }
    if (r == 0) P.outcnt[idx] = L;
    __syncthreads();
}

// A warp sorts one segment of up to 32 * R entries in registers (element e = r * 32 + lane), merges the runs of
// equal neighbour with the fixed-point rule (segmented suffix sums over the register tile) and writes the
// merged entries back to the start of the segment, neighbours ascending.
template <int R>
__device__ void emit_sort_regs(const SchurParams& P, size_t idx, int lv, long long off) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    uint64_t a[R];
    uint32_t wmaxb = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int e = r * 32 + lane;
        a[r] = e < lv ? P.raw[off + e] : RLAP_PAD_A;
        if (e < lv) wmaxb = max(wmaxb, (uint32_t)a[r]);
    }
    warp_sort_regs<R>(a);
    // heads of runs
    unsigned headm[R];
    bool anydup = false;
    {
        uint32_t carry = 0xffffffffu;   // neighbour id of element e - 1 for lane 0 (no vertex has this id)
#pragma unroll
        for (int r = 0; r < R; r++) {
            const uint32_t nb = a_nbr(a[r]);
            uint32_t prev = __shfl_up_sync(RLAP_FULL_MASK, nb, 1);
            if (lane == 0) prev = carry;
            const bool valid = a[r] != RLAP_PAD_A;
            const bool head = valid && prev != nb;
            headm[r] = __ballot_sync(RLAP_FULL_MASK, head);
            anydup |= (headm[r] != __ballot_sync(RLAP_FULL_MASK, valid));
            carry = __shfl_sync(RLAP_FULL_MASK, nb, 31);
        }
    }
    if (anydup) {
        wmaxb = warp_max_u32(wmaxb);
        const int shift = star_shift(__uint_as_float(wmaxb), lv);
        unsigned long long qs[R];
#pragma unroll
        for (int r = 0; r < R; r++) qs[r] = (a[r] != RLAP_PAD_A) ? quantize(a_w(a[r]), shift) : 0ull;
        // segmented suffix sums: after the step with distance d, qs(e) covers the run members in [e, e + 2d).
        // Rows are updated in ascending order, in place: a step only reads rows >= r that are still old.
#pragma unroll
        for (int d = 1; d < 32 * R; d <<= 1) {
#pragma unroll
            for (int r = 0; r < R; r++) {
                unsigned long long oq;
                uint32_t onb;
                if (d < 32) {
                    const int src = (lane + d) & 31;
                    unsigned long long q0 = __shfl_sync(RLAP_FULL_MASK, qs[r], src);
                    uint32_t n0 = __shfl_sync(RLAP_FULL_MASK, a_nbr(a[r]), src);
                    unsigned long long q1 = 0;
                    uint32_t n1 = 0xffffffffu;
                    if (r + 1 < R) {
                        q1 = __shfl_sync(RLAP_FULL_MASK, qs[r + 1], src);
                        n1 = __shfl_sync(RLAP_FULL_MASK, a_nbr(a[r + 1]), src);
                    }
                    const bool wrap = lane + d >= 32;
                    oq = wrap ? q1 : q0;
                    onb = wrap ? n1 : n0;
                } else {
                    const int r2 = r + (d >> 5);
                    oq = (r2 < R) ? qs[r2 < R ? r2 : 0] : 0ull;
                    onb = (r2 < R) ? a_nbr(a[r2 < R ? r2 : 0]) : 0xffffffffu;
                }
                if (a[r] != RLAP_PAD_A && onb == a_nbr(a[r])) qs[r] += oq;
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (a[r] == RLAP_PAD_A) continue;
            const bool head = (headm[r] >> lane) & 1u;
            if (!head) {
                a[r] = ((uint64_t)a_nbr(a[r]) << 32) | (uint64_t)RLAP_DEAD_W;
            } else {
                // merged iff the next element (e + 1) exists and is not the head of a run
                const int e1 = r * 32 + lane + 1;
                bool merged = false;
                if (e1 < lv) {
                    const unsigned hm = (lane == 31) ? ((r + 1 < R) ? headm[r + 1 < R ? r + 1 : 0] : 1u) : (headm[r] >> (lane + 1));
                    merged = (hm & 1u) == 0;
                }
                if (merged) a[r] = ((uint64_t)a_nbr(a[r]) << 32) | (uint64_t)__float_as_uint(dequantize_merged(qs[r], shift));
            }
        }
    }
    int rowbase = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        const bool keep = a[r] != RLAP_PAD_A && !a_dead(a[r]);
        if (keep) P.raw[off + rowbase + __popc(headm[r] & lt)] = a[r];
        rowbase += __popc(headm[r]);
    }
    if (lane == 0) P.outcnt[idx] = rowbase;
}

constexpr int CAP_BIG = 12288;   // largest segment sorted in the shared memory of one SM (k_emit_sort_big)

constexpr int FSORT_MAX = 32;    // fills of a clean survivor
constexpr int FS_LANE = 16;      // fills a single lane sorts in its shared-memory slot

// owner of position p among the 32 ascending row starts a warp holds, one per lane: the last lane whose start is <= p
// (rows without entries share the start of their successor and are never chosen)
__device__ __forceinline__ int owner_of(int start, int p) {
    int lo = 0;
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
        const int r = __shfl_sync(RLAP_FULL_MASK, start, (lo + step) & 31);
        if (lo + step < 32 && r <= p) lo += step;
    }
    return lo;
}

constexpr int FS_NB_MAX = 40;    // longest base row a single lane walks

// Every survivor: sort its fill entries (the tail of its staging segment) by neighbour and look for a multi-edge.
// A warp owns 32 consecutive vertices of one view and reads their counts in one go.
//  * at most FS_LANE fills and a base row of at most FS_NB_MAX entries: the vertex is handled by its lane alone (32
//    independent chains of loads per warp): insertion sort in a shared-memory slot (two fills to the same neighbour
//    are a multi-edge), then one merge walk over the neighbour ids of its base row, eight at a time (a fill parallel
//    to a base edge is a multi-edge);
//  * otherwise, up to 32 fills: the warp sorts them in registers, one vertex after the other, and every fill looks
//    its neighbour up in the base row (binary search).
// No multi-edge: the sorted fills go back in place and the survivor is "clean" (its row count is its live count;
// cursor keeps the fill count). Otherwise, or with more than 32 fills, the survivor takes the merge path
// (cursor = MERGE_PATH) and is listed by size class for the sort kernels.
// (Measured alternatives, profiles/README.md: a warp per vertex for everything 1.9 ms; ranking the staged fills of a
// batch with all lanes plus one coalesced sweep of the batch's base rows against per-owner filters 1.5 - 1.7 ms -
// instruction bound on the per-entry owner and fill searches; this version 1.3 ms per 64 arxiv-shaped views.)
__global__ void __launch_bounds__(256) k_emit_fsort(SchurParams P) {
    __shared__ uint64_t s_slot[8][FS_LANE * 32];
    const int nbv = (P.n + 31) >> 5;                     // batches per view
    const long long nbatch = (long long)P.V * nbv;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const bool failed = run_failed(P);
    uint64_t* sl = s_slot[threadIdx.x >> 5] + lane;    // element e of this lane: sl[e * 32]
    for (long long bt = gw; bt < nbatch; bt += nw) {
        const int view = (int)(bt / nbv), v = (int)(bt % nbv) * 32 + lane;
        const bool inr = v < P.n;
        const long long idx = (long long)view * P.n + (inr ? v : P.n - 1);
        int lv = 0, f = 0;
        long long end = 0;
        const int b = __ldg(P.ptr + (inr ? v : P.n)), nb = inr ? __ldg(P.ptr + v + 1) - b : 0;
        if (inr && !failed) {
            lv = rawcnt_of(P)[idx];
            f = cursor_of(P)[idx];
            end = P.rawoff[idx + 1];
        }
        if (inr && (lv == 0 || f == 0)) P.outcnt[idx] = lv;      // eliminated / isolated, or no fills at all: clean
        int cls = (lv > 0 && f > FSORT_MAX) ? size_class(lv) : -1;
        const bool lanepath = lv > 0 && f > 0 && f <= FS_LANE && nb <= FS_NB_MAX;
        if (lanepath) {
            uint64_t* fp = P.raw + (end - f);
#pragma unroll 4
            for (int i = 0; i < f; i++) sl[i * 32] = fp[i];
            bool dup = false;
            for (int i = 1; i < f; i++) {
                const uint64_t x = sl[i * 32];
                int j = i - 1;
                while (j >= 0) {
                    const uint64_t y = sl[j * 32];
                    if (a_nbr(y) <= a_nbr(x)) { dup |= a_nbr(y) == a_nbr(x); break; }
                    sl[(j + 1) * 32] = y;
                    j--;
                }
                sl[(j + 1) * 32] = x;
            }
            if (!dup) {   // a fill parallel to a base edge of the vertex: both lists ascend, one merge walk
                int i = 0;
                uint32_t fn = a_nbr(sl[0]);
                for (int p0 = 0; p0 < nb && i < f; p0 += 8) {
                    uint32_t c8[8];
#pragma unroll
                    for (int k = 0; k < 8; k++) c8[k] = (p0 + k < nb) ? (uint32_t)__ldg(P.col + b + p0 + k) : 0xffffffffu;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        while (i < f && fn < c8[k]) { i++; fn = i < f ? a_nbr(sl[i * 32]) : 0xffffffffu; }
                        if (i < f && fn == c8[k]) dup = true;
                    }
                }
            }
            if (!dup) {
                for (int i = 0; i < f; i++) fp[i] = sl[i * 32];
                P.outcnt[idx] = lv;
            } else {
                cls = size_class(lv);
            }
        }
        __syncwarp();
        unsigned cand = __ballot_sync(RLAP_FULL_MASK, lv > 0 && f > 0 && f <= FSORT_MAX && !lanepath);
        while (cand) {
            const int k = __ffs(cand) - 1;
            cand &= cand - 1;
            const int kf = __shfl_sync(RLAP_FULL_MASK, f, k), kb = __shfl_sync(RLAP_FULL_MASK, b, k);
            const int knb = __shfl_sync(RLAP_FULL_MASK, nb, k);
            const long long kend = __shfl_sync(RLAP_FULL_MASK, end, k);
            uint64_t a = lane < kf ? P.raw[kend - kf + lane] : RLAP_PAD_A;
            a = warp_sort_u64(a);
            const bool valid = a != RLAP_PAD_A;
            const uint32_t nbr = a_nbr(a);
            const uint32_t prev = __shfl_up_sync(RLAP_FULL_MASK, nbr, 1);
            bool d2 = valid && lane > 0 && prev == nbr;                // two fills to the same neighbour
            if (valid) {                                               // a fill parallel to a base edge of the vertex
                int lo = 0, hi = knb;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if ((uint32_t)__ldg(P.col + kb + mid) < nbr) lo = mid + 1; else hi = mid;
                }
                d2 |= lo < knb && (uint32_t)__ldg(P.col + kb + lo) == nbr;
            }
            if (!__any_sync(RLAP_FULL_MASK, d2)) {
                if (valid) P.raw[kend - kf + lane] = a;
                if (lane == k) P.outcnt[idx] = lv;
            } else if (lane == k) {
                cls = size_class(lv);
            }
        }
        // merge path: dense per-class lists, one tail bump per class and warp pass
        if (cls >= 0) cursor_of(P)[idx] = MERGE_PATH;
        if (__any_sync(RLAP_FULL_MASK, cls >= 0)) {
#pragma unroll
            for (int c = 0; c < N_CLASS; c++) {
                const unsigned m = __ballot_sync(RLAP_FULL_MASK, cls == c);
                if (m == 0) continue;
                int pos0 = 0;
                if (lane == __ffs(m) - 1) pos0 = atomicAdd(class_tail(P, c), __popc(m));
                pos0 = __shfl_sync(RLAP_FULL_MASK, pos0, __ffs(m) - 1);
                if (cls == c) class_list(P, c)[pos0 + __popc(m & lt)] = (unsigned int)idx;
            }
        }
        __syncwarp();
    }
}

// segments of at most 512 entries: one warp each, registers only. One kernel per size class (32, 64, 128, 256, 512
// entries = 1, 2, 4, 8, 16 keys per lane) so that the small classes, which hold most segments, run at their own
// register budget.
template <int R>
__global__ void __launch_bounds__(256, (R <= 4 ? 4 : 2)) k_emit_sort_mid(SchurParams P) {
    constexpr int CLS = size_class(32 * R);
    const int gw = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nw = (int)(((long long)gridDim.x * blockDim.x) >> 5);
    const int end = *class_tail(P, CLS);
    const unsigned int* list = class_list(P, CLS);
    for (int it = gw; it < end; it += nw) {
        const unsigned int idx = list[it];
        emit_sort_regs<R>(P, idx, rawcnt_of(P)[idx], P.rawoff[idx]);
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS, 2) k_emit_sort_block(SchurParams P) {
    extern __shared__ __align__(16) uint64_t smem[];
    __shared__ CtaScratch cs;
    const int end = *class_tail(P, 4);
    const unsigned int* list = class_list(P, 4);
    for (int it = (int)blockIdx.x; it < end; it += (int)gridDim.x) {
        emit_sort_staged(P, list[it], cta_buf(smem), &cs);
        __syncthreads();
    }
    // segments beyond the shared memory of an SM: the NSLOT blocks that own a global scratch slot
    if ((int)blockIdx.x < NSLOT) {
        const int end5 = *class_tail(P, 5);
        const unsigned int* list5 = class_list(P, 5);
        for (int it = (int)blockIdx.x; it < end5; it += NSLOT) {
            const unsigned int idx = list5[it];
            if (rawcnt_of(P)[idx] <= CAP_BIG) continue;
            emit_sort_staged(P, idx, scratch_buf(P), &cs);
            __syncthreads();
        }
    }
}

// segments of CAP_CTA + 1 .. CAP_BIG entries (the hubs that survive): one block per SM with most of its shared
// memory as the staging area (keys + fixed-point weights), instead of the global scratch slots
__global__ void __launch_bounds__(BLOCK_THREADS, 1) k_emit_sort_big(SchurParams P) {
    extern __shared__ __align__(16) uint64_t smem[];
    __shared__ CtaScratch cs;
    StarBuf sb;
    sb.A = smem; sb.Q = smem + CAP_BIG; sb.K = sb.Q; sb.cap = CAP_BIG;
    const int end = *class_tail(P, 5);
    const unsigned int* list = class_list(P, 5);
    for (int it = (int)blockIdx.x; it < end; it += (int)gridDim.x) {
        const unsigned int idx = list[it];
        if (rawcnt_of(P)[idx] > CAP_BIG) continue;
        emit_sort_staged(P, idx, sb, &cs);
        __syncthreads();
    }
}

// Final rows. A warp owns 32 consecutive vertices of one view.
//  * clean survivors (no multi-edge) whose sorted fills fit the warp's shared-memory area: their rows are their alive
//    base entries and their fills, merged by rank. The base rows of the 32 vertices are one contiguous stretch of the
//    CSR, which the warp sweeps 32 entries at a time - coalesced, no dependence on the row lengths. An alive base
//    entry goes to (alive base entries of its row before it) + (fills of its owner with a smaller neighbour: a binary
//    search in shared memory), and bumps a per-owner histogram over that fill count; fill i then goes to
//    i + (alive base entries with a smaller neighbour) = i + the histogram's prefix up to i. Nothing is staged or sorted.
//  * clean survivors beyond the area: the warp merges one vertex at a time by rank (shuffle binary searches).
//  * merge-path survivors: copy of the merged staging segment.
constexpr int WF_CAP = 448;                 // staged fills per warp
constexpr int WH_STRIDE = FSORT_MAX + 1;    // histogram bins per vertex: 0 .. fills
constexpr int WR_WARPS = 4;
__global__ void __launch_bounds__(WR_WARPS * 32) k_emit_write(SchurParams P, int* out_row, int* out_col, float* out_w,
                                                              double* out_f64, const int* __restrict__ newid) {
    __shared__ uint64_t s_fill[WR_WARPS][WF_CAP];
    __shared__ int s_hist[WR_WARPS][32 * WH_STRIDE];
    if (run_failed(P)) return;
    const int nbv = (P.n + 31) >> 5;                     // batches per view
    const long long nbatch = (long long)P.V * nbv;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const bool check = (P.flags & 8) != 0;
    uint64_t* sfill = s_fill[threadIdx.x >> 5];
    int* shist = s_hist[threadIdx.x >> 5];
    // newid (optional): compact ids of the view's vertices (rlap_schur_relabel), applied to both ends of every row
    const int* nid = nullptr;
    auto put = [&](long long w, uint32_t r, int c, float wt) {
        if (nid) { r = (uint32_t)__ldg(nid + r); c = __ldg(nid + c); }
        if (out_row) {
            __stcs(out_row + w, (int)r);
            if (out_col) __stcs(out_col + w, c);      // NULL: the caller rebuilds the columns from the column pointers
            if (out_w) __stcs(out_w + w, wt);         // NULL: an unweighted view
        }
        if (out_f64) {
            out_f64[w * 3 + 0] = (double)r;
            out_f64[w * 3 + 1] = (double)c;
            out_f64[w * 3 + 2] = (double)wt;
        }
    };
    auto mismatch = [&](long long vidx, int got, int want) {   // RLAP_FLAG_CHECK_LIVE: alive base entries + fills must be the live count
        atomicAdd(P.stats + 7, 1ull);
        atomicMax(P.stats + 6, ((unsigned long long)(unsigned)vidx << 32) | ((unsigned long long)(unsigned)(got & 0xffff) << 16) | (unsigned)(want & 0xffff));
    };
    for (long long bt = gw; bt < nbatch; bt += nw) {
        const int view = (int)(bt / nbv), v = (int)(bt % nbv) * 32 + lane;
        const bool inr = v < P.n;
        const long long idx = (long long)view * P.n + (inr ? v : P.n - 1);
        const size_t vb = (size_t)view * (size_t)P.n;
        nid = newid ? newid + vb : nullptr;
        const int b = __ldg(P.ptr + (inr ? v : P.n)), nb = inr ? __ldg(P.ptr + v + 1) - b : 0;
        int L = 0, f = 0;
        long long dst = 0, src = 0, end = 0;
        if (inr) {
            L = P.outcnt[idx];
            f = cursor_of(P)[idx];
            dst = P.outoff[idx];
            src = P.rawoff[idx];
            end = P.rawoff[idx + 1];
        }
        if (!__any_sync(RLAP_FULL_MASK, L > 0)) continue;
        // ---- flat tier: clean survivors, as many as the fill area holds (in lane order)
        const bool clean = L > 0 && f != MERGE_PATH;
        int foff = clean ? f : 0;    // exclusive prefix of the fill counts of the clean survivors
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(RLAP_FULL_MASK, foff, d);
            if (lane >= d) foff += t;
        }
        const bool flat = clean && foff <= WF_CAP;      // foff is still inclusive here
        foff -= clean ? f : 0;
        const int ff = flat ? f : 0;
        const int ftot = __reduce_max_sync(RLAP_FULL_MASK, flat ? foff + f : 0);
        // fills of the flat survivors -> shared memory, all lanes busy whatever the split between vertices
        for (int t0 = 0; t0 < ftot; t0 += 32) {      // uniform trip count: the searches are warp-wide shuffles
            const int t = t0 + lane;
            // owner of staged fill t: the last lane whose prefix is <= t (a lane that stages nothing shares the prefix of
            // its successor, and the search resolves equals to the last one)
            int lo = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const int r = __shfl_sync(RLAP_FULL_MASK, foff, (lo + step) & 31);
                if (lo + step < 32 && r <= t) lo += step;
            }
            const long long oend = __shfl_sync(RLAP_FULL_MASK, end, lo);
            const int of = __shfl_sync(RLAP_FULL_MASK, ff, lo), oo = __shfl_sync(RLAP_FULL_MASK, foff, lo);
            if (t < ftot) sfill[t] = __ldcs((const unsigned long long*)P.raw + (oend - of + (t - oo)));
        }
        for (int t = lane; t < 32 * WH_STRIDE; t += 32) shist[t] = 0;
        __syncwarp();
        if (__any_sync(RLAP_FULL_MASK, flat)) {
            const int p_begin = __shfl_sync(RLAP_FULL_MASK, b, 0);
            const int p_end = __shfl_sync(RLAP_FULL_MASK, b + nb, 31);
            int run = 0;       // alive base entries of flat survivors seen so far
            int rs = 0;        // value of `run` at the start of this lane's row
            // Software pipeline over the steps of the sweep: the ids / weights of step s + 2 and the state look-ups of
            // step s + 1 are in flight while step s is ranked and written (the look-up needs the id: two round trips
            // per step otherwise, exposed 14 times per batch).
            uint32_t c2 = 0xffffffffu, c1 = 0xffffffffu;   // ids of the steps two / one ahead
            float w2 = 0.f, w1 = 0.f;
            int o1 = 0;
            bool al1 = false;                             // owner and liveness of the step one ahead
            auto load_cw = [&](int p0, uint32_t& c, float& w) {
                const int p = p0 + lane;
                c = 0xffffffffu; w = 0.f;
                if (p < p_end) { c = (uint32_t)__ldg(P.col + p); w = __ldg(P.w + p); }
            };
            auto look_up = [&](int p0, uint32_t c, int& o, bool& alive) {
                const int p = p0 + lane;
                o = owner_of(b, p);
                const bool oflat = __shfl_sync(RLAP_FULL_MASK, (int)flat, o) != 0;
                alive = p < p_end && oflat && P.state[vb + c] != 2;
            };
            load_cw(p_begin, c1, w1);
            load_cw(p_begin + 32, c2, w2);
            look_up(p_begin, c1, o1, al1);
            for (int p0 = p_begin; p0 < p_end; p0 += 32) {
                const uint32_t c = c1;
                const float w = w1;
                const int o = o1;
                const bool alive = al1;
                c1 = c2; w1 = w2;
                load_cw(p0 + 64, c2, w2);
                look_up(p0 + 32, c1, o1, al1);
                const unsigned mask = __ballot_sync(RLAP_FULL_MASK, alive);
                // rows that start inside this step note how many alive entries came before them
                if (b >= p0 && b < p0 + 32) rs = run + __popc(mask & ((1u << (b - p0)) - 1u));
                const int ors = __shfl_sync(RLAP_FULL_MASK, rs, o);
                const int of = __shfl_sync(RLAP_FULL_MASK, ff, o), oo = __shfl_sync(RLAP_FULL_MASK, foff, o);
                const long long odst = __shfl_sync(RLAP_FULL_MASK, dst, o);
                if (alive) {
                    int lo = 0, hi = of;     // fills of the owner with a smaller neighbour
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if (a_nbr(sfill[oo + mid]) < c) lo = mid + 1; else hi = mid;
                    }
                    put(odst + (run + __popc(mask & lt) - ors) + lo, c, (int)(bt % nbv) * 32 + o, w);
                    atomicAdd(shist + o * WH_STRIDE + lo, 1);
                }
                run += __popc(mask);
            }
            __syncwarp();
            // prefix of every owner's histogram: entry i = alive base entries with fewer than or exactly i smaller fills,
            // i.e. the base entries that precede fill i
            if (flat) {
                int acc = 0;
                for (int i = 0; i <= f; i++) { acc += shist[lane * WH_STRIDE + i]; shist[lane * WH_STRIDE + i] = acc; }
                if (check && acc + f != L) mismatch(idx, acc + f, L);
            }
            __syncwarp();
            for (int t0 = 0; t0 < ftot; t0 += 32) {
                const int t = t0 + lane;
                int lo = 0;
#pragma unroll
                for (int step = 16; step > 0; step >>= 1) {
                    const int r = __shfl_sync(RLAP_FULL_MASK, foff, (lo + step) & 31);
                    if (lo + step < 32 && r <= t) lo += step;
                }
                const int oo = __shfl_sync(RLAP_FULL_MASK, foff, lo);
                const long long odst = __shfl_sync(RLAP_FULL_MASK, dst, lo);
                if (t < ftot) {
                    const int i = t - oo;
                    const uint64_t a = sfill[t];
                    put(odst + i + shist[lo * WH_STRIDE + i], a_nbr(a), (int)(bt % nbv) * 32 + lo, a_w(a));
                }
            }
            __syncwarp();
        }
        // ---- cooperative tier: the survivors the flat sweep did not take
        unsigned todo = __ballot_sync(RLAP_FULL_MASK, L > 0 && !flat);
        while (todo) {
            const int k = __ffs(todo) - 1;
            todo &= todo - 1;
            const int kL = __shfl_sync(RLAP_FULL_MASK, L, k), kf = __shfl_sync(RLAP_FULL_MASK, f, k);
            const int kv = (int)(bt % nbv) * 32 + k;
            const long long kdst = __shfl_sync(RLAP_FULL_MASK, dst, k);
            if (kf == MERGE_PATH) {
                const long long ksrc = __shfl_sync(RLAP_FULL_MASK, src, k);
                for (int o = lane; o < kL; o += 32) {
                    const uint64_t a = __ldcs((const unsigned long long*)P.raw + ksrc + o);
                    put(kdst + o, a_nbr(a), kv, a_w(a));
                }
                continue;
            }
            const int kb = __shfl_sync(RLAP_FULL_MASK, b, k), knb = __shfl_sync(RLAP_FULL_MASK, nb, k);
            const long long kend = __shfl_sync(RLAP_FULL_MASK, end, k);
            // sorted fills, one per lane; a lane without one holds the largest id, so it never counts as "smaller"
            const uint64_t fa = lane < kf ? __ldcs((const unsigned long long*)P.raw + kend - kf + lane) : RLAP_PAD_A;
            const uint32_t fnbr = a_nbr(fa);
            int cb = 0;     // alive base entries with a smaller neighbour than this lane's fill
            int run = 0;    // alive base entries of the chunks done so far
            for (int p0 = 0; p0 < knb; p0 += 32) {
                const int p = p0 + lane;
                uint32_t c = 0xffffffffu;
                float w = 0.f;
                bool alive = false;
                if (p < knb) {
                    c = (uint32_t)__ldg(P.col + kb + p);
                    w = __ldg(P.w + kb + p);
                    alive = P.state[vb + c] != 2;
                }
                const unsigned mask = __ballot_sync(RLAP_FULL_MASK, alive);
                // fills with a smaller neighbour than this lane's base entry
                int lo = 0, hi = kf;
#pragma unroll
                for (int it = 0; it < 6; it++) {
                    const int mid = (lo + hi) >> 1;
                    const uint32_t fm = __shfl_sync(RLAP_FULL_MASK, fnbr, mid & 31);
                    if (lo < hi) { if (fm < c) lo = mid + 1; else hi = mid; }
                }
                if (alive) put(kdst + run + __popc(mask & lt) + lo, c, kv, w);
                // base entries of this chunk with a smaller neighbour than this lane's fill (the chunk is ascending)
                int lo2 = 0, hi2 = 32;
#pragma unroll
                for (int it = 0; it < 6; it++) {
                    const int mid = (lo2 + hi2) >> 1;
                    const uint32_t cm = __shfl_sync(RLAP_FULL_MASK, c, mid & 31);
                    if (lo2 < hi2) { if (cm < fnbr) lo2 = mid + 1; else hi2 = mid; }
                }
                cb += __popc(mask & (lo2 >= 32 ? 0xffffffffu : ((1u << lo2) - 1u)));
                run += __popc(mask);
            }
            if (lane < kf) put(kdst + lane + cb, fnbr, kv, a_w(fa));
            if (check && lane == 0 && run + kf != kL) mismatch((long long)view * P.n + kv, run + kf, kL);
        }
    }
}

// ---- survivor compaction + relabelling (the step the reference's adapters run after the op: torch.unique of the
// output's node ids + subgraph(relabel_nodes=True), scripts/augmentor_benchmarks.py:149-155, rlap_vc_spectral.py:43-51)
// newid[view * n + v] = rank of v among the vertices of the view that have at least one row, -1 for the others
__global__ void k_relabel_flags(SchurParams P) {
    const long long VN = (long long)P.V * P.n;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < VN) rawcnt_of(P)[idx] = P.outcnt[idx] > 0 ? 1 : 0;
}
__global__ void k_relabel_base(const int* scan, long long n, long long V, long long* base) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v <= V) base[v] = scan[v * n];
}
__global__ void k_relabel_final(SchurParams P, int* newid, const long long* base, long long* view_nodes) {
    const long long VN = (long long)P.V * P.n;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < VN) {
        const long long view = idx / P.n;
        newid[idx] = rawcnt_of(P)[idx] ? (int)(newid[idx] - base[view]) : -1;
    }
    if (view_nodes && idx < P.V) view_nodes[idx] = base[idx + 1] - base[idx];
}

cudaError_t launch_relabel(const SchurParams& P, int* newid, long long* base_dev, long long* view_nodes, cudaStream_t stream) {
    const long long VN = (long long)P.V * P.n;
    k_relabel_flags<<<(unsigned)((VN + 255) / 256), 256, 0, stream>>>(P);
    cudaError_t e = launch_exclusive_scan<int>(P.blk, VN, newid, P.blocksum, nullptr, stream);
    if (e != cudaSuccess) return e;
    k_relabel_base<<<(unsigned)((P.V + 1 + 127) / 128), 128, 0, stream>>>(newid, P.n, P.V, base_dev);
    k_relabel_final<<<(unsigned)((VN + 255) / 256), 256, 0, stream>>>(P, newid, base_dev, view_nodes);
    return cudaGetLastError();
}

// column pointers of every view: colptr[view * (n + 1) + v] = rows of `view` that precede column v (v = n: all rows)
__global__ void k_emit_colptr(SchurParams P, int* colptr) {
    const long long VN1 = (long long)P.V * (P.n + 1);
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= VN1) return;
    const long long view = t / (P.n + 1), v = t % (P.n + 1);
    colptr[t] = (int)(P.outoff[view * P.n + v] - P.outoff[view * P.n]);
}

// ---------------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------------

// -DRLAP_DEBUG with RLAP_DEBUG_SYNC=1: synchronise after every emission kernel and name the one that failed
#ifdef RLAP_DEBUG
#include <stdio.h>
#define DBG_SYNC(name)                                                                        \
    do {                                                                                      \
        if (getenv("RLAP_DEBUG_SYNC")) {                                                      \
            cudaError_t _de = cudaStreamSynchronize(stream);                                  \
            if (_de != cudaSuccess) { fprintf(stderr, "rlap debug: %s failed: %s\n", name, cudaGetErrorString(_de)); return _de; } \
        }                                                                                     \
    } while (0)
#else
#define DBG_SYNC(name) do {} while (0)
#endif

// aux[0..5] / aux_ev[0..6]: side streams and events of the calling thread and device (api.cu). The seven sort kernels of
// the merge path work on disjoint lists of a few hundred to a few thousand segments each - small, latency-bound
// launches: forked onto the side streams they overlap instead of queueing behind one another.
cudaError_t launch_emit_count(const SchurParams& P, long long* total_dev, cudaStream_t stream, cudaStream_t* aux,
                              cudaEvent_t* aux_ev) {
    const size_t smem = (size_t)3 * CAP_CTA * sizeof(uint64_t);
    const size_t smem_big = (size_t)2 * CAP_BIG * sizeof(uint64_t);
    {
        static std::mutex mu;
        static PerDeviceOnce once;
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(mu);
        if (once.first(dev)) {
            cudaFuncSetAttribute(k_emit_sort_block, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            cudaFuncSetAttribute(k_emit_sort_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big);
        }
    }
    const long long VN = (long long)P.V * P.n;
    cudaError_t e = cudaMemsetAsync(P.ctr + CTR_EMIT_C0, 0, N_CLASS * sizeof(int), stream);
    if (e != cudaSuccess) return e;
    k_emit_prep<<<(unsigned)((VN + 255) / 256), 256, 0, stream>>>(P);
    DBG_SYNC("k_emit_prep");
    e = launch_exclusive_scan<long long>(P.blk, VN, P.rawoff, P.blocksum, nullptr, stream);
    if (e != cudaSuccess) return e;
    {
        long long work = P.pool_cap / 2;
        long long bx = (work + 256 * 4 - 1) / (256 * 4);
        if (bx < 1) bx = 1;
        if (bx > 148 * 8) bx = 148 * 8;
        const long long by = P.V < MAX_GRID_Y ? P.V : MAX_GRID_Y;
        k_emit_scatter<<<dim3((unsigned)bx, (unsigned)by), 256, 0, stream>>>(P);
        DBG_SYNC("k_emit_scatter");
        bx = ((long long)P.V * ((P.n + 31) / 32) + 7) / 8;   // one warp per 32 vertices of a view
        if (bx < 1) bx = 1;
        if (bx > 148 * 16) bx = 148 * 16;
        k_emit_fsort<<<(unsigned)bx, 256, 0, stream>>>(P);
        DBG_SYNC("k_emit_fsort");
        k_emit_base<<<148 * 8, 256, 0, stream>>>(P);   // list driven: a warp per merge-path vertex
        DBG_SYNC("k_emit_base");
    }
    int blocks = 296;   // two 512-thread blocks per SM
    {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) blocks = 2 * sms;
    }
    e = cudaEventRecord(aux_ev[6], stream);           // fork: the lists and the staged base entries are complete
    if (e != cudaSuccess) return e;
    for (int i = 0; i < 6; i++) {
        e = cudaStreamWaitEvent(aux[i], aux_ev[6], 0);
        if (e != cudaSuccess) return e;
    }
    k_emit_sort_mid<1><<<148 * 4, 256, 0, stream>>>(P);
    k_emit_sort_mid<2><<<148 * 4, 256, 0, aux[0]>>>(P);
    k_emit_sort_mid<4><<<148 * 4, 256, 0, aux[1]>>>(P);
    k_emit_sort_mid<8><<<148 * 2, 256, 0, aux[2]>>>(P);
    k_emit_sort_mid<16><<<148 * 2, 256, 0, aux[3]>>>(P);
    k_emit_sort_block<<<blocks / 2, BLOCK_THREADS, smem, aux[4]>>>(P);
    k_emit_sort_big<<<blocks / 4, BLOCK_THREADS, smem_big, aux[5]>>>(P);
    for (int i = 0; i < 6; i++) {                     // join
        e = cudaEventRecord(aux_ev[i], aux[i]);
        if (e != cudaSuccess) return e;
        e = cudaStreamWaitEvent(stream, aux_ev[i], 0);
        if (e != cudaSuccess) return e;
    }
    DBG_SYNC("k_emit_sort_*");
    return launch_exclusive_scan<long long>(P.outcnt, VN, P.outoff, P.blocksum, total_dev, stream);
}

cudaError_t launch_emit_colptr(const SchurParams& P, int* colptr, cudaStream_t stream) {
    const long long VN1 = (long long)P.V * (P.n + 1);
    k_emit_colptr<<<(unsigned)((VN1 + 255) / 256), 256, 0, stream>>>(P, colptr);
    return cudaGetLastError();
}

cudaError_t launch_emit_write(const SchurParams& P, int* out_row, int* out_col, float* out_w, double* out_f64,
                              const int* newid, cudaStream_t stream) {
    long long bx = ((long long)P.V * ((P.n + 31) / 32) + WR_WARPS - 1) / WR_WARPS;  // one warp per 32 vertices of a view
    if (bx < 1) bx = 1;
    if (bx > 148 * 32) bx = 148 * 32;
    k_emit_write<<<(unsigned)bx, WR_WARPS * 32, 0, stream>>>(P, out_row, out_col, out_w, out_f64, newid);
    DBG_SYNC("k_emit_write");
    return cudaGetLastError();
}

}  // namespace rlap
