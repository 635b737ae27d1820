// star.cuh — star staging shared by the elimination and emission kernels: shared-memory buffers,
// sort + multi-edge merge of a staged star, and the register-resident (warp shuffle) variants used
// for stars of at most 32 entries, one star per warp and one entry per lane.
#pragma once
#include "rlap_device.cuh"
#include "schur.cuh"
#include "introsort.cuh"

namespace rlap {

__device__ __forceinline__ void set_status(const SchurParams& P, int code) { atomicCAS(P.ctr + CTR_STATUS, 0, code); }

__device__ __forceinline__ StarBuf cta_buf(uint64_t* smem) {
    StarBuf sb;
    sb.A = smem;
    sb.Q = smem + CAP_CTA;
    sb.K = smem + 2 * CAP_CTA;
    sb.cap = CAP_CTA;
    return sb;
}
__device__ __forceinline__ StarBuf scratch_buf(const SchurParams& P) {
    StarBuf sb;
    sb.A = P.scratch + (size_t)((int)blockIdx.x - P.gblock0) * 3 * (size_t)P.scratch_cap;
    sb.Q = sb.A + P.scratch_cap;
    sb.K = sb.Q + P.scratch_cap;
    sb.cap = P.scratch_cap;
    return sb;
}

// Quantise, pad to a power of two, sort by neighbour and merge multi-edges in place: the first entry
// of every run keeps the summed fixed-point weight (and, if the run has more than one entry, the
// dequantised fp32 weight); the others are marked dead (weight word RLAP_DEAD_W, Q = 0) but keep the
// neighbour id. Returns the number of distinct neighbours; *P2_out = padded length.
// merge the runs of equal neighbour of a star already sorted by A; Q is (re)computed here
template <bool CTA>
__device__ int star_merge_sorted(StarBuf sb, int lraw, int shift, CtaScratch* cs) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    for (int i = r; i < lraw; i += gs) sb.Q[i] = quantize(a_w(sb.A[i]), shift);
    g_sync<CTA>();
    int L = 0;
    if (CTA) {
        if (threadIdx.x == 0) cs->icount = 0;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    for (int base = 0; base < lraw; base += gs) {
        int i = base + r;
        bool act = i < lraw;
        uint64_t a = act ? sb.A[i] : RLAP_PAD_A;
        uint32_t nb = a_nbr(a);
        bool headf = act && (i == 0 || a_nbr(sb.A[i - 1]) != nb);
        unsigned long long qs = 0;
        int c = 0;
        if (headf) {
            int j = i;
            do { qs += sb.Q[j]; c++; j++; } while (j < lraw && a_nbr(sb.A[j]) == nb);
        }
        unsigned m = __ballot_sync(RLAP_FULL_MASK, headf);
        g_sync<CTA>();  // every read of this chunk's runs is done before anything is rewritten
        if (act) {
            if (headf) {
                sb.Q[i] = qs;
                if (c > 1) sb.A[i] = ((uint64_t)nb << 32) | (uint64_t)__float_as_uint(dequantize_merged(qs, shift));
            } else {
                sb.Q[i] = 0;
                sb.A[i] = ((uint64_t)nb << 32) | (uint64_t)RLAP_DEAD_W;
            }
        }
        if (CTA) {
            if (lane == 0 && m) atomicAdd(&cs->icount, __popc(m));
        } else {
            L += __popc(m);
        }
    }
    g_sync<CTA>();
    if (CTA) L = cs->icount;
    g_sync<CTA>();
    return L;
}

template <bool CTA>
__device__ int star_sort_merge(StarBuf sb, int lraw, int shift, CtaScratch* cs, int* P2_out) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    const int P2 = next_pow2(lraw);
    for (int i = r; i < P2; i += gs) {
        if (i >= lraw) { sb.A[i] = RLAP_PAD_A; sb.Q[i] = 0; }
        sb.K[i] = ~0ull;
    }
    g_sync<CTA>();
    g_bitonic_sort_keys<CTA>(sb.A, P2);
    *P2_out = P2;
    return star_merge_sorted<CTA>(sb, lraw, shift, cs);
}

// ---------------------------------------------------------------------------------------------
// o_n = asc / desc: ties among more than 16 merged neighbours (DESIGN.md §3.3, introsort.cuh)
// ---------------------------------------------------------------------------------------------
// The partition loop of libstdc++'s std::sort is run by ONE warp of the group (introsort.cuh: long ranges 32 + 32
// elements per step, short ranges one per lane), out of line: its stacks live in local memory and must not cost the
// persistent kernel registers. Generic pointers: the arrays may be shared memory or the global scratch slot.
struct DeviceWarp {                 // the warp primitives introsort_loop_arrange_warp is written against
    int lane;
    template <class F> __device__ __forceinline__ unsigned ballot(F f) { return __ballot_sync(RLAP_FULL_MASK, f(lane)); }
    template <class F> __device__ __forceinline__ void each(F f) { f(lane); }
    __device__ __forceinline__ void sync() { __syncwarp(); }
};
// all 32 lanes of a warp call: partition passes over long ranges run 32 + 32 elements at a time, short ranges one
// per lane (introsort.cuh)
template <bool DESC, class Key, class Tag>
__device__ __noinline__ void introsort_arrange_warp(Key* key, Tag* tag, int n) {
    DeviceWarp wp;
    wp.lane = (int)(threadIdx.x & 31);
    introsort_loop_arrange_warp<DESC, Key, Tag, DeviceWarp>(wp, key, tag, n);
}

// On entry (after star_sort_merge): A sorted by neighbour with the merged-away duplicates marked dead in place,
// Q the fixed-point weights, K = ~0 everywhere. On return the L live records stand in [0, L) in the arrangement the
// partition loop leaves, K[i] = i for them: the o_n sort that follows (by Q, then K) is the stable sort that
// std::__final_insertion_sort performs, i.e. exactly the order the reference's std::sort produces from the
// id-ordered input (preconditioner.cc:275-303).
// `work`: shared-memory workspace of `work_bytes` for a star that lives in the global scratch slot (the loop then runs
// on a copy of the keys with 16-bit tags instead of moving records through L2), nullptr otherwise.
template <bool CTA, bool DESC>
__device__ void star_tie_order(StarBuf sb, int lraw, int L, int P2, uint64_t* work, int work_bytes) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    if (L < lraw) g_bitonic_sort<CTA, SORT_KEY>(sb, P2);   // K is constant: live records first, by neighbour
    if (work != nullptr && L <= 65535 && (long long)L * 10 <= (long long)work_bytes) {
        uint64_t* wk = work;
        uint16_t* wt = (uint16_t*)(work + L);
        for (int i = r; i < L; i += gs) { wk[i] = sb.Q[i]; wt[i] = (uint16_t)i; }
        g_sync<CTA>();
        if (!CTA || threadIdx.x < 32) introsort_arrange_warp<DESC, uint64_t, uint16_t>(wk, wt, L);
        g_sync<CTA>();
        for (int p = r; p < L; p += gs) sb.K[wt[p]] = (uint64_t)p;
    } else {
        if (!CTA || threadIdx.x < 32) introsort_arrange_warp<DESC, uint64_t, uint64_t>(sb.Q, sb.A, L);
        g_sync<CTA>();
        for (int i = r; i < L; i += gs) sb.K[i] = (uint64_t)i;
    }
    g_sync<CTA>();
}

// Register tile of 32 lanes (one merged neighbour per head lane of `hmask`, in neighbour order, q its fixed-point
// weight): returns the lane's position in the same arrangement (0 for lanes outside hmask). The loop only looks at
// the order and the ties of the weights, so it runs on 8-bit keys (how many of the star's weights are smaller) and
// 8-bit tags in `slot`: 96 bytes of shared memory the warp owns (the tile's own staged fills, consumed by now).
// Warp-collective.
template <bool DESC>
__device__ __noinline__ uint32_t warp_tie_order(unsigned long long q, unsigned hmask, uint8_t* slot) {
    const int lane = threadIdx.x & 31;
    const int L = __popc(hmask);
    const bool live = (hmask >> lane) & 1u;
    const int ci = __popc(hmask & ((1u << lane) - 1u));
    int smaller = 0;
    for (unsigned m = hmask; m; m &= m - 1) {
        const unsigned long long v = __shfl_sync(RLAP_FULL_MASK, q, __ffs(m) - 1);
        smaller += (v < q) ? 1 : 0;
    }
    uint8_t* k8 = slot;
    uint8_t* t8 = slot + 32;
    uint8_t* p8 = slot + 64;
    __syncwarp();
    if (live) { k8[ci] = (uint8_t)smaller; t8[ci] = (uint8_t)ci; }
    __syncwarp();
    DeviceWarp wp;
    wp.lane = lane;
    introsort_loop_arrange_warp<DESC, uint8_t, uint8_t, DeviceWarp>(wp, k8, t8, L);
    __syncwarp();
    if (lane < L) p8[t8[lane]] = (uint8_t)lane;
    __syncwarp();
    return live ? (uint32_t)p8[ci] : 0u;
}

// ---------------------------------------------------------------------------------------------
// register-resident stars: one entry per lane
// ---------------------------------------------------------------------------------------------

// ascending bitonic sort of one 64-bit key per lane across the warp
__device__ __forceinline__ uint64_t warp_sort_u64(uint64_t a) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            uint64_t o = __shfl_xor_sync(RLAP_FULL_MASK, a, j);
            bool take_min = (((lane & j) == 0) == ((lane & k) == 0));
            bool lt = a < o;
            a = (take_min == lt) ? a : o;
        }
    }
    return a;
}

// Merge the runs of equal neighbour of a SORTED register star (a = PAD beyond the entries).
// On return every entry has its fixed-point weight *q, and head lanes hold the merged entry (a with the merged fp32
// weight, *q = summed fixed-point weight, *mult = run length); the other entries are marked dead (weight word
// RLAP_DEAD_W, *q = 0) and keep *mult = 1 (0 for padding). Returns the head mask.
__device__ __forceinline__ unsigned warp_merge_sorted(uint64_t& a, unsigned long long& q, int& shift, int& mult) {
    const int lane = threadIdx.x & 31;
    const bool valid = a != RLAP_PAD_A;
    const uint32_t nb = a_nbr(a);
    const uint32_t pnb = __shfl_up_sync(RLAP_FULL_MASK, nb, 1);
    const bool head = valid && (lane == 0 || pnb != nb);
    const unsigned vmask = __ballot_sync(RLAP_FULL_MASK, valid);
    const unsigned hmask = __ballot_sync(RLAP_FULL_MASK, head);
    q = 0;
    shift = 0;
    mult = valid ? 1 : 0;
    if (vmask == 0) return 0;
    const uint32_t wmaxb = warp_max_u32(valid ? (uint32_t)a : 0u);
    shift = star_shift(__uint_as_float(wmaxb), __popc(vmask));
    q = valid ? quantize(a_w(a), shift) : 0ull;
    if (hmask != vmask) {
        unsigned long long qs = q;
        int cnt = mult;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long oq = __shfl_down_sync(RLAP_FULL_MASK, qs, d);
            int oc = __shfl_down_sync(RLAP_FULL_MASK, cnt, d);
            uint32_t onb = __shfl_down_sync(RLAP_FULL_MASK, nb, d);
            bool ov = (vmask >> ((lane + d) & 31)) & 1u;
            if (valid && lane + d < 32 && ov && onb == nb) { qs += oq; cnt += oc; }
        }
        if (head) {
            q = qs;
            mult = cnt;
            if (cnt > 1) a = ((uint64_t)nb << 32) | (uint64_t)__float_as_uint(dequantize_merged(qs, shift));
        } else if (valid) {
            q = 0;
            a = ((uint64_t)nb << 32) | (uint64_t)RLAP_DEAD_W;
        }
    }
    return hmask;
}

// ascending bitonic sort of (k, t, a) triples, one per lane, with payload q
__device__ __forceinline__ void warp_sort_ktaq(uint64_t& k, uint64_t& t, uint64_t& a, unsigned long long& q) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll
        for (int j = kk >> 1; j > 0; j >>= 1) {
            uint64_t ok = __shfl_xor_sync(RLAP_FULL_MASK, k, j);
            uint64_t ot = __shfl_xor_sync(RLAP_FULL_MASK, t, j);
            uint64_t oa = __shfl_xor_sync(RLAP_FULL_MASK, a, j);
            unsigned long long oq = __shfl_xor_sync(RLAP_FULL_MASK, q, j);
            bool take_min = (((lane & j) == 0) == ((lane & kk) == 0));
            bool lt = (k != ok) ? (k < ok) : ((t != ot) ? (t < ot) : (a < oa));
            bool keep = (take_min == lt);
            k = keep ? k : ok;
            t = keep ? t : ot;
            a = keep ? a : oa;
            q = keep ? q : oq;
        }
    }
}

// first lane index in [0, L) whose C exceeds r (L if none); every lane may ask for a different r
__device__ __forceinline__ int warp_upper_bound(unsigned long long C, int L, unsigned long long r) {
    int lo = 0, hi = L;
#pragma unroll
    for (int it = 0; it < 6; it++) {
        int mid = (lo + hi) >> 1;
        unsigned long long cm = __shfl_sync(RLAP_FULL_MASK, C, mid & 31);
        if (lo < hi) {
            if (cm > r) hi = mid; else lo = mid + 1;
        }
    }
    return lo;
}

// ---------------------------------------------------------------------------------------------
// a warp sorts 32 * R keys held in registers: element e = r * 32 + lane. Compare-exchange partners at
// distance >= 32 live in the same lane (pure register work), closer ones are reached by shuffles.
// No shared memory, no barriers.
// ---------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ void warp_sort_regs(uint64_t (&a)[R]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 2; k <= 32 * R; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int jr = j >> 5;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    if ((r & jr) == 0) {
                        const int r2 = r | jr;
                        const bool up = (((r << 5) & k) == 0);   // lane bits are below k's bit here
                        const uint64_t x = a[r], y = a[r2];
                        const bool sw = up ? (y < x) : (x < y);
                        a[r] = sw ? y : x;
                        a[r2] = sw ? x : y;
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const uint64_t o = __shfl_xor_sync(RLAP_FULL_MASK, a[r], j);
                    const bool up = ((((r << 5) | lane) & k) == 0);
                    const bool take_min = (((lane & j) == 0) == up);
                    const bool lt = a[r] < o;
                    a[r] = (take_min == lt) ? a[r] : o;
                }
            }
        }
    }
}

}  // namespace rlap
