// rlap_device.cuh — device-side building blocks shared by the rLap kernels (sm_100a).
//
// Everything here is the GPU half of the "keyed" specification in DESIGN.md §3: counter-based
// randomness (Philox4x32-10), 64-bit fixed-point star arithmetic (order-independent sums) and
// group-cooperative (warp or CTA) sort / scan over a star staged in shared (or global) memory.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rlap {

#define RLAP_FULL_MASK 0xffffffffu

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11)
// ---------------------------------------------------------------------------------------------
enum { TAG_ORDER = 1, TAG_STAR = 2, TAG_PICK = 3 };

__device__ __forceinline__ uint4 philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2,
                                               uint32_t c3) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}

// o_v = random: keyed pseudo-random permutation of a graph's vertices (8-round balanced Feistel
// network, cycle-walked into [0, n_g)). Stands in for std::shuffle + pop (preconditioner.cc:588-613).
struct RankPerm {
    uint32_t rk[8];
    uint32_t hb, mask, ng;
    __device__ __forceinline__ void init(uint32_t k0, uint32_t k1, uint32_t graph, uint32_t view, uint32_t n_g) {
        uint4 a = philox4x32_10(k0, k1, graph, 0u, view, TAG_ORDER);
        uint4 b = philox4x32_10(k0, k1, graph, 1u, view, TAG_ORDER);
        rk[0] = a.x; rk[1] = a.y; rk[2] = a.z; rk[3] = a.w;
        rk[4] = b.x; rk[5] = b.y; rk[6] = b.z; rk[7] = b.w;
        uint32_t bits = 2;
        while (bits < 32 && ((unsigned long long)1 << bits) < (unsigned long long)n_g) bits += 2;
        hb = bits / 2;
        mask = (hb >= 32) ? 0xffffffffu : ((1u << hb) - 1u);
        ng = n_g;
    }
    __device__ __forceinline__ uint32_t perm(uint32_t x) const {
        uint32_t L = x >> hb, R = x & mask;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            uint32_t t = fmix32(R * 0x9E3779B1u + rk[r]) & mask;
            uint32_t nr = L ^ t;
            L = R; R = nr;
        }
        return (L << hb) | R;
    }
    __device__ __forceinline__ uint32_t rank(uint32_t local) const {
        uint32_t x = local;
        do { x = perm(x); } while (x >= ng);
        return x;
    }
};

// ---------------------------------------------------------------------------------------------
// fixed-point star arithmetic
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int ceil_log2_i(int x) { return x <= 1 ? 0 : 32 - __clz(x - 1); }

__device__ __forceinline__ double pow2d(int e) {  // exact 2^e for -1022 <= e <= 1023
    return __hiloint2double((1023 + e) << 20, 0);
}
// shift for a star with `lraw` raw entries and largest weight wmax (> 0): the sum of all
// q = rint(w * 2^shift) stays below 2^62.
__device__ __forceinline__ int star_shift(float wmax, int lraw) {
    int ex;
    frexp((double)wmax, &ex);  // wmax = f * 2^ex, f in [0.5, 1)
    return 62 - ceil_log2_i(lraw) - ex;
}
__device__ __forceinline__ unsigned long long quantize(float w, int shift) {
    return __double2ull_rn(__dmul_rn((double)w, pow2d(shift)));
}
__device__ __forceinline__ float dequantize(unsigned long long q, int shift) {
    return __double2float_rn(__dmul_rn(__ull2double_rn(q), pow2d(-shift)));
}

// fp32 weight of a merged multi-edge. Never zero: with a dynamic range beyond 2^38 inside one star the sum could
// round to 0 on one endpoint's side only and the edge would lose one direction at the next ingest (zero weights
// are dropped, reader.cc:50); the smallest positive float keeps both directions.
__device__ __forceinline__ float dequantize_merged(unsigned long long q, int shift) {
    float w = dequantize(q, shift);
    return w > 0.f ? w : __uint_as_float(1u);
}

__device__ __forceinline__ uint64_t pack_a(uint32_t nbr, float w) {
    return ((uint64_t)nbr << 32) | (uint64_t)__float_as_uint(w);
}
__device__ __forceinline__ uint32_t a_nbr(uint64_t a) { return (uint32_t)(a >> 32); }
__device__ __forceinline__ float a_w(uint64_t a) { return __uint_as_float((uint32_t)a); }
#define RLAP_DEAD_W 0xffffffffu                   // low word of a merged-away duplicate (a NaN pattern)
#define RLAP_PAD_A 0xffffffffffffffffull          // padding entry
__device__ __forceinline__ bool a_dead(uint64_t a) { return (uint32_t)a == RLAP_DEAD_W; }

// ---------------------------------------------------------------------------------------------
// group abstraction: a "group" is one warp (CTA = false) or the whole thread block (CTA = true)
// ---------------------------------------------------------------------------------------------
template <bool CTA> __device__ __forceinline__ int g_rank() { return CTA ? (int)threadIdx.x : (int)(threadIdx.x & 31); }
template <bool CTA> __device__ __forceinline__ int g_size() { return CTA ? (int)blockDim.x : 32; }
template <bool CTA> __device__ __forceinline__ void g_sync() {
    if (CTA) __syncthreads(); else __syncwarp();
}

// star staging area: three 64-bit arrays of `cap` entries each (shared memory, or global scratch)
struct StarBuf {
    uint64_t* A;   // (nbr << 32) | weight bits   [dead duplicates: low word = RLAP_DEAD_W]
    uint64_t* Q;   // fixed-point weight
    uint64_t* K;   // sort key (o_n = random) / cumulative sums
    int cap;
};

// block-level scratch used by the CTA-group reductions / scans
struct CtaScratch {
    unsigned long long wsum[32];
    unsigned long long carry;
    int icount;
};

__device__ __forceinline__ unsigned long long warp_incl_scan_u64(unsigned long long v) {
    int lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(RLAP_FULL_MASK, v, d);
        if (lane >= d) v += t;
    }
    return v;
}
__device__ __forceinline__ uint32_t warp_max_u32(uint32_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = max(v, __shfl_xor_sync(RLAP_FULL_MASK, v, d));
    return v;
}

// group-wide max of a uint32 (all threads of the group must call; result valid in all)
template <bool CTA>
__device__ __forceinline__ uint32_t g_max_u32(uint32_t v, CtaScratch* cs) {
    v = warp_max_u32(v);
    if (!CTA) return v;
    int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) cs->wsum[w] = v;
    __syncthreads();
    uint32_t r = (lane < nw) ? (uint32_t)cs->wsum[lane] : 0u;
    r = warp_max_u32(r);
    return r;
}

// In-place inclusive scan of src[0..len) into dst[0..len) (dst may alias src). Group cooperative.
template <bool CTA>
__device__ __forceinline__ void g_incl_scan_u64(const uint64_t* src, uint64_t* dst, int len, CtaScratch* cs) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    unsigned long long carry = 0;
    for (int base = 0; base < len; base += gs) {
        int i = base + r;
        unsigned long long v = (i < len) ? src[i] : 0ull;
        unsigned long long s = warp_incl_scan_u64(v);
        if (CTA) {
            int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
            __syncthreads();
            if (lane == 31) cs->wsum[w] = s;
            __syncthreads();
            unsigned long long add = 0;
            for (int k = 0; k < w; k++) add += cs->wsum[k];
            unsigned long long tot = 0;
            for (int k = 0; k < nw; k++) tot += cs->wsum[k];
            s += add + carry;
            carry += tot;
        } else {
            s += carry;
            carry = __shfl_sync(RLAP_FULL_MASK, s, 31);
        }
        if (i < len) dst[i] = s;
    }
    g_sync<CTA>();
}

// ---------------------------------------------------------------------------------------------
// group-cooperative bitonic sort of the star records (A, Q, K move together)
// ---------------------------------------------------------------------------------------------
enum { SORT_BY_A = 0, SORT_ASC = 1, SORT_DESC = 2, SORT_KEY = 3 };

template <int MODE>
__device__ __forceinline__ bool rec_less(uint64_t a1, uint64_t q1, uint64_t k1, uint64_t a2, uint64_t q2, uint64_t k2) {
    if (MODE == SORT_BY_A) return a1 < a2;
    // live entries first; dead duplicates and padding (both have low word 0xffffffff) last
    bool d1 = a_dead(a1), d2 = a_dead(a2);
    if (d1 != d2) return d2;
    if (d1) return a1 < a2;
    // asc / desc: ties by the secondary key K (equal for all entries of a star with <= 16 neighbours, above that the
    // position std::sort's partition loop leaves the entry at: star_tie_order, DESIGN.md §3.3), then by neighbour id
    if (MODE == SORT_ASC && q1 != q2) return q1 < q2;
    if (MODE == SORT_DESC && q1 != q2) return q1 > q2;
    return (k1 != k2) ? (k1 < k2) : (a1 < a2);
}

// P = power of two >= number of records; records [len, P) must be padding (A = RLAP_PAD_A).
template <bool CTA, int MODE>
__device__ __forceinline__ void g_bitonic_sort(StarBuf sb, int P) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = r; t < (P >> 1); t += gs) {
                // t-th compare-exchange pair of this stage: i has bit j clear
                int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                int l = i | j;
                bool up = ((i & k) == 0);
                uint64_t a1 = sb.A[i], a2 = sb.A[l], q1 = sb.Q[i], q2 = sb.Q[l];
                uint64_t k1 = (MODE != SORT_BY_A) ? sb.K[i] : 0, k2 = (MODE != SORT_BY_A) ? sb.K[l] : 0;
                bool sw = up ? rec_less<MODE>(a2, q2, k2, a1, q1, k1) : rec_less<MODE>(a1, q1, k1, a2, q2, k2);
                if (sw) {
                    sb.A[i] = a2; sb.A[l] = a1; sb.Q[i] = q2; sb.Q[l] = q1;
                    if (MODE != SORT_BY_A) { sb.K[i] = k2; sb.K[l] = k1; }
                }
            }
            g_sync<CTA>();
        }
    }
}

// key-only variant: sorts A ascending, nothing else moves
template <bool CTA>
__device__ __forceinline__ void g_bitonic_sort_keys(uint64_t* A, int P) {
    const int gs = g_size<CTA>(), r = g_rank<CTA>();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = r; t < (P >> 1); t += gs) {
                int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                int l = i | j;
                bool up = ((i & k) == 0);
                uint64_t a1 = A[i], a2 = A[l];
                if (up ? (a2 < a1) : (a1 < a2)) { A[i] = a2; A[l] = a1; }
            }
            g_sync<CTA>();
        }
    }
}

__device__ __forceinline__ int next_pow2(int x) { return x <= 1 ? 1 : 1 << (32 - __clz(x - 1)); }

// first index in C[0..len) with C[idx] > r  (len if none)
__device__ __forceinline__ int upper_bound_u64(const uint64_t* C, int len, unsigned long long r) {
    int lo = 0, hi = len;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (C[mid] > r) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// cache-global (L2) loads for arrays that other SMs mutate during a persistent kernel
__device__ __forceinline__ int ldcg_i32(const int* p) { return __ldcg(p); }
__device__ __forceinline__ uint8_t ldcg_u8(const uint8_t* p) { return __ldcg(p); }

}  // namespace rlap
