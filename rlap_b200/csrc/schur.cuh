// schur.cuh — parameter block shared by the elimination / emission kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rlap {

// tiers: a star with at most CAP_WARP raw live entries is handled by one warp in shared memory,
// up to CAP_CTA by one thread block in shared memory (the block's warp buffers overlaid), larger
// ones by one thread block in its global-memory scratch slot (up to scratch_cap).
constexpr int BLOCK_THREADS = 512;
constexpr int WARPS_PER_BLOCK = BLOCK_THREADS / 32;
constexpr int CAP_WARP = 128;
constexpr int CAP_CTA = CAP_WARP * WARPS_PER_BLOCK;  // 2048
constexpr int SEL_BLOCK = 1024;                       // ids per block of the truncation search
// the elimination kernel runs smaller blocks than the streaming kernels: four 256-thread blocks per SM, i.e. the blocks
// of four different view groups, so that a group waiting at its barrier leaves the SM to three others
#ifndef RLAP_ELIM_THREADS
#define RLAP_ELIM_THREADS 256
#endif
constexpr int ELIM_THREADS = RLAP_ELIM_THREADS;
constexpr int ELIM_WARPS = ELIM_THREADS / 32;
#ifndef RLAP_ELIM_CTAS
#define RLAP_ELIM_CTAS (1024 / RLAP_ELIM_THREADS)
#endif
constexpr int ELIM_CTAS_PER_SM = RLAP_ELIM_CTAS;
constexpr int ELIM_CAP_CTA = CAP_WARP * ELIM_WARPS;   // largest star one block of the elimination kernel holds in shared memory

constexpr int STAGE_CAP = 128;                        // staged fill-list entries per lane (shared-memory path of the warps)
constexpr int HUB_DEG = 64;                           // input entries from which a vertex gets HUB_HEADS fill lists (o_v = random)
constexpr int HUB_HEADS = 32;
constexpr int NSLOT = 8;                              // blocks that own a global scratch slot

// Work lists are append-only over the whole run. Items appended during round r land at
// base + atomicAdd(ctr[CTR_WCNT0 + r % 3]); the base is a value every block knows, and a counter
// is only read after the grid barrier that ends its round and reset two rounds later, so no block
// ever reads a count that another block may still be bumping.
enum {
    CTR_WCNT0 = 0,       // work-list appends, rotating by round % 3
    CTR_DCNT0 = 3,       // deferred (big star) appends, rotating by round % 3
    CTR_STATUS = 6,      // first error seen by a kernel (rlap_status)
    CTR_ACTIVE0 = 7,     // degree mode: any segment still active, by round parity
    CTR_ACTIVE1 = 8,
    CTR_OVF0 = 9,        // degree mode: some segment selected more candidates than it may remove
    CTR_OVF1 = 10,
    CTR_ROUNDS = 11,
    CTR_EMIT_C0 = 12,    // emission: tails of the seven size-class lists (12..18; the elimination is over by then)
    CTR_LOW0 = 14,       // degree mode: low-list tails, by round parity
    CTR_LOW1 = 15,
    CTR_LOWOVF0 = 16,    // degree mode: the low list of that parity overflowed (every segment rescans)
    CTR_LOWOVF1 = 17,
    CTR_STEAL0 = 18,     // elimination phase: cursor of the part of the work list any warp may fetch (18..20, by round % 3)
    CTR_BAR = 21,        // barrier of the view group: arrivals (21) and generation (22)
    CTR_SCNT0 = 24,      // o_v = random: stars left to the shared-memory pass of the round (24..26, by round % 3)
    CTR_SSTEAL0 = 27,    // ... and the cursor the warps fetch them with (27..29, by round % 3)
    CTR_COUNT = 32
};

struct RoundCtx {
    int wl_base;   // where items appended in this round start
    int wslot;     // ctr index of this round's work-list counter
    int dl_base;
    int dslot;
    int sslot;     // ctr index of this round's shared-tail cursor
    int sl_top;    // o_v = random: the round's shared-memory stars are listed downwards from dl[sl_top - 1]
    int s2slot;    // ctr index of their count
    int c2slot;    // ctr index of the cursor they are fetched with
};
enum { ST_FILLS = 0, ST_POOL_MAX = 1, ST_MAXSTAR = 2, ST_DEFERRED = 3, ST_RAW = 4,
       ST_T_INIT = 8, ST_T_A = 9, ST_T_B = 10, ST_T_C = 11, ST_T_D1 = 12, ST_T_D2 = 13,
       ST_W_INIT = 16 /* .. 21: warp-nanoseconds spent waiting at the grid barrier that ends each phase (flags & 128) */,
       ST_DBG = 24 /* .. 29: debug (flags & 512): thread 0's time in the parts of phase B (setup, list, scan, flush), ns */,
       ST_COUNT = 32 };

struct SchurParams {
    // coalesced graph (shared by all views, immutable)
    int n;
    long long nnz;
    const int* ptr;
    const int* col;
    const float* w;
    int G;
    const int* gptr;   // [G+1]
    const int* teff;   // [G] min(num_remove, n_g - 1), or min(num_remove, m_g) for a graph with a protected vertex
    const int* gid;    // [n] graph of a vertex, or nullptr when G == 1
    const int* ucount; // keep mask: [n + 1] number of unprotected vertices below v (v is protected iff
                       // ucount[v + 1] == ucount[v]); nullptr without a mask
    // run
    int o_v, o_n, flags;
    uint32_t k0, k1;
    uint32_t view_base;
    int V;
    // per view state, all indexed [view * n + v]
    uint8_t* state;    // 0 kept (not eligible, or protected), 1 pending, 2 eliminated, 4 pending and isolated
    int* lh;           // [V*n][2] interleaved: live = number of raw entries whose neighbour is not eliminated
                       // (RLAP_LIVE_DEAD once the vertex itself is eliminated), head = head of the appended fill-entry
                       // list (pool index, -1 = empty). One 8-byte record: the dead test of a neighbour, the update of
                       // its live counter and the exchange of its list head touch the same 32-byte sector.
    int* rank;         // o_v = random: rank in the keyed permutation
    int* blk;          // o_v = random: pending lower-ranked eligible neighbours (raw multiplicity)
    int* candround;    // degree / coarsen: last round in which the vertex was selected
    int* outcnt;       // emission: merged row count
    long long* outoff; // emission: [V*n + 1] exclusive prefix of outcnt
    // emission staging: the live entries of every surviving vertex, owner-major, contiguous
    long long* rawoff; // [V*n + 1] exclusive prefix of the live counts of surviving vertices
    uint64_t* raw;     // [raw_cap] (nbr << 32) | weight bits
    long long raw_cap;
    // fill-entry pool: pool[view * pool_cap + p] = {nbr, weight bits, next, owner}
    int4* pool;
    long long pool_cap;
    unsigned long long* pool_cursor;  // [V]
    // per (view, graph) segment state, indexed [view * G + g]   (degree / coarsen)
    int* rem;
    int* lvl;          // key level established by the segment's last full scan (DESIGN.md §4: low lists)
    int* minkey;       // [2][V*G]: minimum key of the round over the low list / over a full scan
    int* cntI;
    int* ovfseg;
    unsigned int* thresh;
    int* blockcnt;     // [ceil(V*n / SEL_BLOCK)]
    // work lists (append-only over the whole run)
    unsigned int* wl;
    unsigned int* dl;
    unsigned int* low;  // [2][low_cap] degree / coarsen: vertices whose key may be <= lvl (ping-pong by round parity)
    long long low_cap;
    unsigned int* deadbits;   // [V][nw32] one bit per vertex: eliminated. The dead test of a neighbour reads this instead of
    int nw32;                 // its 8-byte (live, head) record: 21 KB per arxiv view, resident in L2 whatever else streams
    int* ctr;          // [CTR_COUNT]
    unsigned long long* stats;  // [ST_COUNT]
    // the blocks [gblock0, gblock0 + gblocks) of the launch work on this parameter block (a view group)
    int gblock0, gblocks;
    // global scratch for stars larger than CAP_CTA: slot b = 3 * scratch_cap u64 for block b
    uint64_t* scratch;
    int scratch_cap;
    uint64_t* stage;     // [blocks of the launch][ELIM_WARPS][32][STAGE_CAP]: fill lists walked ahead by single lanes
    int stage_cap;       // STAGE_CAP, or 0 when the workspace holds no staging area
    // o_v = random: vertices of at least HUB_DEG input entries keep HUB_HEADS fill lists instead of one (a fill goes to
    // list `pool slot % HUB_HEADS`), so that a warp walks a hub's fills 32 chains at a time
    const int* hubidx;   // [n] row of the vertex in the head table or -1 (shared by the views); nullptr for the other orders
    const int* hubcount; // number of rows in use
    int* hubheads;       // [V][nhmax][HUB_HEADS]
    int nhmax;
    long long* blocksum;  // scan scratch
};

constexpr int RLAP_LIVE_DEAD = -0x40000000;

// "first call on this device" latch for per-device set-up (function attributes are per device, and a process may use
// several devices from several threads)
struct PerDeviceOnce {
    unsigned long long done[4] = {0, 0, 0, 0};   // 256 device ordinals
    // returns true exactly once per device ordinal; callers serialise through their own lock
    bool first(int dev) {
        if (dev < 0 || dev >= 256) return true;
        const unsigned long long bit = 1ull << (dev & 63);
        if (done[dev >> 6] & bit) return false;
        done[dev >> 6] |= bit;
        return true;
    }
};
__host__ __device__ __forceinline__ int* live_p(const SchurParams& P, size_t i) { return P.lh + 2 * i; }
__host__ __device__ __forceinline__ int* head_p(const SchurParams& P, size_t i) { return P.lh + 2 * i + 1; }
#ifdef __CUDACC__
// neighbour u of `view` eliminated?
__device__ __forceinline__ bool is_dead(const SchurParams& P, int view, unsigned u) {
    return (__ldcg(P.deadbits + (size_t)view * (size_t)P.nw32 + (u >> 5)) >> (u & 31u)) & 1u;
}
__device__ __forceinline__ void mark_dead(const SchurParams& P, int view, unsigned v) {
    atomicOr(P.deadbits + (size_t)view * (size_t)P.nw32 + (v >> 5), 1u << (v & 31u));
}
#endif

}  // namespace rlap
