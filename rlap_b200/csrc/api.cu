// api.cu — the C ABI declared in include/rlap_b200.h: workspace layout, launch orchestration,
// status handling and the host-buffer entry point that mirrors approximate_cholesky_cpu
// (rlap/csrc/py_api_binder.cc:54-69).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <thread>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/rlap_b200.h"
#include "ingest.cuh"
#include "scan.cuh"
#include "schur.cuh"

namespace rlap {
cudaError_t launch_hub_index(int n, const int* ptr, int* hubidx, int* count, cudaStream_t stream);
cudaError_t launch_setup_graphs(int n, int G, const int* gptr, const long long* num_remove, const int* ucount, int* gid,
                                int* teff, cudaStream_t stream);
cudaError_t launch_count_unprotected(int n, const uint8_t* keep, int* flag, int* ucount, long long* blocksum,
                                     cudaStream_t stream);
cudaError_t eliminate_grid(int* blocks_out, int o_v, int o_n, int flags);
cudaError_t launch_eliminate(const SchurParams* groups_host, int K, int blocks, int o_v, int o_n, int flags,
                             cudaStream_t stream);
int eliminate_max_groups();
int eliminate_max_blocks();
cudaError_t launch_emit_colptr(const SchurParams& P, int* colptr, cudaStream_t stream);
cudaError_t launch_combine_groups(int K, const int* gctr, const unsigned long long* gstats, int* ctr,
                                  unsigned long long* stats, cudaStream_t stream);
constexpr int EMIT_AUX = 6;   // side streams of the emission's merge-path sort kernels
cudaError_t launch_emit_count(const SchurParams& P, long long* total_dev, cudaStream_t stream, cudaStream_t* aux,
                              cudaEvent_t* aux_ev);
cudaError_t launch_emit_write(const SchurParams& P, int* out_row, int* out_col, float* out_w, double* out_f64,
                              const int* newid, cudaStream_t stream);
cudaError_t launch_relabel(const SchurParams& P, int* newid, long long* base_dev, long long* view_nodes, cudaStream_t stream);
}  // namespace rlap

using namespace rlap;

static thread_local std::string g_last_cuda_error;

static int cuda_fail(cudaError_t e, const char* where) {
    g_last_cuda_error = std::string(where) + ": " + cudaGetErrorString(e);
    return RLAP_ERR_CUDA;
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t _e = (call);                                   \
        if (_e != cudaSuccess) return cuda_fail(_e, #call);        \
    } while (0)

// Results that the host needs after a stream synchronisation (status, counts, view offsets) are written by a tiny
// kernel straight into mapped pinned host memory. A cudaMemcpyAsync would work too, but device-to-host copies of all
// streams share the copy engine's FIFO: a few bytes of status would queue behind a caller's bulk transfer of the
// previous batch (measured: 30 ms per call while 1.7 GB of views were in flight).
struct Mailbox {
    long long* host = nullptr;   // also valid on the device (unified addressing)
    size_t words = 0;
    int ensure(size_t need) {
        if (need <= words) return 0;
        if (host) cudaFreeHost(host);
        host = nullptr;
        words = 0;
        size_t w = need < 4096 ? 4096 : need * 2;
        cudaError_t e = cudaHostAlloc((void**)&host, w * sizeof(long long), cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) return 1;
        words = w;
        return 0;
    }
};

// Streams, events and the mailbox belong to the device that was current when they were created: one set per
// (host thread, device), created on first use on that device.
constexpr int MAX_GROUPS = 64;     // view groups of one call (the parameter table of the launch, schur.cu)
struct ThreadDevice {
    Mailbox mail;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    cudaStream_t aux[EMIT_AUX] = {nullptr};          // created on first use on this device
    cudaEvent_t aux_ev[EMIT_AUX + 1] = {nullptr};
    std::vector<int> gp;
    std::vector<SchurParams> groups;   // host copy of the parameter blocks of the view groups
};
static ThreadDevice* thread_device() {
    static thread_local std::unordered_map<int, ThreadDevice*> per_dev;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    auto it = per_dev.find(dev);
    if (it != per_dev.end()) return it->second;
    ThreadDevice* td = new ThreadDevice();   // lives as long as the thread's CUDA context use: never freed
    per_dev[dev] = td;
    return td;
}

__global__ void k_export_ingest(const int* status, const long long* total, const double* acc, long long* out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        out[0] = *status;
        out[1] = *total;
        out[2] = __double_as_longlong(acc[0]);
        out[3] = __double_as_longlong(acc[1]);
        __threadfence_system();
    }
}

// out: [0..CTR_COUNT) counters, [CTR_COUNT .. +ST_COUNT) stats, then V pool cursors, then V + 1 view offsets
__global__ void k_export_views(const int* ctr, const unsigned long long* stats, const unsigned long long* pool_cursor,
                               const long long* outoff, long long n, long long V, long long* out) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < CTR_COUNT) out[t] = ctr[t];
    if (t < ST_COUNT) out[CTR_COUNT + t] = (long long)stats[t];
    if (t < V) out[CTR_COUNT + ST_COUNT + t] = (long long)pool_cursor[t];
    if (t <= V) out[CTR_COUNT + ST_COUNT + V + t] = outoff[t * n];
    __threadfence_system();
}

// bump allocator over a caller-provided workspace (256-byte aligned pieces)
struct Carver {
    char* base;
    size_t off;
    explicit Carver(void* b) : base((char*)b), off(0) {}
    template <typename T>
    T* take(size_t count) {
        off = (off + 255) & ~(size_t)255;
        T* p = base ? (T*)(base + off) : (T*)nullptr;
        off += count * sizeof(T);
        return p;
    }
};

extern "C" {

const char* rlap_status_string(int s) {
    switch (s) {
        case RLAP_OK: return "ok";
        case RLAP_ERR_INVALID_ARG: return "invalid argument";
        case RLAP_ERR_ID_RANGE: return "node id out of range";
        case RLAP_ERR_SELF_LOOP: return "self loop in edge list";
        case RLAP_ERR_ASYMMETRIC: return "adjacency matrix is not symmetric";
        case RLAP_ERR_POOL_OVERFLOW: return "fill-edge pool overflow (raise pool_cap)";
        case RLAP_ERR_STAR_TOO_LARGE: return "vertex star larger than scratch capacity (raise scratch_cap)";
        case RLAP_ERR_WORKSPACE: return "workspace too small";
        case RLAP_ERR_CUDA: return "CUDA error";
        case RLAP_ERR_NEGATIVE_WEIGHT: return "negative or non-finite edge weight";
        case RLAP_ERR_INTERNAL: return "internal invariant failed (elimination round bound exceeded)";
        default: return "unknown status";
    }
}
const char* rlap_last_cuda_error(void) { return g_last_cuda_error.c_str(); }
int rlap_version(void) { return 1; }

// ------------------------------------------------------------------------------------------ ingest
// largest raw row (duplicates included) the global-scratch path of the ingest accepts: max(n, 4096) entries, never
// more than e. A vertex with more incident input entries than the graph has vertices is a degenerate multigraph;
// it is reported as RLAP_ERR_STAR_TOO_LARGE (sizing the NSLOT scratch slots for e entries each would cost 24 e
// bytes per slot: 24 GB for the products-shaped graph).
// The sorts pad a row to the next power of two inside its slot: the capacity is one.
static long long pow2_at_least(long long x) {
    long long p = 1;
    while (p < x) p <<= 1;
    return p;
}
static long long ingest_scratch_cap(long long n, long long e) {
    long long c = n > 4096 ? n : 4096;
    if (c > e) c = e;
    if (c < CAP_CTA + 1) c = CAP_CTA + 1;
    return pow2_at_least(c);
}

struct IngestLayout {
    IngestParams P;
    size_t bytes;
    int* zero_begin;
    size_t zero_bytes;
};

static IngestLayout ingest_layout(long long n, long long e, void* ws) {
    IngestLayout L;
    memset(&L, 0, sizeof(L));
    Carver c(ws);
    IngestParams& P = L.P;
    P.n = n;
    P.e = e;
    // zeroed block: cnt, cursor, small scalars
    P.cnt = c.take<int>((size_t)n);
    P.cursor = c.take<int>((size_t)n);
    P.dl_tail = c.take<int>(1);
    P.status = c.take<int>(1);
    P.sym_acc = c.take<double>(2);
    P.total_dev = c.take<long long>(1);
    size_t zero_end = c.off;
    L.zero_begin = P.cnt;
    L.zero_bytes = zero_end;
    P.rawptr = c.take<int>((size_t)n + 1);
    P.cnt2 = c.take<int>((size_t)n);
    P.rkey = c.take<uint64_t>((size_t)e);
    P.rw = c.take<float>((size_t)e);
    P.tcol = c.take<int>((size_t)e);
    P.tw = c.take<float>((size_t)e);
    P.dl = c.take<unsigned int>((size_t)n);
    P.blocksum = c.take<long long>((size_t)scan_blocks(n));
    P.scratch_cap = (int)ingest_scratch_cap(n, e);
    P.scratch = c.take<uint64_t>((size_t)NSLOT * 3 * (size_t)P.scratch_cap);
    L.bytes = c.off + 256;
    return L;
}

int rlap_ingest_workspace_bytes(int64_t n, int64_t e, size_t* bytes) {
    if (n < 0 || e < 0 || !bytes || n >= (1LL << 31) - 1 || e >= (1LL << 31) - 1) return RLAP_ERR_INVALID_ARG;
    *bytes = ingest_layout(n, e, nullptr).bytes;
    return RLAP_OK;
}

int rlap_ingest(const int64_t* src, const int64_t* dst, const float* w, int64_t e, int64_t n, int32_t* csr_ptr,
                int32_t* csr_col, float* csr_w, int64_t* nnz_out, int flags, void* workspace, size_t workspace_bytes,
                void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    if (n < 0 || e < 0 || n >= (1LL << 31) - 1 || e >= (1LL << 31) - 1 || !csr_ptr || !nnz_out || !workspace)
        return RLAP_ERR_INVALID_ARG;
    if (e > 0 && (!src || !dst || !csr_col || !csr_w)) return RLAP_ERR_INVALID_ARG;
    IngestLayout L = ingest_layout(n, e, workspace);
    if (workspace_bytes < L.bytes) return RLAP_ERR_WORKSPACE;
    IngestParams& P = L.P;
    P.src = (const long long*)src;
    P.dst = (const long long*)dst;
    P.w = w;
    P.ptr = csr_ptr;
    P.col = csr_col;
    P.wout = csr_w;
    P.validate = (flags & RLAP_FLAG_NO_VALIDATE) ? 0 : 1;
    CK(cudaMemsetAsync(L.zero_begin, 0, L.zero_bytes, stream));
    CK(launch_ingest_stage1(P, stream));
    struct { int status; long long total; double acc[2]; } h;
    ThreadDevice* td = thread_device();
    if (!td) return cuda_fail(cudaErrorInvalidDevice, "cudaGetDevice");
    Mailbox& g_mail = td->mail;
    if (g_mail.ensure(8)) return cuda_fail(cudaErrorMemoryAllocation, "cudaHostAlloc(mailbox)");
    k_export_ingest<<<1, 32, 0, stream>>>(P.status, P.total_dev, P.sym_acc, g_mail.host);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(stream));
    h.status = (int)g_mail.host[0];
    h.total = g_mail.host[1];
    memcpy(&h.acc[0], &g_mail.host[2], sizeof(double));
    memcpy(&h.acc[1], &g_mail.host[3], sizeof(double));
    *nnz_out = h.total;
    if (h.status != 0) return h.status;
    // relative Frobenius tolerance 1e-6 (the reference uses Eigen's 1e-12 on float64 data)
    if (P.validate && h.acc[0] > 1e-12 * h.acc[1]) return RLAP_ERR_ASYMMETRIC;
    return RLAP_OK;
}

// ------------------------------------------------------------------------------------------- views
struct SchurLayout {
    SchurParams P;
    size_t bytes;
    int* gptr_dev;
    long long* nrem_dev;
    int* gid_dev;
    int* teff_dev;
    long long* total_dev;
    long long* viewptr_dev;   // [V+1]
    long long G, V, pool_cap, scratch_cap;
    int* gctr;                 // [MAX_GROUPS][CTR_COUNT] control blocks of the view groups
    unsigned long long* gstats; // [MAX_GROUPS][ST_COUNT]
    int* hubidx_dev;           // o_v = random: row of every vertex in the hub head table
    int* hubcount_dev;
    uint64_t* gscratch;        // one scratch slot per block that may own one (NSLOT per group at most)
    int* unprot_dev;           // keep mask (RLAP_FLAG_KEEP): [n] 1 = unprotected, scanned into ucount_dev [n + 1]
    int* ucount_dev;
};

// The views of one call are eliminated by ONE cooperative launch of k_eliminate whose blocks are partitioned into view
// groups, each with its own share of the views, its own lists and counters and its own barrier: views are
// independent, and a barrier over all of them makes every phase of every view wait for the slowest chain of any view
// (45 % of the warp time in the single-barrier profile, profiles/README.md). A group of one block has no global
// barrier at all.
constexpr int MAX_SCRATCH_SLOTS = 1280;  // >= blocks of a launch
static long long default_pool_cap(long long nnz) { return 2 * nnz + 4096; }
static long long default_scratch_cap(long long n) {
    long long c = n < 65536 ? n : 65536;
    if (c < CAP_CTA + 1) c = CAP_CTA + 1;
    return c;     // schur_layout rounds every capacity, the caller's too, up to a power of two
}

static SchurLayout schur_layout(long long n, long long nnz, long long G, long long V, long long pool_cap,
                                long long scratch_cap, int flags, void* ws) {
    const bool full_clique = (flags & RLAP_FLAG_FULL_CLIQUE) != 0;
    SchurLayout L;
    memset(&L, 0, sizeof(L));
    if (pool_cap <= 0) pool_cap = default_pool_cap(nnz);
    if (scratch_cap <= 0) scratch_cap = default_scratch_cap(n);
    // a star is padded to the next power of two inside its slot (star_sort_merge): a slot of any other size would let
    // the padding of its three arrays run into each other
    scratch_cap = pow2_at_least(scratch_cap);
    L.G = G; L.V = V; L.pool_cap = pool_cap; L.scratch_cap = scratch_cap;
    Carver c(ws);
    SchurParams& P = L.P;
    const size_t VN = (size_t)V * (size_t)n, VG = (size_t)V * (size_t)G;
    P.n = (int)n;
    P.nnz = nnz;
    P.G = (int)G;
    P.V = (int)V;
    P.ctr = c.take<int>(CTR_COUNT);
    P.stats = c.take<unsigned long long>(ST_COUNT);
    L.gctr = c.take<int>((size_t)MAX_GROUPS * CTR_COUNT);
    L.gstats = c.take<unsigned long long>((size_t)MAX_GROUPS * ST_COUNT);
    L.total_dev = c.take<long long>(1);
    L.viewptr_dev = c.take<long long>((size_t)V + 1);
    L.gptr_dev = c.take<int>((size_t)G + 1);
    L.nrem_dev = c.take<long long>((size_t)G);
    L.teff_dev = c.take<int>((size_t)G);
    L.gid_dev = c.take<int>(G > 1 ? (size_t)n : 1);
    P.nw32 = (int)((n + 31) / 32);
    P.deadbits = c.take<unsigned int>((size_t)V * (size_t)P.nw32);
    P.state = c.take<uint8_t>(VN);
    P.lh = c.take<int>(2 * VN);
    P.rank = c.take<int>(VN);
    P.blk = c.take<int>(VN);
    P.candround = c.take<int>(VN);
    P.outcnt = c.take<int>(VN);
    P.outoff = c.take<long long>(VN + 1);
    P.rawoff = c.take<long long>(VN + 1);
    // live entries never exceed the input's outside full-clique mode (DESIGN.md §3.6); the full-clique
    // test mode may keep every pool entry alive as well
    P.raw_cap = (long long)V * (nnz + (full_clique ? pool_cap : 0)) + 1;
    P.raw = c.take<uint64_t>((size_t)P.raw_cap);
    P.pool = c.take<int4>((size_t)V * (size_t)pool_cap);
    P.pool_cap = pool_cap;
    P.pool_cursor = c.take<unsigned long long>((size_t)V);
    P.rem = c.take<int>(VG);
    P.lvl = c.take<int>(VG);
    P.minkey = c.take<int>(2 * VG);
    P.cntI = c.take<int>(VG);
    P.ovfseg = c.take<int>(VG);
    P.thresh = c.take<unsigned int>(VG);
    // work lists and scratch: one region per view group inside each array (slack for MAX_GROUPS regions)
    P.blockcnt = c.take<int>((VN + SEL_BLOCK - 1) / SEL_BLOCK + 2 * MAX_GROUPS + 2);
    P.wl = c.take<unsigned int>(2 * VN + MAX_GROUPS + 1);
    P.dl = c.take<unsigned int>(VN + MAX_GROUPS + 1);
    P.low_cap = (long long)(2 * VN + 64);
    P.low = c.take<unsigned int>(4 * VN + 128 * (size_t)MAX_GROUPS);
    {
        // a group's first min(NSLOT, blocks of the group) blocks own a slot each: never more slots than blocks
        const long long slots = V * NSLOT < MAX_SCRATCH_SLOTS ? V * NSLOT : MAX_SCRATCH_SLOTS;
        P.scratch = c.take<uint64_t>((size_t)slots * 3 * (size_t)scratch_cap);
        L.gscratch = P.scratch;
    }
    P.scratch_cap = (int)scratch_cap;
    {
        // staging rows of the warps' shared-memory path: one per lane of every warp the launch can have (the grid never
        // exceeds one block per 256 vertex-views, rlap_schur_views)
        long long sb = (V * n + 255) / 256;
        if (sb < 1) sb = 1;
        if (sb > MAX_SCRATCH_SLOTS) sb = MAX_SCRATCH_SLOTS;
        P.stage = c.take<uint64_t>((size_t)sb * ELIM_WARPS * 32 * (size_t)STAGE_CAP);
        P.stage_cap = STAGE_CAP;
    }
    {
        // o_v = random: head table of the hubs; a vertex needs HUB_DEG input entries for a row
        P.nhmax = (int)(nnz / HUB_DEG + 1);
        L.hubidx_dev = c.take<int>((size_t)n);
        L.hubcount_dev = c.take<int>(1);
        P.hubheads = c.take<int>((size_t)V * (size_t)P.nhmax * HUB_HEADS);
        P.hubidx = nullptr;
        P.hubcount = nullptr;
    }
    P.blocksum = c.take<long long>((size_t)scan_blocks((long long)VN));
    if (flags & RLAP_FLAG_KEEP) {   // last, so that the pieces above sit where they sit without a mask
        L.unprot_dev = c.take<int>((size_t)n);
        L.ucount_dev = c.take<int>((size_t)n + 1);
    }
    P.gptr = L.gptr_dev;
    P.teff = L.teff_dev;
    P.gid = G > 1 ? L.gid_dev : nullptr;
    L.bytes = c.off + 256;
    return L;
}

static int check_dims(int64_t n, int64_t nnz, int64_t G, int64_t V, int64_t pool_cap, int64_t scratch_cap) {
    if (n < 1 || nnz < 0 || G < 1 || V < 1 || pool_cap < 0 || scratch_cap < 0) return RLAP_ERR_INVALID_ARG;
    if (n >= (1LL << 31) - 1 || nnz >= (1LL << 31) - 1) return RLAP_ERR_INVALID_ARG;
    if (V * n >= (1LL << 30)) return RLAP_ERR_INVALID_ARG;  // work-list positions are 32-bit
    long long pc = pool_cap > 0 ? pool_cap : default_pool_cap(nnz);
    if (pc >= (1LL << 31) - 1) return RLAP_ERR_INVALID_ARG;
    if (G > n) return RLAP_ERR_INVALID_ARG;
    return RLAP_OK;
}

int rlap_schur_workspace_bytes(int64_t n, int64_t nnz, int64_t n_graphs, int64_t n_views, int64_t pool_cap,
                               int64_t scratch_cap, int flags, size_t* bytes) {
    if (!bytes) return RLAP_ERR_INVALID_ARG;
    int st = check_dims(n, nnz, n_graphs, n_views, pool_cap, scratch_cap);
    if (st) return st;
    *bytes = schur_layout(n, nnz, n_graphs, n_views, pool_cap, scratch_cap, flags, nullptr).bytes;
    return RLAP_OK;
}

static std::mutex g_layout_mutex;
static std::unordered_map<void*, SchurLayout> g_layouts;  // workspace -> layout of the last eliminate call

__global__ void k_gather_view_ptr(const long long* outoff, long long n, long long V, long long* viewptr) {
    long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v <= V) viewptr[v] = outoff[v * n];
}

int rlap_schur_eliminate_keep(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                              int64_t n_graphs, const int64_t* graph_ptr, const int64_t* num_remove, int o_v, int o_n,
                              uint64_t seed, int64_t view_base, int64_t n_views, int flags, int64_t pool_cap,
                              int64_t scratch_cap, void* workspace, size_t workspace_bytes, int64_t* view_rows,
                              int64_t* stats, const uint8_t* keep, void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    if (keep) flags |= RLAP_FLAG_KEEP;
    int st = check_dims(n, nnz, n_graphs, n_views, pool_cap, scratch_cap);
    if (st) return st;
    if (!csr_ptr || !graph_ptr || !num_remove || !workspace || !view_rows) return RLAP_ERR_INVALID_ARG;
    if (nnz > 0 && (!csr_col || !csr_w)) return RLAP_ERR_INVALID_ARG;
    if (o_v < 0 || o_v > 2 || o_n < 0 || o_n > 2 || view_base < 0) return RLAP_ERR_INVALID_ARG;
    // view ids are 32-bit words of the Philox counter: a larger id would wrap onto view (id mod 2^32)
    if (view_base > (1LL << 32) - n_views) return RLAP_ERR_INVALID_ARG;
    if (graph_ptr[0] != 0 || graph_ptr[n_graphs] != n) return RLAP_ERR_INVALID_ARG;
    for (int64_t g = 0; g < n_graphs; g++)
        if (graph_ptr[g + 1] < graph_ptr[g]) return RLAP_ERR_INVALID_ARG;
    SchurLayout L = schur_layout(n, nnz, n_graphs, n_views, pool_cap, scratch_cap, flags, workspace);
    if (workspace_bytes < L.bytes) return RLAP_ERR_WORKSPACE;
    SchurParams& P = L.P;
    P.ptr = csr_ptr;
    P.col = csr_col;
    P.w = csr_w;
    P.o_v = o_v;
    P.o_n = o_n;
    P.flags = flags;
    P.k0 = (uint32_t)seed;
    P.k1 = (uint32_t)(seed >> 32);
    P.view_base = (uint32_t)view_base;
    ThreadDevice* td = thread_device();
    if (!td) return cuda_fail(cudaErrorInvalidDevice, "cudaGetDevice");
    Mailbox& g_mail = td->mail;
    {
        // the converted graph pointers live until the next call of this thread; this call synchronises the stream
        // before it returns, so no extra synchronisation (which would drain the caller's queued work) is needed here
        std::vector<int>& gp = td->gp;
        gp.resize((size_t)n_graphs + 1);
        for (int64_t g = 0; g <= n_graphs; g++) gp[(size_t)g] = (int)graph_ptr[g];
        CK(cudaMemcpyAsync(L.gptr_dev, gp.data(), sizeof(int) * gp.size(), cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(L.nrem_dev, num_remove, sizeof(long long) * (size_t)n_graphs, cudaMemcpyHostToDevice, stream));
    }
    CK(cudaMemsetAsync(P.ctr, 0, sizeof(int) * CTR_COUNT, stream));
    CK(cudaMemsetAsync(P.stats, 0, sizeof(unsigned long long) * ST_COUNT, stream));
    if (keep) {
        CK(launch_count_unprotected((int)n, keep, L.unprot_dev, L.ucount_dev, P.blocksum, stream));
        P.ucount = L.ucount_dev;
    }
    CK(launch_setup_graphs((int)n, (int)n_graphs, L.gptr_dev, L.nrem_dev, P.ucount, n_graphs > 1 ? L.gid_dev : nullptr,
                           L.teff_dev, stream));
    if (o_v == 0) {
        CK(launch_hub_index((int)n, csr_ptr, L.hubidx_dev, L.hubcount_dev, stream));
        P.hubidx = L.hubidx_dev;
        P.hubcount = L.hubcount_dev;
    }
    // device-side timing of the two phases (read back with the counts; no extra synchronisation)
    cudaEvent_t* ev = td->ev;
    if (!ev[0]) for (int i = 0; i < 3; i++) CK(cudaEventCreate(&ev[i]));
    CK(cudaEventRecord(ev[0], stream));
    {
        // view groups (DESIGN.md §4): K groups share the blocks of one cooperative launch
        int blocks = 0;
        CK(eliminate_grid(&blocks, o_v, o_n, flags));
        if (blocks > eliminate_max_blocks()) blocks = eliminate_max_blocks();
        if (blocks > MAX_SCRATCH_SLOTS) blocks = MAX_SCRATCH_SLOTS;
        {
            // small inputs (the reference's 100-node example, a batch of molecule-sized graphs): about 256 vertices per
            // block, so that a single small view runs in ONE block - no global barrier, every phase a __syncthreads
            long long want = (n_views * n + 255) / 256;
            if (want < 1) want = 1;
            if (want < blocks) blocks = (int)want;
        }
        // every view its own group, up to the number of groups the launch's parameter table holds; more views are
        // dealt out evenly (elimination time per view does not depend on the split: 98 / 92 / 83 us per arxiv-shaped
        // view with 64 / 128 / 148 groups, profiles/README.md)
        long long K = n_views;
        if (K > eliminate_max_groups()) K = eliminate_max_groups();
#ifdef RLAP_DEBUG
        if (const char* env = getenv("RLAP_GROUPS")) { K = atoll(env); }
#endif
        if (K > n_views) K = n_views;
        if (K > blocks) K = blocks;
        if (K < 1) K = 1;
        std::vector<SchurParams>& groups = td->groups;
        groups.assign((size_t)K, P);
        CK(cudaMemsetAsync(L.gctr, 0, sizeof(int) * CTR_COUNT * (size_t)K, stream));
        CK(cudaMemsetAsync(L.gstats, 0, sizeof(unsigned long long) * ST_COUNT * (size_t)K, stream));
        const long long G = n_graphs;
        long long slot0 = 0;
        for (long long g = 0; g < K; g++) {
            const long long v0 = n_views * g / K, v1 = n_views * (g + 1) / K, Vg = v1 - v0;
            SchurParams& Q = groups[(size_t)g];
            const size_t o = (size_t)v0 * (size_t)n, og = (size_t)v0 * (size_t)G;
            Q.V = (int)Vg;
            Q.view_base = P.view_base + (uint32_t)v0;
            Q.deadbits += (size_t)v0 * (size_t)P.nw32;
            Q.state += o; Q.lh += 2 * o; Q.rank += o; Q.blk += o; Q.candround += o;
            Q.outoff += o;                                         // phase A's (round, key) snapshots live here
            Q.pool += (size_t)v0 * (size_t)P.pool_cap;
            Q.pool_cursor += v0;
            Q.hubheads += (size_t)v0 * (size_t)P.nhmax * HUB_HEADS;
            Q.rem += og; Q.lvl += og; Q.cntI += og; Q.ovfseg += og; Q.thresh += og;
            Q.minkey += 2 * og;                                    // [2][Vg * G] inside the [2 * V * G] array
            Q.blockcnt += o / SEL_BLOCK + 2 * (size_t)g;
            Q.wl += 2 * o + (size_t)g;
            Q.dl += o + (size_t)g;
            Q.low += 4 * o + 128 * (size_t)g;
            Q.low_cap = (long long)(2 * (size_t)Vg * (size_t)n + 64);
            Q.ctr = L.gctr + (size_t)g * CTR_COUNT;
            Q.stats = L.gstats + (size_t)g * ST_COUNT;
            Q.gblock0 = (int)((long long)blocks * g / K);
            Q.gblocks = (int)((long long)blocks * (g + 1) / K) - Q.gblock0;
            Q.scratch = L.gscratch + (size_t)slot0 * 3 * (size_t)L.scratch_cap;
            slot0 += Q.gblocks < NSLOT ? Q.gblocks : NSLOT;
        }
        CK(launch_eliminate(groups.data(), (int)K, blocks, o_v, o_n, flags, stream));
        CK(launch_combine_groups((int)K, L.gctr, L.gstats, P.ctr, P.stats, stream));
    }
#ifdef RLAP_DEBUG
    if (getenv("RLAP_DEBUG_SYNC")) {
        cudaError_t de = cudaStreamSynchronize(stream);
        if (de != cudaSuccess) return cuda_fail(de, "k_eliminate (debug sync)");
    }
#endif
    CK(cudaEventRecord(ev[1], stream));
    if (!td->aux[0]) {
        for (int i = 0; i < EMIT_AUX; i++) CK(cudaStreamCreateWithFlags(&td->aux[i], cudaStreamNonBlocking));
        for (int i = 0; i <= EMIT_AUX; i++) CK(cudaEventCreateWithFlags(&td->aux_ev[i], cudaEventDisableTiming));
    }
    CK(launch_emit_count(P, L.total_dev, stream, td->aux, td->aux_ev));
    CK(cudaEventRecord(ev[2], stream));
    const size_t mail_words = (size_t)CTR_COUNT + ST_COUNT + 2 * (size_t)n_views + 2;
    if (g_mail.ensure(mail_words)) return cuda_fail(cudaErrorMemoryAllocation, "cudaHostAlloc(mailbox)");
    {
        long long work = n_views + 1 > CTR_COUNT ? n_views + 1 : CTR_COUNT;
        if (work < ST_COUNT) work = ST_COUNT;
        k_export_views<<<(unsigned)((work + 127) / 128), 128, 0, stream>>>(P.ctr, P.stats, P.pool_cursor, P.outoff, n,
                                                                          n_views, g_mail.host);
    }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(stream));
    std::vector<long long> vp((size_t)n_views + 1);
    int hctr[CTR_COUNT];
    unsigned long long hstats[ST_COUNT];
    std::vector<unsigned long long> hcur((size_t)n_views);
    for (int i = 0; i < CTR_COUNT; i++) hctr[i] = (int)g_mail.host[i];
    for (int i = 0; i < ST_COUNT; i++) hstats[i] = (unsigned long long)g_mail.host[CTR_COUNT + i];
    for (int64_t v = 0; v < n_views; v++) hcur[(size_t)v] = (unsigned long long)g_mail.host[CTR_COUNT + ST_COUNT + v];
    for (int64_t v = 0; v <= n_views; v++) vp[(size_t)v] = g_mail.host[CTR_COUNT + ST_COUNT + n_views + v];
    for (int64_t v = 0; v < n_views; v++) view_rows[v] = vp[(size_t)v + 1] - vp[(size_t)v];
    if (stats) {
        unsigned long long pmax = 0;
        for (auto c : hcur) pmax = c > pmax ? c : pmax;
        stats[0] = hctr[CTR_ROUNDS];
        stats[1] = (int64_t)hstats[ST_FILLS];
        stats[2] = (int64_t)pmax;
        stats[3] = (int64_t)hstats[ST_MAXSTAR];
        stats[4] = (int64_t)hstats[ST_RAW];
        stats[5] = vp[(size_t)n_views];
        stats[6] = L.pool_cap;
        float ms_elim = 0.f, ms_count = 0.f;
        cudaEventElapsedTime(&ms_elim, ev[0], ev[1]);
        cudaEventElapsedTime(&ms_count, ev[1], ev[2]);
        stats[7] = (int64_t)(ms_elim * 1000.0f);   // k_eliminate, microseconds
        stats[8] = (int64_t)(ms_count * 1000.0f);  // emission count pass + scan, microseconds
        for (int i = 0; i < 6; i++) stats[9 + i] = (int64_t)(hstats[ST_T_INIT + i] / 1000);  // phase times, us
        stats[15] = (int64_t)hstats[7];  // RLAP_FLAG_CHECK_LIVE: vertices whose scattered count != live counter
    }
#ifdef RLAP_DEBUG
    if ((flags & 128) && getenv("RLAP_DEBUG_TIMERS")) {   // mean barrier wait per warp and phase, microseconds
        int blocks = 0;
        eliminate_grid(&blocks, o_v, o_n, flags);
        const double nwarps = (double)blocks * ELIM_WARPS;
        static const char* nm[6] = {"init", "A", "B", "C", "D1", "D2"};
        fprintf(stderr, "rlap timers (us): k_eliminate %.0f |", 0.0 + (double)(stats ? stats[7] : 0));
        for (int i = 0; i < 6; i++)
            fprintf(stderr, " %s %.0f (wait %.0f)", nm[i], hstats[ST_T_INIT + i] / 1e3, hstats[ST_W_INIT + i] / 1e3 / nwarps);
        fprintf(stderr, " | stars on the shared-memory warp path %llu\n", hstats[ST_DEFERRED]);
        if (flags & 512)
            fprintf(stderr, "rlap phase B, thread 0 of the slowest group (us): setup %.0f list %.0f scan %.0f flush %.0f tail %.0f barrier %.0f\n",
                    hstats[ST_DBG] / 1e3, hstats[ST_DBG + 1] / 1e3, hstats[ST_DBG + 2] / 1e3, hstats[ST_DBG + 3] / 1e3,
                    hstats[ST_DBG + 4] / 1e3, hstats[ST_DBG + 5] / 1e3);
    }
#endif
    {
        // the layout is what rlap_schur_emit / rlap_schur_colptr need to find the results in the workspace; a failed
        // run leaves nothing to emit
        std::lock_guard<std::mutex> lk(g_layout_mutex);
        if (hctr[CTR_STATUS] != 0) g_layouts.erase(workspace); else g_layouts[workspace] = L;
    }
    if (hctr[CTR_STATUS] != 0) return hctr[CTR_STATUS];
    return RLAP_OK;
}

int rlap_schur_eliminate(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                         int64_t n_graphs, const int64_t* graph_ptr, const int64_t* num_remove, int o_v, int o_n,
                         uint64_t seed, int64_t view_base, int64_t n_views, int flags, int64_t pool_cap,
                         int64_t scratch_cap, void* workspace, size_t workspace_bytes, int64_t* view_rows,
                         int64_t* stats, void* stream_v) {
    return rlap_schur_eliminate_keep(n, nnz, csr_ptr, csr_col, csr_w, n_graphs, graph_ptr, num_remove, o_v, o_n, seed,
                                     view_base, n_views, flags, pool_cap, scratch_cap, workspace, workspace_bytes,
                                     view_rows, stats, nullptr, stream_v);
}

static int find_layout(void* workspace, SchurLayout& L) {
    std::lock_guard<std::mutex> lk(g_layout_mutex);
    auto it = g_layouts.find(workspace);
    if (it == g_layouts.end()) return RLAP_ERR_INVALID_ARG;
    L = it->second;
    return RLAP_OK;
}

int rlap_schur_emit_ids(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                        int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* out_row, int32_t* out_col,
                        float* out_w, double* out_f64, const int32_t* newid, void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    SchurLayout L;
    if (find_layout(workspace, L)) return RLAP_ERR_INVALID_ARG;
    if (L.P.n != n || L.P.nnz != nnz || L.V != n_views || workspace_bytes < L.bytes) return RLAP_ERR_INVALID_ARG;
    if (L.P.ptr != csr_ptr || L.P.col != csr_col || L.P.w != csr_w) return RLAP_ERR_INVALID_ARG;
    if ((out_col || out_w) && !out_row) return RLAP_ERR_INVALID_ARG;   // out_col and out_w may be NULL on their own
    if (!out_row && !out_f64) return RLAP_ERR_INVALID_ARG;
    CK(launch_emit_write(L.P, out_row, out_col, out_w, out_f64, newid, stream));
    return RLAP_OK;
}

int rlap_schur_emit(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                    int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* out_row, int32_t* out_col,
                    float* out_w, double* out_f64, void* stream_v) {
    return rlap_schur_emit_ids(n, nnz, csr_ptr, csr_col, csr_w, n_views, workspace, workspace_bytes, out_row, out_col, out_w,
                               out_f64, nullptr, stream_v);
}

int rlap_schur_relabel(int64_t n, int64_t nnz, int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* newid,
                       int64_t* view_nodes, void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    SchurLayout L;
    if (find_layout(workspace, L)) return RLAP_ERR_INVALID_ARG;
    if (L.P.n != n || L.P.nnz != nnz || L.V != n_views || workspace_bytes < L.bytes || !newid) return RLAP_ERR_INVALID_ARG;
    CK(launch_relabel(L.P, newid, L.viewptr_dev, (long long*)view_nodes, stream));
    return RLAP_OK;
}

int rlap_schur_release(void* workspace) {
    std::lock_guard<std::mutex> lk(g_layout_mutex);
    g_layouts.erase(workspace);
    return RLAP_OK;
}

int rlap_schur_colptr(int64_t n, int64_t nnz, int64_t n_views, void* workspace, size_t workspace_bytes,
                      int32_t* colptr, void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    SchurLayout L;
    {
        std::lock_guard<std::mutex> lk(g_layout_mutex);
        auto it = g_layouts.find(workspace);
        if (it == g_layouts.end()) return RLAP_ERR_INVALID_ARG;
        L = it->second;
    }
    if (L.P.n != n || L.P.nnz != nnz || L.V != n_views || workspace_bytes < L.bytes || !colptr) return RLAP_ERR_INVALID_ARG;
    CK(launch_emit_colptr(L.P, colptr, stream));
    return RLAP_OK;
}

// Host side of the column-pointer output: rebuilds the `col` array of the packed rows from the per-view column
// pointers with n_threads threads (a fill at memory speed; it replaces a third of the device-to-host traffic).
int rlap_expand_cols_host(const int32_t* colptr, int64_t n_views, int64_t n, const int64_t* view_ptr, int32_t* out_col,
                          int n_threads) {
    if (!colptr || !view_ptr || !out_col || n_views < 0 || n < 1) return RLAP_ERR_INVALID_ARG;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 64) n_threads = 64;
    const long long total_rows = view_ptr[n_views];
    auto work = [&](int t) {
        // thread t fills an equal share [r0, r1) of the rows: locate the view and the column of r0, then run forward
        long long r0 = total_rows * t / n_threads;
        const long long r1 = total_rows * (t + 1) / n_threads;
        if (r0 >= r1) return;
        long long lo = 0, hi = n_views;               // last view with view_ptr[view] <= r0
        while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (view_ptr[mid] <= r0) lo = mid; else hi = mid; }
        long long view = lo;
        while (r0 < r1) {
            const int32_t* cp = colptr + view * (n + 1);
            const long long vbase = view_ptr[view], vrows = view_ptr[view + 1] - vbase;
            const long long rel0 = r0 - vbase, rel1 = (r1 - vbase < vrows) ? r1 - vbase : vrows;
            long long a0 = 0, a1 = n;                 // last column with cp[col] <= rel0
            while (a1 - a0 > 1) { const long long mid = (a0 + a1) >> 1; if (cp[mid] <= rel0) a0 = mid; else a1 = mid; }
            int32_t* dst = out_col + vbase;
            long long r = rel0;
            for (long long v = a0; v < n && r < rel1; v++) {
                const long long e = cp[v + 1] < rel1 ? cp[v + 1] : rel1;
                for (; r < e; r++) dst[r] = (int32_t)v;
            }
            r0 = vbase + rel1;
            view++;
        }
    };
    if (n_threads == 1) { work(0); return RLAP_OK; }
    std::vector<std::thread> th;
    th.reserve((size_t)n_threads);
    for (int t = 0; t < n_threads; t++) th.emplace_back(work, t);
    for (auto& x : th) x.join();
    return RLAP_OK;
}

// --------------------------------------------------------------------------- host-buffer entry point
__global__ void k_unpack_edge_info(const double* ei, long long e, long long* src, long long* dst, float* w) {
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < e) {
        src[p] = (long long)ei[p * 3 + 0];
        dst[p] = (long long)ei[p * 3 + 1];
        w[p] = (float)ei[p * 3 + 2];
    }
}

struct DevBuf {
    void* p = nullptr;
    cudaStream_t s;
    explicit DevBuf(cudaStream_t st) : s(st) {}
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 1, s); }
    ~DevBuf() { if (p) cudaFreeAsync(p, s); }
};

int rlap_approximate_cholesky_host(const double* edge_info, int64_t e, int64_t num_nodes, int64_t num_remove,
                                   const char* o_v, const char* o_n, uint64_t seed, double** out, int64_t* rows) {
    if (!out || !rows || !o_v || !o_n || e < 0 || num_nodes < 1 || (e > 0 && !edge_info)) return RLAP_ERR_INVALID_ARG;
    int ov = !strcmp(o_v, "random") ? 0 : !strcmp(o_v, "degree") ? 1 : !strcmp(o_v, "coarsen") ? 2 : -1;
    int on = !strcmp(o_n, "asc") ? 0 : !strcmp(o_n, "desc") ? 1 : !strcmp(o_n, "random") ? 2 : -1;
    if (ov < 0 || on < 0) return RLAP_ERR_INVALID_ARG;
    {   // keep freed blocks cached in the device's default pool: repeated calls do not hit cudaMalloc
        static std::mutex mu;
        static PerDeviceOnce once;
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(mu);
        if (once.first(dev)) {
            cudaMemPool_t mp;
            if (cudaDeviceGetDefaultMemPool(&mp, dev) == cudaSuccess) {
                uint64_t thr = UINT64_MAX;
                cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr);
            }
        }
    }
    cudaStream_t s = 0;
    *out = nullptr;
    *rows = 0;
    const int64_t n = num_nodes;
    DevBuf d_ei(s), d_src(s), d_dst(s), d_w(s), d_ptr(s), d_col(s), d_cw(s), d_ws(s), d_ws2(s), d_out(s);
    CK(d_ei.alloc(sizeof(double) * 3 * (size_t)e));
    CK(d_src.alloc(sizeof(long long) * (size_t)e));
    CK(d_dst.alloc(sizeof(long long) * (size_t)e));
    CK(d_w.alloc(sizeof(float) * (size_t)e));
    CK(d_ptr.alloc(sizeof(int) * ((size_t)n + 1)));
    CK(d_col.alloc(sizeof(int) * (size_t)e));
    CK(d_cw.alloc(sizeof(float) * (size_t)e));
    size_t wsb = 0;
    int st = rlap_ingest_workspace_bytes(n, e, &wsb);
    if (st) return st;
    CK(d_ws.alloc(wsb));
    if (e > 0) {
        CK(cudaMemcpyAsync(d_ei.p, edge_info, sizeof(double) * 3 * (size_t)e, cudaMemcpyHostToDevice, s));
        k_unpack_edge_info<<<(unsigned)((e + 255) / 256), 256, 0, s>>>((const double*)d_ei.p, e, (long long*)d_src.p,
                                                                      (long long*)d_dst.p, (float*)d_w.p);
        CK(cudaGetLastError());
    }
    int64_t nnz = 0;
    st = rlap_ingest((const int64_t*)d_src.p, (const int64_t*)d_dst.p, (const float*)d_w.p, e, n, (int32_t*)d_ptr.p,
                     (int32_t*)d_col.p, (float*)d_cw.p, &nnz, 0, d_ws.p, wsb, s);
    if (st) return st;
    int64_t gp[2] = {0, n};
    int64_t nr[1] = {num_remove};
    int64_t vrows = 0;
    int64_t pool_cap = 0, scratch_cap = 0;
    size_t wsb2 = 0;
    struct Release {   // the registered layout must not outlive the workspace, whatever the exit path
        void* ws;
        ~Release() { rlap_schur_release(ws); }
    };
    for (int attempt = 0;; attempt++) {
        st = rlap_schur_workspace_bytes(n, nnz, 1, 1, pool_cap, scratch_cap, 0, &wsb2);
        if (st) return st;
        DevBuf ws2(s);
        CK(ws2.alloc(wsb2));
        Release rel{ws2.p};
        st = rlap_schur_eliminate(n, nnz, (int32_t*)d_ptr.p, (int32_t*)d_col.p, (float*)d_cw.p, 1, gp, nr, ov, on, seed,
                                  0, 1, 0, pool_cap, scratch_cap, ws2.p, wsb2, &vrows, nullptr, s);
        if (st == RLAP_ERR_POOL_OVERFLOW && attempt < 6) {
            pool_cap = (pool_cap ? pool_cap : 2 * nnz + 4096) * 2;
            continue;
        }
        if (st == RLAP_ERR_STAR_TOO_LARGE && scratch_cap == 0) {   // a star beyond the default scratch: a star never exceeds nnz entries
            scratch_cap = nnz + 1;
            continue;
        }
        if (st) return st;
        CK(d_out.alloc(sizeof(double) * 3 * (size_t)vrows));
        st = rlap_schur_emit(n, nnz, (int32_t*)d_ptr.p, (int32_t*)d_col.p, (float*)d_cw.p, 1, ws2.p, wsb2, nullptr,
                             nullptr, nullptr, (double*)d_out.p, s);
        if (st) return st;
        double* h = (double*)malloc(sizeof(double) * 3 * (size_t)(vrows > 0 ? vrows : 1));
        if (!h) return RLAP_ERR_INVALID_ARG;
        cudaError_t ce = cudaMemcpyAsync(h, d_out.p, sizeof(double) * 3 * (size_t)vrows, cudaMemcpyDeviceToHost, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) { free(h); return cuda_fail(ce, "copy of the result to the host"); }
        *out = h;
        *rows = vrows;
        return RLAP_OK;
    }
}

void rlap_free_host(void* p) { free(p); }

}  // extern "C"
