/* rlap_b200.h — C ABI of the B200-native rLap randomized Schur-complement augmentor.
 *
 * This is the drop-in boundary for ONE path of kvignesh1420/rlap: what sits behind
 * rlap.ops.approximate_cholesky (rlap/ops.py:7-58), i.e. the torch-dispatcher kernel
 * extension_cpp::approximate_cholesky (rlap/csrc/py_api_binder.cc:54-69,80-88) and the C++
 * classes it drives (ApproximateCholesky::setup / ::getSchurComplement, rlap/csrc/factorizers.h:24-48).
 * Plain pointers and sizes only; no torch types. The library is librlap_b200.so
 * (rlap_b200/csrc/, nvcc -gencode arch=compute_100a,code=sm_100a). INTEGRATION.md shows the
 * reference-side bindings.
 *
 * Conventions
 *  - Every function returns an rlap_status (0 = ok). Nothing ever calls exit() (the reference
 *    exit(0)s the interpreter on asymmetric input, factorizers.cc:19-22; here that is
 *    RLAP_ERR_ASYMMETRIC).
 *  - "device" pointers are CUDA device memory of the current device; `stream` is a cudaStream_t
 *    passed as void* (NULL = default stream). Calls are stream ordered; the only host
 *    synchronisations are the ones that return a count/status to the host, documented below.
 *  - The caller owns all memory, including workspaces (sizes from the *_workspace_bytes queries).
 *  - A graph may be a disjoint union of `n_graphs` independent graphs (vertex ranges
 *    graph_ptr[g]..graph_ptr[g+1]); every graph g gets its own num_remove[g], its own ordering and
 *    the reference's cap t = min(num_remove, n_g - 1) (preconditioner.cc:358,723,846).
 *    n_graphs = 1 with graph_ptr = {0, n} is the reference's semantics (a PyG batch treated as
 *    one graph, scripts/graph_shared.py:139-146).
 *  - Which vertices survive can also be named: rlap_schur_eliminate_keep takes a keep mask (protected vertices are
 *    never eliminated), which turns full-clique mode into an exact Kron reduction onto any terminal set.
 */
#ifndef RLAP_B200_H
#define RLAP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    RLAP_OK = 0,
    RLAP_ERR_INVALID_ARG = 1,     /* bad enum / null pointer / negative size                        */
    RLAP_ERR_ID_RANGE = 2,        /* node id outside [0, num_nodes)                                 */
    RLAP_ERR_SELF_LOOP = 3,       /* (v,v) entry with non-zero weight (undefined in the reference)  */
    RLAP_ERR_ASYMMETRIC = 4,      /* adjacency not symmetric (reference: print + exit(0))           */
    RLAP_ERR_POOL_OVERFLOW = 5,   /* fill-edge pool too small: retry with a larger pool_cap         */
    RLAP_ERR_STAR_TOO_LARGE = 6,  /* a vertex star exceeded the scratch capacity (scratch_cap)      */
    RLAP_ERR_WORKSPACE = 7,       /* workspace smaller than the *_workspace_bytes answer            */
    RLAP_ERR_CUDA = 8,            /* CUDA runtime error (see rlap_last_cuda_error)                  */
    RLAP_ERR_NEGATIVE_WEIGHT = 9, /* weight < 0 or not finite                                       */
    RLAP_ERR_INTERNAL = 10        /* an internal invariant failed (round bound exceeded): a bug     */
} rlap_status;

/* o_v: vertex elimination order (factorizers.cc:56-64). o_n: neighbour order (prec.cc:295-307). */
enum { RLAP_OV_RANDOM = 0, RLAP_OV_DEGREE = 1, RLAP_OV_COARSEN = 2 };
enum { RLAP_ON_ASC = 0, RLAP_ON_DESC = 1, RLAP_ON_RANDOM = 2 };

/* flags */
enum {
    RLAP_FLAG_FULL_CLIQUE = 1,   /* replace sampling by full clique elimination: exact Schur complement */
    RLAP_FLAG_SHARED_ORDER = 2,  /* o_v=random: all views share view 0's vertex permutation              */
    RLAP_FLAG_NO_VALIDATE = 4,   /* rlap_ingest: skip the symmetry check                                 */
    RLAP_FLAG_CHECK_LIVE = 8,    /* self-check: count the surviving vertices whose emitted entry count differs
                                    from the live counter the elimination maintained (stats[15], must be 0)  */
    RLAP_FLAG_KEEP = 16          /* rlap_schur_workspace_bytes: room for a keep mask (rlap_schur_eliminate_keep) */
};

const char* rlap_status_string(int status);
const char* rlap_last_cuda_error(void);
int rlap_version(void);

/* ---- ingest: COO -> coalesced CSR  (replaces EdgeInfoMatrixReader::Read, reader.cc:42-61, and the
 * validation half of Factorizer::computeLaplacian, factorizers.cc:18-22) -------------------------
 * src/dst: device int64[e] = edge_index[0], edge_index[1] (rlap/ops.py:47); w: device float32[e] or
 * NULL for unit weights (ops.py:45-46). Zero weights are dropped, duplicates (src,dst) are summed in
 * order of appearance, entry (src -> dst) is stored in dst's segment with neighbour ids ascending
 * (the reference's column-compressed layout). Outputs: csr_ptr device int32[n+1], csr_col device
 * int32[>=e], csr_w device float[>=e]; *nnz_out (host) receives the coalesced entry count.
 * Synchronises `stream` once to return status and nnz. */
int rlap_ingest_workspace_bytes(int64_t n, int64_t e, size_t* bytes);
int rlap_ingest(const int64_t* src, const int64_t* dst, const float* w, int64_t e, int64_t n,
                int32_t* csr_ptr, int32_t* csr_col, float* csr_w, int64_t* nnz_out, int flags,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- views: ordering + elimination (replaces {Random,Priority,Coarsening}Preconditioner::
 * getSchurComplement, preconditioner.cc:348-476, 713-825, 835-957) --------------------------------
 * Produces n_views independent views (view ids view_base .. view_base+n_views-1; randomness is a
 * pure function of (seed, view id, vertex, neighbour), so results do not depend on how views are
 * sharded over GPUs). The limits of one call: view ids are 32-bit (view_base + n_views <= 2^32,
 * RLAP_ERR_INVALID_ARG otherwise) and n_views * n < 2^30 (work-list positions are 32-bit).
 * graph_ptr: HOST int64[n_graphs+1]; num_remove: HOST int64[n_graphs].
 * pool_cap: fill-edge pool entries per view (0 = default 2*nnz + 4096). scratch_cap: largest star
 * (raw live entries) the global scratch path accepts (0 = default min(n, 65536); rounded up to a power of two, the
 * size a star is padded to when it is sorted; a larger star returns
 * RLAP_ERR_STAR_TOO_LARGE and the caller retries with scratch_cap = nnz + 1, as rlap_approximate_cholesky_host does).
 * After rlap_schur_eliminate returns, view_rows (HOST int64[n_views]) holds the number of output
 * rows of every view. Synchronises `stream` once. */
int rlap_schur_workspace_bytes(int64_t n, int64_t nnz, int64_t n_graphs, int64_t n_views, int64_t pool_cap,
                               int64_t scratch_cap, int flags, size_t* bytes);
int rlap_schur_eliminate(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                         int64_t n_graphs, const int64_t* graph_ptr, const int64_t* num_remove, int o_v, int o_n,
                         uint64_t seed, int64_t view_base, int64_t n_views, int flags, int64_t pool_cap,
                         int64_t scratch_cap, void* workspace, size_t workspace_bytes, int64_t* view_rows,
                         int64_t* stats /* HOST int64[16] or NULL, see below */, void* stream);
/* stats: [0] rounds, [1] fill edges, [2] max pool entries used by a view, [3] largest merged star,
 * [4] raw adjacency entries read at elimination, [5] output rows, [6] pool_cap used,
 * [7] elimination kernel time (us, CUDA events), [8] emission count pass time (us),
 * [9..14] time inside the elimination kernel (us): init, min-key scan, candidate selection, truncation,
 * warp-level elimination, block-level elimination; [15] (only with RLAP_FLAG_CHECK_LIVE) number of
 * surviving vertices whose scattered entry count differs from their live counter: must be 0. */

/* ---- views onto a caller-chosen vertex set (no reference counterpart: the reference only takes a count) ----------
 * rlap_schur_eliminate with one more argument: keep, device uint8[n] or NULL. A nonzero keep[v] protects v: it is
 * never eliminated, in every view of the call. For graph g with m_g unprotected vertices the cap becomes
 * t_g = min(max(num_remove[g], 0), m_g) when g has a protected vertex (every unprotected vertex may go) and stays
 * min(max(num_remove[g], 0), n_g - 1) otherwise. o_v = random ranks the unprotected vertices of g (numbered by ascending
 * id) with the same keyed permutation over m_g; degree / coarsen take the minimum key, the bucket and the independent
 * set over the alive unprotected vertices only. With RLAP_FLAG_FULL_CLIQUE and num_remove >= m_g the result is the
 * exact Schur complement onto the protected set (a Kron reduction). A non-NULL keep needs a workspace sized with
 * flags | RLAP_FLAG_KEEP; keep = NULL is rlap_schur_eliminate, bit for bit. keep is read before the call returns. */
int rlap_schur_eliminate_keep(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                              int64_t n_graphs, const int64_t* graph_ptr, const int64_t* num_remove, int o_v, int o_n,
                              uint64_t seed, int64_t view_base, int64_t n_views, int flags, int64_t pool_cap,
                              int64_t scratch_cap, void* workspace, size_t workspace_bytes, int64_t* view_rows,
                              int64_t* stats, const uint8_t* keep, void* stream);

/* ---- emission (replaces the output assembly, preconditioner.cc:435-457 / 789-810 / 916-934) ------
 * Writes the rows of all views back to back, view after view, each view sorted by (col, row):
 * (row = neighbour, col = surviving vertex, weight), both directions present, original node ids.
 * Either the packed device buffers (out_row/out_col int32, out_w float32) or out_f64 (device
 * double[rows,3], the reference's [E',3] float64 layout, py_api_binder.cc:33-51) or both may be
 * given; pass NULL for the ones not wanted (out_col alone may be NULL too: see rlap_schur_colptr; out_w alone may
 * be NULL for an unweighted view, which is what the reference's GCL adapters keep, scripts/augmentor_benchmarks.py:88-96).
 * Must follow rlap_schur_eliminate on the same workspace.
 * Does not synchronise. */
int rlap_schur_emit(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                    int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* out_row, int32_t* out_col,
                    float* out_w, double* out_f64, void* stream);

/* ---- column-pointer output (for consumers behind a PCIe link) -------------------------------------
 * The rows of a view are sorted by (col, row), so `col` is implied by the number of rows per column.
 * rlap_schur_emit with out_col = NULL writes rows and weights only; rlap_schur_colptr writes
 * colptr[view * (n + 1) + v] = number of rows of `view` whose column is < v (device int32[n_views * (n + 1)],
 * colptr[view * (n + 1) + n] = rows of the view): 4 (n + 1) bytes per view instead of 4 bytes per row.
 * rlap_expand_cols_host rebuilds col (HOST int32[rows], views back to back at view_ptr[view], HOST int64[n_views + 1])
 * from a HOST copy of colptr with n_threads host threads. No reference counterpart: the reference never
 * leaves the host (py_api_binder.cc:54-69). */
int rlap_schur_colptr(int64_t n, int64_t nnz, int64_t n_views, void* workspace, size_t workspace_bytes,
                      int32_t* colptr, void* stream);

/* ---- survivor compaction + relabelling (the step the reference's adapters run right after the op:
 * torch.unique over the output's node ids + subgraph(relabel_nodes=True), scripts/augmentor_benchmarks.py:149-155,
 * scripts/rlap_vc_spectral.py:43-51) ----------------------------------------------------------------------------
 * rlap_schur_relabel writes newid (device int32[n_views * n + 1], one spare entry): newid[view * n + v] = rank of v
 * among the vertices of `view` that own at least one output row (ascending id, the order torch.unique returns), -1
 * for the others; view_nodes (device int64[n_views] or NULL) receives the number of such vertices per view.
 * rlap_schur_emit_ids is rlap_schur_emit with both ends of every row passed through newid (NULL: plain ids).
 * Neither synchronises. */
int rlap_schur_relabel(int64_t n, int64_t nnz, int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* newid,
                       int64_t* view_nodes, void* stream);
int rlap_schur_emit_ids(int64_t n, int64_t nnz, const int32_t* csr_ptr, const int32_t* csr_col, const float* csr_w,
                        int64_t n_views, void* workspace, size_t workspace_bytes, int32_t* out_row, int32_t* out_col,
                        float* out_w, double* out_f64, const int32_t* newid, void* stream);

/* Forget the results rlap_schur_eliminate left in `workspace`. Call it before the workspace memory is freed or
 * reused: rlap_schur_emit / rlap_schur_colptr refuse a workspace that was released (the library keeps no
 * reference to caller memory afterwards). No reference counterpart (the reference returns one heap matrix). */
int rlap_schur_release(void* workspace);
int rlap_expand_cols_host(const int32_t* colptr, int64_t n_views, int64_t n, const int64_t* view_ptr, int32_t* out_col,
                          int n_threads);

/* ---- host-buffer entry point: the exact shape of approximate_cholesky_cpu (py_api_binder.cc:54-69)
 * edge_info: HOST row-major double[e,3] (row, col, weight) as rlap/ops.py:47 packs it. Allocates
 * device memory internally, copies in, runs ingest + one view + emission on the current device,
 * copies the [rows,3] double result into a malloc'ed HOST buffer (*out, free with rlap_free_host).
 * `seed` replaces the reference's unseedable std::random_device / fixed mt19937_64 stream. */
int rlap_approximate_cholesky_host(const double* edge_info, int64_t e, int64_t num_nodes, int64_t num_remove,
                                   const char* o_v, const char* o_n, uint64_t seed, double** out, int64_t* rows);
void rlap_free_host(void* p);

#ifdef __cplusplus
}
#endif
#endif /* RLAP_B200_H */
