/*
 * dcr.h — C ABI of libdcr.so, the B200 (sm_100a) library behind the reference's BFC / SDRF entry points.
 *
 * Reference = jakubbober/discrete-curvature-rewiring (read at /root/reference).  The reference has no FFI:
 * its hot path is two numba.cuda kernels plus torch calls driven from Python.  Each function below names the
 * reference interface (file:line) whose work it takes over; the Python modules that keep the reference's
 * module paths and signatures (discrete-curvature-rewiring_b200/{curvature,rewiring,utils}) bind these
 * symbols through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all memory
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it (no host sync) unless
 *     the comment says "synchronises"
 *   - return value: 0 = ok, non-zero = error (message via dcr_last_error(), thread-local)
 *   - graphs are simple (no self-loops, no multi-edges), node ids 0..n-1, given as a CSR with int32 row offsets and
 *     int32 SORTED column indices; unless a function says otherwise the graph is UNDIRECTED (both directions of every
 *     edge present); a "directed entry" is one slot of colidx, an "undirected edge" is a directed entry with row < col,
 *     numbered in CSR order (edge id).  The *_directed entry points and DCR_SDRF_MODE_BFC_DIRECTED take an asymmetric
 *     0/1 adjacency as TWO sorted CSRs: successors (rows of A) and predecessors (rows of A^T)
 */
#ifndef DCR_H_
#define DCR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCR_VERSION 1

/* status codes written by the SDRF loop into dcr_sdrf_result.status */
#define DCR_SDRF_OK 0             /* all requested iterations ran (or the loop hit one of its own `break`s)      */
#define DCR_SDRF_NEED_HOST 1      /* the uniform lies within `guard` of a CDF boundary: host must decide (App. E.3) */
#define DCR_SDRF_PROB_NAN 2       /* softmax overflow/underflow -> NaN probabilities (numpy: ValueError)          */
#define DCR_SDRF_PROB_SUM 3       /* probabilities do not sum to 1 (numpy: ValueError)                            */
#define DCR_SDRF_REMOVE_NONEDGE 4 /* argmax fell on a non-edge and exceeded removal_bound (networkx: NetworkXError) */
#define DCR_SDRF_NO_UNIFORM 5     /* ran out of host-supplied uniforms                                            */
#define DCR_SDRF_ARENA_FULL 6     /* adjacency arena exhausted (create with a larger max_additions)               */
#define DCR_SDRF_TOO_MANY_CANDIDATES 7 /* (deg x+1)(deg y+1) exceeds the candidate scratch of the state          */
#define DCR_SDRF_EMPTY_GRAPH 8    /* classical loop on a graph without edges (python: min() of an empty sequence)  */

/* loop flavours of dcr_sdrf_create_mode */
#define DCR_SDRF_MODE_BFC 0          /* sdrf_cuda_bfc(..., is_undirected=True)   rewiring/sdrf_cuda_bfc.py:14-93        */
#define DCR_SDRF_MODE_BFC_DIRECTED 1 /* sdrf_cuda_bfc(..., is_undirected=False)  :47-49, :72-73, :87-88                 */
#define DCR_SDRF_MODE_1D 2           /* sdrf_no_cuda(curv_type='1d')             rewiring/sdrf_no_cuda.py:9-68          */
#define DCR_SDRF_MODE_AUGMENTED 3    /* sdrf_no_cuda(curv_type='augmented')      curvature/classical_curvatures.py:17-21 */
#define DCR_SDRF_MODE_HAANTJES 4     /* sdrf_no_cuda(curv_type='haantjes')       curvature/classical_curvatures.py:22-26 */

const char* dcr_last_error(void);
int dcr_version(void);
/* Measurement aid (no reference counterpart): a one-thread kernel that spins ~100 us on `stream` and writes the SM
 * clock it observed (clock64 / globaltimer, MHz) to *out_mhz (device memory). */
int dcr_sm_clock_probe(float* out_mhz, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Dense <-> CSR for the legacy dense-matrix signatures.
 * Replaces the dense `A` argument handling of curvature/bfc_cuda.py:51-57 and :144-150.
 * ---------------------------------------------------------------------------------------------------------- */

/* Pass 1: per-row non-zero counts of the fp32 row-major matrix A[n,n] into row_counts[n], and validation
 * flags OR-ed into *flags: bit0 = some value is neither 0 nor 1, bit1 = non-zero diagonal, bit2 = asymmetric. */
int dcr_dense_count(const float* A, int n, int32_t* row_counts, int32_t* flags, void* stream);
/* Pass 2: fill sorted colidx given rowptr[n+1] (exclusive scan of row_counts, done by the caller). */
int dcr_dense_fill(const float* A, int n, const int32_t* rowptr, int32_t* colidx, void* stream);
/* C[n,n] = 0 everywhere, then C[row, colidx[p]] = vals[p] for every directed entry p
 * (the dense `C` the reference returns, bfc_cuda.py:16-18,46-48,65). */
int dcr_scatter_dense(const int32_t* rowptr, const int32_t* colidx, int n, const float* vals, float* C,
                      void* stream);

/* The undirected edge list of a symmetric sorted CSR — the entries with row < col, in CSR order: edge e = (esrc[e],
 * edst[e]) — derived on the device (what `for v1, v2 in G.edges` enumerates, curvature/bfc_naive.py:49, for a graph
 * given as a CSR).  dcr_csr_upper_count writes per row the number of entries beyond the diagonal (int64); the caller
 * turns them into INCLUSIVE prefix sums (offsets_incl[v] = edges of rows 0..v); dcr_csr_upper_fill writes the nnz/2
 * edges.  Lets an end-to-end caller upload rowptr / colidx only. */
int dcr_csr_upper_count(const int32_t* rowptr, const int32_t* colidx, int n, int64_t* counts, void* stream);
int dcr_csr_upper_fill(const int32_t* rowptr, const int32_t* colidx, int n, const int64_t* offsets_incl, int32_t* esrc,
                       int32_t* edst, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * cuda-flavour BFC over CSR.  Replaces _balanced_forman_curvature (curvature/bfc_cuda.py:11-48) and its host
 * wrapper balanced_forman_curvature (:51-65) for symmetric 0/1 adjacency without self-loops.
 * Outputs are per DIRECTED ENTRY p in [entry_lo, entry_hi) (arrays are indexed by p, full length nnz):
 *   tri[p]    = A2[i,j]           (#common neighbours)           int32
 *   sharp[p]  = sharp_ij          (bfc_cuda.py:31-44)            int32
 *   lam[p]    = lambda_ij                                       int32
 *   c64[p]    = the fp64 value before the fp32 stores            double   (may be NULL)
 *   c32[p]    = the fp32 value the compiled kernel stores        float    (two roundings, SURVEY App. A.3)
 * `tri` must hold ALL entries' supports before the curvature pass: call dcr_bfc_support first (it fills
 * tri[0..nnz)), then dcr_bfc_cuda_flavour for the wanted entry range.
 * ---------------------------------------------------------------------------------------------------------- */
int dcr_bfc_support(const int32_t* rowptr, const int32_t* colidx, int n, int32_t* tri, int64_t entry_lo,
                    int64_t entry_hi, void* stream);
int dcr_bfc_cuda_flavour(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* tri,
                         int32_t* sharp, int32_t* lam, double* c64, float* c32, int64_t entry_lo,
                         int64_t entry_hi, void* stream);

/* The same kernel for an ASYMMETRIC 0/1 adjacency without self-loops (a directed simple graph; is_undirected=False
 * callers, curvature/bfc_cuda.py:20-25 take d_in[i] and d_out[j]): out_* = CSR of the successors (rows of A), in_* =
 * CSR of the predecessors (rows of A^T), both sorted.  Per entry p of the successor CSR: tri[p] = A2[i,j] =
 * #{m : i -> m -> j}, sharp / lam by the loop of :31-44 (lam is no longer d_max), c64 / c32 as above.  tri, sharp, lam,
 * c64 may be NULL; no support pass is needed before. */
int dcr_bfc_cuda_flavour_directed(const int32_t* out_rowptr, const int32_t* out_colidx, const int32_t* in_rowptr,
                                  const int32_t* in_colidx, int n, int32_t* tri, int32_t* sharp, int32_t* lam,
                                  double* c64, float* c32, int64_t entry_lo, int64_t entry_hi, void* stream);

/* Dense-regime alternative to dcr_bfc_support (n <= 32768): A2 = A·A on the tensor cores (tcgen05 kind::i8, TMA,
 * TMEM), replacing `torch.matmul(A, A)` of curvature/bfc_cuda.py:53,146; the fused epilogue writes only the entries
 * that sit on an edge, in CSR order — tri[0..nnz) is identical to dcr_bfc_support's.
 * The product is symmetric: only the upper-triangular tiles are computed and mirrored.
 * workspace: dcr_bfc_support_tc_workspace_bytes(n, nnz) bytes of device memory (int8 image of A + per-block offsets). */
int64_t dcr_bfc_support_tc_workspace_bytes(int n, int64_t nnz);
int dcr_bfc_support_tc(const int32_t* rowptr, const int32_t* colidx, int n, int64_t nnz, int32_t* tri, void* workspace,
                       int64_t workspace_bytes, void* stream);
/* The whole cuda flavour in the dense regime (same outputs as dcr_bfc_support + dcr_bfc_cuda_flavour over all
 * entries): A2 = A·A and T1 = (A ∧ [A2 == 1])·A on the tensor cores, then an elementwise closing pass. */
int64_t dcr_bfc_cuda_flavour_tc_workspace_bytes(int n, int64_t nnz);
int dcr_bfc_cuda_flavour_tc(const int32_t* rowptr, const int32_t* colidx, int n, int64_t nnz, int32_t* tri,
                            int32_t* sharp, int32_t* lam, double* c64, float* c32, void* workspace,
                            int64_t workspace_bytes, void* stream);

/* Measurement aid (no reference counterpart): dense int8 tensor rate of this GPU, TOP/s, measured with the product
 * kernel's own instruction (tcgen05.mma kind::i8, M128 N128 K32) on tiles resident in shared memory — the denominator of
 * the tensor roofline in bench.py.  *out_tops is device memory (fp64); synchronises. */
int dcr_tc_int8_peak(double* out_tops, void* stream);

/* Small dense graphs (n <= 1024: the WebKB shapes of configs 1-2): balanced_forman_curvature(A, C) of
 * curvature/bfc_cuda.py:51-65 straight from the dense fp32 A — rows bit-packed once, then one kernel computes supports,
 * the "support == 1" counts and the closing formula per entry and writes ALL n*n entries of C (+0.0 off-edge).  Two
 * launches and no host round trip, where the CSR route is launch-bound.  *flags receives the validation bits of
 * dcr_dense_count (the caller zeroes it and decides what to do with a non-zero value; C is then left untouched).
 * workspace: dcr_bfc_cuda_dense_small_workspace_bytes(n) bytes of device memory. */
int64_t dcr_bfc_cuda_dense_small_workspace_bytes(int n);
int dcr_bfc_cuda_dense_small(const float* A, int n, float* C, int32_t* flags, void* workspace,
                             int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * paper-flavour BFC over CSR.  Replaces bfc_edge / bfc (curvature/bfc_naive.py:7-40, :43-52).
 * Undirected edges are given explicitly: edge e = (esrc[e], edst[e]).  One call handles the strided subset
 * e = e_first + t*e_stride, t in [0,count) (single GPU: e_first=0, e_stride=1, count=E; rank r of W ranks:
 * e_first=r, e_stride=W) and writes the COMPACT outputs out_*[t]:  tri, sq_i (#squares at esrc), sq_j
 * (#squares at edst), gamma (0 where the reference never computes it), bfc (fp64, evaluated left to right
 * as bfc_naive.py:31-32,39-40).  Edges are classed, grouped by tested endpoint and ordered on the device inside
 * the call.  rowptr/colidx must be a SORTED CSR of a simple undirected graph (both directions present).
 * scratch: opaque device workspace of dcr_bfc_paper_scratch_bytes(n, max_degree, count) bytes (plan, orderings,
 * run tables, and the global-memory match hashes: a few hundred MB for the benchmark graphs; contents need not be
 * preserved or initialised between calls); max_degree = the largest row length of the CSR.
 * Graphs of up to 262144 nodes use an exact shared-memory bitmap of the tested endpoint's neighbours, larger ones a
 * hashed bitmap + table (dcr_bfc_paper_set_mode forces the latter; results are identical, the parity tests run both).
 * Threading: passes on the same device are serialised while they enqueue (a per-device mutex guards the fork/join
 * streams of the pass); passes on different devices are independent.
 * ---------------------------------------------------------------------------------------------------------- */
int64_t dcr_bfc_paper_scratch_bytes(int n, int max_degree, int64_t count);
int dcr_bfc_paper(const int32_t* rowptr, const int32_t* colidx, int n, int max_degree, const int32_t* esrc,
                  const int32_t* edst, int64_t e_first, int64_t e_stride, int64_t count, int32_t* out_tri,
                  int32_t* out_sq_i, int32_t* out_sq_j, int32_t* out_gamma, double* out_bfc, void* scratch,
                  int64_t scratch_bytes, void* ev_edge_begin, void* ev_edge_end, void* stream);
/* ev_edge_begin / ev_edge_end: optional cudaEvent_t (NULL = none) recorded on `stream` around the edge kernels
 * (the gather-bound part; the planning kernels before them are O(E)) — used by bench.py for the roofline. */

/* Membership mode of dcr_bfc_paper: 0 = automatic (exact shared-memory bitmap of the tested endpoint's neighbours for
 * graphs of up to 262144 nodes, hashed bitmap + table beyond), 1 = always the hashed structures.  Results are identical;
 * the parity tests run both.  Process-wide; returns the previous mode.  The initial mode is 0 unless the environment
 * variable DCR_PAPER_MODE=hashed was set when the library was loaded. */
int dcr_bfc_paper_set_mode(int mode);

/* Work estimate per undirected edge (entries streamed + per-head + per-edge terms) for cutting the edge list into
 * contiguous ranges of equal work (one range per GPU).  node_s_scratch: n int64 of device scratch. */
int dcr_bfc_paper_edge_cost(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* esrc, const int32_t* edst,
                            int64_t n_edges, int64_t* out_cost, int64_t* node_s_scratch, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Multi-GPU full-graph BFC over contiguous edge ranges (SURVEY.md §8e row 1; north_star: "shards naturally by edge
 * range ... curvature shards all-gathered over NVLink").  The reference has no multi-GPU path; this replaces what a
 * caller would otherwise do with bfc_naive.bfc (curvature/bfc_naive.py:43-52) per shard plus an all-gather.
 * A dcr_comm owns, on this rank's GPU, the FULL result arrays indexed by edge id — bfc f64[chunk] | tri | sq_i | sq_j |
 * gamma int32[chunk], chunk = dcr_comm_chunk() >= n_edges — in one cudaMalloc'ed buffer that the peer ranks map through
 * CUDA IPC (NVLink / NVSwitch peer memory).  dcr_bfc_paper_sharded computes the edges [e_lo, e_lo + count) and its
 * closing kernel stores every result at the edge's position in EVERY rank's buffer (compute + all-gather fused, no
 * staging copy, no re-interleave); device-side flags order it against the peers (no host synchronisation).  When the
 * work enqueued by the call has run, the local buffer holds the results of ALL ranks' ranges for this pass.  Every rank
 * must make the same sequence of calls.  world == 1 needs no connect.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct dcr_comm dcr_comm;
int dcr_comm_create(int rank, int world, int64_t n_edges, dcr_comm** out);
/* 64-byte CUDA IPC handle of this rank's buffer (host memory) — exchange them with any host-side all-gather */
int dcr_comm_handle(dcr_comm* comm, void* handle64_host);
/* handles_host: world x 64 bytes, rank r's handle at offset 64*r; maps the peers' buffers */
int dcr_comm_connect(dcr_comm* comm, const void* handles_host);
void* dcr_comm_buffer(dcr_comm* comm);          /* device pointer of the local result buffer */
int64_t dcr_comm_chunk(dcr_comm* comm);         /* entries per array inside the buffer */
int dcr_comm_error(dcr_comm* comm);             /* synchronises; non-zero if a hand-shake timed out (a peer never arrived) */
int dcr_comm_destroy(dcr_comm* comm);
int dcr_bfc_paper_sharded(const int32_t* rowptr, const int32_t* colidx, int n, int max_degree, const int32_t* esrc,
                          const int32_t* edst, int64_t e_lo, int64_t count, dcr_comm* comm, void* scratch,
                          int64_t scratch_bytes, void* ev_edge_begin, void* ev_edge_end, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * cuda-flavour BFC, one work item per UNDIRECTED edge (the fast path at full-graph scale) and its multi-GPU form
 * (SURVEY.md §8e row 2).  Replaces balanced_forman_curvature (curvature/bfc_cuda.py:51-65) for a symmetric 0/1 adjacency
 * given as a sorted CSR plus its undirected edge list (esrc[e] < edst[e], CSR order).  C[i,j] = C[j,i] is computed once.
 *   aux: dcr_bfc_cuda_edges_aux_ints(nnz, n_edges) int32 of device memory filled ONCE per graph by
 *        dcr_bfc_cuda_edges_prepare (directed entry -> edge id, and the list of hub-hub edges that get a whole CTA).
 *   dcr_bfc_cuda_edges: edges [e_lo, e_lo + count); outputs are indexed by EDGE ID (full-length arrays).  phases bit 0 =
 *        supports tri[e] = A2[i,j], bit 1 = sharp / lam / c64 / c32 (needs tri of ALL edges: run bit 0 over the whole
 *        graph first, or all-gather it).  sharp, lam, c64 may be NULL.
 *   dcr_bfc_cuda_sharded: both phases for this rank's range with the exchange fused into the kernels: supports are
 *        stored into every rank's dcr_comm buffer (the all-gather of `tri` between the two passes of §8e), the ranks meet
 *        on device-side flags, the results follow the same way.  Afterwards the local buffer holds, for ALL edges,
 *        c64 f64[chunk] | tri | sharp | lam int32[chunk] | c32 float[chunk].  Every rank makes the same sequence of calls.
 * ---------------------------------------------------------------------------------------------------------- */
int64_t dcr_bfc_cuda_edges_aux_ints(int64_t nnz, int64_t n_edges);
int dcr_bfc_cuda_edges_prepare(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* esrc,
                               const int32_t* edst, int64_t n_edges, int64_t nnz, int32_t* aux, void* stream);
int dcr_bfc_cuda_edges(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* esrc, const int32_t* edst,
                       int64_t nnz, const int32_t* aux, int64_t e_lo, int64_t count, int32_t* tri, int32_t* sharp,
                       int32_t* lam, double* c64, float* c32, int phases, void* stream);
int dcr_bfc_cuda_sharded(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* esrc, const int32_t* edst,
                         int64_t nnz, const int32_t* aux, int64_t e_lo, int64_t count, dcr_comm* comm, void* stream);

/* Multi-GPU epilogue of the NCCL route (strided shards): `gathered` = the all-gathered per-rank result blocks, rank r's block at byte offset
 * r*chunk*24 laid out as bfc[chunk] f64 | tri[chunk] | sq_i[chunk] | sq_j[chunk] | gamma[chunk] int32, where
 * local index t of rank r is edge e = r + t*world.  Writes the full-graph arrays indexed by edge id. */
int dcr_bfc_paper_unshard(const void* gathered, int world, int64_t chunk, int64_t n_edges, int32_t* out_tri,
                          int32_t* out_sq_i, int32_t* out_sq_j, int32_t* out_gamma, double* out_bfc, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Candidate scoring.  Replaces _balanced_forman_post_delta / balanced_forman_post_delta
 * (curvature/bfc_cuda.py:68-141, :144-159): D[I,J] for i = i_nb[I], j = j_nb[J]; masked cells = -1000.
 * `tri` = supports of all directed entries (dcr_bfc_support).  D is row-major [n_i, n_j] fp32.
 * ---------------------------------------------------------------------------------------------------------- */
int64_t dcr_post_delta_workspace_bytes(int n, int n_i, int n_j);
int dcr_post_delta(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* tri, int x, int y,
                   const int32_t* i_nb, int n_i, const int32_t* j_nb, int n_j, float* D, void* workspace,
                   int64_t workspace_bytes, void* stream);
/* workspace: dcr_post_delta_workspace_bytes(n, n_i, n_j) bytes of device memory (what all cells share: base terms over
 * N(x) / N(y), positions of the list entries).  One CTA fills it, then up to two CTAs per SM score the cells. */

/* Asymmetric A (see dcr_bfc_cuda_flavour_directed): i_nb are usually the successors of x plus x, j_nb the predecessors
 * of y plus y (rewiring/sdrf_cuda_bfc.py:48-49). */
int dcr_post_delta_directed(const int32_t* out_rowptr, const int32_t* out_colidx, const int32_t* in_rowptr,
                            const int32_t* in_colidx, int n, int x, int y, const int32_t* i_nb, int n_i,
                            const int32_t* j_nb, int n_j, float* D, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * SDRF loop.  Replaces the loop body of sdrf_cuda_bfc (rewiring/sdrf_cuda_bfc.py:37-91) including
 * utils/softmax.py:4-10 and the np.random.choice draw (:64-68), for is_undirected=True.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct dcr_sdrf dcr_sdrf;

typedef struct dcr_sdrf_result {
    int32_t status;          /* DCR_SDRF_*                                                                      */
    int32_t iterations_done; /* iterations fully executed by this call (log records written)                   */
    int32_t draws_used;      /* uniforms consumed by this call                                                  */
    int32_t stopped;         /* 1 if the loop took one of the reference's `break`s (:76-77, :89-91)            */
    int32_t pending_n;       /* NEED_HOST: number of candidates of the pending iteration                        */
    int32_t pending_x, pending_y;
    int32_t reserved;
} dcr_sdrf_result;

/* One log record per executed iteration: int32[8] = {x, y, n_candidates, k, l, choice, removed_x, removed_y}
 * (k = l = choice = -1 when nothing was added; removed_* = -1 when nothing was removed). */
#define DCR_SDRF_LOG_INTS 8

/* Build the device state from a host CSR in NETWORKX ADJACENCY ORDER (order_host[rowptr_host[v]..] lists the
 * neighbours of v in insertion order, sdrf_cuda_bfc.py:31-33,45-46); synchronises.  max_additions bounds the
 * number of edge insertions over the lifetime of the state (arena sizing).
 * Self-loops: the reference keeps a self-loop of the input in G (:31) but not in A (:29), so such a node meets ITSELF
 * in G.neighbors(v) and appears twice in its own candidate list (:45-46).  A list may therefore contain v itself, once,
 * at its insertion position: the entry lives in the insertion-order row only (no adjacency entry, no curvature), is
 * exported by dcr_sdrf_export_order, and is removed when the (0,0) fallback of the removal step hits a loop 0-0. */
int dcr_sdrf_create(int n, const int32_t* rowptr_host, const int32_t* order_host, int64_t max_additions,
                    dcr_sdrf** out);
/* The other loop flavours (DCR_SDRF_MODE_*).  BFC_DIRECTED: rowptr/order list the SUCCESSORS of every node in
 * networkx insertion order (G.successors, sdrf_cuda_bfc.py:48) and in_rowptr/in_order the PREDECESSORS (G.predecessors,
 * :49); no repeated entries (to_dense_adj would sum them into a weight); a node with a self-loop lists itself in BOTH
 * its successor and its predecessor list (see dcr_sdrf_create).
 * 1D / AUGMENTED / HAANTJES: the loop of sdrf_no_cuda over the undirected graph rowptr/order (adjacency order of
 * to_networkx(data, to_undirected=True)); in_* are ignored.  dcr_sdrf_run's log record then holds the (x, y) of
 * min(G.edges) (x <= y), the sorted (k, l) that was added and the removed edge; removal_bound is compared in fp64.
 * Here a node that lists itself has a LOOP EDGE (u,u) of G.edges with a curvature of its own (degree + 2, the node its
 * own neighbour): it can be the minimum edge (x == y) and the removed edge. */
int dcr_sdrf_create_mode(int n, int mode, const int32_t* rowptr_host, const int32_t* order_host,
                         const int32_t* in_rowptr_host, const int32_t* in_order_host, int64_t max_additions,
                         dcr_sdrf** out);
void dcr_sdrf_destroy(dcr_sdrf* s);
/* Run up to `loops` iterations.  uniforms[draw_offset + t] is the t-th uniform of this call (device, fp64).
 * forced_choice >= 0 forces the candidate index of the FIRST iteration of this call (host re-decision after
 * DCR_SDRF_NEED_HOST); guard = half-width of the CDF-boundary zone that triggers NEED_HOST (0 disables).
 * log: device int32[loops][8]; result: device dcr_sdrf_result. */
int dcr_sdrf_run(dcr_sdrf* s, int loops, int remove_edges, double removal_bound, double tau,
                 const double* uniforms, int64_t n_uniforms, int forced_choice, double guard, int32_t* log,
                 dcr_sdrf_result* result, void* stream);
/* Batched runs: `count` independent loops in ONE launch, one persistent CTA per run (runs beyond one per SM wait for
 * a free SM).  Each record carries what dcr_sdrf_run takes per run; remove_edges and guard apply to every run.  `runs`
 * is a host array; the library packs one device descriptor per run into `workspace` (device memory of at least
 * dcr_sdrf_batch_workspace_bytes(count) bytes, 8-byte aligned, reusable once the launch has been consumed in stream
 * order) with one host-to-device copy on `stream`, then launches; it allocates nothing.  Status 1 before any launch
 * for count < 1, a null state, the same state twice, states of different DCR_SDRF_MODE_* or a short workspace.
 * Every run then behaves exactly as its own dcr_sdrf_run call would. */
typedef struct dcr_sdrf_batch_run {      /* one run of dcr_sdrf_run_batch; pointers are device pointers */
    dcr_sdrf* state;
    int32_t loops, forced_choice;        /* as in dcr_sdrf_run                                          */
    double removal_bound, tau;
    const double* uniforms; int64_t n_uniforms;
    int32_t* log;                        /* int32[loops][8]                                              */
    dcr_sdrf_result* result;
} dcr_sdrf_batch_run;
int64_t dcr_sdrf_batch_workspace_bytes(int count);
int dcr_sdrf_run_batch(const dcr_sdrf_batch_run* runs, int count, int remove_edges, double guard,
                       void* workspace, int64_t workspace_bytes, void* stream);
/* Improvements (fp64 of the fp32 differences, candidate order) of the pending iteration after NEED_HOST. */
int dcr_sdrf_pending_improvements(dcr_sdrf* s, double* out, int64_t capacity, void* stream);
/* Current number of directed entries (synchronises). */
int64_t dcr_sdrf_nnz(dcr_sdrf* s);
/* Export the current graph: rowptr[n+1], and per directed entry in NETWORKX ORDER the neighbour id
 * (`order_out`), plus, in SORTED order per row, colidx / curvature (fp32, cuda flavour) / support. */
int dcr_sdrf_export(dcr_sdrf* s, int32_t* rowptr, int32_t* order_out, int32_t* colidx_sorted, float* c32_sorted,
                    int32_t* tri_sorted, void* stream);

/* Insertion-order rows INCLUDING the self entries (see dcr_sdrf_create): rowptr_order[n+1] and order_out[rowptr_order[n]]
 * (at most nnz + n entries).  dcr_sdrf_export refuses order_out for a state that has self entries. */
int dcr_sdrf_export_order(dcr_sdrf* s, int32_t* rowptr_order, int32_t* order_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DCR_H_ */
