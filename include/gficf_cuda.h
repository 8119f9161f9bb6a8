/* gficf_cuda.h -- C ABI of the B200-native Phenograph Jaccard edge-weighting path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no R / Rcpp / torch
 * types.  The library behind it (gficf_b200/libgficf_cuda.so, built by nvcc for
 * sm_100a) replaces the bodies of the two native functions that gficf's Rcpp
 * shims call:
 *
 *   rcpp_parallel_jaccard_coef(NumericMatrix mat, bool printOutput)
 *       reference: src/rcpp_parallel_jaccard_coeff.cpp:58-80 (worker :24-55),
 *       bound from R through src/RcppExports.cpp:61-70
 *   jaccard_coeff(NumericMatrix idx, bool printOutput)
 *       reference: src/jaccard_coeff.cpp:19-45,
 *       bound from R through src/RcppExports.cpp:36-45
 *
 * Conventions (all the reference's):
 *   idx  n x k doubles, COLUMN-major (element (i,j) at idx[j*n+i]), values are
 *        1-based neighbour ids (R coerces uwot's integer matrix to REALSXP at
 *        src/RcppExports.cpp:40,65)
 *   out  (n*k) x 3 doubles, COLUMN-major, i.e. three contiguous arrays of
 *        E = n*k doubles: from[], to[], weight[]
 *        (rcpp_parallel_jaccard_coeff.cpp:67, jaccard_coeff.cpp:21)
 *
 * Every function returns 0 on success and a GFICF_E_* code otherwise; when an
 * `err` buffer is supplied a NUL-terminated message is written to it.  Nothing
 * here calls the R API, longjmps or throws across the boundary.  There is no
 * CPU fallback: without a usable CUDA device the calls fail with
 * GFICF_E_CUDA.
 */
#ifndef GFICF_CUDA_H
#define GFICF_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes ------------------------------------------------------- */
#define GFICF_OK 0
#define GFICF_E_ARG 1    /* bad argument (null pointer, negative size, unknown mode ...)   */
#define GFICF_E_RANGE 2  /* a neighbour id is NaN, non-integer or outside [1,n]: the        */
                         /* reference indexes out of bounds there (UB at                    */
                         /* rcpp_parallel_jaccard_coeff.cpp:28 / jaccard_coeff.cpp:30)      */
#define GFICF_E_CUDA 3   /* CUDA runtime / driver error, or no device                       */
#define GFICF_E_NCCL 4   /* NCCL could not be loaded or a collective failed                 */
#define GFICF_E_LIMIT 5  /* size beyond what the path supports (n*k or n >= 2^31, as in the */
                         /* reference, whose row index is an `int`)                         */

/* ---- output modes ------------------------------------------------------- */
/* Fixed slots, multiset intersection: output row r = i*k+j, rows with an empty
 * intersection stay (0,0,0).  = rcpp_parallel_jaccard_coef
 * (rcpp_parallel_jaccard_coeff.cpp:41-52). */
#define GFICF_MODE_PARALLEL 0
/* Compacted rows, unique-set intersection: a row is emitted (r++) only when
 * u>0, trailing rows stay zero.  = jaccard_coeff (jaccard_coeff.cpp:33-39). */
#define GFICF_MODE_SERIAL 1

/* ---- flag bits reported by the device kernels (d_flags) ------------------ */
#define GFICF_FLAG_BAD_ID 1u     /* layout pre-pass met an id that is NaN / non-integer / out of [1,n] */
#define GFICF_FLAG_DUP_ID 2u     /* some row lists the same id twice: the exact kernels must be used  */
#define GFICF_FLAG_HASH_FAIL 4u  /* a row found no collision-free hash: the exact kernels must be used */

/* ======================================================================== *
 *  Host-buffer entry points (what the Rcpp functions call)
 * ======================================================================== */

/* The whole path on host buffers: H2D of idx, layout pre-pass, Jaccard
 * kernel(s), D2H of the three output columns.  `out` is fully written
 * (the caller need not zero it).  n_devices >= 1 shards cell rows over that
 * many GPUs of this node (NCCL all-gather of the int32 index slabs, each GPU
 * returns its own edge slab); n_devices == 0 uses the value set by
 * gficf_cuda_set_devices() (default 1).
 *
 * Replaces: rcpp_parallel_jaccard_coef body (mode 0) and jaccard_coeff body
 * (mode 1; always one device, its rows are compacted across the whole matrix).
 * If n_written is non-NULL it receives the number of emitted rows in mode 1
 * (the reference's final r) and -1 in mode 0. */
int gficf_cuda_jaccard(const double* idx_colmajor, int64_t n, int32_t k, double* out_colmajor,
                       int32_t n_devices, int32_t mode, int64_t* n_written, char* err,
                       size_t errlen);

/* Same call on an INTEGER matrix (R INTSXP: int32, column-major, 1-based; NA_integer_ is rejected
 * like any out-of-range id).  uwot hands clustcells() an integer matrix, which the reference's
 * shim coerces to double first (src/RcppExports.cpp:65); taking it as it is halves the H2D bytes
 * (SURVEY 8f row 2). */
int gficf_cuda_jaccard_i32(const int32_t* idx_colmajor, int64_t n, int32_t k, double* out_colmajor,
                           int32_t n_devices, int32_t mode, int64_t* n_written, char* err,
                           size_t errlen);

/* Device-count option that R/clustCells.R's new `n.gpu` argument sets without
 * changing the arity of the registered .Call routines
 * (src/RcppExports.cpp:85-92).  Also read once from the environment variable
 * GFICF_CUDA_DEVICES. */
int gficf_cuda_set_devices(int32_t n_devices);
int gficf_cuda_get_devices(void);
/* Number of visible CUDA devices (0 if none / no driver). */
int gficf_cuda_device_count(void);

/* Page-locked host buffers so that the H2D / D2H legs run at PCIe speed
 * without a staging copy (ordinary pageable memory is accepted everywhere,
 * it is staged through internal pinned buffers). */
int gficf_cuda_host_alloc(void** p, size_t bytes);
int gficf_cuda_host_free(void* p);
/* Page-lock memory the caller already owns (e.g. a shared-memory mapping that several
 * ranks read their rows from / write their slabs to). */
int gficf_cuda_host_register(void* p, size_t bytes);
int gficf_cuda_host_unregister(void* p);

/* Drop the cached device / pinned workspaces and NCCL communicators. */
int gficf_cuda_release(void);

/* Timings (milliseconds, CUDA events) of the last gficf_cuda_jaccard call on
 * this thread: [0] H2D, [1] layout pre-pass, [2] Jaccard kernel(s),
 * [3] D2H / output phase (overlapped portion included), [4] whole call wall-clock,
 * [5] index all-gather (n_devices>1), [6] kernels launched, [7] bytes copied device -> host. */
int gficf_cuda_last_timings(double* ms8);

/* How the last gficf_cuda_jaccard / _i32 / _rank call on this thread produced its output columns:
 * *out_mode 1 = dma (the device wrote 24 B/edge, the copy engine moved them), 2 = host (only the
 * 1-byte intersection counts crossed PCIe; host threads wrote from = i+1, to = idx(i,j),
 * weight = table[u] straight into the caller's matrix, bit-identical by construction), 3 = hybrid
 * (both at once, (column, row-chunk) pieces claimed dynamically); *host_share = share of the pieces
 * written by host threads; *d2h_bytes / *h2d_bytes = bytes that crossed PCIe towards the host / the
 * device (an f64 matrix is narrowed to int32 on the host while it streams -- its values are integer
 * ids -- so it costs 4 bytes per id; GFICF_CUDA_H2D_NARROW=0 sends the doubles).  The mode is chosen
 * per call: hybrid for page-locked output, host for pageable output (what R passes), dma for k > 255
 * or the serial export; GFICF_CUDA_OUT_MODE=dma|host|hybrid overrides, GFICF_CUDA_EXPAND_THREADS
 * sets the number of host threads. */
int gficf_cuda_last_output(int32_t* out_mode, double* host_share, double* d2h_bytes, double* h2d_bytes);

/* The host half of the counts-over-PCIe output on its own: rows [row_lo,row_hi) of the fixed-slot
 * export written into out_colmajor ((n*k) x 3) from the caller's matrix (elem_bytes 8 = double,
 * 4 = int32; column-major, 1-based) and the rows' intersection counts as the device kernels produce
 * them (gficf_cuda_jaccard_counts_dev, k <= 255; counts[(i-row_lo)*k + j]).  Pure host code, no
 * device needed: for hosts that collect the 1-byte counts themselves (several nodes, a job queue).
 * Replaces the stores rcpp_parallel_jaccard_coeff.cpp:48-52.  n_threads <= 0: automatic. */
int gficf_cuda_expand_host(const void* idx_colmajor, int32_t elem_bytes, int64_t n, int32_t k,
                           const uint8_t* counts, int64_t row_lo, int64_t row_hi, double* out_colmajor,
                           int32_t n_threads);

/* ======================================================================== *
 *  One process per GPU (MPI-style hosts, torchrun): every rank calls the same
 *  function on the SAME host matrices (shared memory mapped by all ranks, or
 *  any buffers when a rank only needs its own rows) and handles its own row slab:
 *  H2D of its rows, layout pre-pass, NCCL all-gather of the int32 index slabs,
 *  fused kernel, D2H of its edge slab -- so the PCIe legs of the ranks run in
 *  parallel.  The communicator is built from an id created on one rank and
 *  distributed by the host framework.
 * ======================================================================== */
#define GFICF_COMM_ID_BYTES 128
int gficf_cuda_comm_unique_id(void* id128);
int gficf_cuda_comm_init_rank(const void* id128, int32_t nranks, int32_t rank, int32_t device,
                              char* err, size_t errlen);
int gficf_cuda_comm_destroy(void);
/* Collective over the communicator: rank r reads rows [r*ceil(n/R), ...) of
 * idx_colmajor and writes the same rows' edges into out_colmajor (parallel-export
 * semantics, rcpp_parallel_jaccard_coeff.cpp:24-55).  Errors (bad ids, CUDA failures)
 * are agreed on by all ranks before anyone returns. */
int gficf_cuda_jaccard_rank(const double* idx_colmajor, int64_t n, int32_t k, double* out_colmajor,
                            char* err, size_t errlen);

/* ======================================================================== *
 *  Peer-memory gather (fused compute + gather over NVLink, one process per GPU):
 *  the host rank allocates the count buffer and exports it (CUDA IPC); the other
 *  ranks map it and pass the mapped pointer as the output of their count kernel, so
 *  the kernel's epilogue stores its 1-byte results straight into the host rank's HBM.
 *  gficf_cuda_signal_dev raises a flag in that buffer when the stream reaches it,
 *  gficf_cuda_wait_dev holds a stream until a flag reaches a value (bounded spin;
 *  GFICF_FLAG_PEER_TIMEOUT on give-up): the one ack per step of the protocol below.
 * ======================================================================== */
#define GFICF_IPC_HANDLE_BYTES 64
#define GFICF_FLAG_PEER_TIMEOUT 8u
int gficf_cuda_ipc_alloc(size_t bytes, void** dptr, void* handle64); /* cudaMalloc + zero + export */
int gficf_cuda_ipc_open(const void* handle64, void** dptr);          /* map a peer's allocation   */
int gficf_cuda_ipc_close(void* dptr);
int gficf_cuda_ipc_free(void* dptr);
int gficf_cuda_signal_dev(uint32_t* d_flag, uint32_t value, void* stream);
int gficf_cuda_wait_dev(const uint32_t* d_flag, uint32_t expected, uint32_t* d_flags, void* stream);

/* The gather itself (no data flags, no fences, one launch per rank and step;
 * gficf_b200.sharding.PeerGather).  Every count byte carries the step's parity in bit 7
 * (`tag` = 0x00 / 0x80, alternating from step to step; k <= 127), so a byte is its own ready flag:
 *   gficf_cuda_jaccard_counts_tagged_dev   the count kernel of gficf_cuda_jaccard_counts_dev, storing
 *                                          u | tag (d_u: typically the host rank's mapped buffer).  For
 *                                          k <= 32 a warp owns groups of 8 consecutive rows and sends a
 *                                          group with 16-byte vector stores (few full NVLink packets
 *                                          instead of one or two <= 30-byte packets per row: what keeps
 *                                          7 peers from saturating one GPU's ingress packet rate);
 *                                          tag | GFICF_TAG_ROW_STORES keeps row-by-row byte stores (the
 *                                          faster kernel by ~15 %: the better choice up to ~4 peers)
 *   gficf_cuda_expand_stream_dev           host rank: expands the rows of n_seg row segments (one per
 *                                          contributing rank; seg_lo/seg_hi are HOST arrays of absolute
 *                                          rows) while the peers are still storing into d_u, polling each
 *                                          byte until its parity equals `tag`.  d_u, d_from, d_to, d_w are
 *                                          indexed by ABSOLUTE edge number i*k+j.  timeout_ms bounds
 *                                          every spin (0: GFICF_CUDA_PEER_TIMEOUT_MS, default 20000);
 *                                          GFICF_FLAG_PEER_TIMEOUT in *d_flags means the output is invalid. */
#define GFICF_TAG_ROW_STORES 0x100u
int gficf_cuda_jaccard_counts_tagged_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                         int64_t row_hi, uint8_t* d_u, uint32_t tag, uint32_t* d_flags,
                                         void* stream);
int gficf_cuda_expand_stream_dev(const int32_t* d_idx_i32, int32_t k, const int64_t* seg_lo,
                                 const int64_t* seg_hi, int32_t n_seg, const uint8_t* d_u, double* d_from,
                                 double* d_to, double* d_w, uint32_t tag, int64_t timeout_ms,
                                 uint32_t* d_flags, void* stream);

/* ======================================================================== *
 *  Device-buffer entry points (resident data: the benchmarked kernels, and
 *  the building blocks a multi-process (one rank per GPU) caller shards with)
 *  All pointers are device pointers on the CURRENT device; `stream` is a
 *  cudaStream_t passed as void* (NULL = default stream).  Asynchronous.
 * ======================================================================== */

/* Row stride (in int32 elements) of the device index layout for a given k:
 * rows are padded so that every row is read with 16-byte vector loads and
 * never straddles an extra 64-byte DRAM burst (k<=4:4, <=8:8, <=16:16, <=32:32,
 * else k rounded up to a multiple of 16).  Pad entries hold -2. */
int32_t gficf_cuda_row_stride(int32_t k);

/* Layout pre-pass for rows [row_lo,row_hi): n x k f64 column-major 1-based
 * (device copy of the R matrix, leading dimension ld_rows >= row count held;
 * element (i,j) of the FULL matrix is at d_idx_f64[j*ld_rows + (i-ld_row0)])
 * -> int32 row-major 0-based with gficf_cuda_row_stride(k) ints per row,
 * written at d_idx_i32[i*stride ...].  Validates ids (sets GFICF_FLAG_BAD_ID
 * in *d_flags).
 * Replaces the per-edge strided row copies of
 * rcpp_parallel_jaccard_coeff.cpp:30-36. */
int gficf_cuda_layout_dev(const double* d_idx_f64, int64_t ld_rows, int64_t ld_row0, int64_t n,
                          int32_t k, int64_t row_lo, int64_t row_hi, int32_t* d_idx_i32,
                          uint32_t* d_flags, void* stream);

/* Same, from an int32 n x k ROW-major 0-based matrix with k ints per row
 * (what a GPU kNN would hand over): pads rows, validates ids in [0,n). */
int gficf_cuda_pad_dev(const int32_t* d_idx_dense, int64_t n, int32_t k, int64_t row_lo,
                       int64_t row_hi, int32_t* d_idx_i32, uint32_t* d_flags, void* stream);

/* Jaccard edges of rows [row_lo,row_hi), gathering from the full padded index
 * (all n rows must be resident).  Fixed-slot output (mode 0 semantics):
 * d_from/d_to/d_w point at the slab's first element, i.e. edge (i,j) is
 * written at [(i-row_lo)*k + j].  Sets GFICF_FLAG_DUP_ID / GFICF_FLAG_HASH_FAIL
 * in *d_flags when the fast kernel's result must not be used (then call
 * gficf_cuda_jaccard_exact_dev).
 * Replaces JCoefficient::operator() (rcpp_parallel_jaccard_coeff.cpp:24-55). */
int gficf_cuda_jaccard_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                           int64_t row_hi, double* d_from, double* d_to, double* d_w,
                           uint32_t* d_flags, void* stream);

/* Same rows, but only the intersection counts u (one byte per edge when
 * k<=255, two bytes for 255<k<=1024; layout [(i-row_lo)*k+j]); the compact form
 * that crosses NVLink / feeds gficf_cuda_expand_dev.  GFICF_E_LIMIT for k>1024
 * (use gficf_cuda_jaccard_exact_dev). */
int gficf_cuda_jaccard_counts_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                  int64_t row_hi, uint8_t* d_u, uint32_t* d_flags, void* stream);

/* Exact (any input: duplicate ids inside a row allowed; any k <= 65535) counts
 * for rows [row_lo,row_hi): set_semantics==0 -> multiset min-count intersection
 * (std::set_intersection, rcpp_parallel_jaccard_coeff.cpp:41-46);
 * set_semantics==1 -> number of distinct common ids (Rcpp::intersect,
 * jaccard_coeff.cpp:33).  d_u holds uint8 per edge when k<=255, else uint16.
 * Slow path, O(k^2) per edge. */
int gficf_cuda_jaccard_exact_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                 int64_t row_hi, int32_t set_semantics, void* d_u, void* stream);

/* Counts -> edge rows for rows [row_lo,row_hi) (d_u: uint8 per edge when
 * k<=255, else uint16; d_from/d_to/d_w point at the slab's first element).
 * mode 0: fixed slots, edge (i,j) at [(i-row_lo)*k+j], zeros where u==0.
 * mode 1: rows with u>0 compacted in (i,j) order from element 0 on, the tail
 *         up to the slab's (row_hi-row_lo)*k rows zero-filled; d_scratch must
 *         hold gficf_cuda_expand_scratch_bytes(slab edges) bytes and the
 *         emitted-row count is stored to *d_n_written (int64, device memory).
 * Replaces the conditional stores rcpp_parallel_jaccard_coeff.cpp:48-52 /
 * jaccard_coeff.cpp:34-39. */
int gficf_cuda_expand_dev(const int32_t* d_idx_i32, int32_t k, int64_t row_lo, int64_t row_hi,
                          const void* d_u, int32_t mode, double* d_from, double* d_to, double* d_w,
                          void* d_scratch, int64_t* d_n_written, void* stream);
size_t gficf_cuda_expand_scratch_bytes(int64_t slab_edges);

/* ---- the step after the path (SURVEY 8f row 1): counts -> the graph the community detection
 * reads.  Replaces, on the device, relations[relations[,3]>0,] + igraph::graph.data.frame +
 * as_adjacency_matrix (parallel edges summed) of R/clustCells.R:66-69,81 and the strictly-lower-
 * triangle scan of src/RModularityOptimizer.cpp:67-83. ---- */
#define GFICF_FLAG_ISOLATED 16u /* informational: some cell keeps no edge of its own (u == 0 on its whole row) */
/* Count kernel that also sets bit 7 of an edge's byte when the edge is mutual (i is in N(t)); k <= 127. */
int gficf_cuda_jaccard_counts_mutual_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                         int64_t row_hi, uint8_t* d_um, uint32_t* d_flags, void* stream);
/* CSC of the strictly lower triangle of the symmetric weighted adjacency matrix over igraph's vertex
 * numbering (first appearance in c(from, to) of the kept rows: cells with an edge of their own in
 * cell order, then cells that only appear as targets in order of the first edge naming them; cells
 * in no kept edge are not vertices):
 *   d_colptr[n+1] (int64; entries beyond the vertex count repeat the total), d_row / d_w with capacity
 *   cap >= n*k entries, rows ascending inside a column (column = node1, row = node2 of the
 *   reference's edge list, both vertex ids), d_vertex_cell[n] (vertex id -> 1-based cell id; may be
 *   NULL), *d_n_vertices (device int64; may be NULL).  d_um covers all n rows.
 * Valid when *d_flags stays free of GFICF_FLAG_DUP_ID / _HASH_FAIL. */
size_t gficf_cuda_snn_scratch_bytes(int64_t n, int64_t cap);
int gficf_cuda_snn_lower_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, const uint8_t* d_um,
                             int64_t* d_colptr, int32_t* d_row, double* d_w, int64_t cap,
                             int32_t* d_vertex_cell, int64_t* d_n_vertices, void* d_scratch,
                             uint32_t* d_flags, void* stream);
/* The same step on HOST buffers, from the caller's kNN matrix (elem_bytes 8 = double, 4 = int32;
 * column-major, 1-based) to the arrays RunModularityClusteringCpp's edge-list loop produces
 * (src/RModularityOptimizer.cpp:67-88): H2D, layout pre-pass, count kernel with the mutual bit, the
 * graph kernels, D2H of colptr / row / weight / vertex map -- 12 bytes per undirected edge instead of
 * the 24 bytes per directed edge slot of the edge matrix.  colptr has n+1 entries (the first
 * *n_vertices + 1 are meaningful), row / w have capacity cap (n*k always suffices); *nnz receives
 * the number of entries.  GFICF_E_LIMIT: k > 127 or a row lists an id twice (use gficf_cuda_jaccard
 * and the host graph build there).  One device. */
int gficf_cuda_snn_lower(const void* idx_colmajor, int32_t elem_bytes, int64_t n, int32_t k,
                         int64_t* colptr, int32_t* row, double* w, int64_t cap, int32_t* vertex_cell,
                         int64_t* n_vertices, int64_t* nnz, char* err, size_t errlen);

/* ---- another step of the package that clustcells()'s labels feed (SURVEY 8f row 4): two-sided
 * Mann-Whitney U per gene with tie correction and continuity correction, and the log2 fold change.
 * Replaces the body of rcpp_parallel_WMU_test (src/rcpp_parallel_mann_whitney.cpp:106-127, worker
 * :12-103; helpers src/mann_whitney.cpp:17-131; caller R/deGenes.R:44-54).
 * mat_x: n_genes x n1, mat_y: n_genes x n2 doubles, COLUMN-major (R matrices: genes are rows, the cells
 * of the cluster / of all other clusters are columns); out: n_genes x 2 column-major --
 * column 0 the p-value, column 1 log2(mean(x+1) / mean(y+1)).  The device sorts every gene's
 * n1+n2 values (CTA per gene, radix sort) and produces the continuity-corrected z and the mean
 * ratio in exact integer / correctly-rounded arithmetic; the normal cdf (GSL in the reference,
 * restated from the published algorithm) and log2 are evaluated on the host, once per gene.
 * Values must not be NaN (the reference's sort is undefined there). ---- */
int gficf_cuda_wmu_test(const double* mat_x, const double* mat_y, int64_t n_genes, int64_t n1, int64_t n2,
                        double* out, char* err, size_t errlen);

/* The loop of findClusterMarkers (R/deGenes.R:44-54) in one call: for every cluster c, cluster c's cells
 * against all other cells.  mat: n_genes x n_cells doubles, COLUMN-major; cluster: n_cells 0-based ids
 * in [0, n_clusters); out: n_genes x 2 x n_clusters doubles, column-major.  Block c (out + c*2*n_genes)
 * is, bit for bit, what gficf_cuda_wmu_test returns for mat[, cluster == c] against
 * mat[, cluster != c] (both with the cells in ascending order).  The matrix is uploaded once and each
 * gene sorted once: its ranks, tie groups, tie term and distinct count do not depend on the split,
 * only the per-cluster rank sums and the two fold-change means do.
 * GFICF_E_ARG: negative size, null pointer, n_clusters < 2, an id outside [0, n_clusters) or a cluster
 * without cells.  GFICF_E_LIMIT: more than 8192 clusters (12 bytes of rank-sum accumulators per cluster
 * in each CTA's shared memory) or n_cells >= 2^31.  Timings as for gficf_cuda_wmu_test.  One device. */
int gficf_cuda_wmu_markers(const double* mat, int64_t n_genes, int64_t n_cells, const int32_t* cluster,
                           int32_t n_clusters, double* out, char* err, size_t errlen);

/* gficf_cuda_wmu_markers on a sparse matrix: genes x cells in compressed-column form, the slots of R's
 * dgCMatrix as they are -- colptr = p (n_cells + 1 entries, colptr[0] = 0, never decreasing), row = i
 * (0-based gene of each stored value, strictly increasing inside a column), x = the stored values;
 * nnz = colptr[n_cells].  cluster, n_clusters, out and the timings as for gficf_cuda_wmu_markers, and out
 * equals, bit for bit, what gficf_cuda_wmu_markers returns for the densified matrix.  Stored zeros (and
 * -0.0) are zeros.  Only the stored values cross PCIe (12 bytes each, plus 4 per cell for colptr); the device
 * turns them gene-major (stable radix sort by gene), and the rank and means kernels read only them.
 * Device memory: 41.5 bytes per stored value (12 of input, 29.5 of transpose scratch that also holds the
 * gene-major copy), 12 per cell and 12 per gene, the n_genes x n_clusters results (16 bytes each), and the
 * rank kernel's sort scratch of 24 bytes x the largest number of stored values of a gene, per resident CTA.
 * GFICF_E_ARG: as gficf_cuda_wmu_markers, and a malformed matrix -- colptr[0] != 0 or colptr decreasing
 * (checked on the host before any upload), a row id outside [0, n_genes) or row ids not strictly increasing
 * in a column (checked on the device before any kernel indexes with them).  GFICF_E_LIMIT: as
 * gficf_cuda_wmu_markers, and n_genes >= 2^31 - 1.  One device. */
int gficf_cuda_wmu_markers_csc(const int32_t* colptr, const int32_t* row, const double* x, int64_t n_genes,
                               int64_t n_cells, const int32_t* cluster, int32_t n_clusters, double* out, char* err,
                               size_t errlen);

/* ---- the data-parallel pieces of the community detection that reads the graph (SURVEY 8f row 3;
 * reference src/ModularityOptimizer.cpp).  The sequential, RNG-ordered local moving loop (:484-583)
 * stays on the host; these are the steps around it that touch every edge:
 *   gficf_cuda_network_dev          matrixToNetwork :761-806 + Network ctor :169-188: the lower-triangle
 *                                   CSC of gficf_cuda_snn_lower_dev (node1 = column < node2 = row, rows
 *                                   ascending) -> symmetric CSR firstNeighborIndex / neighbor / edgeWeight,
 *                                   nodeWeight (= total edge weight per node :272-284), and
 *                                   *d_total_w = getTotalEdgeWeight() :268-270
 *   gficf_cuda_network_quality_dev  VOSClusteringTechnique::calcQualityFunction :462-482 for a clustering
 *                                   (cluster ids 0..n_clusters-1; self_links = the network's
 *                                   totalEdgeWeightSelfLinks), plus the cluster weights it forms
 *   gficf_cuda_network_reduce_dev   Network::createReducedNetwork :322-373 (nodes per cluster :106-118):
 *                                   one node per cluster, neighbours in the reference's order of first
 *                                   appearance; *d_r_self_links = the reduced network's
 *                                   totalEdgeWeightSelfLinks (self_links of the parent plus every edge that
 *                                   stays inside a cluster), *d_r_total_w = its getTotalEdgeWeight()
 * Parity: every output is bit-identical to the reference.  Per-node / per-cluster / per-cluster-pair
 * sums are added in the reference's order by one warp; the sums the reference forms sequentially over
 * the whole edge list (total edge weight, the intra-cluster weight of the quality function, the
 * self-link total) are replayed exactly: inside one binade of the running sum every addition is an
 * integer increment, which composes associatively, and the few additions that cross a binade are done
 * in floating point (network_kernels.cuh).
 * Device pointers on the current device; d_first has n_nodes + 1 int64 entries; neighbour and cluster ids
 * are int32 (the reference's int); n_edges = d_first[n_nodes], the directed edge count, below 2^31.
 * d_scratch: gficf_cuda_network_scratch_bytes(n_nodes, n_items) bytes with n_items >= nnz (network) or
 * n_edges (quality, reduce).  Flags raised in *d_flags (zero it first): GFICF_FLAG_NET_WEIGHT -- an edge
 * weight that is not > 0 and finite; GFICF_FLAG_NET_RANGE -- an entry that is not strictly below the
 * diagonal, or a row / cluster id out of range; the outputs are then unspecified.
 * All three synchronise `stream` (the sequential sums and two entry counts are read back while they
 * run).  reduce returns the number of reduced (directed) edges in *n_reduced_edges -- GFICF_E_LIMIT
 * with the needed number there when r_cap is too small. ---- */
#define GFICF_FLAG_NET_WEIGHT 32u
#define GFICF_FLAG_NET_RANGE 64u
size_t gficf_cuda_network_scratch_bytes(int64_t n_nodes, int64_t n_items);
int gficf_cuda_network_dev(const int64_t* d_colptr, const int32_t* d_row, const double* d_w, int64_t n_vertices,
                           int64_t nnz, int64_t* d_first, int32_t* d_neighbor, double* d_edge_w, double* d_node_w,
                           double* d_total_w, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                           void* stream);
int gficf_cuda_network_quality_dev(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                                   const double* d_node_w, int64_t n_nodes, int64_t n_edges,
                                   const int32_t* d_cluster, int32_t n_clusters, double resolution,
                                   double self_links, const double* d_total_w, double* d_cluster_w,
                                   double* d_quality, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                                   void* stream);
int gficf_cuda_network_reduce_dev(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                                  const double* d_node_w, int64_t n_nodes, int64_t n_edges,
                                  const int32_t* d_cluster, int32_t n_clusters, double self_links,
                                  int64_t* d_r_first, int32_t* d_r_neighbor, double* d_r_edge_w, int64_t r_cap,
                                  double* d_r_node_w, double* d_r_self_links, double* d_r_total_w,
                                  int64_t* n_reduced_edges, void* d_scratch, size_t scratch_bytes,
                                  uint32_t* d_flags, void* stream);

/* Caps the resident CTAs per SM of the persistent Jaccard kernels launched from THIS thread (0 = what
 * the occupancy allows: the default).  For callers that run two of them side by side on different
 * streams: the peer gather's peers count most of their rows with 3 CTAs per SM while a 1-CTA-per-SM
 * fused kernel stores finished doubles of the other rows straight into the host rank's output. */
int gficf_cuda_set_launch_ctas_per_sm(int32_t ctas_per_sm);

/* Launch geometry of the last fast-kernel launch on this thread (for the
 * bench record): grid, block, dynamic smem bytes, kernels launched. */
int gficf_cuda_last_launch(int32_t* grid, int32_t* block, int32_t* smem_bytes, int32_t* variant);

/* Library / build identification, e.g. "gficf_cuda 0.1 sm_100a". */
const char* gficf_cuda_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GFICF_CUDA_H */
