// network_plan.h -- the launch sequences of the network kernels (network_kernels.cuh) and their
// scratch layout.  Included by gficf_cuda.cu (after its error helpers) for the product, and by
// tests/cuda_emu/network_emu.cpp with GFICF_CUDA_EMU defined, so the SAME sequence of launches is
// what the CPU test suite runs against the oracle and what runs on the B200.
#pragma once
#include "gficf_cuda.h"
#include "network_kernels.cuh"
#include "plan_common.h"

namespace gficf {

// number of bits needed for values in [0, max_value]
inline int bits_for(long long max_value) {
  int b = 0;
  while (max_value > 0) {
    ++b;
    max_value >>= 1;
  }
  return b;
}

// scratch of the network entry points: nn = node capacity, cap = item capacity (entries of the
// lower triangle / directed edges of the network, whichever call is the largest; >= nn)
struct NetScratch {
  unsigned long long* keys[2];
  unsigned* vals[2];
  unsigned* aux;  // column of a lower entry / network edge of a cross entry
  unsigned* perm;  // nodes sorted by cluster
  int* head;
  unsigned* seg_start;
  long long* seg_id;
  unsigned long long* seg_key;
  double* seg_w;
  int* hist;
  long long* offsets;
  long long* block_sums;
  long long* total;
  int* cnt;
  long long *ptr_a, *ptr_b;
  double* dbl_b;  // (cw * cw) * resolution per cluster
  SeqState* seq_state;
  SeqFn* seq_fn;
  double* sums;  // [0] intra-cluster weight of calcQualityFunction
  long long* ptr_c;  // first traversal position of every node of the cluster-sorted list
  int* cnt_b;        // its degree
  size_t bytes;
};

inline NetScratch net_scratch_layout(char* base, long long nn, long long cap) {
  NetScratch s;
  ScratchCarver c{base};
  if (cap < nn) cap = nn;
  const long long n_tiles = (cap + kRadixTile - 1) / kRadixTile + 1;
  const long long scan_len = (256 * n_tiles > cap ? 256 * n_tiles : cap) + 1;
  for (int b = 0; b < 2; ++b) s.keys[b] = c.take<unsigned long long>(cap);
  for (int b = 0; b < 2; ++b) s.vals[b] = c.take<unsigned>(cap);
  s.aux = c.take<unsigned>(cap);
  s.perm = c.take<unsigned>(nn);
  s.head = c.take<int>(cap);
  s.seg_start = c.take<unsigned>(cap);
  s.seg_id = c.take<long long>(cap + 1);
  s.seg_key = c.take<unsigned long long>(cap);
  s.seg_w = c.take<double>(cap);
  s.hist = c.take<int>(256 * n_tiles);
  s.offsets = c.take<long long>(256 * n_tiles + 1);
  s.block_sums = c.take<long long>(scan_len / kScanBlock + 2);
  s.total = c.take<long long>(1);
  s.cnt = c.take<int>(nn + 1);
  s.ptr_a = c.take<long long>(nn + 1);
  s.ptr_b = c.take<long long>(nn + 1);
  s.dbl_b = c.take<double>(nn + 1);
  s.seq_state = c.take<SeqState>(1);
  s.seq_fn = c.take<SeqFn>(kSeqMaxBlocks);
  s.sums = c.take<double>(8);
  s.ptr_c = c.take<long long>(nn + 1);
  s.cnt_b = c.take<int>(nn + 1);
  s.bytes = c.bytes;
  return s;
}

struct NetCtx {
  net_stream_t st;
  NetScratch sc;
  unsigned* flags;
  int max_ctas;  // cap of the grid-stride launches (a multiple of the SM count on the device)
};

inline long long net_grid(const NetCtx& cx, long long items, int per_cta) {
  long long g = (items + per_cta - 1) / per_cta;
  if (g < 1) g = 1;
  return g < cx.max_ctas ? g : cx.max_ctas;
}

// exclusive scan of m int counts into int64 offsets; out[m] = total
inline void net_scan(const NetCtx& cx, const int* cnt, long long m, long long* out) {
  if (m <= 0) {
    net_zero(cx.st, out, 8);
    return;
  }
  const long long nb = (m + kScanBlock - 1) / kScanBlock;
  long long* block_sums = cx.sc.block_sums;
  long long* total = cx.sc.total;
  GFICF_LAUNCH(cx.st, scan_block_sums_kernel, nb, kScanBlock, cnt, m, block_sums);
  GFICF_LAUNCH(cx.st, compact_scan_kernel, 1, 1024, block_sums, nb, total);
  GFICF_LAUNCH(cx.st, scan_finish_kernel, nb, kScanBlock, cnt, m, block_sums, total, out);
}

// stable sort of (keys[start], vals[start])[0, n) by the low nbits of the key; returns the buffer
// index that holds the result
inline int net_radix_sort(const NetCtx& cx, int start, long long n, int nbits) {
  int cur = start;
  if (n <= 1) return cur;
  const long long n_tiles = (n + kRadixTile - 1) / kRadixTile;
  const long long grid = n_tiles < cx.max_ctas ? n_tiles : cx.max_ctas;
  for (int shift = 0; shift < nbits; shift += 8) {
    const unsigned long long* kin = cx.sc.keys[cur];
    const unsigned* vin = cx.sc.vals[cur];
    unsigned long long* kout = cx.sc.keys[cur ^ 1];
    unsigned* vout = cx.sc.vals[cur ^ 1];
    int* hist = cx.sc.hist;
    long long* offsets = cx.sc.offsets;
    GFICF_LAUNCH(cx.st, radix_hist_kernel, grid, kRadixThreads, kin, n, shift, n_tiles, hist);
    net_scan(cx, hist, 256 * n_tiles, offsets);
    GFICF_LAUNCH(cx.st, radix_scatter_kernel, grid, kRadixThreads, kin, vin, kout, vout, n, shift, n_tiles,
                 (const long long*)offsets);
    cur ^= 1;
  }
  return cur;
}

// out[0] = scale * (((s0 + x[0]) + x[1]) + ... + x[n-1]), every addition rounded like the sequential
// loop rounds it (network_kernels.cuh, "The reference's whole-graph sums, bit for bit").  x >= 0.
// Synchronises the stream (the position is read back every kSeqBatch steps).
#ifdef GFICF_CUDA_EMU
constexpr int kSeqBatch = 2;
#else
constexpr int kSeqBatch = 24;
#endif
inline void net_seq_sum(const NetCtx& cx, const double* x, long long n, double s0, double scale, double* out) {
  SeqState* st = cx.sc.seq_state;
  SeqFn* bf = cx.sc.seq_fn;
  unsigned* flags = cx.flags;
  const long long grid = cx.max_ctas < kSeqMaxBlocks ? cx.max_ctas : kSeqMaxBlocks;
  GFICF_LAUNCH(cx.st, seq_init_kernel, 1, 32, st, s0);
  long long t0 = 0;
  do {
    for (int it = 0; it < kSeqBatch; ++it) {
      GFICF_LAUNCH(cx.st, seq_blocks_kernel, grid, kSeqThreads, x, n, (const SeqState*)st, bf, flags);
      GFICF_LAUNCH(cx.st, seq_advance_kernel, 1, kSeqThreads, x, n, st, (const SeqFn*)bf, scale, out, flags);
    }
    net_read(cx.st, &t0, &st->t0, 8);
  } while (t0 < n);
}

// Clustering::getNodesPerCluster (:106-118): sc.perm = nodes grouped by cluster, ascending inside
// a cluster; sc.ptr_a[c] = start of cluster c
inline void net_nodes_per_cluster(const NetCtx& cx, const int* cluster, long long n_nodes, int n_clusters) {
  const NetScratch& sc = cx.sc;
  net_zero(cx.st, sc.cnt, (size_t)(n_clusters + 1) * 4);
  GFICF_LAUNCH(cx.st, net_cluster_keys_kernel, net_grid(cx, n_nodes, 256), 256, cluster, n_nodes, n_clusters,
               sc.keys[0], sc.vals[0], sc.cnt, cx.flags);
  net_scan(cx, sc.cnt, n_clusters, sc.ptr_a);
  const int b = net_radix_sort(cx, 0, n_nodes, bits_for((long long)n_clusters - 1));
  net_copy(cx.st, sc.perm, sc.vals[b], (size_t)n_nodes * 4);
}

// matrixToNetwork + Network constructor.  first[nv+1], neighbor[2 nnz], edge_w[2 nnz], node_w[nv],
// total_w[1] (= getTotalEdgeWeight).
inline void net_build(const NetCtx& cx, const long long* colptr, const int* row, const double* w, long long nv,
                      long long nnz, long long* first, int* neighbor, double* edge_w, double* node_w,
                      double* total_w) {
  const NetScratch& sc = cx.sc;
  int* col_of = (int*)sc.aux;
  net_zero(cx.st, sc.cnt, (size_t)(nv + 1) * 4);
  GFICF_LAUNCH(cx.st, net_col_keys_kernel, net_grid(cx, nv * 32, 256), 256, colptr, row, nv, col_of, sc.keys[0],
               sc.vals[0], sc.cnt, cx.flags);
  net_scan(cx, sc.cnt, nv, sc.ptr_a);
  const int b = net_radix_sort(cx, 0, nnz, bits_for(nv - 1));
  GFICF_LAUNCH(cx.st, net_first_kernel, net_grid(cx, nv + 1, 256), 256, colptr, (const long long*)sc.ptr_a, nv,
               first);
  GFICF_LAUNCH(cx.st, net_fill_kernel, net_grid(cx, nnz, 256), 256, colptr, row, w, (const long long*)sc.ptr_a,
               (const int*)col_of, (const unsigned long long*)sc.keys[b], (const unsigned*)sc.vals[b], nnz,
               neighbor, edge_w);
  GFICF_LAUNCH(cx.st, net_node_weight_kernel, net_grid(cx, nv * 32, 256), 256, (const long long*)first,
               (const double*)edge_w, nv, node_w, cx.flags);
  net_seq_sum(cx, edge_w, 2 * nnz, 0.0, 0.5, total_w);
}

// calcQualityFunction.  cluster_w[n_clusters] and q[1] are outputs.  Needs item capacity n_edges.
inline void net_quality(const NetCtx& cx, const long long* first, const int* neighbor, const double* edge_w,
                        const double* node_w, long long n_nodes, long long n_edges, const int* cluster,
                        int n_clusters, double resolution, double self_links, const double* total_w,
                        double* cluster_w, double* q) {
  const NetScratch& sc = cx.sc;
  double* y = sc.seg_w;
  GFICF_LAUNCH(cx.st, net_intra_mask_kernel, net_grid(cx, n_nodes * 32, 256), 256, first, neighbor, edge_w, cluster,
               n_nodes, y);
  net_seq_sum(cx, y, n_edges, 0.0, 1.0, sc.sums + 0);
  net_nodes_per_cluster(cx, cluster, n_nodes, n_clusters);
  GFICF_LAUNCH(cx.st, net_cluster_weight_kernel, net_grid(cx, (long long)n_clusters * 32, 256), 256, (const long long*)sc.ptr_a,
               (const unsigned*)sc.perm, node_w, n_clusters, resolution, cluster_w, sc.dbl_b);
  GFICF_LAUNCH(cx.st, net_quality_final_kernel, 1, 32, (const double*)(sc.sums + 0), (const double*)sc.dbl_b,
               n_clusters, total_w, self_links, q);
}

// createReducedNetwork.  Outputs: r_first[n_clusters+1], r_neighbor / r_edge_w (capacity r_cap
// entries), r_node_w[n_clusters], r_self_links[1] = totalEdgeWeightSelfLinks of the reduced network
// (the parent's value `self_links` plus, in traversal order, every edge that stays inside a cluster,
// :329/:351), r_total_w[1] = getTotalEdgeWeight of the reduced network.  Returns the number of
// reduced edges, or -1 when r_cap is too small (*n_needed then holds the number).  Synchronises the
// stream (entry counts and the positions of the sequential sums are read back).
inline long long net_reduce(const NetCtx& cx, const long long* first, const int* neighbor, const double* edge_w,
                            const double* node_w, long long n_nodes, long long n_edges, const int* cluster,
                            int n_clusters, double self_links, long long* r_first, int* r_neighbor,
                            double* r_edge_w, long long r_cap, double* r_node_w, double* r_self_links,
                            double* r_total_w, long long* n_needed) {
  const NetScratch& sc = cx.sc;
  net_nodes_per_cluster(cx, cluster, n_nodes, n_clusters);
  GFICF_LAUNCH(cx.st, net_cluster_weight_kernel, net_grid(cx, (long long)n_clusters * 32, 256), 256, (const long long*)sc.ptr_a,
               (const unsigned*)sc.perm, node_w, n_clusters, 0.0, r_node_w, (double*)nullptr);
  GFICF_LAUNCH(cx.st, rn_count_kernel, net_grid(cx, n_nodes * 32, 256), 256, first, neighbor, cluster,
               (const unsigned*)sc.perm, n_nodes, sc.cnt, sc.cnt_b);
  net_scan(cx, sc.cnt, n_nodes, sc.ptr_b);
  net_scan(cx, sc.cnt_b, n_nodes, sc.ptr_c);
  GFICF_LAUNCH(cx.st, rn_intra_mask_kernel, net_grid(cx, n_nodes * 32, 256), 256, first, neighbor, edge_w, cluster,
               (const unsigned*)sc.perm, (const long long*)sc.ptr_c, n_nodes, sc.seg_w);
  net_seq_sum(cx, sc.seg_w, n_edges, self_links, 1.0, r_self_links);
  long long n_cross = 0;
  net_read(cx.st, &n_cross, sc.ptr_b + n_nodes, 8);
  *n_needed = 0;
  if (n_cross == 0) {
    net_zero(cx.st, r_first, (size_t)(n_clusters + 1) * 8);
    net_zero(cx.st, r_total_w, 8);
    return 0;
  }
  const int cbits = bits_for((long long)n_clusters - 1);
  GFICF_LAUNCH(cx.st, rn_emit_kernel, net_grid(cx, n_nodes * 32, 256), 256, first, neighbor, cluster,
               (const unsigned*)sc.perm, (const long long*)sc.ptr_b, n_nodes, cbits, sc.keys[0], sc.vals[0],
               sc.aux);
  const int b = net_radix_sort(cx, 0, n_cross, 2 * cbits);
  GFICF_LAUNCH(cx.st, rn_heads_kernel, net_grid(cx, n_cross, 256), 256, (const unsigned long long*)sc.keys[b],
               n_cross, sc.head);
  net_scan(cx, sc.head, n_cross, sc.seg_id);
  long long n_seg = 0;
  net_read(cx.st, &n_seg, sc.seg_id + n_cross, 8);
  *n_needed = n_seg;
  if (n_seg > r_cap) return -1;
  net_zero(cx.st, sc.cnt, (size_t)(n_clusters + 1) * 4);
  GFICF_LAUNCH(cx.st, rn_seg_start_kernel, net_grid(cx, n_cross, 256), 256, (const int*)sc.head,
               (const long long*)sc.seg_id, n_cross, sc.seg_start);
  GFICF_LAUNCH(cx.st, rn_segments_kernel, net_grid(cx, n_seg * 32, 256), 256, (const unsigned long long*)sc.keys[b],
               (const unsigned*)sc.vals[b], (const unsigned*)sc.seg_start, (const unsigned*)sc.aux, edge_w, n_cross,
               n_seg, cbits, sc.seg_key, sc.seg_w, sc.keys[b ^ 1], sc.vals[b ^ 1], sc.cnt);
  const int b2 = net_radix_sort(cx, b ^ 1, n_seg, bits_for(n_cross - 1));
  GFICF_LAUNCH(cx.st, rn_write_kernel, net_grid(cx, n_seg, 256), 256, (const unsigned*)sc.vals[b2],
               (const unsigned long long*)sc.seg_key, (const double*)sc.seg_w, n_seg, cbits, r_neighbor, r_edge_w);
  net_scan(cx, sc.cnt, n_clusters, r_first);
  net_seq_sum(cx, r_edge_w, n_seg, 0.0, 0.5, r_total_w);
  return n_seg;
}

// ---------------------------------------------------------------------------------------------
// bodies of the C entry points gficf_cuda_network_*_dev (argument checks included, so that the
// emulated test build exercises them too); `max_ctas`: 8 x the SM count on the device
// ---------------------------------------------------------------------------------------------
inline bool net_make_ctx(NetCtx* cx, void* d_scratch, size_t scratch_bytes, long long nn, long long cap,
                         unsigned* d_flags, net_stream_t st, int max_ctas) {
  if (!d_scratch || !d_flags || scratch_bytes < net_scratch_layout(nullptr, nn, cap).bytes) return false;
  cx->st = st;
  cx->sc = net_scratch_layout((char*)d_scratch, nn, cap);
  cx->flags = d_flags;
  cx->max_ctas = max_ctas;
  return true;
}

inline int net_entry_network(const int64_t* d_colptr, const int32_t* d_row, const double* d_w, int64_t n_vertices,
                             int64_t nnz, int64_t* d_first, int32_t* d_neighbor, double* d_edge_w, double* d_node_w,
                             double* d_total_w, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                             net_stream_t st, int max_ctas) {
  if (!d_colptr || !d_row || !d_w || !d_first || !d_neighbor || !d_edge_w || !d_node_w || !d_total_w)
    return GFICF_E_ARG;
  if (n_vertices < 1 || nnz < 1) return GFICF_E_ARG;  // "Matrix contained no network data" (RModularityOptimizer.cpp:84)
  if (n_vertices >= 0x7fffffffLL || 2 * nnz >= 0x7fffffffLL) return GFICF_E_LIMIT;  // the reference's int indices
  NetCtx cx;
  if (!net_make_ctx(&cx, d_scratch, scratch_bytes, n_vertices, nnz, d_flags, st, max_ctas)) return GFICF_E_ARG;
  net_build(cx, (const long long*)d_colptr, d_row, d_w, n_vertices, nnz, (long long*)d_first, d_neighbor, d_edge_w,
            d_node_w, d_total_w);
  net_check_launches();
  return GFICF_OK;
}

inline int net_entry_quality(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                             const double* d_node_w, int64_t n_nodes, int64_t n_edges, const int32_t* d_cluster,
                             int32_t n_clusters, double resolution, double self_links, const double* d_total_w,
                             double* d_cluster_w,
                             double* d_quality, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                             net_stream_t st, int max_ctas) {
  if (!d_first || !d_neighbor || !d_edge_w || !d_node_w || !d_cluster || !d_total_w || !d_cluster_w || !d_quality)
    return GFICF_E_ARG;
  if (n_nodes < 1 || n_edges < 0 || n_clusters < 1 || n_clusters > n_nodes) return GFICF_E_ARG;
  if (n_nodes >= 0x7fffffffLL || n_edges >= 0x7fffffffLL) return GFICF_E_LIMIT;
  NetCtx cx;
  if (!net_make_ctx(&cx, d_scratch, scratch_bytes, n_nodes, n_edges, d_flags, st, max_ctas)) return GFICF_E_ARG;
  net_quality(cx, (const long long*)d_first, d_neighbor, d_edge_w, d_node_w, n_nodes, n_edges, d_cluster,
              n_clusters, resolution, self_links, d_total_w, d_cluster_w, d_quality);
  net_check_launches();
  return GFICF_OK;
}

inline int net_entry_reduce(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                            const double* d_node_w, int64_t n_nodes, int64_t n_edges, const int32_t* d_cluster,
                            int32_t n_clusters, double self_links, int64_t* d_r_first, int32_t* d_r_neighbor,
                            double* d_r_edge_w, int64_t r_cap, double* d_r_node_w, double* d_r_self_links,
                            double* d_r_total_w,
                            int64_t* n_reduced_edges, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                            net_stream_t st, int max_ctas) {
  if (!d_first || !d_neighbor || !d_edge_w || !d_node_w || !d_cluster || !d_r_first || !d_r_neighbor ||
      !d_r_edge_w || !d_r_node_w || !d_r_self_links || !d_r_total_w || !n_reduced_edges)
    return GFICF_E_ARG;
  if (n_nodes < 1 || n_edges < 0 || n_clusters < 1 || n_clusters > n_nodes || r_cap < 0) return GFICF_E_ARG;
  if (n_nodes >= 0x7fffffffLL || n_edges >= 0x7fffffffLL) return GFICF_E_LIMIT;
  NetCtx cx;
  if (!net_make_ctx(&cx, d_scratch, scratch_bytes, n_nodes, n_edges, d_flags, st, max_ctas)) return GFICF_E_ARG;
  long long needed = 0;
  const long long r = net_reduce(cx, (const long long*)d_first, d_neighbor, d_edge_w, d_node_w, n_nodes, n_edges,
                                 d_cluster, n_clusters, self_links, (long long*)d_r_first, d_r_neighbor, d_r_edge_w,
                                 r_cap, d_r_node_w, d_r_self_links, d_r_total_w, &needed);
  net_check_launches();
  *n_reduced_edges = r < 0 ? needed : r;
  return r < 0 ? GFICF_E_LIMIT : GFICF_OK;  // r_cap too small: *n_reduced_edges holds the number needed
}

}  // namespace gficf
