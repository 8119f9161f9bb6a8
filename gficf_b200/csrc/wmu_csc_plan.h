// wmu_csc_plan.h -- host half of gficf_cuda_wmu_markers_csc that the CPU test suite shares with the product:
// the cluster lists the means kernel reads, the scratch layout, and the launch sequence that turns a
// compressed-column (dgCMatrix) genes x cells matrix gene-major on the device.  Included by gficf_cuda.cu
// (after its error helpers) and by tests/cuda_emu/wmu_markers_sparse_emu.cpp with GFICF_CUDA_EMU defined.
//
// Transpose: every entry gets key = its gene (row id, checked first: wmu_csc_keys_kernel) and payload = its
// index; the stable LSD radix sort of the network kernels (net_radix_sort, bits_for(n_genes - 1) bits) puts
// the entries of a gene together in column order, i.e. cells ascending, and the gene pointers are the scan of
// the per-gene counts.  Stability matters: the means chains walk a gene's cells in order.
#pragma once
#include <vector>

#include "network_plan.h"
#include "wmu_kernels.cuh"

namespace gficf {

// Per-cluster cell lists: size[c] (cells of c), crank[cell] = rank of the cell inside its own cluster,
// members = cells grouped by cluster, ascending inside a cluster, starting at cptr[c].  Ids must be valid.
struct WmuClusterLists {
  std::vector<long long> size, cptr;
  std::vector<int> crank, members;
};

inline WmuClusterLists wmu_cluster_lists(const int* cluster, long long n_cells, int n_clusters) {
  WmuClusterLists l;
  l.size.assign((size_t)n_clusters, 0);
  l.crank.resize((size_t)n_cells);
  for (long long i = 0; i < n_cells; ++i) l.crank[(size_t)i] = (int)l.size[(size_t)cluster[i]]++;
  l.cptr.assign((size_t)n_clusters + 1, 0);
  for (int c = 0; c < n_clusters; ++c) l.cptr[(size_t)c + 1] = l.cptr[(size_t)c] + l.size[(size_t)c];
  l.members.resize((size_t)n_cells);
  for (long long i = 0; i < n_cells; ++i)
    l.members[(size_t)(l.cptr[(size_t)cluster[i]] + l.crank[(size_t)i])] = (int)i;
  return l;
}

// Device scratch of the transpose for nnz entries and n_genes genes.  `sort` holds what net_scan and
// net_radix_sort use (keys[2], vals[2], hist, offsets, block_sums, total); its other pieces stay null.
// 29.5 bytes per stored value (keys 16, payloads 8, column 4, digit histograms and offsets 1.5) plus 12
// bytes per gene.
struct WmuCscScratch {
  NetScratch sort;
  unsigned* col_of;
  int* gene_cnt;
  long long* gene_ptr;  // [n_genes + 1]
  unsigned* flags;
  size_t bytes;
};

inline WmuCscScratch wmu_csc_layout(char* base, long long n_genes, long long nnz) {
  WmuCscScratch s;
  memset(&s, 0, sizeof s);
  size_t off = 0;
  auto take = [&](size_t b) {
    char* p = base + off;
    off += (b + GFICF_NET_REDZONE + 255) / 256 * 256;
    GFICF_NET_PIECE(p, b);
    return p;
  };
  const long long n = nnz > 1 ? nnz : 1;
  const long long n_tiles = (n + kRadixTile - 1) / kRadixTile + 1;
  const long long scan_len = (256 * n_tiles > n_genes ? 256 * n_tiles : n_genes) + 1;
  for (int b = 0; b < 2; ++b) s.sort.keys[b] = (unsigned long long*)take((size_t)n * 8);
  for (int b = 0; b < 2; ++b) s.sort.vals[b] = (unsigned*)take((size_t)n * 4);
  s.sort.hist = (int*)take((size_t)(256 * n_tiles) * 4);
  s.sort.offsets = (long long*)take((size_t)(256 * n_tiles + 1) * 8);
  s.sort.block_sums = (long long*)take((size_t)(scan_len / kScanBlock + 2) * 8);
  s.sort.total = (long long*)take(8);
  s.col_of = (unsigned*)take((size_t)n * 4);
  s.gene_cnt = (int*)take((size_t)(n_genes > 1 ? n_genes : 1) * 4);
  s.gene_ptr = (long long*)take((size_t)(n_genes + 1) * 8);
  s.flags = (unsigned*)take(4);
  s.bytes = off;
  return s;
}

// The stored values gene-major: gene g's are ent_x[gene_ptr[g] .. gene_ptr[g + 1]) at cells ent_cell[...],
// ascending.  Both live in the sort's key buffers, free once the sort is done.
struct WmuGeneMajor {
  const unsigned* ent_cell;
  const double* ent_x;
};

// colptr / row / x: device copies of the matrix; colptr must already be checked (starts at 0, never
// decreases, ends at nnz).  Raises kFlagCscRow in *sc.flags for a row id out of range or out of order; the
// result is then meaningless but every access stayed in bounds.
inline WmuGeneMajor wmu_csc_to_genes(net_stream_t st, const WmuCscScratch& sc, int max_ctas, const int* colptr,
                                     const int* row, const double* x, long long n_genes, long long n_cells,
                                     long long nnz) {
  NetCtx cx;
  cx.st = st;
  cx.sc = sc.sort;
  cx.flags = sc.flags;
  cx.max_ctas = max_ctas;
  net_zero(st, sc.gene_cnt, (size_t)n_genes * 4);
  net_zero(st, sc.flags, 4);
  GFICF_LAUNCH(st, wmu_csc_keys_kernel, net_grid(cx, n_cells * 32, 256), 256, colptr, row, n_cells, n_genes,
               sc.col_of, sc.sort.keys[0], sc.sort.vals[0], sc.gene_cnt, sc.flags);
  net_scan(cx, sc.gene_cnt, n_genes, sc.gene_ptr);
  const int b = net_radix_sort(cx, 0, nnz, bits_for(n_genes - 1));
  unsigned* ent_cell = reinterpret_cast<unsigned*>(sc.sort.keys[b]);
  double* ent_x = reinterpret_cast<double*>(sc.sort.keys[b ^ 1]);
  GFICF_LAUNCH(st, wmu_csc_gather_kernel, net_grid(cx, nnz, 256), 256, (const unsigned*)sc.sort.vals[b],
               (const unsigned*)sc.col_of, x, nnz, ent_cell, ent_x);
  return WmuGeneMajor{ent_cell, ent_x};
}

// threads per CTA of wmu_markers_csr_means_kernel: one per cluster, up to 128
inline int wmu_csr_means_threads(int n_clusters) {
  const int w = (n_clusters + 31) / 32;
  return 32 * (w < 4 ? w : 4);
}

}  // namespace gficf
