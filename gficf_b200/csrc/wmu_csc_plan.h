// wmu_csc_plan.h -- the Mann-Whitney calls' launch sequences (wmu_kernels.cuh) and host finish, shared by the product
// and the CPU test suite: the rank + means launches of gficf_cuda_wmu_test, gficf_cuda_wmu_markers and
// gficf_cuda_wmu_markers_csc, the cluster lists and device transpose of the compressed-column call, and the
// p-value / log2 finish of all three.  Included by gficf_cuda.cu (after its error helpers) and by the
// tests/cuda_emu/wmu*_emu.cpp harnesses with GFICF_CUDA_EMU defined.  Grids come from the caller (the product
// sizes them from the occupancy of the rank kernels).
//
// Transpose: every entry gets key = its gene (row id, checked first: wmu_csc_keys_kernel) and payload = its
// index; the stable LSD radix sort of the network kernels (net_radix_sort, bits_for(n_genes - 1) bits) puts
// the entries of a gene together in column order, i.e. cells ascending, and the gene pointers are the scan of
// the per-gene counts.  Stability matters: the means chains walk a gene's cells in order.
#pragma once
#include <math.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "host_stats.h"
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
  ScratchCarver c{base};
  const long long n = nnz > 1 ? nnz : 1;
  const long long n_tiles = (n + kRadixTile - 1) / kRadixTile + 1;
  const long long scan_len = (256 * n_tiles > n_genes ? 256 * n_tiles : n_genes) + 1;
  for (int b = 0; b < 2; ++b) s.sort.keys[b] = c.take<unsigned long long>(n);
  for (int b = 0; b < 2; ++b) s.sort.vals[b] = c.take<unsigned>(n);
  s.sort.hist = c.take<int>(256 * n_tiles);
  s.sort.offsets = c.take<long long>(256 * n_tiles + 1);
  s.sort.block_sums = c.take<long long>(scan_len / kScanBlock + 2);
  s.sort.total = c.take<long long>(1);
  s.col_of = c.take<unsigned>(n);
  s.gene_cnt = c.take<int>(n_genes > 1 ? n_genes : 1);
  s.gene_ptr = c.take<long long>(n_genes + 1);
  s.flags = c.take<unsigned>(1);
  s.bytes = c.bytes;
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

// longest gene of the gene-major values: the rank kernel's per-CTA scratch holds 2 x this many items
inline long long wmu_gene_cap(const long long* gene_ptr, long long n_genes) {
  long long cap = 1;
  for (long long g = 0; g < n_genes; ++g) cap = std::max(cap, gene_ptr[g + 1] - gene_ptr[g]);
  return cap;
}

// Rank + means of one split (gficf_cuda_wmu_test): genes x n1 cells against genes x n2 cells.  `grid` CTAs
// of wmu_rank_kernel, each with 2 (n1 + n2) keys and 3 (n1 + n2) + 2 payload words of sort scratch.
inline void wmu_test_launch(net_stream_t st, int grid, const double* x, const double* y, long long n_genes,
                            long long n1, long long n2, unsigned long long* keys, unsigned* pay, double* z,
                            double* ratio, int* single) {
  GFICF_LAUNCH(st, wmu_rank_kernel, grid, kWmuThreads, x, y, n_genes, n1, n2, keys, pay, z, single);
  GFICF_LAUNCH(st, wmu_means_kernel, (n_genes + kMeanGenes - 1) / kMeanGenes, kMeanThreads, x, y, n_genes, n1, n2,
               ratio);
}

// Rank + means of every cluster against the rest (gficf_cuda_wmu_markers) on a dense genes x n_cells matrix;
// sort scratch per CTA as in wmu_test_launch.  z and ratio hold n_clusters blocks of n_genes.
inline void wmu_markers_launch(net_stream_t st, int grid, const double* mat, long long n_genes, long long n_cells,
                               const int* cluster, const long long* size, int n_clusters, unsigned long long* keys,
                               unsigned* pay, double* z, double* ratio, int* single) {
  GFICF_LAUNCH_EX(st, wmu_markers_rank_kernel, grid, 1, kWmuThreads, (size_t)n_clusters * kWmuClusterSmemBytes, mat,
                  n_genes, n_cells, cluster, size, n_clusters, keys, pay, z, single);
  GFICF_LAUNCH_EX(st, wmu_markers_means_kernel, (n_genes + kMeanGenes - 1) / kMeanGenes,
                  (n_clusters + kMarkClusters - 1) / kMarkClusters, kMarkThreads, 0, mat, n_genes, n_cells, cluster,
                  size, n_clusters, ratio);
}

// threads per CTA of wmu_markers_csr_means_kernel: one per cluster, up to 128
inline int wmu_csr_means_threads(int n_clusters) {
  const int w = (n_clusters + 31) / 32;
  return 32 * (w < 4 ? w : 4);
}

// The same on the gene-major values of a compressed-column matrix (gficf_cuda_wmu_markers_csc); sort scratch
// per CTA: 2 cap keys and 2 cap payload words, cap = wmu_gene_cap.  crank / members / size / cptr are the
// device copies of wmu_cluster_lists.
inline void wmu_markers_csc_launch(net_stream_t st, int grid, const WmuGeneMajor& gm, const long long* gene_ptr,
                                   long long n_genes, long long n_cells, const int* cluster, const int* crank,
                                   const int* members, const long long* size, const long long* cptr, int n_clusters,
                                   long long cap, unsigned long long* keys, unsigned* pay, double* z, double* ratio,
                                   int* single) {
  GFICF_LAUNCH_EX(st, wmu_markers_csr_rank_kernel, grid, 1, kWmuThreads, (size_t)n_clusters * kWmuClusterSmemBytes,
                  gm.ent_x, gm.ent_cell, gene_ptr, n_genes, n_cells, cluster, size, n_clusters, cap, keys, pay, z,
                  single);
  const int mthreads = wmu_csr_means_threads(n_clusters);
  GFICF_LAUNCH_EX(st, wmu_markers_csr_means_kernel, n_genes, (n_clusters + mthreads - 1) / mthreads, mthreads, 0,
                  gm.ent_x, gm.ent_cell, gene_ptr, n_genes, n_cells, cluster, crank, members, cptr, n_clusters,
                  ratio);
}

// Host finish of the three calls: the two transcendental steps per (gene, cluster), getPvalue
// (mann_whitney.cpp:101-110) and log2 (:100).  z_ratio = z | ratio, each n_clusters blocks of n_genes;
// block c of out is cluster c's n_genes x 2 result (one split: n_clusters = 1).  Clusters are spread over
// host threads when there are many values.
inline void wmu_finish(const double* z_ratio, const int* single, long long n_genes, int n_clusters, double* out) {
  const long long C = n_clusters;
  const size_t zc = (size_t)n_genes * C;
  auto finish = [&](long long c_lo, long long c_hi) {
    for (long long c = c_lo; c < c_hi; ++c) {
      const double* z = z_ratio + (size_t)c * n_genes;
      const double* ratio = z_ratio + zc + (size_t)c * n_genes;
      double* o = out + (size_t)c * 2 * n_genes;
      for (long long g = 0; g < n_genes; ++g) {
        o[g] = single[g] ? 1.0 : gficf_host::wmu_pvalue(z[g]);
        o[n_genes + g] = log2(ratio[g]);
      }
    }
  };
  const long long nthreads =
      std::min<long long>({C, (long long)std::max(1u, std::thread::hardware_concurrency()), 16LL,
                           std::max(1LL, (long long)zc / 16384)});
  if (nthreads <= 1) {
    finish(0, C);
  } else {
    std::vector<std::thread> th;
    for (long long t = 0; t < nthreads; ++t) th.emplace_back(finish, C * t / nthreads, C * (t + 1) / nthreads);
    for (auto& x : th) x.join();
  }
}

}  // namespace gficf
