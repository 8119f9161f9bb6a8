// wmu_markers_sparse_emu.cpp -- the device half of gficf_cuda_wmu_markers_csc (gficf_b200/csrc/wmu_csc_plan.h:
// transpose to gene-major, then wmu_markers_csr_rank_kernel and wmu_markers_csr_means_kernel of
// wmu_kernels.cuh) compiled as plain C++ against the CUDA emulation, followed by the host half of the call
// (host_stats.cpp: normal cdf, log2).  TEST INFRASTRUCTURE; built and loaded by
// tests/test_wmu_markers_sparse_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
//   tests/cuda_emu/wmu_markers_sparse_emu.cpp gficf_b200/csrc/host_stats.cpp
// Cluster ids and colptr must already be valid (those checks are the library's host code; the test calls it
// for them); the row ids are checked by the emulated transpose, as on the device.
#include <math.h>

#include <vector>

#include "host_stats.h"
#include "wmu_csc_plan.h"

using namespace gficf;

namespace {
// the transpose's scratch: 0xA5 filled (never assumed zero); with GFICF_NET_ASAN every piece is fenced by a
// poisoned red zone
struct Scratch {
  std::vector<char> mem;
  WmuCscScratch sc;
  Scratch(long long n_genes, long long nnz) {
    mem.assign(wmu_csc_layout(nullptr, n_genes, nnz).bytes, (char)0xA5);
#ifdef GFICF_NET_ASAN
    __asan_poison_memory_region(mem.data(), mem.size());
#endif
    sc = wmu_csc_layout(mem.data(), n_genes, nnz);
  }
  ~Scratch() {
#ifdef GFICF_NET_ASAN
    __asan_unpoison_memory_region(mem.data(), mem.size());
#endif
  }
};
}  // namespace

extern "C" {

double emu_ones_run(double s, long long m) { return wmu_ones_run(s, m); }

// The whole call on host memory.  Returns the transpose's flags; out is written only when they are 0.
unsigned emu_wmu_markers_csc(const int* colptr, const int* row, const double* x, long long n_genes, long long n_cells,
                             const int* cluster, int n_clusters, double* out, int grid, int max_ctas) {
  const long long N = n_cells, C = n_clusters, nnz = colptr[N];
  Scratch s(n_genes, nnz);
  const WmuGeneMajor gm = wmu_csc_to_genes(0, s.sc, max_ctas, colptr, row, x, n_genes, N, nnz);
  if (*s.sc.flags) return *s.sc.flags;
  const WmuClusterLists cl = wmu_cluster_lists(cluster, N, n_clusters);
  const long long* gptr = s.sc.gene_ptr;
  long long cap = 1;
  for (long long g = 0; g < n_genes; ++g) cap = gptr[g + 1] - gptr[g] > cap ? gptr[g + 1] - gptr[g] : cap;
  if (grid > n_genes) grid = (int)n_genes;
  std::vector<unsigned long long> keys((size_t)grid * 2 * cap, 0xA5A5A5A5A5A5A5A5ull);
  std::vector<unsigned> pay((size_t)grid * 2 * cap, 0xA5A5A5A5u);
  std::vector<double> z((size_t)n_genes * C), ratio((size_t)n_genes * C);
  std::vector<int> single(n_genes);
  unsigned long long* d_keys = keys.data();
  unsigned* d_pay = pay.data();
  double *d_z = z.data(), *d_ratio = ratio.data();
  int* d_single = single.data();
  const long long *d_size = cl.size.data(), *d_cptr = cl.cptr.data();
  const int *d_crank = cl.crank.data(), *d_members = cl.members.data();
  cuda_emu::launch(
      (unsigned)grid, kWmuThreads,
      [=] {
        wmu_markers_csr_rank_kernel(gm.ent_x, gm.ent_cell, gptr, n_genes, N, cluster, d_size, n_clusters, cap, d_keys,
                                    d_pay, d_z, d_single);
      },
      (size_t)C * kWmuClusterSmemBytes);
  const int mthreads = wmu_csr_means_threads(n_clusters);
  cuda_emu::launch((unsigned)n_genes, (unsigned)mthreads,
                   [=] {
                     wmu_markers_csr_means_kernel(gm.ent_x, gm.ent_cell, gptr, n_genes, N, cluster, d_crank,
                                                  d_members, d_cptr, n_clusters, d_ratio);
                   },
                   0, (unsigned)((C + mthreads - 1) / mthreads));
  for (long long c = 0; c < C; ++c)  // as in gficf_cuda_wmu_markers_csc
    for (long long g = 0; g < n_genes; ++g) {
      out[c * 2 * n_genes + g] = single[g] ? 1.0 : gficf_host::wmu_pvalue(z[c * n_genes + g]);
      out[c * 2 * n_genes + n_genes + g] = log2(ratio[c * n_genes + g]);
    }
  return 0;
}

}  // extern "C"
