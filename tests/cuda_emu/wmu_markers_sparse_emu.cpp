// wmu_markers_sparse_emu.cpp -- gficf_cuda_wmu_markers_csc's transpose, launches and host finish
// (gficf_b200/csrc/wmu_csc_plan.h) on the CUDA emulation.  TEST INFRASTRUCTURE; built and loaded by
// tests/test_wmu_markers_sparse_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
//   tests/cuda_emu/wmu_markers_sparse_emu.cpp gficf_b200/csrc/host_stats.cpp
// Cluster ids and colptr must already be valid (those checks are the library's host code; the test calls it
// for them); the row ids are checked by the emulated transpose, as on the device.
#include <vector>

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
  const long long cap = wmu_gene_cap(s.sc.gene_ptr, n_genes);
  if (grid > n_genes) grid = (int)n_genes;
  std::vector<unsigned long long> keys((size_t)grid * 2 * cap, 0xA5A5A5A5A5A5A5A5ull);
  std::vector<unsigned> pay((size_t)grid * 2 * cap, 0xA5A5A5A5u);
  std::vector<double> z_ratio((size_t)n_genes * C * 2);
  std::vector<int> single(n_genes);
  wmu_markers_csc_launch(0, grid, gm, s.sc.gene_ptr, n_genes, N, cluster, cl.crank.data(), cl.members.data(),
                         cl.size.data(), cl.cptr.data(), n_clusters, cap, keys.data(), pay.data(), z_ratio.data(),
                         z_ratio.data() + (size_t)n_genes * C, single.data());
  wmu_finish(z_ratio.data(), single.data(), n_genes, n_clusters, out);
  return 0;
}

}  // extern "C"
