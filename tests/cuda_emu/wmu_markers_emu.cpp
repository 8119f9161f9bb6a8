// wmu_markers_emu.cpp -- the one-vs-rest kernels of gficf_cuda_wmu_markers (gficf_b200/csrc/wmu_kernels.cuh)
// compiled as plain C++ against the CUDA emulation, followed by the host half of the call (host_stats.cpp:
// normal cdf, log2).  TEST INFRASTRUCTURE; built and loaded by tests/test_wmu_markers_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -shared -fPIC
//   tests/cuda_emu/wmu_markers_emu.cpp gficf_b200/csrc/host_stats.cpp
// Ids must already be valid (the argument checks are the library's; the test calls it for those).
#include <math.h>

#include <vector>

#include "host_stats.h"
#include "wmu_kernels.cuh"

using namespace gficf;

extern "C" void emu_wmu_markers(const double* mat, long long n_genes, long long n_cells, const int* cluster,
                                int n_clusters, double* out, int grid) {
  const long long N = n_cells, C = n_clusters;
  if (grid > n_genes) grid = (int)n_genes;
  std::vector<long long> size((size_t)C, 0);
  for (long long i = 0; i < N; ++i) ++size[(size_t)cluster[i]];
  std::vector<unsigned long long> keys((size_t)grid * 2 * N, 0xA5A5A5A5A5A5A5A5ull);
  std::vector<unsigned> pay((size_t)grid * (3 * N + 2), 0xA5A5A5A5u);
  std::vector<double> z((size_t)n_genes * C), ratio((size_t)n_genes * C);
  std::vector<int> single(n_genes);
  unsigned long long* d_keys = keys.data();
  unsigned* d_pay = pay.data();
  double *d_z = z.data(), *d_ratio = ratio.data();
  int* d_single = single.data();
  const long long* d_size = size.data();
  cuda_emu::launch(
      (unsigned)grid, kWmuThreads,
      [=] { wmu_markers_rank_kernel(mat, n_genes, N, cluster, d_size, n_clusters, d_keys, d_pay, d_z, d_single); },
      (size_t)C * kWmuClusterSmemBytes);
  cuda_emu::launch((unsigned)((n_genes + kMeanGenes - 1) / kMeanGenes), kMarkThreads,
                   [=] { wmu_markers_means_kernel(mat, n_genes, N, cluster, d_size, n_clusters, d_ratio); }, 0,
                   (unsigned)((C + kMarkClusters - 1) / kMarkClusters));
  for (long long c = 0; c < C; ++c)  // as in gficf_cuda_wmu_markers
    for (long long g = 0; g < n_genes; ++g) {
      out[c * 2 * n_genes + g] = single[g] ? 1.0 : gficf_host::wmu_pvalue(z[c * n_genes + g]);
      out[c * 2 * n_genes + n_genes + g] = log2(ratio[c * n_genes + g]);
    }
}
