// wmu_markers_emu.cpp -- gficf_cuda_wmu_markers' launches and host finish (gficf_b200/csrc/wmu_csc_plan.h) on the
// CUDA emulation.  TEST INFRASTRUCTURE; built and loaded by tests/test_wmu_markers_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
//   tests/cuda_emu/wmu_markers_emu.cpp gficf_b200/csrc/host_stats.cpp
// Ids must already be valid (the argument checks are the library's; the test calls it for those).
#include <vector>

#include "wmu_csc_plan.h"

using namespace gficf;

extern "C" void emu_wmu_markers(const double* mat, long long n_genes, long long n_cells, const int* cluster,
                                int n_clusters, double* out, int grid) {
  const long long N = n_cells;
  const size_t zc = (size_t)n_genes * n_clusters;
  if (grid > n_genes) grid = (int)n_genes;
  const WmuClusterLists cl = wmu_cluster_lists(cluster, N, n_clusters);
  std::vector<unsigned long long> keys((size_t)grid * 2 * N, 0xA5A5A5A5A5A5A5A5ull);
  std::vector<unsigned> pay((size_t)grid * (3 * N + 2), 0xA5A5A5A5u);
  std::vector<double> z_ratio(zc * 2);
  std::vector<int> single(n_genes);
  wmu_markers_launch(0, grid, mat, n_genes, N, cluster, cl.size.data(), n_clusters, keys.data(), pay.data(),
                     z_ratio.data(), z_ratio.data() + zc, single.data());
  wmu_finish(z_ratio.data(), single.data(), n_genes, n_clusters, out);
}
