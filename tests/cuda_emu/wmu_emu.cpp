// wmu_emu.cpp -- gficf_cuda_wmu_test's launches and host finish (gficf_b200/csrc/wmu_csc_plan.h) on the CUDA
// emulation.  TEST INFRASTRUCTURE; built and loaded by tests/test_wmu_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
//   tests/cuda_emu/wmu_emu.cpp gficf_b200/csrc/host_stats.cpp
#include <vector>

#include "wmu_csc_plan.h"

using namespace gficf;

extern "C" void emu_wmu_test(const double* mat_x, const double* mat_y, long long n_genes, long long n1, long long n2,
                             double* out, int grid) {
  const long long N = n1 + n2;
  if (grid > n_genes) grid = (int)n_genes;
  std::vector<unsigned long long> keys((size_t)grid * 2 * N, 0xA5A5A5A5A5A5A5A5ull);
  std::vector<unsigned> pay((size_t)grid * (3 * N + 2), 0xA5A5A5A5u);
  std::vector<double> z_ratio((size_t)n_genes * 2);
  std::vector<int> single(n_genes);
  wmu_test_launch(0, grid, mat_x, mat_y, n_genes, n1, n2, keys.data(), pay.data(), z_ratio.data(),
                  z_ratio.data() + n_genes, single.data());
  wmu_finish(z_ratio.data(), single.data(), n_genes, 1, out);
}
