// snn_emu.cpp -- the graph build of gficf_cuda_snn_lower_dev through its own launch sequence
// (gficf_b200/csrc/snn_plan.h) on the CUDA emulation.  TEST INFRASTRUCTURE; built and loaded by
// tests/test_snn_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
#include <vector>

#include "snn_plan.h"

using namespace gficf;

// idx: n x kp int32 (0-based, padded rows), um: n*k bytes (count | mutual << 7).  Outputs sized by the
// caller: colptr[n+1], row / w [n*k], vertex_cell[n].  Returns the flags; *n_vertices, *nnz are set.
// max_ctas caps the grid-stride launches, sort_ctas is the grid of the shared-memory column sort.
extern "C" unsigned emu_snn_lower(const int* idx, long long n, int k, int kp, const unsigned char* um,
                                  long long* colptr, int* row, double* w, int* vertex_cell,
                                  long long* n_vertices, long long* nnz, int max_ctas, int sort_ctas) {
  // scratch is never assumed initialised: every 32-bit word starts as 1, non-zero (a missing zero fill shows)
  // and below every edge number (so does a missing 0xFF fill of the first-appearance minima)
  std::vector<unsigned> scratch(snn_scratch_layout(nullptr, n, n * k).bytes / 4, 1u);
  unsigned flags = 0;
  snn_lower(0, snn_scratch_layout((char*)scratch.data(), n, n * k), max_ctas, sort_ctas, idx, n, k, kp, um, colptr,
            row, w, vertex_cell, n_vertices, &flags);
  *nnz = colptr[*n_vertices];
  return flags;
}
