// wmu_markers_multi_emu.cpp -- gficf_cuda_wmu_markers_csc_devices's plan (gficf_b200/csrc/wmu_csc_plan.h) on the
// CUDA emulation, with D emulated devices: column slabs, the transpose of each slab, the gene ranges and exchange
// table, the exchange as copies between per-device buffers, wmu_regroup_kernel, the rank + means launches of
// each gene range and the finish into its rows.  TEST INFRASTRUCTURE; built and loaded by
// tests/test_wmu_markers_multi_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -Iinclude -shared -fPIC
//   tests/cuda_emu/wmu_markers_multi_emu.cpp gficf_b200/csrc/host_stats.cpp
// Cluster ids and colptr must already be valid (the library's host code checks them); the row ids are checked
// by the emulated transpose of each slab, as on the devices.
#include <memory>
#include <vector>

#include "wmu_csc_plan.h"

using namespace gficf;

namespace {
// 0xA5 filled: nothing the plan reads is assumed zero
template <class T>
std::vector<T> junk(long long n) {
  std::vector<T> v((size_t)(n > 0 ? n : 1));
  memset(v.data(), 0xA5, v.size() * sizeof(T));
  return v;
}

// what one emulated device holds of its column slab: the upload and the transpose's scratch
struct Slab {
  std::vector<int> colptr, row;
  std::vector<double> x;
  std::vector<char> mem;
  WmuCscScratch sc;
  WmuGeneMajor gm;
};
}  // namespace

extern "C" {

void emu_cell_slabs(const int* colptr, long long n_cells, int D, long long* c) {
  const std::vector<long long> v = wmu_cell_slabs(colptr, n_cells, D);
  memcpy(c, v.data(), v.size() * 8);
}

void emu_gene_ranges(const long long* G, long long n_genes, int D, long long* g) {
  const std::vector<long long> v = wmu_gene_ranges(G, n_genes, D);
  memcpy(g, v.data(), v.size() * 8);
}

// The whole call on D = min(D, n_genes) emulated devices.  Returns the OR of the slabs' transpose flags; out is
// written only when it is 0.  grid: rank-kernel CTAs per device (at most its genes), max_ctas: the persistent
// grids of the transpose and the regroup.
unsigned emu_wmu_markers_csc_devices(const int* colptr, const int* row, const double* x, long long n_genes,
                                     long long n_cells, const int* cluster, int n_clusters, int D, double* out,
                                     int grid, int max_ctas) {
  const long long N = n_cells, C = n_clusters;
  if (D > n_genes) D = (int)n_genes;
  const std::vector<long long> c = wmu_cell_slabs(colptr, N, D);
  std::vector<std::unique_ptr<Slab>> slabs;
  std::vector<const long long*> gptr;
  unsigned flags = 0;
  for (int r = 0; r < D; ++r) {
    slabs.emplace_back(new Slab);
    Slab& s = *slabs.back();
    const long long n = c[(size_t)r + 1] - c[(size_t)r], v0 = colptr[c[(size_t)r]], nnz = colptr[c[(size_t)r + 1]] - v0;
    for (long long j = 0; j <= n; ++j) s.colptr.push_back(colptr[c[(size_t)r] + j] - (int)v0);
    s.row.assign(row + v0, row + v0 + nnz);
    s.x.assign(x + v0, x + v0 + nnz);
    s.mem.assign(wmu_csc_layout(nullptr, n_genes, nnz).bytes, (char)0xA5);
    s.sc = wmu_csc_layout(s.mem.data(), n_genes, nnz);
    s.gm = wmu_csc_to_genes(0, s.sc, max_ctas, s.colptr.data(), s.row.data(), s.x.data(), n_genes, n, nnz);
    flags |= *s.sc.flags;
    gptr.push_back(s.sc.gene_ptr);
  }
  if (flags) return flags;
  const WmuExchange xp = wmu_exchange_plan(gptr, n_genes);
  const WmuClusterLists cl = wmu_cluster_lists(cluster, N, n_clusters);
  const std::vector<long long> cell0(c.begin(), c.end() - 1);
  for (int d = 0; d < D; ++d) {
    const long long g0 = xp.g[(size_t)d], ng = xp.g[(size_t)d + 1] - g0, nr = xp.nrecv[(size_t)d];
    std::vector<unsigned> rcell = junk<unsigned>(nr), ecell = junk<unsigned>(nr);
    std::vector<double> rx = junk<double>(nr), ex = junk<double>(nr);
    for (int r = 0; r < D; ++r) {
      const size_t i = (size_t)r * D + d;
      memcpy(rcell.data() + xp.recv[i], slabs[(size_t)r]->gm.ent_cell + xp.send[i], (size_t)xp.cnt[i] * 4);
      memcpy(rx.data() + xp.recv[i], slabs[(size_t)r]->gm.ent_x + xp.send[i], (size_t)xp.cnt[i] * 8);
    }
    std::vector<long long> src, dst;
    wmu_regroup_tables(xp, gptr, d, &src, &dst);
    const WmuGeneMajor gm = D == 1 ? WmuGeneMajor{rcell.data(), rx.data()}
                                   : wmu_regroup(0, max_ctas, rcell.data(), rx.data(), src.data(), dst.data(),
                                                 cell0.data(), D, ng, ecell.data(), ex.data());
    const long long cap = wmu_gene_cap(dst.data(), ng);
    const int gd = (int)std::min<long long>(grid, ng);
    std::vector<unsigned long long> keys = junk<unsigned long long>((long long)gd * 2 * cap);
    std::vector<unsigned> pay = junk<unsigned>((long long)gd * 2 * cap);
    std::vector<double> z_ratio((size_t)(ng * C * 2));
    std::vector<int> single((size_t)ng);
    wmu_markers_csc_launch(0, gd, gm, dst.data(), ng, N, cluster, cl.crank.data(), cl.members.data(),
                           cl.size.data(), cl.cptr.data(), n_clusters, cap, keys.data(), pay.data(), z_ratio.data(),
                           z_ratio.data() + (size_t)(ng * C), single.data());
    wmu_finish(z_ratio.data(), single.data(), ng, n_clusters, out, g0, n_genes);
  }
  return 0;
}

}  // extern "C"
