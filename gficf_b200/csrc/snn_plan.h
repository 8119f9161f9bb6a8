// snn_plan.h -- the scratch layout and launch sequence of the graph build (snn_kernels.cuh), the body of
// gficf_cuda_snn_lower_dev.  Included by gficf_cuda.cu (after its error helpers) and by
// tests/cuda_emu/snn_emu.cpp with GFICF_CUDA_EMU defined, so the CPU test suite runs the same launches as the
// B200.  Scans are the network plan's (net_scan).
#pragma once
#include "network_plan.h"
#include "snn_kernels.cuh"

namespace gficf {

// scratch of the graph build for n cells and cap entries (all pieces 256-byte aligned)
struct SnnScratch {
  int *act, *vid;
  unsigned* first;
  // cnt_b | cnt | cursor | big_cols | n_big: one piece, zeroed by one fill
  char* zeroed;
  size_t zeroed_bytes;
  int *cnt_b, *cnt, *cursor, *big_cols, *n_big;
  long long *off_a, *off_b, *nv;
  NetScratch scan;  // block_sums and total of net_scan; its other pieces stay null
  SnnEntry* entries;
  size_t bytes;
};

inline SnnScratch snn_scratch_layout(char* base, long long n, long long cap) {
  SnnScratch s;
  ScratchCarver c{base};
  s.act = c.take<int>(n);
  s.vid = c.take<int>(n);
  s.first = c.take<unsigned>(n);
  const size_t a = align256((size_t)n * 4), a_big = align256((size_t)(cap / kSnnWarpRankMax + 2) * 4);
  s.zeroed_bytes = 3 * a + a_big + 4;
  s.zeroed = c.take<char>(s.zeroed_bytes);
  s.cnt_b = (int*)s.zeroed;
  s.cnt = (int*)(s.zeroed + a);
  s.cursor = (int*)(s.zeroed + 2 * a);
  s.big_cols = (int*)(s.zeroed + 3 * a);
  s.n_big = (int*)(s.zeroed + 3 * a + a_big);
  s.off_a = c.take<long long>(n + 1);
  s.off_b = c.take<long long>(n + 1);
  s.scan = NetScratch{};
  s.scan.block_sums = c.take<long long>((n + kScanBlock - 1) / kScanBlock + 2);
  s.scan.total = c.take<long long>(1);
  s.nv = c.take<long long>(1);
  s.entries = c.take<SnnEntry>(cap);
  s.bytes = c.bytes;
  return s;
}

// idx: n x row_stride(k) padded rows, um: n*k count bytes with the mutual bit.  Outputs colptr[n+1],
// row / w [entries], vertex_cell[n] (may be null), *nv (sc.nv when nv is null); flags are raised in *flags.
// max_ctas caps the grid-stride launches; sort_ctas is the grid of snn_sort_big_kernel, which needs
// kSnnSmemSortMax * 12 bytes of dynamic shared memory.
inline void snn_lower(net_stream_t st, const SnnScratch& sc, int max_ctas, int sort_ctas, const int* idx, long long n,
                      int k, int kp, const unsigned char* um, long long* colptr, int* row, double* w, int* vertex_cell,
                      long long* nv, unsigned* flags) {
  NetCtx cx;
  cx.st = st;
  cx.sc = sc.scan;
  cx.flags = flags;
  cx.max_ctas = max_ctas;
  if (!nv) nv = sc.nv;
  const long long grid_w = net_grid(cx, n * 32, 256);  // warp per row / column
  const long long grid_t = net_grid(cx, n, 256);
  net_zero(st, sc.zeroed, sc.zeroed_bytes);
  net_fill(st, sc.first, 0xff, (size_t)n * 4);
  // 1. igraph's vertex numbering (first appearance in c(from, to) of the kept rows)
  GFICF_LAUNCH(st, snn_active_kernel, grid_w, 256, um, n, k, sc.act, flags);
  net_scan(cx, sc.act, n, sc.off_a);
  GFICF_LAUNCH(st, snn_vertex_ids_kernel, grid_t, 256, n, (const int*)sc.act, (const long long*)sc.off_a,
               (const long long*)sc.off_b, sc.vid, 0, (int*)nullptr, nv);
  GFICF_LAUNCH(st, snn_targets_kernel<0>, grid_w, 256, idx, um, n, k, kp, (const int*)sc.act,
               (const long long*)sc.off_a, sc.first, sc.cnt_b, (const long long*)sc.off_b, sc.vid);
  GFICF_LAUNCH(st, snn_targets_kernel<1>, grid_w, 256, idx, um, n, k, kp, (const int*)sc.act,
               (const long long*)sc.off_a, sc.first, sc.cnt_b, (const long long*)sc.off_b, sc.vid);
  net_scan(cx, sc.cnt_b, n, sc.off_b);
  GFICF_LAUNCH(st, snn_targets_kernel<2>, grid_w, 256, idx, um, n, k, kp, (const int*)sc.act,
               (const long long*)sc.off_a, sc.first, sc.cnt_b, (const long long*)sc.off_b, sc.vid);
  GFICF_LAUNCH(st, snn_vertex_ids_kernel, grid_t, 256, n, (const int*)sc.act, (const long long*)sc.off_a,
               (const long long*)sc.off_b, sc.vid, 1, vertex_cell, nv);
  // 2. entries per column, column pointers, scatter, rows ascending inside a column
  GFICF_LAUNCH(st, snn_edges_kernel<false>, grid_w, 256, idx, um, n, k, kp, (const int*)sc.vid, sc.cnt,
               (const long long*)nullptr, (SnnEntry*)nullptr);
  net_scan(cx, sc.cnt, n, colptr);
  GFICF_LAUNCH(st, snn_edges_kernel<true>, grid_w, 256, idx, um, n, k, kp, (const int*)sc.vid, sc.cursor,
               (const long long*)colptr, sc.entries);
  GFICF_LAUNCH(st, snn_sort_columns_kernel, grid_w, 256, (const long long*)colptr, (const long long*)nv,
               (const SnnEntry*)sc.entries, row, w, sc.big_cols, sc.n_big);
  GFICF_LAUNCH_EX(st, snn_sort_big_kernel, sort_ctas, 1, 256, kSnnSmemSortMax * 12, (const long long*)colptr,
                  (const SnnEntry*)sc.entries, row, w, (const int*)sc.big_cols, (const int*)sc.n_big);
}

}  // namespace gficf
