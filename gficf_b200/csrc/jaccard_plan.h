// jaccard_plan.h -- which kernel, grid and shared memory every call of the Jaccard path launches
// (jaccard_kernels.cuh): row stride, the count kernel for each k, layout pre-pass, exact kernel, expand,
// compaction and the streaming expand.  Included by gficf_cuda.cu (after its error helpers) and by
// tests/cuda_emu/jaccard_emu.cpp with GFICF_CUDA_EMU defined, so the CPU test suite runs the same dispatch
// as the B200.
#pragma once
#include <stdint.h>
#include <stdlib.h>

#include "jaccard_kernels.cuh"
#include "plan_common.h"

namespace gficf {

// k > 32: rows are padded to a multiple of GFICF_WIDE_ROW_INTS ints.  16 (64 bytes): a row never
// straddles an extra 64-byte DRAM burst; 8 (32 bytes, whole sectors): k = 100 fetches 416 instead of
// 448 bytes per gathered row (A/B in profiles/r02_wide_k.md).
#ifndef GFICF_WIDE_ROW_INTS
#define GFICF_WIDE_ROW_INTS 16
#endif
inline int32_t row_stride(int32_t k) {
  if (k <= 4) return 4;
  if (k <= 8) return 8;
  if (k <= 16) return 16;
  if (k <= 32) return 32;
  return (k + GFICF_WIDE_ROW_INTS - 1) / GFICF_WIDE_ROW_INTS * GFICF_WIDE_ROW_INTS;
}

// Table slots per warp-group.  A multiplier is collision free with probability ~exp(-k^2/2/slots)
// (0.37 at slots = k^2/2, 0.14 at k=128 in 4096 slots); a failed try costs warp 0 ~150 cycles of a
// ~20k-cycle row, so the smaller table (more resident warp-groups) wins.
#ifndef GFICF_WIDE_MAX_LOG_TS
#define GFICF_WIDE_MAX_LOG_TS 12
#endif
inline int wide_log_ts(int k) {
  const int want = k <= 45 ? 10 : (k <= 64 ? 11 : (k <= 90 ? 12 : 13));
  return want < GFICF_WIDE_MAX_LOG_TS ? want : GFICF_WIDE_MAX_LOG_TS;
}

inline size_t wide_smem_bytes(int log_ts) { return (size_t)wide_smem_words(log_ts) * 4 + 129 * sizeof(double); }

// the count kernel that serves k, numbered as gficf_cuda_last_launch reports it: KP (k <= 32),
// 1000 + LOG_TS (k <= 128), 2000 / 2001 (k <= 1024, 8- / 16-bit counts); 0 = no fast kernel
inline int jaccard_variant(int k) {
  if (k <= 4) return 4;
  if (k <= 8) return 8;
  if (k <= 16) return 16;
  if (k <= 32) return 32;
  if (k <= 128) return 1000 + wide_log_ts(k);
  if (k <= kLargeMaxK) return k <= 255 ? 2000 : 2001;
  return 0;
}

// grid, block and shared memory of the last count kernel, and its variant (jaccard_variant)
struct LaunchInfo {
  int grid = 0, block = 0, smem = 0, variant = 0;
};

// what the plan needs from the device: the stream, the SM count, and cta_cap (> 0) to lower the resident
// CTAs per SM of the persistent kernels so that two of them on different streams fit side by side
// (gficf_cuda_set_launch_ctas_per_sm).  Every count kernel launched is recorded in *last.
struct JacCtx {
  net_stream_t st;
  int sms;
  int cta_cap;
  LaunchInfo* last;
};

// persistent grid: resident CTAs per SM x SM count, capped by the work
template <typename K>
inline int persistent_grid(const JacCtx& cx, K kernel, int block, size_t smem, long long work_ctas) {
  int per_sm = net_occupancy(kernel, block, smem);
  if (per_sm < 1) per_sm = 1;
  if (cx.cta_cap > 0 && per_sm > cx.cta_cap) per_sm = cx.cta_cap;
  long long g = (long long)per_sm * cx.sms;
  if (g > work_ctas) g = work_ctas;
  if (g < 1) g = 1;
  return (int)g;
}

inline int grid_1d(const JacCtx& cx, long long total, int block, int cap_per_sm = 8) {
  long long g = (total + block - 1) / block;
  long long cap = (long long)cx.sms * cap_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

template <int KP, int CO, bool SKIP>
inline LaunchInfo launch_small_t(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, double* f,
                                 double* t, double* w, uint8_t* u, unsigned* flags, unsigned tag) {
  auto kern = jaccard_small_k_kernel<KP, CO, SKIP>;
  const int block = kSmallWarps * 32;
  const int lg_group = CO == 3 ? 3 : 0;  // CO == 3: groups of 8 rows (8k bytes: whole 8- or 16-byte vectors)
  const long long work = CO == 3 ? (((hi - lo) >> lg_group) + 1 + kSmallWarps - 1) / kSmallWarps
                                 : (hi - lo + kSmallWarps - 1) / kSmallWarps;
  const int grid = persistent_grid(cx, kern, block, 0, work);
  GFICF_LAUNCH(cx.st, kern, grid, block, idx, k, lo, hi, f, t, w, u, flags, tag, lg_group);
  return {grid, block, (int)(sizeof(unsigned) * kSmallWarps * SmallK<KP>::TS + 33 * 8)};
}

// the pad-skipping variant costs registers, so it is used only when a whole 16-byte piece of every
// row is padding (k <= KP-4, e.g. k=25..28 in 32-int rows); k=30 keeps the lean variant
template <int KP, int CO>
inline LaunchInfo launch_small(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, double* f,
                               double* t, double* w, uint8_t* u, unsigned* flags, unsigned tag) {
  if (KP > 4 && k <= KP - 4) return launch_small_t<KP, CO, true>(cx, idx, k, lo, hi, f, t, w, u, flags, tag);
  return launch_small_t<KP, CO, false>(cx, idx, k, lo, hi, f, t, w, u, flags, tag);
}

template <int LOG_TS, int CO>
inline LaunchInfo launch_wide(const JacCtx& cx, const int* idx, int k, int kp, long long lo, long long hi, double* f,
                              double* t, double* w, uint8_t* u, unsigned* flags, unsigned tag) {
  auto kern = jaccard_wide_k_kernel<LOG_TS, CO>;
  const size_t smem = wide_smem_bytes(LOG_TS);
  net_max_dynamic_smem(kern, smem);
  const int block = kWideWarps * 32;
  const int grid = persistent_grid(cx, kern, block, smem, hi - lo);
  GFICF_LAUNCH_EX(cx.st, kern, grid, 1, block, smem, idx, k, kp, lo, hi, f, t, w, u, flags, tag);
  return {grid, block, (int)smem};
}

template <bool CO>
inline LaunchInfo launch_large(const JacCtx& cx, const int* idx, int k, int kp, long long lo, long long hi, double* f,
                               double* t, double* w, void* u, unsigned* flags) {
  const size_t smem = large_smem_bytes();
  const int block = kLargeWarps * 32;
  if (k <= 255) {
    auto kern = jaccard_large_k_kernel<uint8_t, CO>;
    net_max_dynamic_smem(kern, smem);
    const int grid = persistent_grid(cx, kern, block, smem, hi - lo);
    GFICF_LAUNCH_EX(cx.st, kern, grid, 1, block, smem, idx, k, kp, lo, hi, f, t, w, (uint8_t*)u, flags);
    return {grid, block, (int)smem};
  }
  auto kern = jaccard_large_k_kernel<uint16_t, CO>;
  net_max_dynamic_smem(kern, smem);
  const int grid = persistent_grid(cx, kern, block, smem, hi - lo);
  GFICF_LAUNCH_EX(cx.st, kern, grid, 1, block, smem, idx, k, kp, lo, hi, f, t, w, (uint16_t*)u, flags);
  return {grid, block, (int)smem};
}

// fast kernels; returns false when k is outside their range.  CO: 0 = (from,to,w) doubles,
// 1 = counts, 2 = counts with the mutual-neighbour bit (k <= 127), 3 = tagged counts in groups of 8 rows
template <int CO>
inline bool launch_fast(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, double* f, double* t,
                        double* w, void* u_any, unsigned* flags, unsigned tag = 0) {
  uint8_t* u = (uint8_t*)u_any;  // one byte per edge for k <= 255, two above
  if (CO == 2 && k > 127) return false;  // bit 7 of the count byte carries the mutual flag
  if (tag && ((CO != 1 && CO != 3) || k > 127)) return false;  // ... or the epoch bit of the streaming gather
  if (CO == 3 && k > 32) return false;                           // grouped vector stores: the k <= 32 kernel only
  if (hi <= lo) return true;
  const int kp = row_stride(k);
  const int variant = jaccard_variant(k);
  LaunchInfo l;
  switch (variant) {
    case 4: l = launch_small<4, CO>(cx, idx, k, lo, hi, f, t, w, u, flags, tag); break;
    case 8: l = launch_small<8, CO>(cx, idx, k, lo, hi, f, t, w, u, flags, tag); break;
    case 16: l = launch_small<16, CO>(cx, idx, k, lo, hi, f, t, w, u, flags, tag); break;
    case 32: l = launch_small<32, CO>(cx, idx, k, lo, hi, f, t, w, u, flags, tag); break;
    case 1010: l = launch_wide<10, CO>(cx, idx, k, kp, lo, hi, f, t, w, u, flags, tag); break;
    case 1011: l = launch_wide<11, CO>(cx, idx, k, kp, lo, hi, f, t, w, u, flags, tag); break;
    case 1012: l = launch_wide<12, CO>(cx, idx, k, kp, lo, hi, f, t, w, u, flags, tag); break;
    case 1013: l = launch_wide<13, CO>(cx, idx, k, kp, lo, hi, f, t, w, u, flags, tag); break;
    case 2000:
    case 2001:
      if (CO == 2) return false;
      l = launch_large<(CO != 0)>(cx, idx, k, kp, lo, hi, f, t, w, u_any, flags);
      break;
    default: return false;
  }
  l.variant = variant;
  *cx.last = l;
  net_check_launches();
  return true;
}

// layout pre-pass of rows [lo, hi): ld_rows x k column-major source whose first row is row ld_row0
template <typename T>
inline void launch_layout(const JacCtx& cx, const T* src, long long ld_rows, long long ld_row0, long long n, int k,
                          long long lo, long long hi, int* dst, unsigned* flags) {
  if (hi <= lo) return;
  const int kp = row_stride(k);
  int tile_r = kLayoutTileR;
  while (tile_r > 1 && (size_t)tile_r * (kp + 1) * sizeof(int) > 48 * 1024) tile_r /= 2;
  const size_t smem = (size_t)tile_r * (kp + 1) * sizeof(int);
  if (smem > 48 * 1024) net_limit("k too large for the layout pre-pass (k <= 12000)");
  const long long ntiles = (hi - lo + tile_r - 1) / tile_r;
  const long long g = ntiles < (long long)cx.sms * 8 ? ntiles : (long long)cx.sms * 8;
  GFICF_LAUNCH_EX(cx.st, layout_colmajor_kernel<T>, g, 1, kLayoutThreads, smem, src, ld_rows, ld_row0, n, k, kp, lo,
                  hi, dst, flags, tile_r);
  net_check_launches();
}

// rows [lo, hi) of a dense row-major n x k int32 0-based source
inline void launch_pad(const JacCtx& cx, const int* src, long long n, int k, long long lo, long long hi, int* dst,
                       unsigned* flags) {
  if (hi <= lo) return;
  const int kp = row_stride(k);
  const long long total = (hi - lo) * (long long)kp;
  GFICF_LAUNCH(cx.st, pad_i32_kernel, grid_1d(cx, total, 256, 8), 256, src, n, k, kp, lo, hi, dst, flags);
  net_check_launches();
}

inline void launch_exact(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, int set_sem, void* u) {
  if (hi <= lo) return;
  const int kp = row_stride(k);
  const long long total = (hi - lo) * (long long)k;
  const int grid = grid_1d(cx, total, 128, 16);
  if (k <= 255)
    GFICF_LAUNCH(cx.st, jaccard_exact_kernel<uint8_t>, grid, 128, idx, k, kp, lo, hi, set_sem, (uint8_t*)u);
  else
    GFICF_LAUNCH(cx.st, jaccard_exact_kernel<uint16_t>, grid, 128, idx, k, kp, lo, hi, set_sem, (uint16_t*)u);
  net_check_launches();
}

// expand_stream_kernel<W> (W adjacent edges per thread) over ns row segments, the longest of `longest` edges
template <int W>
inline void launch_expand_stream_t(const JacCtx& cx, const int* idx, int k, const StreamSegs& segs, int ns,
                                   long long longest, const uint8_t* u, double* f, double* t, double* w, unsigned tag,
                                   long long spin, unsigned* flags) {
  auto kern = expand_stream_kernel<W>;
  // the resident CTAs are shared evenly by the segments: every sub-grid then advances
  // through its segment at the same rate as the ranks that produce the segments
  int per_sm = net_occupancy(kern, kExpandThreads, 0);
  if (cx.cta_cap > 0 && per_sm > cx.cta_cap) per_sm = cx.cta_cap;  // leave room for a kernel on another stream
  long long gx = (long long)cx.sms * (per_sm > 1 ? per_sm : 1) / ns;
  if (gx < 1) gx = 1;
  const long long need = (longest / W + kExpandThreads - 1) / kExpandThreads;
  if (gx > need) gx = need;
  if (gx < 1) gx = 1;
  GFICF_LAUNCH_EX(cx.st, kern, gx, ns, kExpandThreads, 0, idx, k, row_stride(k), segs, u, f, t, w, tag, spin, flags);
  net_check_launches();
}

// expand_stream_kernel over the row segments [seg_lo[i], seg_hi[i]) (counts and outputs indexed by absolute
// edge number); returns false when a segment is malformed.  spin: bound of the polls in SM clocks.
inline bool launch_expand_stream(const JacCtx& cx, const int* idx, int k, const int64_t* seg_lo,
                                 const int64_t* seg_hi, int n_seg, const uint8_t* u, double* f, double* t, double* w,
                                 unsigned tag, long long spin, unsigned* flags) {
  StreamSegs segs;
  int ns = 0;
  long long longest = 0;
  for (int i = 0; i < n_seg; ++i) {
    if (seg_lo[i] < 0 || seg_hi[i] < seg_lo[i]) return false;
    if (seg_hi[i] == seg_lo[i]) continue;
    segs.lo[ns] = seg_lo[i];
    segs.hi[ns] = seg_hi[i];
    const long long edges = (seg_hi[i] - seg_lo[i]) * (long long)k;
    if (edges > longest) longest = edges;
    ++ns;
  }
  if (!ns) return true;
  // two adjacent edges per thread (16-byte stores) when every output column is 16-byte aligned and every
  // segment starts on an even edge; GFICF_CUDA_STREAM_WIDTH=1 forces the one-edge form (A/B switch)
  bool pair = (((uintptr_t)f | (uintptr_t)t | (uintptr_t)w) & 15) == 0 && ((uintptr_t)u & 1) == 0;
  for (int i = 0; i < ns; ++i) pair = pair && ((segs.lo[i] * (long long)k) & 1) == 0;
  const char* we = getenv("GFICF_CUDA_STREAM_WIDTH");
  if (we && we[0] == '1') pair = false;
  if (pair) launch_expand_stream_t<2>(cx, idx, k, segs, ns, longest, u, f, t, w, tag, spin, flags);
  else launch_expand_stream_t<1>(cx, idx, k, segs, ns, longest, u, f, t, w, tag, spin, flags);
  return true;
}

inline size_t expand_scratch_bytes(long long slab_e) {
  const long long nchunks = (slab_e + kCompactChunk - 1) / kCompactChunk;
  return (size_t)(nchunks + 1) * sizeof(long long);
}

// serial: compaction into the first *n_written edges and a zero tail (scratch: expand_scratch_bytes);
// otherwise every edge in its fixed slot
template <typename CT>
inline void launch_expand_t(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, const CT* u,
                            bool serial, double* f, double* t, double* w, void* scratch, long long* n_written) {
  const int kp = row_stride(k);
  const long long total = (hi - lo) * (long long)k;
  if (total <= 0) return;
  if (!serial) {
    GFICF_LAUNCH(cx.st, expand_fixed_kernel<CT>, grid_1d(cx, total, kExpandThreads, 8), kExpandThreads, idx, k, kp,
                 lo, hi, u, f, t, w);
  } else {
    long long* chunk = (long long*)scratch;
    const long long nchunks = (total + kCompactChunk - 1) / kCompactChunk;
    if (nchunks > 0x7fffffffLL) net_limit("slab too large for compaction");
    GFICF_LAUNCH(cx.st, compact_count_kernel<CT>, nchunks, kCompactThreads, u, total, chunk);
    GFICF_LAUNCH(cx.st, compact_scan_kernel, 1, 1024, chunk, nchunks, n_written);
    GFICF_LAUNCH(cx.st, compact_scatter_kernel<CT>, nchunks, kCompactThreads, idx, k, kp, lo, u, total,
                 (const long long*)chunk, f, t, w);
    GFICF_LAUNCH(cx.st, zero_tail_kernel, grid_1d(cx, total, 256, 8), 256, (const long long*)n_written, total, f, t,
                 w);
  }
  net_check_launches();
}

inline void launch_expand(const JacCtx& cx, const int* idx, int k, long long lo, long long hi, const void* u,
                          bool serial, double* f, double* t, double* w, void* scratch, long long* n_written) {
  if (k <= 255)
    launch_expand_t<uint8_t>(cx, idx, k, lo, hi, (const uint8_t*)u, serial, f, t, w, scratch, n_written);
  else
    launch_expand_t<uint16_t>(cx, idx, k, lo, hi, (const uint16_t*)u, serial, f, t, w, scratch, n_written);
}

}  // namespace gficf
