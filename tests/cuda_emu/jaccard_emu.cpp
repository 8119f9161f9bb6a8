// jaccard_emu.cpp -- the kernels of the Jaccard path itself (gficf_b200/csrc/jaccard_kernels.cuh: layout
// pre-pass, the k <= 32 / k <= 128 / k <= 1024 count kernels in all output modes, the exact kernel,
// expand and compaction) compiled as plain C++ against the CUDA emulation.  TEST INFRASTRUCTURE.  The
// five inline-PTX helpers of the header have plain C++ bodies under GFICF_CUDA_EMU; the dispatch below
// restates launch_fast / launch_expand of gficf_b200/csrc/gficf_cuda.cu with small grids (the kernel it
// picks for each k, emu_jaccard_variant, is compared with the product's gficf_cuda_last_launch on the
// GPU).  Built and loaded by tests/test_jaccard_emu.py and tests/test_jaccard_slabs_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -shared -fPIC
#include <vector>

#include "jaccard_kernels.cuh"

using namespace gficf;

#define LAUNCH(kernel, grid, block, smem, ...) \
  cuda_emu::launch((unsigned)(grid), (unsigned)(block), [=] { kernel(__VA_ARGS__); }, (size_t)(smem))

namespace {
int row_stride(int k) {  // gficf_cuda_row_stride
  if (k <= 4) return 4;
  if (k <= 8) return 8;
  if (k <= 16) return 16;
  if (k <= 32) return 32;
  return (k + 15) / 16 * 16;
}
int wide_log_ts(int k) { return k <= 45 ? 10 : (k <= 64 ? 11 : 12); }

template <int KP, int CO>
void small(const int* idx, int k, long long lo, long long hi, double* f, double* t, double* w, uint8_t* u,
           unsigned* flags, unsigned tag, int grid) {
  const int lg = CO == 3 ? 3 : 0;
  if (KP > 4 && k <= KP - 4) {
    LAUNCH((jaccard_small_k_kernel<KP, CO, true>), grid, kSmallWarps * 32, 0, idx, k, lo, hi, f, t, w, u, flags, tag, lg);
  } else {
    LAUNCH((jaccard_small_k_kernel<KP, CO, false>), grid, kSmallWarps * 32, 0, idx, k, lo, hi, f, t, w, u, flags, tag, lg);
  }
}

template <int LOG_TS, int CO>
void wide(const int* idx, int k, int kp, long long lo, long long hi, double* f, double* t, double* w, uint8_t* u,
          unsigned* flags, unsigned tag, int grid) {
  const size_t smem = (size_t)wide_smem_words(LOG_TS) * 4 + 129 * sizeof(double);
  LAUNCH((jaccard_wide_k_kernel<LOG_TS, CO>), grid, kWideWarps * 32, smem, idx, k, kp, lo, hi, f, t, w, u, flags, tag);
}

// which count kernel serves k, numbered like gficf_cuda_last_launch reports it: KP (k <= 32),
// 1000 + LOG_TS (k <= 128), 2000 / 2001 (k <= 1024, 8- / 16-bit counts); 0 = no fast kernel
int variant(int k) {
  if (k <= 4) return 4;
  if (k <= 8) return 8;
  if (k <= 16) return 16;
  if (k <= 32) return 32;
  if (k <= 128) return 1000 + wide_log_ts(k);
  if (k <= kLargeMaxK) return k <= 255 ? 2000 : 2001;
  return 0;
}

template <int CO>
bool fast(const int* idx, int k, long long lo, long long hi, double* f, double* t, double* w, void* u_any,
          unsigned* flags, unsigned tag, int grid) {
  uint8_t* u = (uint8_t*)u_any;
  if (CO == 2 && k > 127) return false;
  if (tag && ((CO != 1 && CO != 3) || k > 127)) return false;
  if (CO == 3 && k > 32) return false;
  if (hi <= lo) return true;
  const int kp = row_stride(k);
  switch (variant(k)) {
    case 4: small<4, CO>(idx, k, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 8: small<8, CO>(idx, k, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 16: small<16, CO>(idx, k, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 32: small<32, CO>(idx, k, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 1010: wide<10, CO>(idx, k, kp, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 1011: wide<11, CO>(idx, k, kp, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 1012: wide<12, CO>(idx, k, kp, lo, hi, f, t, w, u, flags, tag, grid); break;
    case 2000:
    case 2001: {
      if (CO == 2 || CO == 3) return false;
      const size_t smem = large_smem_bytes();
      if (k <= 255) {
        LAUNCH((jaccard_large_k_kernel<uint8_t, (CO != 0)>), grid, kLargeWarps * 32, smem, idx, k, kp, lo, hi, f, t, w,
               (uint8_t*)u_any, flags);
      } else {
        LAUNCH((jaccard_large_k_kernel<uint16_t, (CO != 0)>), grid, kLargeWarps * 32, smem, idx, k, kp, lo, hi, f, t, w,
               (uint16_t*)u_any, flags);
      }
      break;
    }
    default: return false;
  }
  return true;
}

template <typename CT>
void expand(const int* idx, int k, long long lo, long long hi, const CT* u, int serial, double* f, double* t,
            double* w, long long* n_written, int grid) {
  const int kp = row_stride(k);
  const long long total = (hi - lo) * (long long)k;
  if (total <= 0) return;
  if (!serial) {
    LAUNCH(expand_fixed_kernel<CT>, grid, kExpandThreads, 0, idx, k, kp, lo, hi, u, f, t, w);
    return;
  }
  const long long nchunks = (total + kCompactChunk - 1) / kCompactChunk;
  std::vector<long long> chunk(nchunks + 1, -7);
  long long* d_chunk = chunk.data();
  LAUNCH(compact_count_kernel<CT>, nchunks, kCompactThreads, 0, u, total, d_chunk);
  LAUNCH(compact_scan_kernel, 1, 1024, 0, d_chunk, nchunks, n_written);
  LAUNCH(compact_scatter_kernel<CT>, nchunks, kCompactThreads, 0, idx, k, kp, lo, u, total, (const long long*)d_chunk, f,
         t, w);
  LAUNCH(zero_tail_kernel, grid, 256, 0, (const long long*)n_written, total, f, t, w);
}
}  // namespace

extern "C" {

// mode: 0 fused kernel (from, to, w straight from the count kernel); 1 counts + expand (fixed slots);
//       2 counts + compaction (serial export; counts must come with set semantics: exact kernel);
//       3 exact kernel (multiset) + expand; 4 counts with the mutual bit (returned in `counts`, no expand);
//       5 tagged counts, grouped stores (k <= 32; returned in `counts`)
//       6 / 7 the two halves of the multi-GPU gather on one "device": parity-tagged counts (6: row stores,
//         7: grouped stores, k <= 32) into `counts`, then expand_stream_kernel over three row segments
//         reading them (every byte is already there, so nothing spins); k <= 127
// idx_colmajor: n x k doubles (1-based); out_colmajor: (n*k) x 3.  Returns the flags, or 0x80000000 when
// the fast kernels do not cover k in that mode.
unsigned emu_jaccard(const double* idx_colmajor, long long n, int k, int mode, double* out_colmajor,
                     unsigned char* counts, long long* n_written, int grid) {
  const int kp = row_stride(k);
  const long long E = n * k;
  std::vector<int> idx((size_t)n * kp, 0x5A5A5A5A);
  std::vector<unsigned short> u16((size_t)E + 8, 0xA5A5);
  unsigned flags = 0;
  int* d_idx = idx.data();
  unsigned* d_flags = &flags;
  int tile_r = kLayoutTileR;
  while (tile_r > 1 && (size_t)tile_r * (kp + 1) * sizeof(int) > 48 * 1024) tile_r /= 2;
  LAUNCH(layout_colmajor_kernel<double>, grid, kLayoutThreads, (size_t)tile_r * (kp + 1) * sizeof(int), idx_colmajor, n,
         0LL, n, k, kp, 0LL, n, d_idx, d_flags, tile_r);
  if (flags & kFlagBadId) return flags;
  double *f = out_colmajor, *t = out_colmajor + E, *w = out_colmajor + 2 * E;
  void* u = u16.data();
  bool ok = true;
  if (mode == 0) {
    ok = fast<0>(d_idx, k, 0, n, f, t, w, nullptr, d_flags, 0, grid);
  } else if (mode == 1) {
    ok = fast<1>(d_idx, k, 0, n, nullptr, nullptr, nullptr, u, d_flags, 0, grid);
    if (ok && k <= 255) expand<uint8_t>(d_idx, k, 0, n, (const uint8_t*)u, 0, f, t, w, n_written, grid);
    else if (ok) expand<uint16_t>(d_idx, k, 0, n, (const uint16_t*)u, 0, f, t, w, n_written, grid);
  } else if (mode == 2 || mode == 3) {
    const long long total = E;
    const int g = grid;
    if (k <= 255) {
      LAUNCH(jaccard_exact_kernel<uint8_t>, g, 128, 0, (const int*)d_idx, k, kp, 0LL, n, mode == 2 ? 1 : 0, (uint8_t*)u);
      expand<uint8_t>(d_idx, k, 0, n, (const uint8_t*)u, mode == 2, f, t, w, n_written, grid);
    } else {
      LAUNCH(jaccard_exact_kernel<uint16_t>, g, 128, 0, (const int*)d_idx, k, kp, 0LL, n, mode == 2 ? 1 : 0,
             (uint16_t*)u);
      expand<uint16_t>(d_idx, k, 0, n, (const uint16_t*)u, mode == 2, f, t, w, n_written, grid);
    }
    (void)total;
  } else if (mode == 4) {
    ok = fast<2>(d_idx, k, 0, n, nullptr, nullptr, nullptr, counts, d_flags, 0, grid);
  } else if (mode == 5) {
    ok = fast<3>(d_idx, k, 0, n, nullptr, nullptr, nullptr, counts, d_flags, 0x80u, grid);
  }
  else if (mode == 6 || mode == 7) {
    if (k > 127 || (mode == 7 && k > 32)) return 0x80000000u;
    const unsigned tag = 0x80u;
    ok = mode == 7 ? fast<3>(d_idx, k, 0, n, nullptr, nullptr, nullptr, counts, d_flags, tag, grid)
                   : fast<1>(d_idx, k, 0, n, nullptr, nullptr, nullptr, counts, d_flags, tag, grid);
    StreamSegs segs;
    const long long cut1 = (n / 3) & ~1LL, cut2 = (2 * n / 3) & ~1LL;  // even rows: even first edges for any k
    segs.lo[0] = 0, segs.hi[0] = cut1, segs.lo[1] = cut1, segs.hi[1] = cut2, segs.lo[2] = cut2, segs.hi[2] = n;
    const bool pair = (((uintptr_t)f | (uintptr_t)t | (uintptr_t)w) & 15) == 0 && ((uintptr_t)counts & 1) == 0;
    const unsigned char* cu = counts;
    if (pair) {
      cuda_emu::launch(2, kExpandThreads, [=] { expand_stream_kernel<2>(d_idx, k, kp, segs, cu, f, t, w, tag, 1LL << 40, d_flags); },
                       0, 3);
    } else {
      cuda_emu::launch(2, kExpandThreads, [=] { expand_stream_kernel<1>(d_idx, k, kp, segs, cu, f, t, w, tag, 1LL << 40, d_flags); },
                       0, 3);
    }
  }
  return ok ? flags : 0x80000000u;
}

int emu_jaccard_variant(int k) { return variant(k); }

// emu_jaccard on the row slab [row_lo, row_hi) of an n x k matrix: all n rows are laid out (the gathers
// need them), the kernels run on the slab only, and every output is slab-relative -- from / to / w point
// at the slab's first edge, and so does `counts`, which every count-producing mode uses (uint16 for
// k > 255).  Modes as in emu_jaccard; modes 6 / 7 expand three segments of the slab by absolute edge
// number, as the host rank of the peer gather does.
unsigned emu_jaccard_slab(const double* idx_colmajor, long long n, int k, int mode, long long row_lo,
                          long long row_hi, double* f, double* t, double* w, void* counts, long long* n_written,
                          int grid) {
  const int kp = row_stride(k);
  std::vector<int> idx((size_t)n * kp, 0x5A5A5A5A);
  unsigned flags = 0;
  int* d_idx = idx.data();
  unsigned* d_flags = &flags;
  int tile_r = kLayoutTileR;
  while (tile_r > 1 && (size_t)tile_r * (kp + 1) * sizeof(int) > 48 * 1024) tile_r /= 2;
  LAUNCH(layout_colmajor_kernel<double>, grid, kLayoutThreads, (size_t)tile_r * (kp + 1) * sizeof(int), idx_colmajor, n,
         0LL, n, k, kp, 0LL, n, d_idx, d_flags, tile_r);
  if (flags & kFlagBadId) return flags;
  const long long lo = row_lo, hi = row_hi;
  bool ok = true;
  if (mode == 0) {
    ok = fast<0>(d_idx, k, lo, hi, f, t, w, nullptr, d_flags, 0, grid);
  } else if (mode == 1) {
    ok = fast<1>(d_idx, k, lo, hi, nullptr, nullptr, nullptr, counts, d_flags, 0, grid);
    if (ok && k <= 255) expand<uint8_t>(d_idx, k, lo, hi, (const uint8_t*)counts, 0, f, t, w, n_written, grid);
    else if (ok) expand<uint16_t>(d_idx, k, lo, hi, (const uint16_t*)counts, 0, f, t, w, n_written, grid);
  } else if (mode == 2 || mode == 3) {
    if (hi <= lo) return flags;
    if (k <= 255) {
      LAUNCH(jaccard_exact_kernel<uint8_t>, grid, 128, 0, (const int*)d_idx, k, kp, lo, hi, mode == 2 ? 1 : 0,
             (uint8_t*)counts);
      expand<uint8_t>(d_idx, k, lo, hi, (const uint8_t*)counts, mode == 2, f, t, w, n_written, grid);
    } else {
      LAUNCH(jaccard_exact_kernel<uint16_t>, grid, 128, 0, (const int*)d_idx, k, kp, lo, hi, mode == 2 ? 1 : 0,
             (uint16_t*)counts);
      expand<uint16_t>(d_idx, k, lo, hi, (const uint16_t*)counts, mode == 2, f, t, w, n_written, grid);
    }
  } else if (mode == 4) {
    ok = fast<2>(d_idx, k, lo, hi, nullptr, nullptr, nullptr, counts, d_flags, 0, grid);
  } else if (mode == 5) {
    ok = fast<3>(d_idx, k, lo, hi, nullptr, nullptr, nullptr, counts, d_flags, 0x80u, grid);
  } else if (mode == 6 || mode == 7) {
    if (k > 127 || (mode == 7 && k > 32)) return 0x80000000u;
    const unsigned tag = 0x80u;
    ok = mode == 7 ? fast<3>(d_idx, k, lo, hi, nullptr, nullptr, nullptr, counts, d_flags, tag, grid)
                   : fast<1>(d_idx, k, lo, hi, nullptr, nullptr, nullptr, counts, d_flags, tag, grid);
    if (hi <= lo) return ok ? flags : 0x80000000u;
    // expand_stream_kernel indexes counts and outputs by absolute edge number
    const long long e0 = lo * (long long)k;
    const unsigned char* cu = (const unsigned char*)counts - e0;
    double *fa = f - e0, *ta = t - e0, *wa = w - e0;
    StreamSegs segs;
    const long long cut1 = lo + (hi - lo) / 3, cut2 = lo + 2 * (hi - lo) / 3;
    segs.lo[0] = lo, segs.hi[0] = cut1, segs.lo[1] = cut1, segs.hi[1] = cut2, segs.lo[2] = cut2, segs.hi[2] = hi;
    // the pairwise form needs 16-byte aligned columns and even first edges (gficf_cuda_expand_stream_dev)
    bool pair = (((uintptr_t)fa | (uintptr_t)ta | (uintptr_t)wa) & 15) == 0 && ((uintptr_t)cu & 1) == 0;
    for (int s = 0; s < 3; ++s) pair = pair && ((segs.lo[s] * (long long)k) & 1) == 0;
    if (pair) {
      cuda_emu::launch(2, kExpandThreads, [=] { expand_stream_kernel<2>(d_idx, k, kp, segs, cu, fa, ta, wa, tag, 1LL << 40, d_flags); },
                       0, 3);
    } else {
      cuda_emu::launch(2, kExpandThreads, [=] { expand_stream_kernel<1>(d_idx, k, kp, segs, cu, fa, ta, wa, tag, 1LL << 40, d_flags); },
                       0, 3);
    }
  }
  return ok ? flags : 0x80000000u;
}

// Layout pre-pass of rows [lo, hi) into dst (n x row_stride(k) ints; other rows untouched).
// elem 8 / 4: layout_colmajor_kernel on a slab-shaped column-major source (f64 1-based, or int32
// 1-based with NA = INT_MIN) of hi - lo rows whose first row is row lo (ld_rows = hi - lo,
// ld_row0 = lo).  elem 0: pad_i32_kernel on a dense row-major n x k int32 0-based source.  The
// source is copied into a buffer followed by n invalid ids, so a read past it shows up as a bad id.
unsigned emu_layout_slab(const void* src, int elem, long long n, int k, long long lo, long long hi, int* dst,
                         int grid) {
  const int kp = row_stride(k);
  unsigned flags = 0;
  unsigned* d_flags = &flags;
  if (hi <= lo) return 0;
  int tile_r = kLayoutTileR;
  while (tile_r > 1 && (size_t)tile_r * (kp + 1) * sizeof(int) > 48 * 1024) tile_r /= 2;
  const size_t smem = (size_t)tile_r * (kp + 1) * sizeof(int);
  const long long ld = hi - lo;
  if (elem == 8) {
    std::vector<double> s((size_t)(ld * k + n), -1.0);
    memcpy(s.data(), src, (size_t)(ld * k) * sizeof(double));
    const double* d_src = s.data();
    LAUNCH(layout_colmajor_kernel<double>, grid, kLayoutThreads, smem, d_src, ld, lo, n, k, kp, lo, hi, dst, d_flags,
           tile_r);
  } else if (elem == 4) {
    std::vector<int> s((size_t)(ld * k + n), INT32_MIN);
    memcpy(s.data(), src, (size_t)(ld * k) * sizeof(int));
    const int* d_src = s.data();
    LAUNCH(layout_colmajor_kernel<int>, grid, kLayoutThreads, smem, d_src, ld, lo, n, k, kp, lo, hi, dst, d_flags,
           tile_r);
  } else {
    std::vector<int> s((size_t)(n * k + n), -1);
    memcpy(s.data(), src, (size_t)(n * k) * sizeof(int));
    const int* d_src = s.data();
    LAUNCH(pad_i32_kernel, grid, 256, 0, d_src, n, k, kp, lo, hi, dst, d_flags);
  }
  return flags;
}

}  // extern "C"
