// jaccard_emu.cpp -- the kernels of the Jaccard path itself (gficf_b200/csrc/jaccard_kernels.cuh: layout
// pre-pass, the k <= 32 / k <= 128 / k <= 1024 count kernels in all output modes, the exact kernel,
// expand and compaction) run through the product's own dispatch (gficf_b200/csrc/jaccard_plan.h) on the
// CUDA emulation.  TEST INFRASTRUCTURE: this file only allocates and poisons the buffers.  The five
// inline-PTX helpers of the header have plain C++ bodies under GFICF_CUDA_EMU; `grid` is the emulated SM
// count (one resident CTA per SM).  Built and loaded by tests/test_jaccard_emu.py and
// tests/test_jaccard_slabs_emu.py:
//   g++ -O1 -std=c++17 -ffp-contract=off -DGFICF_CUDA_EMU -Itests/cuda_emu -Igficf_b200/csrc -shared -fPIC
#include <vector>

#include "jaccard_plan.h"

using namespace gficf;

namespace {
JacCtx emu_ctx(int grid) {
  static LaunchInfo last;
  return JacCtx{0, grid, 0, &last};
}

// the padded rows of the whole n x k matrix (1-based doubles, column-major), laid out by the pre-pass
std::vector<int> layout(const JacCtx& cx, const double* idx_colmajor, long long n, int k, unsigned* flags) {
  std::vector<int> idx((size_t)n * row_stride(k), 0x5A5A5A5A);
  launch_layout(cx, idx_colmajor, n, 0LL, n, k, 0LL, n, idx.data(), flags);
  return idx;
}

// modes 0..7 of emu_jaccard on rows [lo, hi) of the laid-out matrix; cut1 / cut2 end the first two of the
// three segments of modes 6 / 7
bool run_mode(const JacCtx& cx, const int* idx, int k, int mode, long long lo, long long hi, double* f, double* t,
              double* w, void* counts, long long* n_written, unsigned* flags, long long cut1, long long cut2) {
  if (mode == 0) return launch_fast<0>(cx, idx, k, lo, hi, f, t, w, nullptr, flags);
  if (mode == 1 || mode == 2 || mode == 3) {
    std::vector<long long> scratch(expand_scratch_bytes((hi - lo) * (long long)k) / sizeof(long long), -7);
    if (mode == 1 && !launch_fast<1>(cx, idx, k, lo, hi, nullptr, nullptr, nullptr, counts, flags)) return false;
    if (mode != 1) launch_exact(cx, idx, k, lo, hi, mode == 2 ? 1 : 0, counts);
    launch_expand(cx, idx, k, lo, hi, counts, mode == 2, f, t, w, scratch.data(), n_written);
    return true;
  }
  if (mode == 4) return launch_fast<2>(cx, idx, k, lo, hi, nullptr, nullptr, nullptr, counts, flags);
  if (mode == 5) return launch_fast<3>(cx, idx, k, lo, hi, nullptr, nullptr, nullptr, counts, flags, 0x80u);
  if (k > 127 || (mode == 7 && k > 32)) return false;
  const unsigned tag = 0x80u;
  const bool ok = mode == 7 ? launch_fast<3>(cx, idx, k, lo, hi, nullptr, nullptr, nullptr, counts, flags, tag)
                            : launch_fast<1>(cx, idx, k, lo, hi, nullptr, nullptr, nullptr, counts, flags, tag);
  // expand_stream_kernel indexes counts and outputs by absolute edge number
  const long long e0 = lo * (long long)k;
  const int64_t seg_lo[3] = {lo, cut1, cut2}, seg_hi[3] = {cut1, cut2, hi};
  launch_expand_stream(cx, idx, k, seg_lo, seg_hi, 3, (const uint8_t*)counts - e0, f - e0, t - e0, w - e0, tag,
                       1LL << 40, flags);
  return ok;
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
  const JacCtx cx = emu_ctx(grid);
  const long long E = n * k;
  unsigned flags = 0;
  const std::vector<int> idx = layout(cx, idx_colmajor, n, k, &flags);
  if (flags & kFlagBadId) return flags;
  std::vector<unsigned short> u16((size_t)E + 8, 0xA5A5);  // the counts of modes 1 to 3
  void* u = mode >= 1 && mode <= 3 ? (void*)u16.data() : (void*)counts;
  const long long cut1 = (n / 3) & ~1LL, cut2 = (2 * n / 3) & ~1LL;  // even rows: even first edges for any k
  const bool ok = run_mode(cx, idx.data(), k, mode, 0, n, out_colmajor, out_colmajor + E, out_colmajor + 2 * E, u,
                           n_written, &flags, cut1, cut2);
  return ok ? flags : 0x80000000u;
}

int emu_jaccard_variant(int k) { return jaccard_variant(k); }

// emu_jaccard on the row slab [row_lo, row_hi) of an n x k matrix: all n rows are laid out (the gathers
// need them), the kernels run on the slab only, and every output is slab-relative -- from / to / w point
// at the slab's first edge, and so does `counts`, which every count-producing mode uses (uint16 for
// k > 255).  Modes as in emu_jaccard; modes 6 / 7 expand three segments of the slab by absolute edge
// number, as the host rank of the peer gather does.
unsigned emu_jaccard_slab(const double* idx_colmajor, long long n, int k, int mode, long long row_lo,
                          long long row_hi, double* f, double* t, double* w, void* counts, long long* n_written,
                          int grid) {
  const JacCtx cx = emu_ctx(grid);
  unsigned flags = 0;
  const std::vector<int> idx = layout(cx, idx_colmajor, n, k, &flags);
  if (flags & kFlagBadId) return flags;
  const long long lo = row_lo, hi = row_hi;
  const bool ok = run_mode(cx, idx.data(), k, mode, lo, hi, f, t, w, counts, n_written, &flags, lo + (hi - lo) / 3,
                           lo + 2 * (hi - lo) / 3);
  return ok ? flags : 0x80000000u;
}

// Layout pre-pass of rows [lo, hi) into dst (n x row_stride(k) ints; other rows untouched).
// elem 8 / 4: layout_colmajor_kernel on a slab-shaped column-major source (f64 1-based, or int32
// 1-based with NA = INT_MIN) of hi - lo rows whose first row is row lo (ld_rows = hi - lo,
// ld_row0 = lo).  elem 0: pad_i32_kernel on a dense row-major n x k int32 0-based source.  The
// source is copied into a buffer followed by n invalid ids, so a read past it shows up as a bad id.
unsigned emu_layout_slab(const void* src, int elem, long long n, int k, long long lo, long long hi, int* dst,
                         int grid) {
  const JacCtx cx = emu_ctx(grid);
  unsigned flags = 0;
  if (hi <= lo) return 0;
  const long long ld = hi - lo;
  if (elem == 8) {
    std::vector<double> s((size_t)(ld * k + n), -1.0);
    memcpy(s.data(), src, (size_t)(ld * k) * sizeof(double));
    launch_layout(cx, (const double*)s.data(), ld, lo, n, k, lo, hi, dst, &flags);
  } else if (elem == 4) {
    std::vector<int> s((size_t)(ld * k + n), INT32_MIN);
    memcpy(s.data(), src, (size_t)(ld * k) * sizeof(int));
    launch_layout(cx, (const int*)s.data(), ld, lo, n, k, lo, hi, dst, &flags);
  } else {
    std::vector<int> s((size_t)(n * k + n), -1);
    memcpy(s.data(), src, (size_t)(n * k) * sizeof(int));
    launch_pad(cx, s.data(), n, k, lo, hi, dst, &flags);
  }
  return flags;
}

}  // extern "C"
