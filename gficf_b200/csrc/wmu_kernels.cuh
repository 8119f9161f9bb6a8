// wmu_kernels.cuh -- Mann-Whitney U per gene on the device (SURVEY section 8f, "next" row 4).
//
// What it replaces (reference = dibbelab/gficf):
//   src/rcpp_parallel_mann_whitney.cpp:27-100   WMU_test::operator(): per gene concatenate the two
//       groups, sort (sort_indexes, mann_whitney.cpp:17-29), average ranks over ties (getRanks
//       :31-54), tie-group sizes (getCounts :65-85), rank sums U1/U2, sigma with the tie
//       correction (getSigma :87-99), continuity-corrected z, and the group means for log2FC
//   called per cluster from R/deGenes.R:44-54 (findClusterMarkers)
//
// Everything here is integer or correctly-rounded IEEE arithmetic, so it is bit-identical to the
// reference's doubles:
//   * rank sums are sums of half-integers below 2^53 -- exact in any order; here 2*R1 is
//     accumulated in 64-bit integers as sum over tie groups of cx * (i + j + 1) (cx = members of
//     group 1 in the group that occupies sorted positions [i, j));
//   * the tie term sum(t^3 - t) is accumulated by the reference sequentially in sorted order in
//     double; below N = 208064 every partial sum is an exact integer < 2^53 and the order is
//     irrelevant (integer accumulation here); above, the non-trivial groups are compacted in order
//     and summed sequentially by one thread, with the reference's rounding ((t*t)*t) - t;
//   * sigma and z use __dmul_rn / __ddiv_rn / __dsqrt_rn in the reference's operation order;
//   * the group means are sequential sums over the cells in their original order (one thread per
//     gene, coalesced because the R matrix is column-major: consecutive genes are adjacent).
// The two transcendental steps -- the normal cdf of z (GSL in the reference) and log2 of the mean
// ratio -- are left to the host wrapper (libm), one evaluation per gene.
//
// findClusterMarkers' loop over clusters is served by one call as well (wmu_markers_rank_kernel,
// wmu_markers_means_kernel): each gene is sorted once and every cluster's rank sum is formed from the
// same sorted order.
//
// Sort: one CTA per gene, least-significant-digit radix sort (8-bit digits, 8 passes, passes whose
// digit is constant are skipped) on order-preserving 64-bit keys with the element's original
// position as payload, ping-pong buffers in global memory (L2 resident for typical N).
// With GFICF_CUDA_EMU defined the header compiles as plain C++ against tests/cuda_emu/cuda_emu.h (the CPU test
// suite runs both kernels that way); the product build never defines it.
#pragma once
#ifdef GFICF_CUDA_EMU
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>

#include "scan_kernels.cuh"  // GFICF_DYNAMIC_SMEM_T

namespace gficf {

constexpr int kWmuThreads = 512;
constexpr int kWmuWarps = kWmuThreads / 32;
constexpr long long kWmuExactTieN = 208064;  // N^3 < 2^53 below this

__device__ __forceinline__ unsigned long long wmu_key(double v) {
  v = v + 0.0;  // -0.0 -> +0.0: they compare equal in the reference (one tie group)
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

struct WmuGeneOut {
  unsigned long long two_r1;  // 2 * (sum of the averaged ranks of group 1)
  double tie_sum;             // sum over tie groups of t^3 - t, the reference's double
  unsigned distinct;          // number of distinct values (nties.size() in the reference)
  unsigned pad;
};

// z (continuity corrected, divided by sigma) from the exact pieces; *single = 1 when all values are
// equal (the reference then leaves pval = 1, rcpp_parallel_mann_whitney.cpp:56)
__device__ __forceinline__ double wmu_z(const WmuGeneOut& o, long long n1, long long n2, int* single) {
  *single = o.distinct <= 1;
  if (*single) return 0.0;
  const long long n = n1 + n2;
  // U1 = R1 - n1(n1+1)/2, U2 = R2 - n2(n2+1)/2 with R1 + R2 = n(n+1)/2: all multiples of 1/2, exact
  const long long two_u1 = (long long)o.two_r1 - n1 * (n1 + 1);
  const long long two_u2 = (n * (n + 1) - (long long)o.two_r1) - n2 * (n2 + 1);
  const double u1 = 0.5 * (double)two_u1, u2 = 0.5 * (double)two_u2;
  const double mu = (double)((unsigned long long)(n1 * n2) / 2ull);  // :86 size_t division, then double
  // getSigma (mann_whitney.cpp:87-99) with n1, n2 as doubles, in its operation order
  const double d1 = (double)n1, d2 = (double)n2;
  const double a = __ddiv_rn(__dmul_rn(d1, d2), 12.0);
  const double np1 = __dadd_rn(__dadd_rn(d1, d2), 1.0);
  const double den = __dmul_rn(__dadd_rn(d1, d2), __dadd_rn(__dadd_rn(d1, d2), -1.0));
  const double sig = __dsqrt_rn(__dmul_rn(a, __dadd_rn(np1, -__ddiv_rn(o.tie_sum, den))));
  double z = u1 < u2 ? u1 - mu : u2 - mu;  // exact
  z = z < 0 ? z + 0.5 : z - 0.5;           // :90 continuity correction, exact
  return __ddiv_rn(z, sig);
}

// ---------------------------------------------------------------------------
// One CTA per gene (persistent over genes).  scratch per CTA: keys[2][N] | pay[2][N] | px[N+1].
//
// Expression matrices are sparse: most of a gene's values are exactly 0, i.e. ONE tie group that
// needs no sorting.  Only the M non-zero values are compacted and sorted; the zeros enter the rank
// sums, the tie term and the distinct-value count analytically as the group that occupies sorted
// positions [n_neg, n_neg + nz) (n_neg = number of negative values, nz = N - M).  Dense input
// simply has M = N.
// ---------------------------------------------------------------------------

// Shared memory of the per-gene sort and tie-group pass (wmu_load, wmu_sort, wmu_tie_groups).
struct WmuSortSmem {
  unsigned hist[256];
  unsigned base[256];
  unsigned short wcnt[kWmuWarps][256];
  unsigned tile_total[256];
  unsigned long long red[kWmuWarps];
  unsigned scan[kWmuWarps];
  unsigned carry, flag, m, z1, neg, negties;
};

// A gene after wmu_load (and wmu_sort): its M non-zero values sorted (keys, payload = the value's position)
// in buffer `cur`; nz = N - M zeros, n_neg negative values, z1 zeros among positions [0, n1).
struct WmuSorted {
  long long M, nz, n_neg, z1;
  int cur;
};

// Load step: the n_items values item(i, &pos) of a gene of N cells (n_items == N for a dense row; the
// stored values for a sparse one, the other N - n_items cells being zeros) -- non-zero values are appended
// in any order to k0 / p0 as (key, position); zeros, stored or not, are counted.  Called by every thread
// of the CTA; ends on a barrier.
template <class Item>
__device__ __forceinline__ WmuSorted wmu_load(long long n_items, long long n1, long long N, unsigned long long* k0,
                                              unsigned* p0, WmuSortSmem& sm, Item item) {
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  if (tid == 0) {
    sm.m = 0;
    sm.z1 = 0;
    sm.neg = 0;
  }
  __syncthreads();
  for (long long t0 = 0; t0 < n_items; t0 += kWmuThreads) {
    const long long i = t0 + tid;
    double v = 0.0;
    unsigned p = 0;
    const bool in = i < n_items;
    if (in) v = item(i, &p);
    const bool nzv = in && v != 0.0;  // -0.0 == 0.0: same tie group as +0.0, like in the reference
    const unsigned m_nz = __ballot_sync(0xffffffffu, nzv);
    const unsigned m_z1 = __ballot_sync(0xffffffffu, in && !nzv && (long long)p < n1);
    const unsigned m_neg = __ballot_sync(0xffffffffu, nzv && v < 0.0);
    unsigned wbase = 0;
    if (lane == 0) {
      if (m_nz) wbase = atomicAdd(&sm.m, __popc(m_nz));
      if (m_z1) atomicAdd(&sm.z1, __popc(m_z1));
      if (m_neg) atomicAdd(&sm.neg, __popc(m_neg));
    }
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if (nzv) {
      const unsigned pos = wbase + __popc(m_nz & lt_mask);
      k0[pos] = wmu_key(v);
      p0[pos] = p;
    }
  }
  __syncthreads();
  WmuSorted s;
  s.M = sm.m;
  s.nz = N - s.M;
  s.z1 = sm.z1;
  s.n_neg = sm.neg;
  s.cur = 0;
  return s;
}

// Gene g's dense row of N values -- positions [0, n1) from mat_x, the rest from mat_y; element (g, c) of a
// column-major matrix sits at g + c * n_genes.
__device__ __forceinline__ WmuSorted wmu_load_dense(const double* __restrict__ mat_x, const double* __restrict__ mat_y,
                                                    long long n_genes, long long g, long long n1, long long N,
                                                    unsigned long long* k0, unsigned* p0, WmuSortSmem& sm) {
  return wmu_load(N, n1, N, k0, p0, sm, [&](long long i, unsigned* p) {
    *p = (unsigned)i;
    return i < n1 ? __ldg(mat_x + g + i * n_genes) : __ldg(mat_y + g + (i - n1) * n_genes);
  });
}

// Sort step: LSD radix sort of the M loaded keys, 8 bits per pass; sets s.cur.  Ends on a barrier.
__device__ __forceinline__ void wmu_sort(WmuSorted& s, unsigned long long* k0, unsigned long long* k1, unsigned* p0,
                                         unsigned* p1, WmuSortSmem& sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long M = s.M;
  int cur = 0;
  for (int pass = 0; pass < 8 && M > 1; ++pass) {
    const int shift = pass * 8;
    if (tid < 256) sm.hist[tid] = 0;
    __syncthreads();
    const unsigned long long* kin = cur ? k1 : k0;
    const unsigned* pin = cur ? p1 : p0;
    unsigned long long* kout = cur ? k0 : k1;
    unsigned* pout = cur ? p0 : p1;
    for (long long t0 = 0; t0 < M; t0 += kWmuThreads) {  // warp-aggregated histogram
      const long long i = t0 + tid;
      const unsigned d = i < M ? ((unsigned)(kin[i] >> shift) & 255u) : 256u + (unsigned)lane;
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      if (i < M && (peers & lt_mask) == 0) atomicAdd(&sm.hist[d], (unsigned)__popc(peers));
    }
    __syncthreads();
    if (tid == 0) sm.flag = 0;
    __syncthreads();
    if (tid < 256 && sm.hist[tid] == (unsigned)M) sm.flag = 1;  // every key has the same digit: nothing moves
    __syncthreads();
    if (sm.flag) continue;
    if (warp == 0) {  // exclusive scan of the 256 counts: 8 per lane
      unsigned c[8], sum = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        c[q] = sm.hist[lane * 8 + q];
        sum += c[q];
      }
      unsigned inc = sum;
#pragma unroll
      for (int m = 1; m < 32; m <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, inc, m);
        if (lane >= m) inc += o;
      }
      unsigned run = inc - sum;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        sm.base[lane * 8 + q] = run;
        run += c[q];
      }
    }
    __syncthreads();
    for (long long t0 = 0; t0 < M; t0 += kWmuThreads) {
      for (int x = tid; x < kWmuWarps * 256; x += kWmuThreads) (&sm.wcnt[0][0])[x] = 0;
      __syncthreads();
      const long long i = t0 + tid;
      const bool valid = i < M;
      unsigned long long key = 0;
      unsigned pay = 0, d = 256u + (unsigned)lane;  // invalid lanes: a digit nobody shares
      if (valid) {
        key = kin[i];
        pay = pin[i];
        d = (unsigned)(key >> shift) & 255u;
      }
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      const unsigned rank_in_warp = __popc(peers & lt_mask);
      if (valid && rank_in_warp == 0) sm.wcnt[warp][d] = (unsigned short)__popc(peers);
      __syncthreads();
      if (tid < 256) {  // exclusive prefix over the warps, per digit
        unsigned acc = 0;
#pragma unroll
        for (int w = 0; w < kWmuWarps; ++w) {
          const unsigned c = sm.wcnt[w][tid];
          sm.wcnt[w][tid] = (unsigned short)acc;
          acc += c;
        }
        sm.tile_total[tid] = acc;
      }
      __syncthreads();
      if (valid) {
        const unsigned pos = sm.base[d] + sm.wcnt[warp][d] + rank_in_warp;
        kout[pos] = key;
        pout[pos] = pay;
      }
      __syncthreads();
      if (tid < 256) sm.base[tid] += sm.tile_total[tid];
    }
    cur ^= 1;
    __syncthreads();
  }
  s.cur = cur;
}

// The tie groups of a sorted gene: the thread that sits on the first element of a group finds the
// group's end by binary search (the keys are sorted), calls on_group(i, j, off) for the group at
// sorted non-zero positions [i, j) and adds the group's tie term and distinct count.  Sorted position
// q of the non-zero array is global position q + off: off = 0 for negative values, nz for positive
// ones (the zeros sit in between).  Thread 0 then adds the zero group and writes out.tie_sum and
// out.distinct.  tie_list (M doubles, free scratch) holds the non-trivial groups' terms in sorted order
// when the tie term is the reference's sequential double sum.  Called by every thread; ends on a barrier.
template <class OnGroup>
__device__ __forceinline__ void wmu_tie_groups(const unsigned long long* __restrict__ keys, const WmuSorted& s,
                                               long long N, double* __restrict__ tie_list, WmuSortSmem& sm,
                                               WmuGeneOut& out, OnGroup on_group) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long M = s.M, nz = s.nz, n_neg = s.n_neg;
  const unsigned long long kZeroKey = 0x8000000000000000ull;  // wmu_key(0.0)
  unsigned long long tie_int = 0;
  unsigned distinct = 0;
  const bool ordered_ties = N >= kWmuExactTieN;
  if (tid == 0) {
    sm.carry = 0;
    sm.negties = 0;
  }
  __syncthreads();
  for (long long t0 = 0; t0 < M; t0 += kWmuThreads) {
    const long long i = t0 + tid;
    bool start = false;
    long long j = 0;
    if (i < M) {
      const unsigned long long key = keys[i];
      start = i == 0 || keys[i - 1] != key;
      if (start) {
        long long lo = i + 1, hi = M;  // first position > i whose key differs
        while (lo < hi) {
          const long long mid = (lo + hi) >> 1;
          if (keys[mid] == key) lo = mid + 1;
          else hi = mid;
        }
        j = lo;
        on_group(i, j, key > kZeroKey ? nz : 0);
        ++distinct;
        const unsigned long long t = (unsigned long long)(j - i);
        if (!ordered_ties) tie_int += t * t * t - t;
      }
    }
    if (ordered_ties) {  // non-trivial groups, compacted in sorted order
      const unsigned f = (start && j - i >= 2) ? 1u : 0u;
      unsigned inc = f;
#pragma unroll
      for (int m = 1; m < 32; m <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, inc, m);
        if (lane >= m) inc += o;
      }
      if (lane == 31) sm.scan[warp] = inc;
      __syncthreads();
      unsigned before = sm.carry;
      for (int w = 0; w < warp; ++w) before += sm.scan[w];
      if (f) {
        const double t = (double)(j - i);
        tie_list[before + inc - 1] = __dadd_rn(__dmul_rn(__dmul_rn(t, t), t), -t);  // ((t*t)*t) - t, :94
        if (i < n_neg) atomicAdd(&sm.negties, 1u);  // groups that precede the zeros
      }
      __syncthreads();
      if (tid == kWmuThreads - 1) sm.carry = before + inc;
      __syncthreads();
    }
  }
  // ---- block reduction of the integer pieces
#pragma unroll
  for (int m = 16; m; m >>= 1) {
    tie_int += __shfl_xor_sync(0xffffffffu, tie_int, m);
    distinct += __shfl_xor_sync(0xffffffffu, distinct, m);
  }
  unsigned long long tie_total = 0;  // thread 0
  if (lane == 0) sm.red[warp] = tie_int;
  __syncthreads();
  if (tid == 0)
    for (int w = 0; w < kWmuWarps; ++w) tie_total += sm.red[w];
  __syncthreads();
  if (lane == 0) sm.red[warp] = distinct;
  __syncthreads();
  if (tid == 0) {
    unsigned long long d = 0;
    for (int w = 0; w < kWmuWarps; ++w) d += sm.red[w];
    // the zeros: one group at sorted positions [n_neg, n_neg + nz); below kWmuExactTieN every partial
    // sum of the tie term is an exact integer < 2^53
    if (nz > 0) {
      d += 1;
      tie_total += (unsigned long long)nz * (unsigned long long)nz * (unsigned long long)nz - (unsigned long long)nz;
    }
    out.distinct = (unsigned)d;
    out.tie_sum = (double)tie_total;
    if (ordered_ties) {  // the reference's sequential double accumulation, in sorted order
      double acc = 0.0;
      const unsigned cnt = sm.carry, negc = sm.negties;
      const double tz = (double)nz;
      for (unsigned q = 0; q < negc; ++q) acc = __dadd_rn(acc, tie_list[q]);
      if (nz >= 2) acc = __dadd_rn(acc, __dadd_rn(__dmul_rn(__dmul_rn(tz, tz), tz), -tz));
      for (unsigned q = negc; q < cnt; ++q) acc = __dadd_rn(acc, tie_list[q]);
      out.tie_sum = acc;
    }
  }
  __syncthreads();
}

// Two groups: positions [0, n1) of every gene (mat_x) against positions [n1, n1 + n2) (mat_y).
__global__ void __launch_bounds__(kWmuThreads, 2)
wmu_rank_kernel(const double* __restrict__ mat_x, const double* __restrict__ mat_y, long long n_genes,
                long long n1, long long n2, unsigned long long* __restrict__ scratch_keys,
                unsigned* __restrict__ scratch_pay, double* __restrict__ out_z,
                int* __restrict__ out_single) {
  __shared__ WmuSortSmem sm;
  __shared__ WmuGeneOut s_out;

  const long long N = n1 + n2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long* const k0 = scratch_keys + (size_t)blockIdx.x * 2 * N;
  unsigned long long* const k1 = k0 + N;
  unsigned* const p0 = scratch_pay + (size_t)blockIdx.x * (3 * N + 2);
  unsigned* const p1 = p0 + N;
  unsigned* const px = p0 + 2 * N;  // [M+1]

  for (long long g = blockIdx.x; g < n_genes; g += gridDim.x) {
    WmuSorted s = wmu_load_dense(mat_x, mat_y, n_genes, g, n1, N, k0, p0, sm);
    wmu_sort(s, k0, k1, p0, p1, sm);
    const long long M = s.M;
    const unsigned long long* keys = s.cur ? k1 : k0;
    const unsigned* pays = s.cur ? p1 : p0;
    // ---- px[p] = number of group-1 elements among sorted non-zero positions [0, p)
    if (tid == 0) sm.carry = 0;
    __syncthreads();
    for (long long t0 = 0; t0 < M; t0 += kWmuThreads) {
      const long long i = t0 + tid;
      const unsigned f = (i < M && (long long)pays[i] < n1) ? 1u : 0u;
      unsigned inc = f;
#pragma unroll
      for (int m = 1; m < 32; m <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, inc, m);
        if (lane >= m) inc += o;
      }
      if (lane == 31) sm.scan[warp] = inc;
      __syncthreads();
      unsigned before = sm.carry;
      for (int w = 0; w < warp; ++w) before += sm.scan[w];
      if (i < M) px[i] = before + inc - f;
      __syncthreads();
      if (tid == kWmuThreads - 1) sm.carry = before + inc;
      __syncthreads();
    }
    if (tid == 0) px[M] = sm.carry;
    __syncthreads();
    // ---- 2 * R1 over the non-zero tie groups: cx group-1 members of a group at global positions
    //      [i + off, j + off) have the averaged rank (i + j + 2 off + 1) / 2 each (1-based)
    unsigned long long two_r1 = 0;
    wmu_tie_groups(keys, s, N, reinterpret_cast<double*>(s.cur ? k0 : k1), sm, s_out,
                   [&](long long i, long long j, long long off) {
                     const unsigned long long cx = px[j] - px[i];
                     two_r1 += cx * (unsigned long long)(i + j + 2 * off + 1);
                   });
#pragma unroll
    for (int m = 16; m; m >>= 1) two_r1 += __shfl_xor_sync(0xffffffffu, two_r1, m);
    if (lane == 0) sm.red[warp] = two_r1;
    __syncthreads();
    if (tid == 0) {
      unsigned long long tr = 0;
      for (int w = 0; w < kWmuWarps; ++w) tr += sm.red[w];
      if (s.nz > 0) tr += (unsigned long long)s.z1 * (unsigned long long)(2 * s.n_neg + s.nz + 1);  // the zeros
      s_out.two_r1 = tr;
      int single;
      const double z = wmu_z(s_out, n1, n2, &single);
      out_z[g] = z;
      out_single[g] = single;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// One-vs-rest for every cluster at once (findClusterMarkers, R/deGenes.R:44-54): cluster c's cells
// against all other cells, for every c.  A gene's values form the same multiset whichever way the
// cells are split, so its sort, tie groups, tie term and distinct count are computed once; only the
// rank sum of each cluster depends on the split.  Every sorted non-zero element finds its tie group
// [lo, hi) by binary search and adds its doubled averaged rank lo + hi + 2 off + 1 to its cluster's
// 64-bit accumulator in shared memory (integer atomics: exact in any order); the zero group adds
// (n_c - nnz_c) (2 n_neg + nz + 1) per cluster.  z per (gene, cluster) then comes from wmu_z with
// n1 = n_c, n2 = N - n_c.
// Dynamic shared memory: two_r1[n_clusters] (u64) | nnz[n_clusters] (u32), kWmuClusterSmemBytes each.
// Scratch per CTA as for wmu_rank_kernel (px unused).  out_z[c * n_genes + g], out_single[g].
// ---------------------------------------------------------------------------
constexpr int kWmuClusterSmemBytes = 12;
constexpr int kWmuMaxClusters = 8192;  // 96 KiB of accumulators: two CTAs still fit an SM's shared memory

// Everything of one gene after its load step, shared by both markers kernels: sort, every cluster's rank
// sum, tie groups, z per (gene, cluster).  The payload of a loaded value is its cell.  s_tr / s_nnz must
// be zero on entry.  Called by every thread; ends on a barrier.
__device__ __forceinline__ void wmu_markers_gene(WmuSorted s, long long g, long long n_genes, long long N,
                                                 const int* __restrict__ cluster,
                                                 const long long* __restrict__ cluster_size, int n_clusters,
                                                 unsigned long long* k0, unsigned long long* k1, unsigned* p0,
                                                 unsigned* p1, unsigned long long* s_tr, unsigned* s_nnz,
                                                 WmuSortSmem& sm, WmuGeneOut& s_out, double* __restrict__ out_z,
                                                 int* __restrict__ out_single) {
  const int tid = threadIdx.x;
  const unsigned long long kZeroKey = 0x8000000000000000ull;  // wmu_key(0.0)
  wmu_sort(s, k0, k1, p0, p1, sm);
  const long long M = s.M;
  const unsigned long long* keys = s.cur ? k1 : k0;
  const unsigned* pays = s.cur ? p1 : p0;
  for (long long i = tid; i < M; i += kWmuThreads) {
    const unsigned long long key = keys[i];
    long long lo = i, hi = i + 1;
    if (i > 0 && keys[i - 1] == key) {  // first position whose key equals this one
      long long a = 0, b = i - 1;
      while (a < b) {
        const long long mid = (a + b) >> 1;
        if (keys[mid] < key) a = mid + 1;
        else b = mid;
      }
      lo = a;
    }
    if (hi < M && keys[hi] == key) {  // first position > i whose key differs
      long long a = hi + 1, b = M;
      while (a < b) {
        const long long mid = (a + b) >> 1;
        if (keys[mid] == key) a = mid + 1;
        else b = mid;
      }
      hi = a;
    }
    const long long off = key > kZeroKey ? s.nz : 0;
    const int c = __ldg(cluster + pays[i]);
    atomicAdd(&s_tr[c], (unsigned long long)(lo + hi + 2 * off + 1));
    atomicAdd(&s_nnz[c], 1u);
  }
  wmu_tie_groups(keys, s, N, reinterpret_cast<double*>(s.cur ? k0 : k1), sm, s_out,
                 [](long long, long long, long long) {});
  for (int c = tid; c < n_clusters; c += kWmuThreads) {
    const long long nc = cluster_size[c];
    WmuGeneOut o = s_out;
    o.two_r1 = s_tr[c] + (unsigned long long)(nc - s_nnz[c]) * (unsigned long long)(2 * s.n_neg + s.nz + 1);
    int single;
    out_z[(size_t)c * n_genes + g] = wmu_z(o, nc, N - nc, &single);
    if (c == 0) out_single[g] = single;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kWmuThreads, 2)
wmu_markers_rank_kernel(const double* __restrict__ mat, long long n_genes, long long n_cells,
                        const int* __restrict__ cluster, const long long* __restrict__ cluster_size, int n_clusters,
                        unsigned long long* __restrict__ scratch_keys, unsigned* __restrict__ scratch_pay,
                        double* __restrict__ out_z, int* __restrict__ out_single) {
  __shared__ WmuSortSmem sm;
  __shared__ WmuGeneOut s_out;
  GFICF_DYNAMIC_SMEM_T(unsigned long long, wmu_cluster_acc);
  unsigned long long* const s_tr = wmu_cluster_acc;
  unsigned* const s_nnz = reinterpret_cast<unsigned*>(wmu_cluster_acc + n_clusters);

  const long long N = n_cells;
  const int tid = threadIdx.x;
  unsigned long long* const k0 = scratch_keys + (size_t)blockIdx.x * 2 * N;
  unsigned long long* const k1 = k0 + N;
  unsigned* const p0 = scratch_pay + (size_t)blockIdx.x * (3 * N + 2);
  unsigned* const p1 = p0 + N;

  for (long long g = blockIdx.x; g < n_genes; g += gridDim.x) {
    for (int c = tid; c < n_clusters; c += kWmuThreads) {
      s_tr[c] = 0;
      s_nnz[c] = 0;
    }
    const WmuSorted s = wmu_load_dense(mat, mat, n_genes, g, N, N, k0, p0, sm);
    wmu_markers_gene(s, g, n_genes, N, cluster, cluster_size, n_clusters, k0, k1, p0, p1, s_tr, s_nnz, sm, s_out,
                     out_z, out_single);
  }
}

// The same for a gene-major sparse matrix (wmu_csc_to_genes below): gene g's stored values are
// ent_x[gene_ptr[g] .. gene_ptr[g + 1]) at cells ent_cell[...], cells ascending; every other cell is 0.
// Only the stored values are read.  Scratch per CTA: keys[2][cap] | pay[2][cap], cap >= the largest
// number of stored values of a gene.
__global__ void __launch_bounds__(kWmuThreads, 2)
wmu_markers_csr_rank_kernel(const double* __restrict__ ent_x, const unsigned* __restrict__ ent_cell,
                            const long long* __restrict__ gene_ptr, long long n_genes, long long n_cells,
                            const int* __restrict__ cluster, const long long* __restrict__ cluster_size,
                            int n_clusters, long long cap, unsigned long long* __restrict__ scratch_keys,
                            unsigned* __restrict__ scratch_pay, double* __restrict__ out_z,
                            int* __restrict__ out_single) {
  __shared__ WmuSortSmem sm;
  __shared__ WmuGeneOut s_out;
  GFICF_DYNAMIC_SMEM_T(unsigned long long, wmu_cluster_acc);
  unsigned long long* const s_tr = wmu_cluster_acc;
  unsigned* const s_nnz = reinterpret_cast<unsigned*>(wmu_cluster_acc + n_clusters);

  const int tid = threadIdx.x;
  unsigned long long* const k0 = scratch_keys + (size_t)blockIdx.x * 2 * cap;
  unsigned long long* const k1 = k0 + cap;
  unsigned* const p0 = scratch_pay + (size_t)blockIdx.x * 2 * cap;
  unsigned* const p1 = p0 + cap;

  for (long long g = blockIdx.x; g < n_genes; g += gridDim.x) {
    for (int c = tid; c < n_clusters; c += kWmuThreads) {
      s_tr[c] = 0;
      s_nnz[c] = 0;
    }
    const long long lo = gene_ptr[g];
    const WmuSorted s = wmu_load(gene_ptr[g + 1] - lo, 0, n_cells, k0, p0, sm, [&](long long i, unsigned* p) {
      *p = __ldg(ent_cell + lo + i);
      return __ldg(ent_x + lo + i);
    });
    wmu_markers_gene(s, g, n_genes, n_cells, cluster, cluster_size, n_clusters, k0, k1, p0, p1, s_tr, s_nnz, sm,
                     s_out, out_z, out_single);
  }
}

// Group means for the fold change: avg(v + 1) with the reference's sequential accumulation
// (std::accumulate from 0.0 over the cells in order, rcpp_parallel_mann_whitney.cpp:97-99,
// mann_whitney.cpp:123-126).  The sum of a gene is inherently sequential, the loading is not: a CTA
// owns 32 adjacent genes; its 8 warps stream tiles of 64 cells x 32 genes (coalesced: the R matrix is
// column-major, 32 adjacent genes are 256 contiguous bytes) through a double-buffered shared-memory
// tile while warp 0 -- one lane per gene -- adds its gene's values in cell order.
// out_ratio[g] = avg1 / avg2.
constexpr int kMeanGenes = 32, kMeanCells = 64, kMeanThreads = 256;

__global__ void __launch_bounds__(kMeanThreads)
wmu_means_kernel(const double* __restrict__ mat_x, const double* __restrict__ mat_y, long long n_genes,
                 long long n1, long long n2, double* __restrict__ out_ratio) {
  __shared__ double tile[2][kMeanCells][kMeanGenes + 1];
  const int tid = threadIdx.x, lane = tid & 31;
  const long long g0 = (long long)blockIdx.x * kMeanGenes;
  const long long N = n1 + n2;
  const long long ntiles = (N + kMeanCells - 1) / kMeanCells;
  auto load_tile = [&](long long t, int buf) {
    for (int x = tid; x < kMeanCells * kMeanGenes; x += kMeanThreads) {
      const int c = x / kMeanGenes, gg = x % kMeanGenes;
      const long long cell = t * kMeanCells + c, gene = g0 + gg;
      double v = 0.0;
      if (cell < N && gene < n_genes)
        v = cell < n1 ? __ldg(mat_x + gene + cell * n_genes) : __ldg(mat_y + gene + (cell - n1) * n_genes);
      tile[buf][c][gg] = v;
    }
  };
  double s1 = 0.0, s2 = 0.0;
  load_tile(0, 0);
  __syncthreads();
  for (long long t = 0; t < ntiles; ++t) {
    const int buf = (int)(t & 1);
    if (tid >= 32) {
      if (t + 1 < ntiles) {  // warps 1..7 fetch the next tile while warp 0 sums this one
        for (int x = tid - 32; x < kMeanCells * kMeanGenes; x += kMeanThreads - 32) {
          const int c = x / kMeanGenes, gg = x % kMeanGenes;
          const long long cell = (t + 1) * kMeanCells + c, gene = g0 + gg;
          double v = 0.0;
          if (cell < N && gene < n_genes)
            v = cell < n1 ? __ldg(mat_x + gene + cell * n_genes) : __ldg(mat_y + gene + (cell - n1) * n_genes);
          tile[buf ^ 1][c][gg] = v;
        }
      }
    } else {
      const long long c_lo = t * kMeanCells;
#pragma unroll 8
      for (int c = 0; c < kMeanCells; ++c) {
        const long long cell = c_lo + c;
        if (cell >= N) break;
        const double v1 = __dadd_rn(tile[buf][c][lane], 1.0);
        if (cell < n1) s1 = __dadd_rn(s1, v1);
        else s2 = __dadd_rn(s2, v1);
      }
    }
    __syncthreads();
  }
  if (tid < 32 && g0 + lane < n_genes)
    out_ratio[g0 + lane] = __ddiv_rn(__ddiv_rn(s1, (double)n1), __ddiv_rn(s2, (double)n2));
}

// Fold-change means of every (gene, cluster) pair: sum(v + 1) over the cluster's cells and over all
// other cells, each sequential in cell order (what the per-cluster call sums over its two submatrices;
// "total minus cluster" would round differently, so every pair is a chain of its own).  Grid: gene
// blocks of kMeanGenes x cluster blocks of kMarkClusters.  A tile of 64 cells x 32 genes (v + 1, the
// reference's first rounding) and the tile's labels are staged once per cluster block, double-buffered
// by kMarkLoaders warps, while warp w adds, lane = gene, for cluster blockIdx.y * kMarkClusters + w.
// out_ratio[c * n_genes + g] = avg_in / avg_out.
constexpr int kMarkClusters = 8, kMarkLoaders = 4, kMarkThreads = 32 * (kMarkClusters + kMarkLoaders);
constexpr int kMarkLoadsPerThread = kMeanCells * kMeanGenes / (32 * kMarkLoaders);

__global__ void __launch_bounds__(kMarkThreads)
wmu_markers_means_kernel(const double* __restrict__ mat, long long n_genes, long long n_cells,
                         const int* __restrict__ cluster, const long long* __restrict__ cluster_size, int n_clusters,
                         double* __restrict__ out_ratio) {
  __shared__ double tile[2][kMeanCells][kMeanGenes + 1];
  __shared__ int lab[2][kMeanCells];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long g0 = (long long)blockIdx.x * kMeanGenes;
  const int c = (int)blockIdx.y * kMarkClusters + warp;  // the cluster of an adding warp
  const long long ntiles = (n_cells + kMeanCells - 1) / kMeanCells;
  // loader thread `ltid` of the CTA's loaders: all values first, then the stores (the loads overlap)
  auto load_tile = [&](long long t, int buf, int ltid) {
    double v[kMarkLoadsPerThread];
#pragma unroll
    for (int q = 0; q < kMarkLoadsPerThread; ++q) {
      const int x = ltid + q * 32 * kMarkLoaders;
      const long long cell = t * kMeanCells + x / kMeanGenes, gene = g0 + x % kMeanGenes;
      v[q] = cell < n_cells && gene < n_genes ? __ldg(mat + gene + cell * n_genes) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < kMarkLoadsPerThread; ++q) {
      const int x = ltid + q * 32 * kMarkLoaders;
      tile[buf][x / kMeanGenes][x % kMeanGenes] = __dadd_rn(v[q], 1.0);
    }
    if (ltid < kMeanCells) {
      const long long cell = t * kMeanCells + ltid;
      lab[buf][ltid] = cell < n_cells ? __ldg(cluster + cell) : -1;
    }
  };
  double s_in = 0.0, s_out = 0.0;
  if (warp >= kMarkClusters) load_tile(0, 0, tid - 32 * kMarkClusters);
  __syncthreads();
  for (long long t = 0; t < ntiles; ++t) {
    const int buf = (int)(t & 1);
    if (warp >= kMarkClusters) {
      if (t + 1 < ntiles) load_tile(t + 1, buf ^ 1, tid - 32 * kMarkClusters);
    } else if (c < n_clusters) {
      const int n_here = (int)(n_cells - t * kMeanCells < kMeanCells ? n_cells - t * kMeanCells : kMeanCells);
#pragma unroll 8
      for (int x = 0; x < n_here; ++x) {
        const double v1 = tile[buf][x][lane];
        if (lab[buf][x] == c) s_in = __dadd_rn(s_in, v1);
        else s_out = __dadd_rn(s_out, v1);
      }
    }
    __syncthreads();
  }
  if (warp < kMarkClusters && c < n_clusters && g0 + lane < n_genes) {
    const long long nc = cluster_size[c];
    out_ratio[(size_t)c * n_genes + g0 + lane] =
        __ddiv_rn(__ddiv_rn(s_in, (double)nc), __ddiv_rn(s_out, (double)(n_cells - nc)));
  }
}

// ---------------------------------------------------------------------------
// Sparse input: a genes x cells matrix in compressed-column form (R's dgCMatrix: colptr = p, row = i,
// x), turned gene-major on the device, then the two markers kernels read only the stored values.
// ---------------------------------------------------------------------------
constexpr unsigned kFlagCscRow = 1u;  // a row id outside [0, n_genes), or row ids not strictly increasing in a column

// Transpose, step 1 (warp per column): checks every row id before anything indexes with it, and writes
// the radix-sort input key = gene, payload = entry index, the entry's cell, and the per-gene counts.
// A bad entry raises kFlagCscRow and gets key 0 (the sort stays in bounds; the call then fails).
__global__ void __launch_bounds__(256)
wmu_csc_keys_kernel(const int* __restrict__ colptr, const int* __restrict__ row, long long n_cells, long long n_genes,
                    unsigned* __restrict__ col_of, unsigned long long* __restrict__ keys, unsigned* __restrict__ vals,
                    int* __restrict__ gene_cnt, unsigned* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  bool bad = false;
  for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < n_cells; c += nwarps) {
    const long long lo = colptr[c], hi = colptr[c + 1];
    for (long long e = lo + lane; e < hi; e += 32) {
      const int r = row[e];
      col_of[e] = (unsigned)c;
      vals[e] = (unsigned)e;
      if (r >= 0 && r < n_genes && (e == lo || row[e - 1] < r)) {
        keys[e] = (unsigned long long)r;
        atomicAdd(gene_cnt + r, 1);
      } else {
        keys[e] = 0;
        bad = true;
      }
    }
  }
  if (bad) atomicOr(flags, kFlagCscRow);
}

// Transpose, step 3 (after the stable sort by gene): sorted position q holds entry vals[q]; the entries of a
// gene keep their column order, so its cells are ascending.
__global__ void __launch_bounds__(256)
wmu_csc_gather_kernel(const unsigned* __restrict__ vals, const unsigned* __restrict__ col_of,
                      const double* __restrict__ x, long long nnz, unsigned* __restrict__ ent_cell,
                      double* __restrict__ ent_x) {
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nnz; q += (long long)gridDim.x * blockDim.x) {
    const unsigned e = vals[q];
    ent_cell[q] = col_of[e];
    ent_x[q] = x[e];
  }
}

// s + 1.0 + 1.0 + ... (m additions, each rounded), replayed in O(binades) steps.  While ulp(s) <= 1, adding
// an integer is exact as long as the result stays within s's binade or reaches its upper end 2^(e+1)
// (s >= 0), or does not pass 0 (s < 0): those steps are taken in one addition.  The step that leaves that
// range is a real addition (where rounding happens).  Above 2^53, s + 1 rounds back to s after at most one
// step (ties to even), and the run stops there.  Bit-identical to the loop, sign of zero included.
__device__ __forceinline__ double wmu_ones_run(double s, long long m) {
  while (m > 0) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(s);
    const int ef = (int)((b >> 52) & 0x7ffu);
    long long t = 0;
    if (ef <= 1023 + 52) {  // ulp(s) <= 1
      t = (b >> 63) ? (long long)(-s)
                    : (long long)__dadd_rn(__longlong_as_double((long long)((unsigned long long)(ef + 1) << 52)), -s);
      if (t > m) t = m;
    }
    if (t > 0) {
      s = __dadd_rn(s, (double)t);
      m -= t;
      continue;
    }
    const double n = __dadd_rn(s, 1.0);
    --m;
    if (n == s || n != n) break;  // a fixed point (or NaN): every further step gives the same
    s = n;
  }
  return s;
}

// Fold-change means from the gene-major sparse matrix: for each (gene, cluster c) the same two sequential
// chains as wmu_markers_means_kernel -- sum(v + 1) over c's cells and over all other cells, in cell order --
// walking only the gene's stored values.  The zeros between two stored values of a chain are a run of
// additions of 1.0, replayed by wmu_ones_run.  Run lengths: in-chain, the difference of the cells' ranks
// inside c (crank[cell], the cell's rank inside its own cluster); out-chain, the difference of the cells'
// positions among the non-c cells, cell - #{c cells below it}, with the count found in c's ascending cell
// list (members[cptr[c] ..]) by a galloping search that only moves forward.
// Thread = cluster blockIdx.y * blockDim.x + threadIdx.x of gene blockIdx.x.
// out_ratio[c * n_genes + g] = avg_in / avg_out.
__global__ void __launch_bounds__(128)
wmu_markers_csr_means_kernel(const double* __restrict__ ent_x, const unsigned* __restrict__ ent_cell,
                             const long long* __restrict__ gene_ptr, long long n_genes, long long n_cells,
                             const int* __restrict__ cluster, const int* __restrict__ crank,
                             const int* __restrict__ members, const long long* __restrict__ cptr, int n_clusters,
                             double* __restrict__ out_ratio) {
  const long long g = blockIdx.x;
  const int c = (int)(blockIdx.y * blockDim.x + threadIdx.x);
  if (c >= n_clusters) return;
  const long long lo = gene_ptr[g], hi = gene_ptr[g + 1];
  const int* const L = members + cptr[c];
  const long long nc = cptr[c + 1] - cptr[c];
  double s_in = 0.0, s_out = 0.0;
  long long in_next = 0, out_next = 0;  // chain positions of the next value of each chain
  long long p = 0;                      // c cells below the current cell: L[0, p) < cell
  long long next_c = nc > 0 ? L[0] : n_cells;  // L[p]
  for (long long q = lo; q < hi; ++q) {
    const long long cell = __ldg(ent_cell + q);
    const double v1 = __dadd_rn(__ldg(ent_x + q), 1.0);
    if (__ldg(cluster + cell) == c) {
      const long long r = __ldg(crank + cell);
      s_in = __dadd_rn(wmu_ones_run(s_in, r - in_next), v1);
      in_next = r + 1;
      p = r + 1;
      next_c = p < nc ? __ldg(L + p) : n_cells;
    } else {
      if (next_c < cell) {  // first index >= p whose cell is above `cell`
        long long a = p + 1, step = 1;  // L[0, a) < cell
        while (a + step <= nc && __ldg(L + a + step - 1) < cell) {
          a += step;
          step <<= 1;
        }
        long long b = a + step - 1 < nc ? a + step - 1 : nc;
        while (a < b) {
          const long long mid = (a + b) >> 1;
          if (__ldg(L + mid) < cell) a = mid + 1;
          else b = mid;
        }
        p = a;
        next_c = p < nc ? __ldg(L + p) : n_cells;
      }
      const long long r = cell - p;
      s_out = __dadd_rn(wmu_ones_run(s_out, r - out_next), v1);
      out_next = r + 1;
    }
  }
  s_in = wmu_ones_run(s_in, nc - in_next);
  s_out = wmu_ones_run(s_out, (n_cells - nc) - out_next);
  out_ratio[(size_t)c * n_genes + g] = __ddiv_rn(__ddiv_rn(s_in, (double)nc), __ddiv_rn(s_out, (double)(n_cells - nc)));
}

}  // namespace gficf
