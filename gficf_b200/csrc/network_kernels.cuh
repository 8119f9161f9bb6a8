// network_kernels.cuh -- the data-parallel pieces of the community detection that consumes the
// Jaccard graph (SURVEY section 8f, "next" row 3), on the device next to the graph they read.
//
// What they replace in the reference (src/ModularityOptimizer.cpp, single-threaded C++):
//   matrixToNetwork              :761-806  lower-triangle edge list -> symmetric CSR network
//   Network::Network             :169-188  node weights = total edge weight per node (:278-284)
//   Network::getTotalEdgeWeight  :268-270
//   VOSClusteringTechnique::calcQualityFunction  :462-482
//   Clustering::getNodesPerCluster               :106-118
//   Network::createReducedNetwork                :322-373
// The sequential, RNG-ordered local moving loop (:484-583) is NOT here: it stays on the host and
// calls these between its passes (INTEGRATION.md section 8).
//
// Parity with the reference, by construction:
//   * all structure (firstNeighborIndex, neighbor order, nodes per cluster, the neighbour order
//     of the reduced network = order of first appearance in the reference's traversal) is integer
//     work and identical;
//   * every floating-point sum the reference forms over one node's, cluster's or cluster pair's
//     list is formed here in the same order from the same start value (warp_ordered_sum: a warp
//     fetches the list in parallel and replays the additions in list order): node weights (the node's
//     neighbour list), cluster weights / reduced node weights (the cluster's nodes ascending),
//     reduced edge weights (the cross edges of one cluster pair in traversal order) -- bit-identical;
//   * the sums the reference forms sequentially over the WHOLE edge list (total edge weight, the
//     intra-cluster weight inside calcQualityFunction, the self-link total of the reduced network)
//     are replayed exactly as well -- see "The reference's whole-graph sums, bit for bit" below --
//     and the subtraction chain over the clusters in calcQualityFunction is done by one thread.
//   Every double these kernels produce is the reference's double.
//
// Ordering primitive: a stable least-significant-digit radix sort over 64-bit keys with a 32-bit
// payload (8-bit digits; per-tile digit histograms, one exclusive scan over (digit, tile), ranked
// scatter).  Stability is what turns "group by key" into "group by key, original order kept", which
// is exactly the order the reference's sequential loops visit things in.
//
// HBM-bound integer/byte work: thread-per-item kernels with coalesced streams, no tensor cores.
// With GFICF_CUDA_EMU defined this header compiles as plain C++ (see scan_kernels.cuh).
#pragma once
#include "scan_kernels.cuh"

namespace gficf {

constexpr unsigned kFlagNetWeight = 32u;  // an edge weight that is not > 0 (the reference's "weight == 0
                                          // means not seen yet" bookkeeping, :342, would behave differently)
constexpr unsigned kFlagNetRange = 64u;   // a row / cluster id outside its range, or a non-lower entry

// ---------------------------------------------------------------------------------------------
// stable LSD radix sort, one 8-bit digit per pass
// ---------------------------------------------------------------------------------------------
constexpr int kRadixThreads = 256;  // == number of digit values: thread t owns digit t in the prefix steps
constexpr int kRadixWarps = kRadixThreads / 32;
constexpr int kRadixRounds = 8;
constexpr int kRadixTile = kRadixThreads * kRadixRounds;

// hist[digit * n_tiles + tile] = keys of the tile with that digit
__global__ void __launch_bounds__(kRadixThreads)
radix_hist_kernel(const unsigned long long* __restrict__ keys, long long n, int shift, long long n_tiles,
                  int* __restrict__ hist) {
  __shared__ unsigned h[256];
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    h[threadIdx.x] = 0;
    __syncthreads();
    const long long base = tile * kRadixTile;
    for (int r = 0; r < kRadixRounds; ++r) {
      const long long i = base + (long long)r * kRadixThreads + threadIdx.x;
      if (i < n) atomicAdd(&h[(unsigned)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(long long)threadIdx.x * n_tiles + tile] = (int)h[threadIdx.x];
    __syncthreads();
  }
}

// offsets = exclusive scan of hist: where the tile's keys with a digit start in the output.
// Inside a tile the keys are ranked in order: rounds in sequence, warps in sequence inside a
// round, lanes in sequence inside a warp (match.any finds the lanes with the same digit).
__global__ void __launch_bounds__(kRadixThreads)
radix_scatter_kernel(const unsigned long long* __restrict__ keys_in, const unsigned* __restrict__ vals_in,
                     unsigned long long* __restrict__ keys_out, unsigned* __restrict__ vals_out, long long n,
                     int shift, long long n_tiles, const long long* __restrict__ offsets) {
  __shared__ long long base[256];
  __shared__ unsigned short wcnt[kRadixWarps][256];
  __shared__ unsigned round_total[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    base[tid] = offsets[(long long)tid * n_tiles + tile];
    for (int r = 0; r < kRadixRounds; ++r) {
      for (int x = tid; x < kRadixWarps * 256; x += kRadixThreads) (&wcnt[0][0])[x] = 0;
      __syncthreads();
      const long long i = tile * kRadixTile + (long long)r * kRadixThreads + tid;
      const bool valid = i < n;
      unsigned long long key = 0;
      unsigned val = 0, d = 256u + (unsigned)lane;  // lanes past the end: a digit nobody shares
      if (valid) {
        key = keys_in[i];
        val = vals_in[i];
        d = (unsigned)(key >> shift) & 255u;
      }
      const unsigned peers = __match_any_sync(kFull, d);
      const unsigned rank_in_warp = (unsigned)__popc(peers & lt_mask);
      if (valid && rank_in_warp == 0) wcnt[warp][d] = (unsigned short)__popc(peers);
      __syncthreads();
      {  // exclusive prefix over the warps, per digit (thread tid owns digit tid)
        unsigned acc = 0;
        for (int w = 0; w < kRadixWarps; ++w) {
          const unsigned c = wcnt[w][tid];
          wcnt[w][tid] = (unsigned short)acc;
          acc += c;
        }
        round_total[tid] = acc;
      }
      __syncthreads();
      if (valid) {
        const long long pos = base[d] + wcnt[warp][d] + rank_in_warp;
        keys_out[pos] = key;
        vals_out[pos] = val;
      }
      __syncthreads();
      base[tid] += round_total[tid];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// The reference's whole-graph sums, bit for bit.  std::accumulate over 10^8 doubles is a chain
// s <- RN(s + x[t]); re-associating it changes the bits (with the few distinct Jaccard weights the
// sequential sum drifts ~n * 2^-53 away from the true sum, 4e-10 at 5e7 terms -- measured).  But
// the chain has structure: while s stays inside one binade [2^e, 2^(e+1)) its spacing is
// ulp = 2^(e-52), s = S * ulp with an integer S, and for x = W * ulp + r (0 <= r < ulp)
//     RN(s + x) = (S + W + c) * ulp,   c = [r > ulp/2], or on a tie (r == ulp/2) the choice that
//                                          makes S + W + c even,
// as long as S + W + c <= 2^53.  So inside a binade every element is an INTEGER increment that
// depends on S only through its parity (ties): a pair (d_even, d_odd).  Such pairs compose
// associatively, hence a block of elements collapses to one pair, blocks are combined in order, and
// the increments are non-negative, so "the first element that leaves the binade" is found by
// walking the block pairs.  That one element is added with a real floating-point add, the binade
// changes, and the walk goes on.  The doubles produced are exactly the sequential chain's.
//   domain: x[t] >= 0 (0 = skipped element), finite; anything else raises kFlagNetWeight.
// s == 0 needs no case of its own: it is S = 0 in binade e = -1022, where a zero element is the
// identity pair and every non-zero element (shift <= 0) saturates, so the walk below finds the first
// non-zero element and its real addition gives 0 + x = x.  A run of leading zeros (masked sums whose
// first entries are all masked out) is thus consumed a window at a time like any other stretch.
// A window of up to 1024 blocks x 4096 elements is processed per step; the window grows while no
// binade boundary is met.  State lives on the device; the host only reads the position back
// every few dozen steps.
// ---------------------------------------------------------------------------------------------
struct SeqFn {
  unsigned long long d0, d1;  // increment of S when S is even / odd; saturates at kSeqClamp
};
struct SeqState {
  long long t0;          // next element
  unsigned long long S;  // s = S * 2^(e-52); S == 0 <=> s == 0
  int e;
  int win_blocks;        // blocks in the next window
  double value;          // s as a double (kept for the caller)
};
constexpr unsigned long long kSeqClamp = 1ull << 54;
constexpr unsigned long long kSeqTop = 1ull << 53;
constexpr int kSeqThreads = 256;
constexpr int kSeqPerThread = 16;
constexpr int kSeqBlock = kSeqThreads * kSeqPerThread;  // 4096 elements
constexpr int kSeqMaxBlocks = 1024;

__device__ __forceinline__ void seq_split(double v, unsigned long long* S, int* e) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  const int ef = (int)((b >> 52) & 0x7ffu);
  const unsigned long long m = b & ((1ull << 52) - 1ull);
  if (ef == 0) {
    *S = m;
    *e = -1022;
  } else {
    *S = m | (1ull << 52);
    *e = ef - 1023;
  }
}

__device__ __forceinline__ double seq_value(unsigned long long S, int e) {
  if (S == 0) return 0.0;
  if (S >> 52) return __longlong_as_double((long long)(((unsigned long long)(e + 1023) << 52) | (S & ((1ull << 52) - 1ull))));
  return __longlong_as_double((long long)S);  // subnormal: e == -1022, no implicit bit
}

// the increment pair of element x while s sits in binade e
__device__ __forceinline__ SeqFn seq_fn(double x, int e, bool* bad) {
  SeqFn f;
  f.d0 = f.d1 = 0;
  if (x == 0.0) return f;
  if (!(x > 0.0) || x > 1.7976931348623157e308) {
    *bad = true;
    return f;
  }
  unsigned long long M;
  int ex;
  seq_split(x, &M, &ex);
  const int shift = e - ex;  // x = M * 2^(ex-52), ulp = 2^(e-52): x / ulp = M / 2^shift
  if (shift <= 0) {
    f.d0 = f.d1 = kSeqClamp;  // x alone reaches the top of the binade
  } else if (shift <= 53) {
    const unsigned long long W = M >> shift;
    const unsigned long long rem = M & ((1ull << shift) - 1ull);
    const unsigned long long half = 1ull << (shift - 1);
    if (rem == half) {
      f.d0 = W + (W & 1ull);
      f.d1 = W + ((W & 1ull) ^ 1ull);
    } else {
      f.d0 = f.d1 = W + (rem > half ? 1ull : 0ull);
    }
  }  // shift >= 54: x is below half an ulp, s absorbs it
  return f;
}

__device__ __forceinline__ unsigned long long seq_apply(unsigned long long S, SeqFn f) {
  const unsigned long long r = S + ((S & 1ull) ? f.d1 : f.d0);
  return r < kSeqClamp ? r : kSeqClamp;
}

// f first, then g
__device__ __forceinline__ SeqFn seq_compose(SeqFn f, SeqFn g) {
  SeqFn r;
  r.d0 = f.d0 >= kSeqClamp ? kSeqClamp : seq_apply(f.d0, g);          // S even: S + d0 has the parity of d0
  r.d1 = f.d1 >= kSeqClamp ? kSeqClamp : seq_apply(f.d1 + 1ull, g) - 1ull;  // S odd: S + d1 has the parity of d1 + 1
  return r;
}

// the pair of elements [lo, lo + 16) (clipped at n), composed in order
__device__ __forceinline__ SeqFn seq_thread_fn(const double* __restrict__ x, long long lo, long long n, int e,
                                               bool* bad) {
  SeqFn f;
  f.d0 = f.d1 = 0;
  for (int q = 0; q < kSeqPerThread; ++q) {
    const long long i = lo + q;
    if (i < n) f = seq_compose(f, seq_fn(x[i], e, bad));
  }
  return f;
}

__global__ void __launch_bounds__(32)
seq_init_kernel(SeqState* __restrict__ st, double s0) {
  if (threadIdx.x == 0) {
    st->t0 = 0;
    seq_split(s0, &st->S, &st->e);
    st->win_blocks = 1;
    st->value = s0;
  }
}

// block_fn[b] = composition of the elements of block b of the current window
__global__ void __launch_bounds__(kSeqThreads)
seq_blocks_kernel(const double* __restrict__ x, long long n, const SeqState* __restrict__ st,
                  SeqFn* __restrict__ block_fn, unsigned* __restrict__ flags) {
  __shared__ SeqFn s_warp[kSeqThreads / 32];
  const long long t0 = st->t0;
  if (t0 >= n) return;  // finished
  const int nb = st->win_blocks, e = st->e;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool bad = false;
  for (int b = blockIdx.x; b < nb; b += gridDim.x) {
    const long long lo = t0 + (long long)b * kSeqBlock + (long long)threadIdx.x * kSeqPerThread;
    SeqFn f = seq_thread_fn(x, lo, n, e, &bad);
    for (int off = 1; off < 32; off <<= 1) {  // ordered tree: lane i absorbs lane i + off
      SeqFn o;
      o.d0 = __shfl_down_sync(kFull, f.d0, off);
      o.d1 = __shfl_down_sync(kFull, f.d1, off);
      if ((lane & (2 * off - 1)) == 0) f = seq_compose(f, o);
    }
    if (lane == 0) s_warp[warp] = f;
    __syncthreads();
    if (threadIdx.x == 0) {
      SeqFn a = s_warp[0];
      for (int w = 1; w < kSeqThreads / 32; ++w) a = seq_compose(a, s_warp[w]);
      block_fn[b] = a;
    }
    __syncthreads();
  }
  if (bad) atomicOr(flags, kFlagNetWeight);
}

// one CTA: walks the block pairs of the window; either the whole window stays inside the binade
// (s moves to its end) or the first block / thread / element that leaves it is located, that
// element is added in floating point and the state continues behind it.  When the last element
// is consumed, out[0] = s * scale.
__global__ void __launch_bounds__(kSeqThreads)
seq_advance_kernel(const double* __restrict__ x, long long n, SeqState* __restrict__ st,
                   const SeqFn* __restrict__ block_fn, double scale, double* __restrict__ out,
                   unsigned* __restrict__ flags) {
  __shared__ SeqFn s_fn[kSeqMaxBlocks];
  __shared__ int s_bstar;
  __shared__ unsigned long long s_S;
  // every thread takes its copy of the state before thread 0 may change it
  const long long t0 = st->t0;
  const unsigned long long S0 = st->S;
  const int e = st->e;
  const int nb = st->win_blocks;
  __syncthreads();
  if (t0 >= n) {
    if (threadIdx.x == 0 && n == 0) out[0] = st->value * scale;
    return;
  }
  bool bad = false;
  for (int b = threadIdx.x; b < nb; b += kSeqThreads) s_fn[b] = block_fn[b];
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long S = S0;
    int bstar = -1;
    for (int b = 0; b < nb; ++b) {
      const unsigned long long nS = seq_apply(S, s_fn[b]);
      if (nS >= kSeqTop) {
        bstar = b;
        break;
      }
      S = nS;
    }
    s_bstar = bstar;
    s_S = S;  // s at the start of block bstar, or at the end of the window
  }
  __syncthreads();
  const int bstar = s_bstar;
  if (bstar < 0) {
    if (threadIdx.x == 0) {
      long long end = t0 + (long long)nb * kSeqBlock;
      if (end > n) end = n;
      st->S = s_S;
      st->value = seq_value(s_S, e);
      st->t0 = end;
      st->win_blocks = 2 * nb < kSeqMaxBlocks ? 2 * nb : kSeqMaxBlocks;
      if (end >= n) out[0] = st->value * scale;
    }
    return;
  }
  // the crossing is inside block bstar: per-thread pairs, then thread 0 walks threads and elements
  const long long blo = t0 + (long long)bstar * kSeqBlock;
  __syncthreads();
  s_fn[threadIdx.x] = seq_thread_fn(x, blo + (long long)threadIdx.x * kSeqPerThread, n, e, &bad);
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long S = s_S;
    int j = 0;
    for (; j < kSeqThreads; ++j) {
      const unsigned long long nS = seq_apply(S, s_fn[j]);
      if (nS >= kSeqTop) break;
      S = nS;
    }
    long long i = blo + (long long)j * kSeqPerThread;
    for (; i < n - 1; ++i) {  // the crossing element exists: the block's pair said so (n - 1 bounds the walk regardless)
      const unsigned long long nS = seq_apply(S, seq_fn(x[i], e, &bad));
      if (nS >= kSeqTop) break;
      S = nS;
    }
    if (i >= n) i = n - 1;  // unreachable with consistent pairs; keeps the read inside the array
    const double s_new = __dadd_rn(seq_value(S, e), x[i]);  // the one real addition of this step
    seq_split(s_new, &st->S, &st->e);
    st->value = s_new;
    st->t0 = i + 1;
    // the next binade is twice as wide: about twice as many elements fit
    long long want = 2 * ((i + 1 - t0) / kSeqBlock + 1);
    st->win_blocks = want < kSeqMaxBlocks ? (int)want : kSeqMaxBlocks;
    if (i + 1 >= n) out[0] = s_new * scale;
  }
  if (bad) atomicOr(flags, kFlagNetWeight);
}

// ---------------------------------------------------------------------------------------------
// Sums in the reference's order.  The reference adds a list front to back into one double; a
// single GPU thread doing that is a chain of dependent, scattered loads.  Here a WARP owns the
// list: its lanes fetch 32 consecutive elements at once (coalesced / independent gathers), then
// every lane replays the same 32 additions in list order from shuffled values -- the additions
// stay sequential (that is what makes the result the reference's), the memory traffic does not.
// fetch(i, &v) returns whether element i takes part (and its value in v).  All 32 lanes call.
// ---------------------------------------------------------------------------------------------
template <class Fetch>
__device__ __forceinline__ double warp_ordered_sum(long long lo, long long hi, int lane, Fetch fetch) {
  double s = 0.0;
  for (long long base = lo; base < hi; base += 32) {
    const long long i = base + lane;
    double v = 0.0;
    bool take = false;
    if (i < hi) take = fetch(i, &v);
    const unsigned m = __ballot_sync(kFull, take);
    if (m == 0) continue;
    const int cnt = hi - base < 32 ? (int)(hi - base) : 32;
    for (int l = 0; l < cnt; ++l) {
      const double x = __shfl_sync(kFull, v, l);
      if ((m >> l) & 1u) s += x;
    }
  }
  return s;
}

// ---------------------------------------------------------------------------------------------
// matrixToNetwork (:761-806): lower-triangle CSC (column = node1 < row = node2, rows ascending
// inside a column -- what gficf_cuda_snn_lower_dev produces and RModularityOptimizer.cpp:67-83
// reads) -> symmetric CSR.  The reference appends, per edge in input order, node2 to node1's
// list and node1 to node2's: node v's list is therefore [columns c < v that hold row v, c
// ascending] followed by [the rows of column v, ascending] -- ascending neighbour ids.
// The first part is the transposed lower triangle: entries grouped by row with the column order
// kept = a stable sort of the entries by row.
// ---------------------------------------------------------------------------------------------

// one warp per column: column id of every entry, sort keys (row) / payload (entry), entries per row
__global__ void __launch_bounds__(256)
net_col_keys_kernel(const long long* __restrict__ colptr, const int* __restrict__ row, long long nv,
                    int* __restrict__ col_of, unsigned long long* __restrict__ keys, unsigned* __restrict__ vals,
                    int* __restrict__ up_cnt, unsigned* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  bool bad = false;
  for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < nv; c += nwarps) {
    const long long lo = colptr[c], hi = colptr[c + 1];
    for (long long e = lo + lane; e < hi; e += 32) {
      const int r = row[e];
      col_of[e] = (int)c;
      vals[e] = (unsigned)e;
      if (r > c && r < nv) {
        keys[e] = (unsigned long long)r;
        atomicAdd(up_cnt + r, 1);
      } else {
        keys[e] = 0;
        bad = true;
      }
    }
  }
  if (bad) atomicOr(flags, kFlagNetRange);
}

// firstNeighborIndex[v] = entries of rows < v in the transposed part + entries of columns < v
__global__ void __launch_bounds__(256)
net_first_kernel(const long long* __restrict__ colptr, const long long* __restrict__ upptr, long long nv,
                 long long* __restrict__ first) {
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v <= nv;
       v += (long long)gridDim.x * blockDim.x)
    first[v] = colptr[v] + upptr[v];
}

// thread s handles sorted entry s (goes into the list of its ROW) and lower entry s (goes into
// the list of its COLUMN).  With first[v] = colptr[v] + upptr[v]:
//   transposed part of v starts at first[v]; sorted entry s is number s - upptr[v] in it -> colptr[v] + s
//   own part of c starts at first[c] + (upptr[c+1] - upptr[c]); entry s is number s - colptr[c] -> upptr[c+1] + s
__global__ void __launch_bounds__(256)
net_fill_kernel(const long long* __restrict__ colptr, const int* __restrict__ row, const double* __restrict__ w,
                const long long* __restrict__ upptr, const int* __restrict__ col_of,
                const unsigned long long* __restrict__ keys_sorted, const unsigned* __restrict__ vals_sorted,
                long long nnz, int* __restrict__ neighbor, double* __restrict__ edge_w) {
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < nnz;
       s += (long long)gridDim.x * blockDim.x) {
    const long long v = (long long)keys_sorted[s];
    const unsigned e = vals_sorted[s];
    const long long p1 = colptr[v] + s;
    neighbor[p1] = col_of[e];
    edge_w[p1] = w[e];
    const int c = col_of[s];
    const long long p2 = upptr[c + 1] + s;
    neighbor[p2] = row[s];
    edge_w[p2] = w[s];
  }
}

// nodeWeight[v] = std::accumulate over v's edge weights from 0.0, in list order (:272-284).  Warp per node.
__global__ void __launch_bounds__(256)
net_node_weight_kernel(const long long* __restrict__ first, const double* __restrict__ edge_w, long long nv,
                       double* __restrict__ node_w, unsigned* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  bool bad = false;
  for (long long v = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); v < nv; v += nwarps) {
    const double s = warp_ordered_sum(first[v], first[v + 1], lane, [&](long long m, double* x) {
      *x = edge_w[m];
      bad |= !(*x > 0.0);
      return true;
    });
    if (lane == 0) node_w[v] = s;
  }
  if (bad) atomicOr(flags, kFlagNetWeight);
}

// ---------------------------------------------------------------------------------------------
// clustering helpers: nodes per cluster (ascending node ids: a stable sort of the nodes by cluster)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
net_cluster_keys_kernel(const int* __restrict__ cluster, long long n_nodes, int n_clusters,
                        unsigned long long* __restrict__ keys, unsigned* __restrict__ vals,
                        int* __restrict__ ccnt, unsigned* __restrict__ flags) {
  bool bad = false;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < n_nodes;
       v += (long long)gridDim.x * blockDim.x) {
    const int c = cluster[v];
    vals[v] = (unsigned)v;
    if (c >= 0 && c < n_clusters) {
      keys[v] = (unsigned long long)c;
      atomicAdd(ccnt + c, 1);
    } else {
      keys[v] = 0;
      bad = true;
    }
  }
  if (bad) atomicOr(flags, kFlagNetRange);
}

// clusterWeight[c] (calcQualityFunction :474-476) == reducedNetwork.nodeWeight[c] (:345): the node
// weights of the cluster's nodes, ascending node id, added from 0.0.  Warp per cluster.
// term[c] = (cw * cw) * resolution, the amount :478 subtracts (term may be null).
__global__ void __launch_bounds__(256)
net_cluster_weight_kernel(const long long* __restrict__ cptr, const unsigned* __restrict__ nodes_sorted,
                          const double* __restrict__ node_w, int n_clusters, double resolution,
                          double* __restrict__ cluster_w, double* __restrict__ term) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < n_clusters; c += nwarps) {
    const double s = warp_ordered_sum(cptr[c], cptr[c + 1], lane, [&](long long t, double* x) {
      *x = node_w[nodes_sorted[t]];
      return true;
    });
    if (lane == 0) {
      cluster_w[c] = s;
      if (term) term[c] = __dmul_rn(__dmul_rn(s, s), resolution);
    }
  }
}

// y[m] = edge weight m if both ends share a cluster, else 0 (a skipped element of the sequential sum
// :465-469).  Warp per node, CSR order.
__global__ void __launch_bounds__(256)
net_intra_mask_kernel(const long long* __restrict__ first, const int* __restrict__ neighbor,
                      const double* __restrict__ edge_w, const int* __restrict__ cluster, long long n_nodes,
                      double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long v = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); v < n_nodes; v += nwarps) {
    const int c = cluster[v];
    for (long long m = first[v] + lane; m < first[v + 1]; m += 32)
      y[m] = cluster[neighbor[m]] == c ? edge_w[m] : 0.0;
  }
}

// :470-481 in the reference's order: q = intra; q += selfLinks; q -= term[c] for c = 0, 1, ...;
// q /= 2 * totalEdgeWeight + selfLinks.  One thread: the subtractions are a chain over the clusters.
__global__ void __launch_bounds__(32)
net_quality_final_kernel(const double* __restrict__ intra_sum, const double* __restrict__ term, int n_clusters,
                         const double* __restrict__ total_edge_w, double self_links, double* __restrict__ q) {
  if (threadIdx.x == 0) {
    double v = __dadd_rn(intra_sum[0], self_links);
    for (int c = 0; c < n_clusters; ++c) v = __dadd_rn(v, -term[c]);
    q[0] = __ddiv_rn(v, __dadd_rn(__dmul_rn(2.0, total_edge_w[0]), self_links));
  }
}

// warp per position t of the cluster-sorted node list: cross edges of the node, and its degree
__global__ void __launch_bounds__(256)
rn_count_kernel(const long long* __restrict__ first, const int* __restrict__ neighbor,
                const int* __restrict__ cluster, const unsigned* __restrict__ nodes_sorted, long long n_nodes,
                int* __restrict__ xcnt, int* __restrict__ deg_t) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_nodes; t += nwarps) {
    const unsigned l = nodes_sorted[t];
    const int i = cluster[l];
    const long long lo = first[l], hi = first[l + 1];
    int cross = 0;
    for (long long base = lo; base < hi; base += 32) {
      const long long m = base + lane;
      cross += __popc(__ballot_sync(kFull, m < hi && cluster[neighbor[m]] != i));
    }
    if (lane == 0) {
      xcnt[t] = cross;
      deg_t[t] = (int)(hi - lo);
    }
  }
}

// y[gbase[t] + j] = weight of the j-th edge of node t (traversal order) if it stays inside the
// cluster, else 0: the sequence :351 adds to totalEdgeWeightSelfLinks
__global__ void __launch_bounds__(256)
rn_intra_mask_kernel(const long long* __restrict__ first, const int* __restrict__ neighbor,
                     const double* __restrict__ edge_w, const int* __restrict__ cluster,
                     const unsigned* __restrict__ nodes_sorted, const long long* __restrict__ gbase,
                     long long n_nodes, double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_nodes; t += nwarps) {
    const unsigned l = nodes_sorted[t];
    const int i = cluster[l];
    const long long lo = first[l], g = gbase[t];
    for (long long m = lo + lane; m < first[l + 1]; m += 32)
      y[g + (m - lo)] = cluster[neighbor[m]] == i ? edge_w[m] : 0.0;
  }
}

// warp per position t: the node's cross edges, compacted in list order behind xbase[t]
__global__ void __launch_bounds__(256)
rn_emit_kernel(const long long* __restrict__ first, const int* __restrict__ neighbor,
               const int* __restrict__ cluster, const unsigned* __restrict__ nodes_sorted,
               const long long* __restrict__ xbase, long long n_nodes, int cluster_bits,
               unsigned long long* __restrict__ keys, unsigned* __restrict__ vals, unsigned* __restrict__ edge_of) {
  const int lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_nodes; t += nwarps) {
    const unsigned l = nodes_sorted[t];
    const int i = cluster[l];
    const long long lo = first[l], hi = first[l + 1];
    long long p = xbase[t];
    for (long long base = lo; base < hi; base += 32) {
      const long long m = base + lane;
      int n = i;
      if (m < hi) n = cluster[neighbor[m]];
      const unsigned mask = __ballot_sync(kFull, n != i);
      if (n != i) {
        const long long q = p + __popc(mask & lt_mask);
        keys[q] = ((unsigned long long)(unsigned)i << cluster_bits) | (unsigned long long)(unsigned)n;
        vals[q] = (unsigned)q;
        edge_of[q] = (unsigned)m;
      }
      p += __popc(mask);
    }
  }
}

__global__ void __launch_bounds__(256)
rn_heads_kernel(const unsigned long long* __restrict__ keys_sorted, long long n_cross, int* __restrict__ head) {
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < n_cross;
       s += (long long)gridDim.x * blockDim.x)
    head[s] = (s == 0 || keys_sorted[s] != keys_sorted[s - 1]) ? 1 : 0;
}

// seg_start[q] = first sorted position of cluster pair q
__global__ void __launch_bounds__(256)
rn_seg_start_kernel(const int* __restrict__ head, const long long* __restrict__ seg_id, long long n_cross,
                    unsigned* __restrict__ seg_start) {
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < n_cross;
       s += (long long)gridDim.x * blockDim.x)
    if (head[s]) seg_start[seg_id[s]] = (unsigned)s;
}

// warp per cluster pair (segment of equal keys): weights added in traversal order
__global__ void __launch_bounds__(256)
rn_segments_kernel(const unsigned long long* __restrict__ keys_sorted, const unsigned* __restrict__ vals_sorted,
                   const unsigned* __restrict__ seg_start, const unsigned* __restrict__ edge_of,
                   const double* __restrict__ edge_w, long long n_cross, long long n_seg, int cluster_bits,
                   unsigned long long* __restrict__ seg_key, double* __restrict__ seg_w,
                   unsigned long long* __restrict__ keys2, unsigned* __restrict__ vals2, int* __restrict__ rcnt) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < n_seg; q += nwarps) {
    const long long lo = seg_start[q];
    const long long hi = q + 1 < n_seg ? (long long)seg_start[q + 1] : n_cross;
    const double sum = warp_ordered_sum(lo, hi, lane, [&](long long j, double* x) {
      *x = edge_w[edge_of[vals_sorted[j]]];
      return true;
    });
    if (lane == 0) {
      const unsigned long long key = keys_sorted[lo];
      seg_key[q] = key;
      seg_w[q] = sum;
      keys2[q] = (unsigned long long)vals_sorted[lo];  // first appearance in the traversal
      vals2[q] = (unsigned)q;
      atomicAdd(rcnt + (int)(key >> cluster_bits), 1);
    }
  }
}

__global__ void __launch_bounds__(256)
rn_write_kernel(const unsigned* __restrict__ vals2_sorted, const unsigned long long* __restrict__ seg_key,
                const double* __restrict__ seg_w, long long n_seg, int cluster_bits, int* __restrict__ r_neighbor,
                double* __restrict__ r_edge_w) {
  const unsigned long long mask = (1ull << cluster_bits) - 1ull;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_seg;
       j += (long long)gridDim.x * blockDim.x) {
    const unsigned q = vals2_sorted[j];
    r_neighbor[j] = (int)(seg_key[q] & mask);
    r_edge_w[j] = seg_w[q];
  }
}

}  // namespace gficf
