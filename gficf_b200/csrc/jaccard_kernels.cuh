// jaccard_kernels.cuh -- sm_100a device kernels of the Phenograph Jaccard path.
//
// What they replace (reference = dibbelab/gficf):
//   layout_colmajor_kernel the per-edge strided row copies out of the column-major
//                          double matrix, src/rcpp_parallel_jaccard_coeff.cpp:30-36
//   jaccard_small_k_kernel JCoefficient::operator() for k<=32,
//   jaccard_wide_k_kernel  and for 32<k<=128, rcpp_parallel_jaccard_coeff.cpp:24-55
//   jaccard_exact_kernel   the same for any k and rows with repeated ids
//                          (std::set_intersection multiset semantics :41-46, or
//                          Rcpp::intersect unique-set semantics, jaccard_coeff.cpp:33)
//   expand_* kernels       the conditional (from,to,w) stores :48-52 and the
//                          compacting stores of jaccard_coeff.cpp:34-39
//
// Design (HBM-bound sparse gather; no tensor cores -- there is no dense
// contraction here):
//   * the index matrix lives in HBM as int32, row-major, 0-based, rows padded to a
//     32-byte sector multiple, so a neighbour row is fetched with 16-byte vector
//     loads (one LDG.128 per lane brings 4 ids; k=30 -> 8 lanes per row, 4 rows
//     per warp instruction);
//   * one warp owns row i: N(i) is put into a per-warp COLLISION-FREE
//     multiplicative hash table in shared memory (a multiplier is searched per
//     row), so membership of each gathered id is one IMAD+SHF+LDS+compare;
//   * all gathers of a row are issued before the first probe (up to 8 LDG.128
//     in flight per lane), the next row's own ids are prefetched;
//   * per-edge counts are packed 4 per register and reduced across the lanes of
//     an edge group by xor-shuffles; lane e ends with u(i, e) and writes
//     from/to/w with coalesced streaming stores (st.global.cs) so that the
//     output does not evict the index matrix from L2.
#pragma once
#include "jaccard_weight.cuh"
#include "scan_kernels.cuh"

// tuning knobs (overridable with -D for A/B runs; defaults are the measured best)
#ifndef GFICF_SMALL_LOG_TS32
#define GFICF_SMALL_LOG_TS32 9   // hash-table slots per warp for 16 < k <= 32: 2^9
#endif
#ifndef GFICF_SMALL_MATCH
#define GFICF_SMALL_MATCH 0      // k<=32: find hash collisions with match.any (1; measured slower: 3.12 vs 3.07 ms at k=30, 1.95 vs 1.55 ms at k=15) or through the table (0)
#endif
#ifndef GFICF_SMALL_WARPS
#define GFICF_SMALL_WARPS 7      // warps (rows in flight) per CTA of the k<=32 kernel
#endif
#ifndef GFICF_WIDE_MINB
#define GFICF_WIDE_MINB 8        // resident CTAs (warp-groups) per SM the 32<k<=128 kernel is compiled for
#endif
#ifndef GFICF_SMALL_MINB
#define GFICF_SMALL_MINB 4       // resident CTAs per SM the k<=32 kernel is compiled for
#endif
#ifndef GFICF_MAX_TRIES
#define GFICF_MAX_TRIES 256      // multipliers the k<=128 kernels try before raising kFlagHashFail (1: tests of that path)
#endif
#include <stdint.h>

namespace gficf {

constexpr int kPadId = -2;              // pad entries of an index row (never equals an id or kEmpty)
constexpr unsigned kEmpty = 0xFFFFFFFFu;  // empty hash slot
constexpr unsigned kFlagBadId = 1u, kFlagDupId = 2u, kFlagHashFail = 4u;
constexpr int kMaxTries = GFICF_MAX_TRIES;
constexpr unsigned kMult0 = 0x9E3779B1u;  // odd; successive multipliers come from an LCG

__device__ __forceinline__ unsigned next_mult(unsigned m) { return (m * 0x2C1B3C6Du + 0x297A2D39u) | 1u; }

__device__ __forceinline__ int4 ldg16(const int* p) {
  return __ldg(reinterpret_cast<const int4*>(p));
}

// 16-byte piece of neighbour row t: base already points at this lane's column offset
__device__ __forceinline__ int4 ldg_row(const char* lane_base, unsigned t, unsigned row_bytes) {
  return __ldg(reinterpret_cast<const int4*>(lane_base + (unsigned long long)t * row_bytes));  // IMAD.WIDE.U32
}

// acc += INC when the table slot of x holds x: ISETP + predicated IADD, no select chain
template <unsigned INC>
__device__ __forceinline__ void add_if_eq(unsigned& acc, unsigned a, unsigned b) {
#ifdef GFICF_CUDA_EMU
  if (a == b) acc += INC;
#else
  asm("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, %1, %2;\n\t@p add.u32 %0, %0, %3;\n\t}"
      : "+r"(acc) : "r"(a), "r"(b), "n"(INC));
#endif
}

__device__ __forceinline__ unsigned smem_addr(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ unsigned lds_u32(unsigned addr) {
#ifdef GFICF_CUDA_EMU
  return *static_cast<const unsigned*>(cuda_emu::smem_ptr(addr));
#else
  unsigned r;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr));
  return r;
#endif
}

// shared address of the table slot of id x: IMAD (multiplicative hash), SHF (top bits), and one
// IMAD for base + 4*slot (kept opaque, otherwise it is split into a mask and an add)
template <int SHIFT>
__device__ __forceinline__ unsigned slot_addr(unsigned tbl32, unsigned x, unsigned mult) {
#ifdef GFICF_CUDA_EMU
  return ((x * mult) >> SHIFT) * 4u + tbl32;
#else
  unsigned a;
  asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(a) : "r"((x * mult) >> SHIFT), "r"(tbl32));
  return a;
#endif
}

// membership probes of the 4 ids of one 16-byte piece against a collision-free table at
// shared address tbl32: per id IMAD (hash), SHF (slot), LEA (address), LDS, ISETP, @p IADD
template <unsigned INC, int SHIFT, bool MUT = false>
__device__ __forceinline__ void probe4(unsigned& acc, unsigned tbl32, unsigned mult, const int4& v,
                                       unsigned self = 0) {
  const unsigned x0 = (unsigned)v.x, x1 = (unsigned)v.y, x2 = (unsigned)v.z, x3 = (unsigned)v.w;
  const unsigned k0 = lds_u32(slot_addr<SHIFT>(tbl32, x0, mult));
  const unsigned k1 = lds_u32(slot_addr<SHIFT>(tbl32, x1, mult));
  const unsigned k2 = lds_u32(slot_addr<SHIFT>(tbl32, x2, mult));
  const unsigned k3 = lds_u32(slot_addr<SHIFT>(tbl32, x3, mult));
  add_if_eq<INC>(acc, k0, x0);
  add_if_eq<INC>(acc, k1, x1);
  add_if_eq<INC>(acc, k2, x2);
  add_if_eq<INC>(acc, k3, x3);
  if (MUT) {  // bit 7 of the edge's byte: the neighbour's own list contains this row (i in N(t))
    add_if_eq<INC * 0x80u>(acc, x0, self);
    add_if_eq<INC * 0x80u>(acc, x1, self);
    add_if_eq<INC * 0x80u>(acc, x2, self);
    add_if_eq<INC * 0x80u>(acc, x3, self);
  }
}

// ---------------------------------------------------------------------------
// Layout pre-pass: f64 column-major 1-based  ->  int32 row-major 0-based, padded.
// One CTA converts a tile of TILE_R rows: coalesced 256-byte column reads into a
// shared-memory tile, then the tile (contiguous in the output) leaves with 16-byte
// stores.
// ---------------------------------------------------------------------------
constexpr int kLayoutTileR = 64;  // rows per tile (halved by the host until the tile fits 48 KB)
constexpr int kLayoutThreads = 256;

// id of one element of the caller's matrix: T = double (R numeric matrix) or int (R integer
// matrix, NA_integer_ = INT_MIN is out of range like any other bad id); returns false for a bad id
template <typename T>
__device__ __forceinline__ bool id_from_r(T d, long long n, int& v);
template <>
__device__ __forceinline__ bool id_from_r<double>(double d, long long n, int& v) {
  // ids must be integers in [1,n]; NaN fails the first comparison
  if (d >= 1.0 && d <= (double)n && d == floor(d)) {
    v = (int)d - 1;  // :28  int k = mat(i,j)-1
    return true;
  }
  return false;
}
template <>
__device__ __forceinline__ bool id_from_r<int>(int d, long long n, int& v) {
  if (d >= 1 && (long long)d <= n) {
    v = d - 1;
    return true;
  }
  return false;
}

template <typename T>
__global__ void __launch_bounds__(kLayoutThreads)
layout_colmajor_kernel(const T* __restrict__ src, long long ld_rows, long long ld_row0, long long n,
                  int k, int kp, long long row_lo, long long row_hi, int* __restrict__ dst,
                  unsigned* __restrict__ flags, int tile_r) {
  GFICF_DYNAMIC_SMEM_T(int, tile);  // [tile_r][kp + 1]
  const int tid = threadIdx.x;
  const int stride = kp + 1;
  const long long ntiles = (row_hi - row_lo + tile_r - 1) / tile_r;
  bool bad = false;
  for (long long tb = blockIdx.x; tb < ntiles; tb += gridDim.x) {
    const long long r0 = row_lo + tb * tile_r;
    const int rows = (int)min((long long)tile_r, row_hi - r0);
    // column reads: thread -> (row r = tid % tile_r, column group tid / tile_r); tile_r is a power of 2
    const int r = tid & (tile_r - 1);
    for (int j = tid / tile_r; j < kp; j += kLayoutThreads / tile_r) {
      int v = kPadId;
      if (j < k && r < rows) {
        const T d = __ldcs(src + (long long)j * ld_rows + (r0 + r - ld_row0));
        if (!id_from_r<T>(d, n, v)) {
          bad = true;
          v = 0;
        }
      }
      tile[r * stride + j] = v;
    }
    __syncthreads();
    // contiguous output: rows*kp ints starting at dst + r0*kp  (kp % 4 == 0, 16B aligned)
    int4* out4 = reinterpret_cast<int4*>(dst + r0 * (long long)kp);
    const int nvec = rows * kp / 4;
    for (int x = tid; x < nvec; x += kLayoutThreads) {
      const int f = x * 4;
      const int rr = f / kp, cc = f - rr * kp;
      const int* t = tile + rr * stride + cc;
      out4[x] = make_int4(t[0], t[1], t[2], t[3]);
    }
    __syncthreads();
  }
  if (bad) atomicOr(flags, kFlagBadId);
}

// int32 dense row-major (k per row, 0-based) -> padded rows.  Validates ids in [0,n).
__global__ void __launch_bounds__(256)
pad_i32_kernel(const int* __restrict__ src, long long n, int k, int kp, long long row_lo,
               long long row_hi, int* __restrict__ dst, unsigned* __restrict__ flags) {
  const long long total = (row_hi - row_lo) * (long long)kp;
  bool bad = false;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < total;
       x += (long long)gridDim.x * blockDim.x) {
    const long long rr = x / kp;
    const int cc = (int)(x - rr * kp);
    int v = kPadId;
    if (cc < k) {
      v = __ldcs(src + (row_lo + rr) * (long long)k + cc);
      if (v < 0 || (long long)v >= n) {
        bad = true;
        v = 0;
      }
    }
    dst[(row_lo + rr) * (long long)kp + cc] = v;
  }
  if (bad) atomicOr(flags, kFlagBadId);
}

// ---------------------------------------------------------------------------
// Fast kernel, k <= 32.  KP = padded row length in {4,8,16,32}.
//   LPE lanes fetch one neighbour row (one int4 each); a warp instruction
//   therefore gathers EPS = 32/LPE rows; S steps cover the KP edge slots.
//   Step s, lane group g works on edge e = g*S + s.
// ---------------------------------------------------------------------------
template <int KP>
struct SmallK {
  static constexpr int LPE = KP / 4;
  static constexpr int EPS = 32 / LPE;
  static constexpr int S = (KP >= EPS) ? KP / EPS : 1;
  // table slots per warp: ~k^2/2 gives a >40% chance that a multiplier is collision free
  static constexpr int LOG_TS = (KP == 32) ? GFICF_SMALL_LOG_TS32 : (KP == 16) ? 7 : 6;
  static constexpr int TS = 1 << LOG_TS;
};

constexpr int kSmallWarps = GFICF_SMALL_WARPS;

// OUT: 0 = (from,to,w) doubles, 1 = counts, 2 = counts with the mutual-neighbour bit (bit 7),
//      3 = tagged counts for the streaming peer gather: a warp owns GROUPS of 8 consecutive rows
//          (lg_group = 3) and sends a group with 16-byte (k even) or 8-byte vector stores -- the
//          destination is a peer GPU's memory, and NVLink carries a few 128-byte packets per group
//          instead of one or two 30-byte partial-sector packets per row (measured: 7 peers storing
//          row by row into one GPU are held to 0.67 ms for a 0.40 ms kernel by the packet rate)
template <int KP, int OUT, bool SKIP>
__global__ void __launch_bounds__(kSmallWarps * 32, GFICF_SMALL_MINB)
jaccard_small_k_kernel(const int* __restrict__ idx, int k, long long row_lo, long long row_hi,
                       double* __restrict__ o_from, double* __restrict__ o_to,
                       double* __restrict__ o_w, uint8_t* __restrict__ o_u,
                       unsigned* __restrict__ flags, unsigned tag, int lg_group) {
  constexpr bool COUNTS_ONLY = OUT != 0;
  constexpr bool MUT = OUT == 2;
  constexpr bool GROUPED = OUT == 3;
  using G = SmallK<KP>;
  constexpr int LPE = G::LPE, S = G::S, TS = G::TS, SHIFT = 32 - G::LOG_TS;
  __shared__ __align__(16) unsigned tbl_all[kSmallWarps][TS];
  __shared__ double lut[COUNTS_ONLY ? 1 : 33];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned* tbl = tbl_all[warp];
#pragma unroll
  for (int x = lane; x < TS; x += 32) tbl[x] = kEmpty;
  if (!COUNTS_ONLY && (int)threadIdx.x <= k) lut[threadIdx.x] = jaccard_weight((int)threadIdx.x, k);
  __syncthreads();

  const long long nwarps = (long long)gridDim.x * kSmallWarps;
  const long long gw = (long long)blockIdx.x * kSmallWarps + warp;
  // rows of this warp, in the order it visits them: round-robin over the grid (neighbouring warps write
  // neighbouring output), or -- GROUPED -- round-robin groups of 2^lg_group consecutive rows
  const int gmask = GROUPED ? (1 << lg_group) - 1 : 0;
  int gr = 0;  // GROUPED: position of `row` inside its group
  unsigned cpk0 = 0, cpk1 = 0;  // GROUPED: the group's count bytes of this lane's edge slot
  // GROUPED: only whole rounds of groups (every warp the same number of them) are grouped; the
  // remaining < nwarps groups' worth of rows are dealt row by row like in the other modes, so the
  // kernel does not end with a few warps working through one more 8-row group each (a 0.45 ms launch
  // would lose ~6 % to that tail)
  const long long main_end =
      GROUPED ? row_lo + ((((row_hi - row_lo) >> lg_group) / nwarps) * nwarps << lg_group) : row_lo;
  long long row = (GROUPED && main_end > row_lo) ? row_lo + (gw << lg_group) : row_lo + gw;
  // the row this warp visits after `r` (which sits at position `pos` of its group)
  auto next_row = [&](long long r, int pos) -> long long {
    if (GROUPED && r < main_end) {
      if (pos != gmask) return r + 1;
      const long long nr = r - gmask + (nwarps << lg_group);
      return nr < main_end ? nr : main_end + gw;
    }
    return r + nwarps;
  };
  // which 16-byte piece of a neighbour row this lane fetches
  const char* lane_base = reinterpret_cast<const char*>(idx + (lane % LPE) * 4);
  // SKIP (chosen by the host when k <= KP-4): a 16-byte piece that holds only pads is never fetched
  const bool piece_on = !SKIP || (lane % LPE) * 4 < k;
  const int grp = lane / LPE;
  const bool valid = lane < k;
  unsigned warp_flags = 0;

  int a_next = (row < row_hi && lane < KP) ? __ldg(idx + row * KP + lane) : kPadId;
  for (; row < row_hi; row = next_row(row, gr), gr = (gr + 1) & gmask) {
    const int a = a_next;  // N(i)[lane], 0-based
    {
      const long long nrow = next_row(row, gr);
      a_next = (nrow < row_hi && lane < KP) ? __ldg(idx + nrow * KP + lane) : kPadId;
    }
    // ---- gather addresses first: the loads do not depend on the hash table
    int4 v[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const int e = grp * S + s;
      const int t = __shfl_sync(kFull, a, e & 31);
      v[s] = (e < k && piece_on) ? ldg_row(lane_base, (unsigned)t, KP * 4)
                                 : make_int4(kPadId, kPadId, kPadId, kPadId);
    }
    // ---- collision-free hash of N(i): search a multiplier
    unsigned mult = kMult0, slot;
    bool dup = false;
    int tries = 0;
#if GFICF_SMALL_MATCH
    // Collisions are found in registers: lanes whose ids hash to the same slot find each other
    // with match.any; a group whose ids differ from its leader's is a collision (try the next
    // multiplier), a group with equal ids is a repeated id.  No shared-memory traffic per try.
    for (;;) {
      slot = ((unsigned)a * mult) >> SHIFT;
      const unsigned peers = __match_any_sync(kFull, valid ? slot : (0x80000000u | (unsigned)lane));
      const int leader = __ffs(peers) - 1;
      const int lkey = __shfl_sync(kFull, a, leader);
      const bool follower = valid && lane != leader;  // shares its slot with a lower lane
      dup |= follower && lkey == a;
      if (!__any_sync(kFull, follower && lkey != a)) break;
      if (++tries == kMaxTries) {
        warp_flags |= kFlagHashFail;
        break;
      }
      mult = next_mult(mult);
    }
#else
    // Collisions are found through the table: every lane stores its lane id in its slot and reads
    // it back.  Lanes of one warp that hash to the same slot store DIFFERENT values to it in the
    // same instruction on purpose -- whichever 32-bit store lands, all the others read a foreign
    // id and report the collision (compute-sanitizer's racecheck flags this write-write hazard).
    for (;;) {
      slot = ((unsigned)a * mult) >> SHIFT;
      if (valid) tbl[slot] = (unsigned)lane;
      __syncwarp();
      const int owner = valid ? (int)tbl[slot] : lane;
      const int okey = __shfl_sync(kFull, a, owner);
      const bool lost = owner != lane;
      const bool coll = lost && okey != a;
      dup |= lost && okey == a;
      if (!__any_sync(kFull, coll)) break;
      if (++tries == kMaxTries) {
        warp_flags |= kFlagHashFail;
        break;
      }
      __syncwarp();
      if (valid) tbl[slot] = kEmpty;
      __syncwarp();
      mult = next_mult(mult);
    }
#endif
    __syncwarp();  // every lane has read its slot's owner before the keys overwrite the lane ids
    if (valid) tbl[slot] = (unsigned)a;
    if (__any_sync(kFull, dup)) warp_flags |= kFlagDupId;
    __syncwarp();
    // ---- probe the gathered ids; counts of up to 4 steps packed per register
    unsigned c_lo = 0, c_hi = 0;
    const unsigned tbl32 = smem_addr(tbl);
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if ((s & 3) == 0) probe4<1u, SHIFT, MUT>(s < 4 ? c_lo : c_hi, tbl32, mult, v[s], (unsigned)row);
      if ((s & 3) == 1) probe4<1u << 8, SHIFT, MUT>(s < 4 ? c_lo : c_hi, tbl32, mult, v[s], (unsigned)row);
      if ((s & 3) == 2) probe4<1u << 16, SHIFT, MUT>(s < 4 ? c_lo : c_hi, tbl32, mult, v[s], (unsigned)row);
      if ((s & 3) == 3) probe4<1u << 24, SHIFT, MUT>(s < 4 ? c_lo : c_hi, tbl32, mult, v[s], (unsigned)row);
    }
#pragma unroll
    for (int m = 1; m < LPE; m <<= 1) {
      c_lo += __shfl_xor_sync(kFull, c_lo, m);
      if (S > 4) c_hi += __shfl_xor_sync(kFull, c_hi, m);
    }
    // lane e wants edge e = g*S+s  ->  group e/S, byte e%S
    unsigned p_lo = c_lo, p_hi = c_hi;
    if (S != LPE) {
      const int src = ((lane / S) * LPE) & 31;
      p_lo = __shfl_sync(kFull, c_lo, src);
      if (S > 4) p_hi = __shfl_sync(kFull, c_hi, src);
    }
    const int sb = lane % S;
    const unsigned word = (S > 4 && sb >= 4) ? p_hi : p_lo;
    const int u = (int)((word >> (8 * (sb & 3))) & 0xFFu);
    __syncwarp();
    if (valid) tbl[slot] = kEmpty;  // leave the table empty for the next row
    // ---- epilogue: lane e writes edge (i, e)
    if (GROUPED && row < main_end) {
      // the row's byte waits in a register (8 rows per group: two packed words per lane); at the end
      // of the group the bytes pass through the -- at this point empty -- hash table to be regrouped
      // into 16-byte (k even) or 8-byte (k odd) vectors: no extra shared memory, which would push the
      // SM's carve-out up a step and take 36 KB of L1 from the lines in flight
      const unsigned val = (unsigned)(u | tag) & 0xFFu;
      if (gr < 4) cpk0 |= val << (8 * gr);
      else cpk1 |= val << (8 * (gr - 4));
      if (gr == gmask) {  // the group is complete
        __syncwarp();  // every lane has erased its key: the table is empty
        uint8_t* stage = reinterpret_cast<uint8_t*>(tbl);
        const int nr = gr + 1;
        if (valid) {
#pragma unroll
          for (int r = 0; r < 8; ++r)
            if (r < nr) stage[r * k + lane] = (uint8_t)((r < 4 ? cpk0 >> (8 * r) : cpk1 >> (8 * (r - 4))) & 0xFFu);
        }
        __syncwarp();
        const int nbytes = nr * k;
        uint8_t* dst = o_u + (row - gr - row_lo) * (long long)k;
        if ((nbytes & 15) == 0 && ((unsigned long long)dst & 15ull) == 0) {
          if (lane < (nbytes >> 4)) reinterpret_cast<uint4*>(dst)[lane] = reinterpret_cast<const uint4*>(stage)[lane];
        } else if ((nbytes & 7) == 0 && ((unsigned long long)dst & 7ull) == 0) {
          if (lane < (nbytes >> 3)) reinterpret_cast<uint2*>(dst)[lane] = reinterpret_cast<const uint2*>(stage)[lane];
        } else {
          for (int x = lane; x < nbytes; x += 32) dst[x] = stage[x];
        }
        __syncwarp();
        tbl[lane] = kEmpty;  // 8 rows x k <= 256 bytes were used: 64 words
        tbl[lane + 32] = kEmpty;
        cpk0 = cpk1 = 0;
      }
    } else if (valid) {
      const long long r = (row - row_lo) * (long long)k + lane;
      if (COUNTS_ONLY) {
        o_u[r] = (uint8_t)(u | tag);  // tag: the epoch bit of the streaming peer gather (else 0)
      } else {
        const bool nz = u > 0;  // :48 if(u>0), else the zero-filled row stays
        __stcs(o_from + r, nz ? (double)(row + 1) : 0.0);
        __stcs(o_to + r, nz ? (double)(a + 1) : 0.0);
        __stcs(o_w + r, lut[u]);
      }
    }
    __syncwarp();
  }
  if (COUNTS_ONLY) __threadfence_system();  // the counts may live in a peer GPU's memory
  if (warp_flags && lane == 0) atomicOr(flags, warp_flags);
}

// ---------------------------------------------------------------------------
// Fast kernel, 32 < k <= 128: a warp-group (one CTA of 4 warps) owns row i.
//   * the row's ids go to shared memory once; warp 0 searches the collision-free
//     multiplier and fills the CTA's hash table while the other warps already have
//     their first gathers in flight (the loads do not depend on the table);
//   * each warp takes a quarter of the row's edges; one load instruction fetches ONE
//     neighbour row (lane l brings ids 4l..4l+3), up to U rows in flight per warp;
//   * the table is shared by the 4 warps, so it costs 4x less shared memory per
//     resident warp than a per-warp table: 24-48 warps per SM stay resident.
// ---------------------------------------------------------------------------
constexpr int kWideWarps = 4;
constexpr int kWideU = 8;  // neighbour rows in flight per warp

// table | 2 x own-row ids | 2 x counts (double-buffered across rows) | multiplier
__host__ __device__ constexpr int wide_smem_words(int log_ts) { return (1 << log_ts) + 256 + 256 + 4; }

// N neighbour rows of one batch: issue the gathers / probe them.  N is a template
// parameter (dispatched on the warp-uniform batch size) so that both are branch-free and the
// compiler can put all 4N shared-memory probes in flight together.
template <int N>
__device__ __forceinline__ void wide_load(int4 (&v)[kWideU], const char* lane_base, const int* ids,
                                          unsigned row_bytes, bool lane_on) {
#pragma unroll
  for (int q = 0; q < N; ++q) {
    const unsigned t = (unsigned)ids[q];
    if (lane_on) v[q] = ldg_row(lane_base, t, row_bytes);  // lanes past the row keep their pads
  }
}

template <int N, int SHIFT, bool MUT>
__device__ __forceinline__ void wide_probe(const int4 (&v)[kWideU], unsigned tbl, unsigned mult,
                                           unsigned& a0, unsigned& a1, unsigned self) {
#pragma unroll
  for (int q = 0; q < N; ++q) {
    if ((q & 3) == 0) probe4<1u, SHIFT, MUT>(q < 4 ? a0 : a1, tbl, mult, v[q], self);
    if ((q & 3) == 1) probe4<1u << 8, SHIFT, MUT>(q < 4 ? a0 : a1, tbl, mult, v[q], self);
    if ((q & 3) == 2) probe4<1u << 16, SHIFT, MUT>(q < 4 ? a0 : a1, tbl, mult, v[q], self);
    if ((q & 3) == 3) probe4<1u << 24, SHIFT, MUT>(q < 4 ? a0 : a1, tbl, mult, v[q], self);
  }
}

#define GFICF_WIDE_DISPATCH(cnt, CALL) \
  switch (cnt) {                       \
    case 8: { constexpr int N = 8; CALL; } break; \
    case 7: { constexpr int N = 7; CALL; } break; \
    case 6: { constexpr int N = 6; CALL; } break; \
    case 5: { constexpr int N = 5; CALL; } break; \
    case 4: { constexpr int N = 4; CALL; } break; \
    case 3: { constexpr int N = 3; CALL; } break; \
    case 2: { constexpr int N = 2; CALL; } break; \
    case 1: { constexpr int N = 1; CALL; } break; \
    default: break;                    \
  }

template <int LOG_TS, int OUT>
__global__ void __launch_bounds__(kWideWarps * 32, GFICF_WIDE_MINB)
jaccard_wide_k_kernel(const int* __restrict__ idx, int k, int kp, long long row_lo,
                      long long row_hi, double* __restrict__ o_from, double* __restrict__ o_to,
                      double* __restrict__ o_w, uint8_t* __restrict__ o_u,
                      unsigned* __restrict__ flags, unsigned tag) {
  constexpr int TS = 1 << LOG_TS, SHIFT = 32 - LOG_TS;
  constexpr bool COUNTS_ONLY = OUT != 0;
  constexpr bool MUT = OUT == 2;  // needs k <= 127 (bit 7 of the count byte)
  GFICF_DYNAMIC_SMEM_T(unsigned, smem_u);
  unsigned* tbl = smem_u;                             // [TS]
  int* srow_base = reinterpret_cast<int*>(tbl + TS);   // [2][128] ids of row i
  int* scnt_base = srow_base + 256;                    // [2][128] u per edge
  unsigned* s_mult = reinterpret_cast<unsigned*>(scnt_base + 256);  // [4]
  double* lut = reinterpret_cast<double*>(s_mult + 4);  // [129]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int x = tid; x < TS; x += blockDim.x) tbl[x] = kEmpty;
  for (int x = tid; x <= k; x += blockDim.x) lut[x] = jaccard_weight(x, k);
  __syncthreads();

  const int c0 = lane * 4;
  const bool lane_on = c0 < k;  // lanes whose 16-byte piece holds only pads never load (nor probe)
  const char* lane_base = reinterpret_cast<const char*>(idx + c0);
  const unsigned row_bytes = (unsigned)kp * 4u;
  // gathered pieces; lanes past the end of a row never load and keep these pads for good
  int4 v[kWideU];
#pragma unroll
  for (int q = 0; q < kWideU; ++q) v[q] = make_int4(kPadId, kPadId, kPadId, kPadId);
  // this warp's share of the row's edges, in nb batches of at most U
  const int e_lo = (warp * k) / kWideWarps, e_hi = ((warp + 1) * k) / kWideWarps;
  const int ne = e_hi - e_lo;
  const int nb = (ne + kWideU - 1) / kWideU;
  const int bsz = nb ? (ne + nb - 1) / nb : 0;
  unsigned warp_flags = 0;

  int a_next = (row_lo + blockIdx.x < row_hi && tid < kp)
                   ? __ldg(idx + (row_lo + blockIdx.x) * (long long)kp + tid) : kPadId;
  int parity = 0;
  for (long long row = row_lo + blockIdx.x; row < row_hi; row += gridDim.x, parity ^= 1) {
    // srow / scnt alternate between two buffers, so the epilogue of row r may still read its
    // buffers while the next row is being staged: 3 block barriers per row instead of 4
    int* srow = srow_base + parity * 128;
    int* scnt = scnt_base + parity * 128;
    srow[tid] = a_next;  // blockDim == 128 == capacity of srow
    {
      const long long nrow = row + gridDim.x;
      a_next = (nrow < row_hi && tid < kp) ? __ldg(idx + nrow * (long long)kp + tid) : kPadId;
    }
    __syncthreads();
    // ---- first batch of gathers (independent of the hash table)
    {
      const int cnt0 = min(bsz, ne);
      GFICF_WIDE_DISPATCH(cnt0, wide_load<N>(v, lane_base, srow + e_lo, row_bytes, lane_on))
    }
    // ---- warp 0: collision-free hash of N(i); lane l owns keys l, l+32, l+64, l+96
    if (warp == 0) {
      int av[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) av[c] = srow[lane + 32 * c];
      unsigned mult = kMult0, slot[4];
      bool dup = false;
      int tries = 0;
      for (;;) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          slot[c] = ((unsigned)av[c] * mult) >> SHIFT;
          if (lane + 32 * c < k) tbl[slot[c]] = (unsigned)(lane + 32 * c);
        }
        __syncwarp();  // whichever writer survives in a slot, every other one sees it lost
        bool coll = false;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (lane + 32 * c < k) {
            const int owner = (int)tbl[slot[c]];
            const int okey = srow[owner];
            const bool lost = owner != lane + 32 * c;
            coll |= lost && okey != av[c];
            dup |= lost && okey == av[c];
          }
        }
        if (!__any_sync(kFull, coll)) break;
        if (++tries == kMaxTries) {
          warp_flags |= kFlagHashFail;
          break;
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (lane + 32 * c < k) tbl[slot[c]] = kEmpty;
        __syncwarp();
        mult = next_mult(mult);
      }
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (lane + 32 * c < k) tbl[slot[c]] = (unsigned)av[c];
      if (__any_sync(kFull, dup)) warp_flags |= kFlagDupId;
      if (lane == 0) s_mult[0] = mult;
    }
    __syncthreads();
    const unsigned mult = s_mult[0];
    const unsigned tbl32 = smem_addr(tbl);

    // ---- this warp's batches
    for (int b = 0; b < nb; ++b) {
      const int e0 = e_lo + b * bsz;
      const int cnt = min(bsz, e_hi - e0);
      unsigned acc[kWideU / 4];
#pragma unroll
      for (int q = 0; q < kWideU / 4; ++q) acc[q] = 0;
      GFICF_WIDE_DISPATCH(cnt, (wide_probe<N, SHIFT, MUT>(v, tbl32, mult, acc[0], acc[1], (unsigned)row)))
      // next batch's gathers fly while this batch's counts are reduced
      if (b + 1 < nb) {
        const int n0 = e0 + bsz;
        const int ncnt = min(bsz, e_hi - n0);
        GFICF_WIDE_DISPATCH(ncnt, wide_load<N>(v, lane_base, srow + n0, row_bytes, lane_on))
      }
#pragma unroll
      for (int m = 1; m < 32; m <<= 1) {
#pragma unroll
        for (int q = 0; q < kWideU / 4; ++q) acc[q] += __shfl_xor_sync(kFull, acc[q], m);
      }
      if (lane < cnt) {
        unsigned word = acc[0];
#pragma unroll
        for (int q = 1; q < kWideU / 4; ++q)
          if ((lane >> 2) == q) word = acc[q];
        scnt[e0 + lane] = (int)((word >> (8 * (lane & 3))) & 0xFFu);
      }
    }
    __syncthreads();
    // ---- epilogue: thread e writes edge (i, e): 8-byte coalesced streaming stores
    if (tid < k) {
      const int u = scnt[tid];
      const long long r = (row - row_lo) * (long long)k + tid;
      if (COUNTS_ONLY) {
        o_u[r] = (uint8_t)(u | tag);
      } else {
        const bool nz = u > 0;
        __stcs(o_from + r, nz ? (double)(row + 1) : 0.0);
        __stcs(o_to + r, nz ? (double)(srow[tid] + 1) : 0.0);
        __stcs(o_w + r, lut[u]);
      }
      tbl[((unsigned)srow[tid] * mult) >> SHIFT] = kEmpty;  // leave the table empty
    }
    // no barrier here: the next row's first barrier orders these erasures before warp 0 rebuilds
  }
  if (COUNTS_ONLY) __threadfence_system();  // the counts may live in a peer GPU's memory
  if (warp_flags && lane == 0) atomicOr(flags, warp_flags);
}

// ---------------------------------------------------------------------------
// Fast kernel, 128 < k <= 1024: a CTA of 8 warps owns row i.  A collision-free table would need
// ~k^2/2 slots, so membership is tested in an open-addressing table (4096 slots, load <= 0.25,
// linear probing: 1.2 probes on average).  Each warp takes every 8th edge; one neighbour row is
// fetched with up to 8 LDG.128 per lane.
// ---------------------------------------------------------------------------
constexpr int kLargeWarps = 8;
constexpr int kLargeMaxK = 1024;
constexpr int kLargeLogTs = 12;
constexpr int kLargeChunks = kLargeMaxK / 128;  // 16-byte pieces per lane per neighbour row

__host__ __device__ constexpr size_t large_smem_bytes() {
  return ((size_t)(1 << kLargeLogTs) + kLargeMaxK + kLargeMaxK / 2) * 4 + (kLargeMaxK + 1) * 8 + 16;
}

template <typename CT, bool COUNTS_ONLY>
__global__ void __launch_bounds__(kLargeWarps * 32)
jaccard_large_k_kernel(const int* __restrict__ idx, int k, int kp, long long row_lo, long long row_hi,
                       double* __restrict__ o_from, double* __restrict__ o_to,
                       double* __restrict__ o_w, CT* __restrict__ o_u, unsigned* __restrict__ flags) {
  constexpr int TS = 1 << kLargeLogTs, SHIFT = 32 - kLargeLogTs;
  GFICF_DYNAMIC_SMEM_T(unsigned, smem_u);
  unsigned* tbl = smem_u;                                              // [TS]
  int* srow = reinterpret_cast<int*>(tbl + TS);                         // [1024] ids of row i
  unsigned short* scnt = reinterpret_cast<unsigned short*>(srow + kLargeMaxK);  // [1024] u per edge
  double* lut = reinterpret_cast<double*>(srow + kLargeMaxK + kLargeMaxK / 2 + 2);  // [k+1]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int x = tid; x <= k; x += blockDim.x) lut[x] = jaccard_weight(x, k);
  const int nchunk = (kp + 127) / 128;
  const char* lane_base = reinterpret_cast<const char*>(idx + lane * 4);
  const unsigned row_bytes = (unsigned)kp * 4u;
  bool dup = false;

  for (long long row = row_lo + blockIdx.x; row < row_hi; row += gridDim.x) {
    for (int x = tid; x < TS; x += blockDim.x) tbl[x] = kEmpty;
    for (int x = tid; x < kp; x += blockDim.x) srow[x] = __ldg(idx + row * (long long)kp + x);
    __syncthreads();
    // ---- insert N(i): linear probing, a slot is claimed with a shared-memory CAS
    for (int x = tid; x < k; x += blockDim.x) {
      const unsigned key = (unsigned)srow[x];
      unsigned s = (key * kMult0) >> SHIFT;
      for (;;) {
        const unsigned old = atomicCAS(&tbl[s], kEmpty, key);
        if (old == kEmpty) break;
        if (old == key) {  // the row lists this id twice
          dup = true;
          break;
        }
        s = (s + 1) & (TS - 1);
      }
    }
    __syncthreads();
    // ---- edges e = warp, warp+8, ...
    for (int e = warp; e < k; e += kLargeWarps) {
      const unsigned t = (unsigned)srow[e];
      int4 v[kLargeChunks];
#pragma unroll
      for (int c = 0; c < kLargeChunks; ++c) {
        v[c] = make_int4(kPadId, kPadId, kPadId, kPadId);
        if (c < nchunk && c * 128 + lane * 4 < kp)
          v[c] = __ldg(reinterpret_cast<const int4*>(lane_base + (unsigned long long)t * row_bytes + c * 512));
      }
      int cnt = 0;
#pragma unroll
      for (int c = 0; c < kLargeChunks; ++c) {
        if (c < nchunk) {  // block-uniform
          const unsigned xs[4] = {(unsigned)v[c].x, (unsigned)v[c].y, (unsigned)v[c].z, (unsigned)v[c].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const unsigned x = xs[q];
            if (x == (unsigned)kPadId) continue;
            unsigned s = (x * kMult0) >> SHIFT;
            for (;;) {
              const unsigned o = tbl[s];
              if (o == x) {
                ++cnt;
                break;
              }
              if (o == kEmpty) break;
              s = (s + 1) & (TS - 1);
            }
          }
        }
      }
#pragma unroll
      for (int m = 16; m; m >>= 1) cnt += __shfl_xor_sync(kFull, cnt, m);
      if (lane == 0) scnt[e] = (unsigned short)cnt;
    }
    __syncthreads();
    // ---- epilogue
    for (int e = tid; e < k; e += blockDim.x) {
      const int u = scnt[e];
      const long long r = (row - row_lo) * (long long)k + e;
      if (COUNTS_ONLY) {
        o_u[r] = (CT)u;
      } else {
        const bool nz = u > 0;
        __stcs(o_from + r, nz ? (double)(row + 1) : 0.0);
        __stcs(o_to + r, nz ? (double)(srow[e] + 1) : 0.0);
        __stcs(o_w + r, lut[u]);
      }
    }
    __syncthreads();
  }
  if (COUNTS_ONLY) __threadfence_system();
  if (dup) atomicOr(flags, kFlagDupId);
}

// ---------------------------------------------------------------------------
// Exact kernel: any k, rows may repeat ids.  One thread per edge, O(k^2).
//   multiset:  u = sum_p [ rank_t(p) < cnt_i(t_p) ]   = sum_v min(cnt_i(v), cnt_t(v))
//   set:       u = sum_p [ rank_t(p)==0 && cnt_i(t_p)>0 ]
// where rank_t(p) = #{q<p : t_q == t_p}.
// ---------------------------------------------------------------------------
template <typename CT>
__global__ void __launch_bounds__(128)
jaccard_exact_kernel(const int* __restrict__ idx, int k, int kp, long long row_lo, long long row_hi,
                     int set_semantics, CT* __restrict__ o_u) {
  const long long total = (row_hi - row_lo) * (long long)k;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < total;
       r += (long long)gridDim.x * blockDim.x) {
    const long long i = row_lo + r / k;
    const int j = (int)(r % k);
    const int* ri = idx + i * (long long)kp;
    const int* rt = idx + (long long)ri[j] * kp;
    int u = 0;
    for (int p = 0; p < k; ++p) {
      const int x = rt[p];
      int rank = 0;
      for (int q = 0; q < p; ++q) rank += rt[q] == x;
      int cnt = 0;
      for (int q = 0; q < k; ++q) cnt += ri[q] == x;
      u += set_semantics ? (rank == 0 && cnt > 0) : (rank < cnt);
    }
    o_u[r] = (CT)u;
  }
}

// ---------------------------------------------------------------------------
// counts -> edge rows, fixed slots (mode 0).  One thread per edge, streaming.
// ---------------------------------------------------------------------------
constexpr unsigned kFlagPeerTimeout = 8u;

constexpr int kExpandThreads = 256;

template <typename CT>
__global__ void __launch_bounds__(kExpandThreads)
expand_fixed_kernel(const int* __restrict__ idx, int k, int kp, long long row_lo, long long row_hi,
                    const CT* d_u, double* __restrict__ o_from, double* __restrict__ o_to,
                    double* __restrict__ o_w) {
  __shared__ double lut[256];
  const bool use_lut = k <= 255;
  if (use_lut && (int)threadIdx.x <= k) lut[threadIdx.x] = jaccard_weight((int)threadIdx.x, k);
  __syncthreads();
  // Grid-stride over the edges (at any moment the whole grid writes ONE contiguous window of each
  // output array: DRAM-page friendly), with a (row, j) walk that needs no division per edge: one
  // division per thread, then fixed increments.
  const long long stride = (long long)gridDim.x * kExpandThreads;
  const long long d_row = stride / k;
  const int d_j = (int)(stride % k);
  const long long e_hi = (row_hi - row_lo) * k;
  const long long g0 = (long long)blockIdx.x * kExpandThreads + threadIdx.x;
  long long row = row_lo + g0 / k;
  int j = (int)(g0 % k);
#pragma unroll 4
  for (long long e = g0; e < e_hi; e += stride) {
    const int u = (int)__ldcg(d_u + e);
    // the id is loaded unconditionally: a load that waits for u first doubles the latency chain
    // (measured 0.98 -> 0.62 ms at 4M x 30, tools/expand_bench.cu)
    const int t = __ldg(idx + row * (long long)kp + j);
    const bool nz = u > 0;
    __stcs(o_from + e, nz ? (double)(row + 1) : 0.0);
    __stcs(o_to + e, nz ? (double)(t + 1) : 0.0);
    __stcs(o_w + e, use_lut ? lut[u] : (nz ? jaccard_weight(u, k) : 0.0));
    row += d_row;
    j += d_j;
    if (j >= k) {
      j -= k;
      ++row;
    }
  }
}

// ---------------------------------------------------------------------------
// Streaming expand of the peer-memory gather (host rank).  The count bytes of the rows in
// segs[0..gridDim.y) are being stored into THIS GPU's memory by the count kernels of peer GPUs
// (NVLink stores from their epilogues) while this kernel runs.  There are no flags and no fences:
// every count byte carries the epoch's parity in bit 7 (`tag`, k <= 127), the buffer still holds the
// other parity from the previous epoch, so a byte IS its own ready flag -- a thread polls its byte
// (volatile load, served by L2, the point of coherence for stores arriving over NVLink) until the
// parity matches.  blockIdx.y selects a segment (one per contributing rank); inside a segment the
// sub-grid walks the rows linearly, like the peer's persistent count kernel does, so it trails the
// producer by a fixed distance and normally never waits.
// A bounded spin: after spin_clocks without progress the thread raises GFICF_FLAG_PEER_TIMEOUT and
// leaves (the output is then invalid and the host side reports the error).
// ---------------------------------------------------------------------------
constexpr int kMaxStreamSegs = 16;
struct StreamSegs {
  long long lo[kMaxStreamSegs], hi[kMaxStreamSegs];
};

__device__ __forceinline__ unsigned ld_volatile_u8(const uint8_t* p) {
#ifdef GFICF_CUDA_EMU
  return *static_cast<const volatile uint8_t*>(p);
#else
  unsigned v;
  asm volatile("ld.volatile.global.u8 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
#endif
}

#ifndef GFICF_STREAM_BATCH
#define GFICF_STREAM_BATCH 2  // edges per thread whose loads are in flight together
#endif
#ifndef GFICF_STREAM_MINB
#define GFICF_STREAM_MINB 8   // resident CTAs per SM the streaming expand is compiled for
#endif
constexpr int kStreamBatch = GFICF_STREAM_BATCH;
#ifndef GFICF_STREAM_STORE
#define GFICF_STREAM_STORE 0  // 0: st.global.cs (evict first), 1: default policy
#endif

template <typename V>
__device__ __forceinline__ void stream_store(V* p, V v) {
#if GFICF_STREAM_STORE == 0
  __stcs(p, v);
#else
  *p = v;
#endif
}

__device__ __forceinline__ unsigned ld_volatile_u16(const uint8_t* p) {
#ifdef GFICF_CUDA_EMU
  return *reinterpret_cast<const volatile unsigned short*>(p);
#else
  unsigned short v;
  asm volatile("ld.volatile.global.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return v;
#endif
}

// W = edges per thread and round that are adjacent in memory: 1 (8-byte stores) or 2 (one 16-bit
// count load, 16-byte stores; needs 16-byte aligned output columns and even segment starts)
template <int W>
__global__ void __launch_bounds__(kExpandThreads, W == 2 ? 6 : GFICF_STREAM_MINB)
expand_stream_kernel(const int* __restrict__ idx, int k, int kp, StreamSegs segs, const uint8_t* d_u,
                     double* __restrict__ o_from, double* __restrict__ o_to, double* __restrict__ o_w,
                     unsigned tag, long long spin_clocks, unsigned* flags) {
  __shared__ double lut[128];
  if ((int)threadIdx.x <= k && threadIdx.x < 128) lut[threadIdx.x] = jaccard_weight((int)threadIdx.x, k);
  __syncthreads();
  const long long e_hi = segs.hi[blockIdx.y] * k;
  const long long stride = (long long)gridDim.x * kExpandThreads * W;
  const long long d_row = stride / k;
  const int d_j = (int)(stride % k);
  const long long g0 = segs.lo[blockIdx.y] * k + ((long long)blockIdx.x * kExpandThreads + threadIdx.x) * W;
  long long row = g0 / k;  // absolute row: d_u, o_* are indexed by absolute edge number
  int j = (int)(g0 % k);
  const unsigned want = W == 2 ? tag * 0x0101u : tag, pmask = W == 2 ? 0x8080u : 0x80u;
  // A thread walks its edges with a grid-wide stride, kStreamBatch items per round: the id loads
  // and the (volatile) count-byte loads of a round are all issued before the first byte is looked
  // at.  One edge per round would make every thread pay a full L2/DRAM round trip per edge, and a
  // thread that trails the producers by less than that could never keep their pace.
  for (long long e = g0; e < e_hi; e += kStreamBatch * stride) {
    long long rows[kStreamBatch];
    int js[kStreamBatch];
    int t[kStreamBatch][W];
    unsigned b[kStreamBatch];
#pragma unroll
    for (int q = 0; q < kStreamBatch; ++q) {
      rows[q] = row;
      js[q] = j;
      const long long eq = e + q * stride;
      if (eq < e_hi) {
        t[q][0] = __ldg(idx + row * (long long)kp + j);  // independent of the count byte
        if (W == 2) {
          const bool wrap = j + 1 >= k;  // the second edge starts the next row
          if (eq + 1 < e_hi) t[q][W - 1] = __ldg(idx + (row + (wrap ? 1 : 0)) * (long long)kp + (wrap ? 0 : j + 1));
          b[q] = eq + 1 < e_hi ? ld_volatile_u16(d_u + eq) : (ld_volatile_u8(d_u + eq) | (want & 0xFF00u));
        } else {
          b[q] = ld_volatile_u8(d_u + eq);
        }
      }
      row += d_row;
      j += d_j;
      if (j >= k) {
        j -= k;
        ++row;
      }
    }
#pragma unroll
    for (int q = 0; q < kStreamBatch; ++q) {
      const long long eq = e + q * stride;
      if (eq >= e_hi) break;
      unsigned bq = b[q];
      if ((bq & pmask) != want) {
        const long long t0 = clock64();
        unsigned ns = 32;
        do {
          __nanosleep(ns);
          if (ns < 1024) ns <<= 1;
          bq = (W == 2 && eq + 1 < e_hi) ? ld_volatile_u16(d_u + eq)
                                         : (ld_volatile_u8(d_u + eq) | (W == 2 ? (want & 0xFF00u) : 0u));
          if ((bq & pmask) != want && clock64() - t0 > spin_clocks) {
            atomicOr(flags, kFlagPeerTimeout);
            return;
          }
        } while ((bq & pmask) != want);
      }
      const int u0 = (int)(bq & 0x7Fu);
      const double f0 = u0 > 0 ? (double)(rows[q] + 1) : 0.0, t0v = u0 > 0 ? (double)(t[q][0] + 1) : 0.0;
      if (W == 2 && eq + 1 < e_hi) {
        const int u1 = (int)((bq >> 8) & 0x7Fu);
        const long long r1 = rows[q] + (js[q] + 1 >= k ? 1 : 0);
        stream_store(reinterpret_cast<double2*>(o_from + eq), make_double2(f0, u1 > 0 ? (double)(r1 + 1) : 0.0));
        stream_store(reinterpret_cast<double2*>(o_to + eq), make_double2(t0v, u1 > 0 ? (double)(t[q][W - 1] + 1) : 0.0));
        stream_store(reinterpret_cast<double2*>(o_w + eq), make_double2(lut[u0], lut[u1]));
      } else {
        stream_store(o_from + eq, f0);
        stream_store(o_to + eq, t0v);
        stream_store(o_w + eq, lut[u0]);
      }
    }
  }
}

// holds the stream until *flag >= expected (bounded spin: after spin_clocks it raises
// GFICF_FLAG_PEER_TIMEOUT instead of hanging the GPU)
__global__ void wait_kernel(const volatile unsigned* flag, unsigned expected, unsigned* flags,
                            long long spin_clocks) {
  const long long t0 = clock64();
  while ((int)(*flag - expected) < 0) {
    if (clock64() - t0 > spin_clocks) {
      atomicOr(flags, kFlagPeerTimeout);
      break;
    }
    __nanosleep(500);
  }
  __threadfence_system();
}

// raises a (possibly peer-resident) flag once everything before it in the stream has finished
__global__ void signal_kernel(unsigned* flag, unsigned value) {
  __threadfence_system();
  *(volatile unsigned*)flag = value;
  __threadfence_system();
}

// ---------------------------------------------------------------------------
// counts -> edge rows, compacted (mode 1): rows with u>0 in (i,j) order, the
// tail zero-filled.  Three passes: per-chunk counts, scan of the chunk counts,
// scatter.
// ---------------------------------------------------------------------------
constexpr int kCompactChunk = 4096;  // edges per CTA
constexpr int kCompactThreads = 256;

template <typename CT>
__global__ void __launch_bounds__(kCompactThreads)
compact_count_kernel(const CT* __restrict__ d_u, long long total, long long* __restrict__ chunk_cnt) {
  __shared__ int wsum[kCompactThreads / 32];
  const long long base = (long long)blockIdx.x * kCompactChunk;
  int c = 0;
  for (int x = threadIdx.x; x < kCompactChunk; x += kCompactThreads) {
    const long long r = base + x;
    c += (r < total) && d_u[r] != 0;
  }
  for (int m = 16; m; m >>= 1) c += __shfl_xor_sync(kFull, c, m);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < kCompactThreads / 32; ++w) s += wsum[w];
    chunk_cnt[blockIdx.x] = s;
  }
}

template <typename CT>
__global__ void __launch_bounds__(kCompactThreads)
compact_scatter_kernel(const int* __restrict__ idx, int k, int kp, long long row_lo,
                       const CT* __restrict__ d_u, long long total,
                       const long long* __restrict__ chunk_off, double* __restrict__ o_from,
                       double* __restrict__ o_to, double* __restrict__ o_w) {
  __shared__ int wsum[kCompactThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long base = (long long)blockIdx.x * kCompactChunk;
  long long off = chunk_off[blockIdx.x];
  for (int x0 = 0; x0 < kCompactChunk; x0 += kCompactThreads) {
    const long long r = base + x0 + threadIdx.x;
    const int u = (r < total) ? (int)d_u[r] : 0;
    const bool nz = u > 0;
    const unsigned b = __ballot_sync(kFull, nz);
    if (lane == 0) wsum[warp] = __popc(b);
    __syncthreads();
    int before = __popc(b & ((1u << lane) - 1u));
    int all = 0;
    for (int w = 0; w < kCompactThreads / 32; ++w) {
      const int s = wsum[w];
      if (w < warp) before += s;
      all += s;
    }
    if (nz) {
      const long long rr = r / k;
      const int j = (int)(r - rr * k);
      const int t = __ldg(idx + (row_lo + rr) * (long long)kp + j);
      const long long o = off + before;
      __stcs(o_from + o, (double)(row_lo + rr + 1));
      __stcs(o_to + o, (double)(t + 1));
      __stcs(o_w + o, jaccard_weight(u, k));
    }
    off += all;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256)
zero_tail_kernel(const long long* __restrict__ n_written, long long total, double* __restrict__ o_from,
                 double* __restrict__ o_to, double* __restrict__ o_w) {
  const long long start = *n_written;
  for (long long r = start + (long long)blockIdx.x * blockDim.x + threadIdx.x; r < total;
       r += (long long)gridDim.x * blockDim.x) {
    o_from[r] = 0.0;
    o_to[r] = 0.0;
    o_w[r] = 0.0;
  }
}

}  // namespace gficf
