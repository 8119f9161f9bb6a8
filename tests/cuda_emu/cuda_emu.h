// cuda_emu.h -- a small emulation of the CUDA execution model on the CPU (TEST INFRASTRUCTURE,
// NOT PRODUCT CODE; only tests/ compiles against it).
//
// Purpose: the container the CPU test suite runs in has no GPU.  Kernels whose source is plain
// C++ plus the CUDA built-ins below (no inline PTX) are compiled with g++ -DGFICF_CUDA_EMU and
// run here, so their indexing, barriers, warp collectives and the order of the launches are
// exercised against the oracle before they ever reach a B200.  It checks LOGIC only: nothing
// about memory ordering between CTAs, performance or resource limits carries over.
//
// Model: one CTA at a time; every CUDA thread is a fibre (ucontext) scheduled round-robin;
// __syncthreads() and the *_sync warp collectives are barriers between fibres.  Being stricter
// than the hardware is intended:
//   * a collective with a partial mask, or one that not all 32 lanes of the warp reach, aborts;
//   * a __syncthreads() that some live thread of the CTA never reaches aborts (deadlock report);
//   * atomics are plain read-modify-writes (fibres never run concurrently): their order is the
//     order in which the fibres run, which the schedule below decides.
// Schedule (emu_set_schedule): in every round the runnable fibres run in ascending threadIdx.x
// (the default), descending, or a permutation drawn afresh each round from a seeded xorshift; the
// CTAs of a launch, over x and y, run in the same kind of order.  A missing barrier where a lower
// thread writes and a higher one reads, an atomic cursor whose order leaks into the output, or a
// CTA that reads what a lower-numbered CTA of the same launch wrote passes in ascending order only.
// Dynamic shared memory is filled with 0xA5 at the start of every CTA.
#pragma once
#include <ucontext.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __launch_bounds__(...)
#define __shared__ static
#define __align__(n) __attribute__((aligned(n)))

namespace cuda_emu {

struct Idx3 {
  unsigned x = 0, y = 0, z = 0;
};
struct Dim3 {
  unsigned x = 1, y = 1, z = 1;
};

enum class St { Runnable, WaitCta, WaitWarp, Done };

struct Fibre {
  ucontext_t ctx;
  St st = St::Runnable;
  unsigned tid = 0;
};

struct WarpState {
  uint64_t slot[32];
  unsigned arrived = 0;
};

struct CtaState {
  std::vector<Fibre> fibres;
  std::vector<WarpState> warps;
  unsigned cta_arrived = 0;
  unsigned live = 0;
  ucontext_t sched;
  Fibre* cur = nullptr;
  std::function<void()> body;
};

inline CtaState* g_cta = nullptr;
inline long long g_launches = 0;

// the order in which runnable fibres (and the CTAs of a launch) are visited
enum Schedule : int { kAscending = 0, kDescending = 1, kRandom = 2 };
inline int g_schedule = kAscending;
inline unsigned long long g_rng = 1;  // xorshift64 state, never 0

inline unsigned long long next_random() {
  g_rng ^= g_rng << 13;
  g_rng ^= g_rng >> 7;
  g_rng ^= g_rng << 17;
  return g_rng;
}

// order[0..n) := the visiting order of n items under the current schedule
inline void schedule_order(std::vector<unsigned>& order, unsigned n) {
  order.resize(n);
  for (unsigned i = 0; i < n; ++i) order[i] = g_schedule == kDescending ? n - 1 - i : i;
  if (g_schedule == kRandom)
    for (unsigned i = n; i > 1; --i) {  // Fisher-Yates
      const unsigned j = (unsigned)(next_random() % i);
      const unsigned t = order[i - 1];
      order[i - 1] = order[j];
      order[j] = t;
    }
}

// the launch's dynamic shared memory (CTAs run one at a time); static so that it lies inside the 32-bit
// window of emulated shared-memory addresses (smem_base below), like the kernels' static __shared__ arrays
constexpr size_t kMaxDynamicSmem = 232 * 1024;
alignas(128) inline unsigned char g_dyn_smem[kMaxDynamicSmem];
inline unsigned char* dynamic_smem() { return g_dyn_smem; }

[[noreturn]] inline void die(const char* msg) {
  fprintf(stderr, "cuda_emu: %s\n", msg);
  abort();
}

inline void yield_to_scheduler() { swapcontext(&g_cta->cur->ctx, &g_cta->sched); }

inline void cta_barrier() {
  CtaState* c = g_cta;
  c->cur->st = St::WaitCta;
  if (++c->cta_arrived == c->live) {
    c->cta_arrived = 0;
    for (auto& f : c->fibres)
      if (f.st == St::WaitCta) f.st = St::Runnable;
    return;  // the last arriver simply goes on
  }
  yield_to_scheduler();
}

inline unsigned warp_live_lanes(CtaState* c, unsigned warp) {
  unsigned n = 0;
  for (unsigned l = 0; l < 32; ++l) {
    const unsigned t = warp * 32 + l;
    if (t < c->fibres.size() && c->fibres[t].st != St::Done) ++n;
  }
  return n;
}

inline void warp_barrier() {
  CtaState* c = g_cta;
  const unsigned warp = c->cur->tid >> 5;
  WarpState& w = c->warps[warp];
  c->cur->st = St::WaitWarp;
  if (warp_live_lanes(c, warp) != 32) die("warp collective reached while lanes of the warp have exited");
  if (++w.arrived == 32) {
    w.arrived = 0;
    for (unsigned l = 0; l < 32; ++l) c->fibres[warp * 32 + l].st = St::Runnable;
    return;
  }
  yield_to_scheduler();
}

inline void fibre_entry() {
  CtaState* c = g_cta;
  c->body();
  // lanes of this warp already wait in a collective that it will never reach (in ascending order the
  // next lane to arrive reports it; in other orders every other lane may have arrived already)
  if (c->warps[c->cur->tid >> 5].arrived) die("warp collective reached while lanes of the warp have exited");
  c->cur->st = St::Done;
  --c->live;
  // a thread that exits while others wait at __syncthreads: the hardware lets the rest proceed
  if (c->live && c->cta_arrived == c->live) {
    c->cta_arrived = 0;
    for (auto& f : c->fibres)
      if (f.st == St::WaitCta) f.st = St::Runnable;
  }
  swapcontext(&c->cur->ctx, &c->sched);
}

}  // namespace cuda_emu

// mode 0 ascending, 1 descending, 2 random(seed): the schedule of every later launch.  Exported from
// every harness library for ctypes (`used` emits the inline definition even where nothing calls it).
extern "C" inline __attribute__((used, visibility("default"))) void emu_set_schedule(int mode,
                                                                                     unsigned long long seed) {
  if (mode < cuda_emu::kAscending || mode > cuda_emu::kRandom) cuda_emu::die("unknown schedule");
  cuda_emu::g_schedule = mode;
  cuda_emu::g_rng = seed * 0x9E3779B97F4A7C15ull + 0x2545F4914F6CDD1Dull;  // any seed, 0 included
  if (cuda_emu::g_rng == 0) cuda_emu::g_rng = 1;
}

inline cuda_emu::Idx3 threadIdx, blockIdx;
inline cuda_emu::Dim3 blockDim, gridDim;

namespace cuda_emu {

constexpr size_t kStackBytes = 64 * 1024;

// run `body` (a call of the kernel function with its arguments) for grid x block threads
template <class F>
void launch(unsigned grid, unsigned block, F&& body, size_t dynamic_smem_bytes = 0, unsigned grid_y = 1) {
  if (dynamic_smem_bytes > kMaxDynamicSmem) die("more dynamic shared memory than an SM has");
  if (block == 0 || block % 32 != 0 || block > 1024) die("block size must be a multiple of 32, at most 1024");
  ++g_launches;
  gridDim = Dim3{grid, grid_y, 1};
  blockDim = Dim3{block, 1, 1};
  CtaState cta;
  cta.body = body;
  cta.fibres.resize(block);
  // fibre stacks are kept between launches (allocating 1024 x 64 KB per launch dominated the run time)
  static std::vector<std::unique_ptr<char[]>> stack_pool;
  while (stack_pool.size() < block) stack_pool.emplace_back(new char[kStackBytes]);
  cta.warps.resize(block / 32);
  g_cta = &cta;
  std::vector<unsigned> ctas, order;
  if ((unsigned long long)grid * grid_y > 0xFFFFFFFFull) die("more CTAs than the emulation numbers");
  schedule_order(ctas, grid * grid_y);  // y-major, like the nested loops of the ascending order
  for (const unsigned c : ctas) {
    blockIdx = Idx3{c % grid, c / grid, 0};
    memset(g_dyn_smem, 0xA5, dynamic_smem_bytes);  // every CTA starts from poison, not its predecessor's data
    cta.live = block;
    cta.cta_arrived = 0;
    for (auto& w : cta.warps) w.arrived = 0;
    for (unsigned t = 0; t < block; ++t) {
      Fibre& f = cta.fibres[t];
      f.st = St::Runnable;
      f.tid = t;
      getcontext(&f.ctx);
      f.ctx.uc_stack.ss_sp = stack_pool[t].get();
      f.ctx.uc_stack.ss_size = kStackBytes;
      f.ctx.uc_link = nullptr;
      makecontext(&f.ctx, (void (*)())fibre_entry, 0);
    }
    while (cta.live) {
      bool ran = false;
      schedule_order(order, block);
      for (const unsigned t : order) {
        Fibre& f = cta.fibres[t];
        if (f.st != St::Runnable) continue;
        ran = true;
        cta.cur = &f;
        threadIdx = Idx3{t, 0, 0};
        swapcontext(&cta.sched, &f.ctx);
      }
      if (!ran && cta.live) die("deadlock: live threads are all waiting (divergent __syncthreads or collective)");
    }
  }
  g_cta = nullptr;
}

template <class T>
inline uint64_t to_raw(T v) {
  static_assert(sizeof(T) <= 8, "collective operand wider than 8 bytes");
  uint64_t r = 0;
  memcpy(&r, &v, sizeof(T));
  return r;
}
template <class T>
inline T from_raw(uint64_t r) {
  T v;
  memcpy(&v, &r, sizeof(T));
  return v;
}

inline void check_mask(unsigned mask) {
  if (mask != 0xFFFFFFFFu) die("collective with a partial member mask (the emulation only accepts full warps)");
}

// every lane publishes a value, then reads the lane it wants
template <class T>
inline T exchange(T v, unsigned src_lane) {
  CtaState* c = g_cta;
  const unsigned tid = c->cur->tid;
  WarpState& w = c->warps[tid >> 5];
  w.slot[tid & 31] = to_raw(v);
  warp_barrier();
  const uint64_t got = w.slot[src_lane & 31];
  warp_barrier();
  return from_raw<T>(got);
}

}  // namespace cuda_emu

// ---- built-ins -------------------------------------------------------------------------------
inline void __syncthreads() { cuda_emu::cta_barrier(); }
inline void __syncwarp(unsigned mask = 0xFFFFFFFFu) {
  cuda_emu::check_mask(mask);
  cuda_emu::warp_barrier();
}

template <class T>
inline T __shfl_sync(unsigned mask, T v, int src) {
  cuda_emu::check_mask(mask);
  return cuda_emu::exchange(v, (unsigned)src);
}
template <class T>
inline T __shfl_up_sync(unsigned mask, T v, unsigned delta) {
  cuda_emu::check_mask(mask);
  const unsigned lane = threadIdx.x & 31;
  return cuda_emu::exchange(v, lane >= delta ? lane - delta : lane);
}
template <class T>
inline T __shfl_down_sync(unsigned mask, T v, unsigned delta) {
  cuda_emu::check_mask(mask);
  const unsigned lane = threadIdx.x & 31;
  return cuda_emu::exchange(v, lane + delta < 32 ? lane + delta : lane);
}
template <class T>
inline T __shfl_xor_sync(unsigned mask, T v, int lane_mask) {
  cuda_emu::check_mask(mask);
  return cuda_emu::exchange(v, (threadIdx.x & 31) ^ (unsigned)lane_mask);
}
inline unsigned __ballot_sync(unsigned mask, int pred) {
  cuda_emu::check_mask(mask);
  cuda_emu::CtaState* c = cuda_emu::g_cta;
  cuda_emu::WarpState& w = c->warps[c->cur->tid >> 5];
  w.slot[c->cur->tid & 31] = pred ? 1 : 0;
  cuda_emu::warp_barrier();
  unsigned m = 0;
  for (unsigned l = 0; l < 32; ++l) m |= (unsigned)(w.slot[l] & 1) << l;
  cuda_emu::warp_barrier();
  return m;
}
inline int __any_sync(unsigned mask, int pred) { return __ballot_sync(mask, pred) != 0; }
inline int __all_sync(unsigned mask, int pred) { return __ballot_sync(mask, pred) == 0xFFFFFFFFu; }
template <class T>
inline unsigned __match_any_sync(unsigned mask, T v) {
  cuda_emu::check_mask(mask);
  cuda_emu::CtaState* c = cuda_emu::g_cta;
  cuda_emu::WarpState& w = c->warps[c->cur->tid >> 5];
  const uint64_t mine = cuda_emu::to_raw(v);
  w.slot[c->cur->tid & 31] = mine;
  cuda_emu::warp_barrier();
  unsigned m = 0;
  for (unsigned l = 0; l < 32; ++l) m |= (unsigned)(w.slot[l] == mine) << l;
  cuda_emu::warp_barrier();
  return m;
}

template <class T>
inline T atomicAdd(T* p, T v) {
  const T old = *p;
  *p = old + v;
  return old;
}
// mixed operand types as CUDA's overload set accepts them, e.g. atomicAdd(unsigned*, int)
inline unsigned atomicAdd(unsigned* p, int v) { return atomicAdd<unsigned>(p, (unsigned)v); }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned v) { return atomicAdd<unsigned long long>(p, v); }
inline unsigned atomicCAS(unsigned* p, unsigned expected, unsigned desired) {
  const unsigned old = *p;
  if (old == expected) *p = desired;
  return old;
}
inline unsigned atomicOr(unsigned* p, unsigned v) {
  const unsigned old = *p;
  *p = old | v;
  return old;
}
inline unsigned atomicMin(unsigned* p, unsigned v) {
  const unsigned old = *p;
  if (v < old) *p = v;
  return old;
}
inline int atomicMax(int* p, int v) {
  const int old = *p;
  if (v > old) *p = v;
  return old;
}

template <class T>
inline T __ldg(const T* p) {
  return *p;
}
inline int __popc(unsigned v) { return __builtin_popcount(v); }
inline int __popcll(unsigned long long v) { return __builtin_popcountll(v); }
inline int __clz(int v) { return v ? __builtin_clz((unsigned)v) : 32; }
inline int __ffs(int v) { return __builtin_ffs(v); }
// correctly rounded IEEE operations (compile the test with -ffp-contract=off)
inline double __dadd_rn(double a, double b) { volatile double r = a + b; return r; }
inline double __dmul_rn(double a, double b) { volatile double r = a * b; return r; }
inline double __ddiv_rn(double a, double b) { volatile double r = a / b; return r; }
inline double __dsqrt_rn(double a) { volatile double r = std::sqrt(a); return r; }
inline long long __double_as_longlong(double v) { return cuda_emu::from_raw<long long>(cuda_emu::to_raw(v)); }
inline double __longlong_as_double(long long v) { return cuda_emu::from_raw<double>(cuda_emu::to_raw(v)); }

// ---- vector types, cache-hinted accesses, fences (what jaccard_kernels.cuh uses) ----------------
struct __attribute__((aligned(8))) int2 { int x, y; };
struct __attribute__((aligned(16))) int4 { int x, y, z, w; };
struct __attribute__((aligned(8))) uint2 { unsigned x, y; };
struct __attribute__((aligned(16))) uint4 { unsigned x, y, z, w; };
struct __attribute__((aligned(16))) double2 { double x, y; };
inline int2 make_int2(int x, int y) { return int2{x, y}; }
inline int4 make_int4(int x, int y, int z, int w) { return int4{x, y, z, w}; }
inline uint2 make_uint2(unsigned x, unsigned y) { return uint2{x, y}; }
inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }
inline double2 make_double2(double x, double y) { return double2{x, y}; }
template <class T> inline T __ldcs(const T* p) { return *p; }
template <class T> inline T __ldcg(const T* p) { return *p; }
template <class T> inline void __stcs(T* p, T v) { *p = v; }
template <class T> inline void __stcg(T* p, T v) { *p = v; }
inline void __threadfence() {}
inline void __threadfence_system() {}
inline void __nanosleep(unsigned) {}
inline long long clock64() { return 0; }
template <class T> inline T min(T a, T b) { return b < a ? b : a; }
template <class T> inline T max(T a, T b) { return a < b ? b : a; }
inline long long min(long long a, int b) { return b < a ? b : a; }
inline long long min(int a, long long b) { return b < a ? b : a; }
// shared-memory "addresses": 32-bit offsets from a fixed base below the library's static data
namespace cuda_emu {
inline char g_smem_anchor = 0;
inline uintptr_t smem_base() { return (uintptr_t)&g_smem_anchor - (1ull << 31); }
inline void* smem_ptr(unsigned addr) { return (void*)(smem_base() + addr); }
}  // namespace cuda_emu
inline size_t __cvta_generic_to_shared(const void* p) { return (size_t)((uintptr_t)p - cuda_emu::smem_base()); }
