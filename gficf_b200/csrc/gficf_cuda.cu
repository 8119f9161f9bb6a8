// gficf_cuda.cu -- C ABI (include/gficf_cuda.h) and host orchestration of the
// B200-native Jaccard path: device workspaces, H2D / D2H pipelines, kernel
// dispatch, multi-GPU row sharding over NCCL.
//
// Replaces the bodies of rcpp_parallel_jaccard_coef
// (reference src/rcpp_parallel_jaccard_coeff.cpp:58-80) and jaccard_coeff
// (src/jaccard_coeff.cpp:19-45).  There is deliberately no CPU fallback.
#include "gficf_cuda.h"  // include/gficf_cuda.h (-I)

#include <cuda_runtime.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "host_expand.h"
#include "host_stats.h"
#include "jaccard_kernels.cuh"
#include "snn_kernels.cuh"
#include "wmu_kernels.cuh"
#include "nccl_dyn.h"

namespace {

using namespace gficf;

// ------------------------------------------------------------------ errors
struct Err {
  int code = GFICF_OK;
  std::string msg;
};

void set_err(char* err, size_t errlen, const std::string& m) {
  if (err && errlen) {
    snprintf(err, errlen, "%s", m.c_str());
  }
}

std::string fmt(const char* f, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof buf, f, ap);
  va_end(ap);
  return buf;
}

#define CU_TRY(expr)                                                                   \
  do {                                                                                 \
    cudaError_t e_ = (expr);                                                           \
    if (e_ != cudaSuccess) {                                                           \
      throw Err{GFICF_E_CUDA, fmt("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                                  __FILE__, __LINE__)};                                \
    }                                                                                  \
  } while (0)

#define NCCL_TRY(expr)                                                                   \
  do {                                                                                   \
    ncclResult_t r_ = (expr);                                                            \
    if (r_ != ncclSuccess) {                                                             \
      throw Err{GFICF_E_NCCL, fmt("%s failed: %s (%s:%d)", #expr,                        \
                                  nccl_dyn::get().GetErrorString(r_), __FILE__, __LINE__)}; \
    }                                                                                    \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize of a kernel, set once per device and host thread
void set_max_dynamic_smem(const void* kernel, size_t bytes) {
  static thread_local std::vector<std::pair<const void*, int>> done;
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  const std::pair<const void*, int> key(kernel, dev);
  if (std::find(done.begin(), done.end(), key) != done.end()) return;
  CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  done.push_back(key);
}

}  // namespace

// the launch plans shared with the CPU emulation (they use CU_TRY, Err and set_max_dynamic_smem)
#include "jaccard_plan.h"
#include "network_plan.h"
#include "snn_plan.h"
#include "wmu_csc_plan.h"

namespace {

// ------------------------------------------------------------------ launch bookkeeping
thread_local LaunchInfo tl_launch;  // the last count kernel of this thread (gficf_cuda_last_launch)
thread_local double tl_timings[8] = {0, 0, 0, 0, 0, 0, 0, 0};
struct OutputInfo {
  int mode = 1;           // OutMode of the last host-buffer call
  double host_share = 0;  // share of the output pieces written by host threads
  double h2d_bytes = 0;   // bytes copied host -> device
};
thread_local OutputInfo tl_output;

struct DevProps {
  bool ok = false;
  int sms = 0;
};
DevProps g_props[64];
std::mutex g_mu;

int sm_count() {
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_mu);
  if (dev < 64 && g_props[dev].ok) return g_props[dev].sms;
  int sms = 0;
  CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (dev < 64) g_props[dev] = {true, sms};
  return sms;
}

// tl_cta_cap (> 0) lowers the resident CTAs per SM of the persistent kernels so that two of them on
// different streams can be resident side by side (gficf_cuda_set_launch_ctas_per_sm)
thread_local int tl_cta_cap = 0;

// bounded spins of the peer-memory kernels: GFICF_CUDA_PEER_TIMEOUT_MS (default 20 s) in SM clocks.
// The clock rate is queried once per device: cudaDevAttrClockRate is one of the attributes the
// driver answers slowly (milliseconds), and this sits on the launch path of every step.
long long peer_spin_clocks(long long timeout_ms) {
  static std::atomic<int> khz_cache[64];
  static std::atomic<long long> env_ms{-1};
  if (timeout_ms <= 0) {
    long long v = env_ms.load();
    if (v < 0) {
      const char* e = getenv("GFICF_CUDA_PEER_TIMEOUT_MS");
      v = e ? atoll(e) : 0;
      if (v <= 0) v = 20000;
      env_ms.store(v);
    }
    timeout_ms = v;
  }
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev));
  int khz = khz_cache[dev & 63].load();
  if (khz <= 0) {
    if (cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev) != cudaSuccess || khz <= 0) khz = 1965000;
    khz_cache[dev & 63].store(khz);
  }
  return timeout_ms * (long long)khz;
}

// the Jaccard plan on the current device and stream
JacCtx jac_ctx(cudaStream_t st) { return JacCtx{st, sm_count(), tl_cta_cap, &tl_launch}; }

// ------------------------------------------------------------------ per-device workspace
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  void need(size_t bytes) {
    if (bytes <= cap) return;
    if (p) CU_TRY(cudaFree(p));
    p = nullptr;
    cap = 0;
    CU_TRY(cudaMalloc(&p, bytes));
    cap = bytes;
  }
  void drop() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  void need(size_t bytes) {
    if (bytes <= cap) return;
    if (p) CU_TRY(cudaFreeHost(p));
    p = nullptr;
    cap = 0;
    CU_TRY(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
    cap = bytes;
  }
  void drop() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

constexpr int kMaxChunks = 32;
constexpr size_t kStageChunk = 4u << 20;  // pageable host memory moves in pieces of this size
constexpr int kStageSlots = 16;           // through a ring of pinned slots (64 MiB per device)
constexpr size_t kSmallCopyBytes = 8u << 20;  // below this, pageable copies go through the driver's own staging

struct DeviceWs {
  int dev = -1;
  bool init = false;
  cudaStream_t s_comp = nullptr, s_copy = nullptr;
  cudaEvent_t ev[8] = {};
  cudaEvent_t ev_chunk[kMaxChunks] = {};
  cudaEvent_t ev_k0[kMaxChunks] = {}, ev_k1[kMaxChunks] = {};
  // in_raw: device copy of the caller's rows (f64 or int32, column-major); small: flags + n_written
  Buf in_raw, idx, out, counts, scratch, small;
  PinBuf ring, h_counts;  // h_counts: the slab's 1-byte counts on the host (counts-over-PCIe output mode)
  cudaEvent_t ev_cnt_done = nullptr, ev_exp = nullptr, ev_dma[4] = {}, ev_ring = nullptr;
  bool ring_used = false;  // ev_ring marks the end of the last staged copy through `ring`
  cudaEvent_t ev_slot[kStageSlots] = {};
  unsigned* h_small = nullptr;  // pinned mirror of `small`

  void ensure(int d) {
    if (init) return;
    dev = d;
    CU_TRY(cudaSetDevice(dev));
    CU_TRY(cudaStreamCreateWithFlags(&s_comp, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&s_copy, cudaStreamNonBlocking));
    for (auto& e : ev) CU_TRY(cudaEventCreate(&e));
    for (auto& e : ev_chunk) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : ev_k0) CU_TRY(cudaEventCreate(&e));
    for (auto& e : ev_k1) CU_TRY(cudaEventCreate(&e));
    for (auto& e : ev_slot) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : ev_dma) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&ev_cnt_done, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&ev_exp, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&ev_ring, cudaEventDisableTiming));
    ring_used = false;
    small.need(64);
    CU_TRY(cudaHostAlloc((void**)&h_small, 64, cudaHostAllocDefault));
    init = true;
  }
  void release() {
    if (!init) return;
    cudaSetDevice(dev);
    cudaDeviceSynchronize();
    in_raw.drop(); idx.drop(); out.drop(); counts.drop(); scratch.drop(); small.drop();
    ring.drop();
    h_counts.drop();
    cudaEventDestroy(ev_cnt_done);
    cudaEventDestroy(ev_exp);
    cudaEventDestroy(ev_ring);
    for (auto& e : ev_dma) cudaEventDestroy(e);
    if (h_small) cudaFreeHost(h_small);
    h_small = nullptr;
    for (auto& e : ev) cudaEventDestroy(e);
    for (auto& e : ev_chunk) cudaEventDestroy(e);
    for (auto& e : ev_k0) cudaEventDestroy(e);
    for (auto& e : ev_k1) cudaEventDestroy(e);
    for (auto& e : ev_slot) cudaEventDestroy(e);
    cudaStreamDestroy(s_comp);
    cudaStreamDestroy(s_copy);
    init = false;
  }
};

constexpr int kMaxDevices = 16;
DeviceWs g_ws[kMaxDevices];
std::mutex g_call_mu;  // one host-level call at a time (workspaces are shared)
int g_default_devices = -1;

struct NcclState {
  int ndev = 0;
  ncclComm_t comms[kMaxDevices] = {};
} g_nccl;

std::atomic<int> g_sharers{1};  // ranks on this host (one process per GPU); they share its cores

// one process per GPU: the communicator built from a unique id the host framework distributes
struct MpState {
  ncclComm_t comm = nullptr;
  int nranks = 0, rank = 0, dev = 0;
} g_mp;

void mp_release() {
  if (g_mp.comm) nccl_dyn::get().CommDestroy(g_mp.comm);
  g_mp = MpState();
  g_sharers.store(1);
}

void nccl_release() {
  if (g_nccl.ndev) {
    for (int i = 0; i < g_nccl.ndev; ++i)
      if (g_nccl.comms[i]) nccl_dyn::get().CommDestroy(g_nccl.comms[i]);
    g_nccl = NcclState();
  }
}

void nccl_ensure(int ndev) {
  if (g_nccl.ndev == ndev) return;
  nccl_release();
  if (!nccl_dyn::get().ok) throw Err{GFICF_E_NCCL, "cannot load libnccl.so.2: " + nccl_dyn::get().why};
  int devs[kMaxDevices];
  for (int i = 0; i < ndev; ++i) devs[i] = i;
  NCCL_TRY(nccl_dyn::get().CommInitAll(g_nccl.comms, ndev, devs));
  g_nccl.ndev = ndev;
}

bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// ------------------------------------------------------------------ pageable host memory
// R hands over ordinary (pageable) memory.  cudaMemcpy on pageable memory is a single-threaded
// staging copy; here the transfer is cut into kStageChunk pieces that go through a ring of pinned
// slots, the host-side memcpy of the pieces is done by a few worker threads in parallel, and the
// DMA of piece j overlaps the memcpy of its neighbours.
struct Seg {
  char* host;
  char* dev;
  size_t bytes;
  cudaEvent_t wait_before;  // the copy stream waits for this event before the segment (or null)
};

std::atomic<int> g_active_devices{1};  // devices of the running host-level call (they share the cores)

int copy_threads() {
  static int t = [] {
    const char* e = getenv("GFICF_CUDA_COPY_THREADS");
    int v = e ? atoi(e) : 0;
    if (v <= 0) {
      // measured on a 16-thread host (4M x 30, pageable in/out, non-temporal copy-out): 2 threads
      // 183 ms, 4: 79, 6: 74, 8: 74, 12: 76, 16: 100 (pinned buffers: 72 ms)
      v = (int)std::thread::hardware_concurrency() / 2;
      v = std::max(2, std::min(8, v));
    }
    return v;
  }();
  return std::max(2, t / std::max(1, g_active_devices.load()));
}

// Device -> pageable host: the destination will not be read again soon, so the pieces are written
// with non-temporal stores (no read-for-ownership of the destination lines).
void copy_out(char* dst, const char* src, size_t bytes) { gficf_host::stream_copy(dst, src, bytes); }

// Threads that write the output columns from the 1-byte counts (counts-over-PCIe output mode).
// The devices / ranks of one call share the host's cores.
int expand_threads() {
  static int t = [] {
    const char* e = getenv("GFICF_CUDA_EXPAND_THREADS");
    int v = e ? atoi(e) : 0;
    if (v <= 0) v = std::max(2, std::min(32, (int)std::thread::hardware_concurrency() - 2));
    return v;
  }();
  return std::max(1, t / std::max(1, g_active_devices.load() * g_sharers.load()));
}

// How the (n*k) x 3 doubles of the parallel export reach the caller's matrix:
//   dma     the device writes all 24 B/edge and the copy engine moves them (r01 path)
//   host    only the 1-byte counts cross PCIe; host threads write the three columns (host_expand.h)
//   hybrid  both at once: (column, row-chunk) pieces are claimed from one list, the host threads from
//           the end that is cheapest for them (from, weight), the copy engine from the other (to)
//   auto    hybrid when the output buffer is page-locked, host when it is pageable (what R passes:
//           a staged DMA would cost the host a 24 B/edge read AND write), dma when k > 255
enum OutMode { kOutAuto = 0, kOutDma, kOutHost, kOutHybrid };
OutMode out_mode_env() {
  const char* e = getenv("GFICF_CUDA_OUT_MODE");
  if (!e) return kOutAuto;
  if (!strcmp(e, "dma")) return kOutDma;
  if (!strcmp(e, "host")) return kOutHost;
  if (!strcmp(e, "hybrid")) return kOutHybrid;
  return kOutAuto;
}

struct Piece {
  char* host;
  char* dev;
  size_t bytes;
  cudaEvent_t wait_before;
};

// narrow (host -> device only): the source holds ids as doubles; the workers convert every piece to
// int32 inside its pinned slot (gficf_host::f64_to_i32) and the copy engine moves HALF the bytes;
// Seg.bytes / Piece.bytes count SOURCE bytes, Seg.dev addresses the int32 destination.
void staged_copy(DeviceWs& ws, const std::vector<Seg>& segs, bool to_device, cudaStream_t st,
                 bool narrow = false) {
  std::vector<Piece> pieces;
  for (const Seg& g : segs) {
    bool first = true;
    for (size_t off = 0; off < g.bytes; off += kStageChunk) {
      pieces.push_back({g.host + off, g.dev + (narrow ? off / 2 : off), std::min(kStageChunk, g.bytes - off),
                        first ? g.wait_before : nullptr});
      first = false;
    }
  }
  const int np = (int)pieces.size();
  if (!np) return;
  // the ring may still be the source / target of DMAs queued by the previous staged copy of this
  // device (two matrices uploaded back to back): wait until those have drained
  if (ws.ring_used) CU_TRY(cudaEventSynchronize(ws.ev_ring));
  ws.ring.need(kStageChunk * kStageSlots);
  char* ring = (char*)ws.ring.p;
  std::vector<std::atomic<int>> host_done(np), dma_issued(np);
  for (int j = 0; j < np; ++j) {
    host_done[j].store(0);
    dma_issued[j].store(0);
  }
  std::atomic<int> next(0);
  std::atomic<bool> failed(false);
  const int dev = ws.dev;
  const int nthreads = std::min(narrow ? expand_threads() : copy_threads(), np);
  auto worker = [&]() {
    cudaSetDevice(dev);
    for (;;) {
      const int j = next.fetch_add(1);
      if (j >= np || failed.load()) return;
      const Piece& pc = pieces[j];
      char* slot = ring + (size_t)(j % kStageSlots) * kStageChunk;
      if (to_device) {
        // the slot is free once the DMA of piece j - kStageSlots has completed
        if (j >= kStageSlots) {
          while (!dma_issued[j - kStageSlots].load(std::memory_order_acquire)) {
            if (failed.load()) return;
            std::this_thread::yield();
          }
          if (cudaEventSynchronize(ws.ev_slot[j % kStageSlots]) != cudaSuccess) failed.store(true);
        }
        if (narrow) gficf_host::f64_to_i32((const double*)pc.host, (int32_t*)slot, pc.bytes / 8);
        else memcpy(slot, pc.host, pc.bytes);
        host_done[j].store(1, std::memory_order_release);
      } else {
        while (!dma_issued[j].load(std::memory_order_acquire)) {
          if (failed.load()) return;
          std::this_thread::yield();
        }
        if (cudaEventSynchronize(ws.ev_slot[j % kStageSlots]) != cudaSuccess) failed.store(true);
        copy_out(pc.host, slot, pc.bytes);
        host_done[j].store(1, std::memory_order_release);
      }
    }
  };
  std::vector<std::thread> pool;
  for (int t = 0; t < nthreads; ++t) pool.emplace_back(worker);
  cudaError_t err = cudaSuccess;
  for (int j = 0; j < np && err == cudaSuccess; ++j) {
    const Piece& pc = pieces[j];
    char* slot = ring + (size_t)(j % kStageSlots) * kStageChunk;
    if (pc.wait_before) err = cudaStreamWaitEvent(st, pc.wait_before, 0);
    // a worker that failed stops marking pieces: never wait for it (failed ends the loop below)
    if (to_device) {
      while (!host_done[j].load(std::memory_order_acquire) && !failed.load()) std::this_thread::yield();
      if (failed.load()) break;
      if (err == cudaSuccess)
        err = cudaMemcpyAsync(pc.dev, slot, narrow ? pc.bytes / 2 : pc.bytes, cudaMemcpyHostToDevice, st);
    } else {
      // the slot is free once piece j - kStageSlots has been copied out by a worker
      if (j >= kStageSlots)
        while (!host_done[j - kStageSlots].load(std::memory_order_acquire) && !failed.load())
          std::this_thread::yield();
      if (failed.load()) break;
      if (err == cudaSuccess) err = cudaMemcpyAsync(slot, pc.dev, pc.bytes, cudaMemcpyDeviceToHost, st);
    }
    if (err == cudaSuccess) err = cudaEventRecord(ws.ev_slot[j % kStageSlots], st);
    dma_issued[j].store(1, std::memory_order_release);
  }
  if (err != cudaSuccess || failed.load()) {
    failed.store(true);
    for (int j = 0; j < np; ++j) {
      dma_issued[j].store(1);
      host_done[j].store(1);
    }
  }
  for (auto& t : pool) t.join();
  if (err == cudaSuccess && cudaEventRecord(ws.ev_ring, st) == cudaSuccess) ws.ring_used = true;
  if (err != cudaSuccess || failed.load())
    throw Err{GFICF_E_CUDA, fmt("staged host copy failed: %s", cudaGetErrorString(err))};
}

// Host -> device of a strided 2-D block (rows x cols doubles, source leading dimension ld_src,
// destination dense with leading dimension rows).  Pinned sources go straight to the copy
// engine; pageable ones through staged_copy.
// Returns the element size of the device copy: an f64 matrix above kSmallCopyBytes arrives as int32
// (narrowed on the host while it streams: half the PCIe bytes), everything else as it is.
bool h2d_narrow_enabled() {
  const char* e = getenv("GFICF_CUDA_H2D_NARROW");
  return !(e && e[0] == '0');
}

size_t h2d_block(DeviceWs& ws, const void* src_v, long long ld_src, void* dst_v, long long rows, int cols,
                 size_t elem, cudaStream_t st, bool ids = true) {
  if (rows <= 0 || cols <= 0) return elem;
  const char* src = (const char*)src_v;
  char* dst = (char*)dst_v;
  const bool small = (size_t)rows * cols * elem <= kSmallCopyBytes;
  // narrowing trades host memory traffic (read 8 + write 4 + DMA read 4 bytes per id instead of a DMA
  // read of 8) for PCIe bytes: a win while ONE link is the bottleneck, a loss when several GPUs'
  // links together outrun the host's memory (measured at 8 ranks: 12.4 ms instead of ~3)
  if (ids && elem == 8 && !small && h2d_narrow_enabled() && g_active_devices.load() * g_sharers.load() == 1) {
    std::vector<Seg> segs;
    for (int c = 0; c < cols; ++c)
      segs.push_back({(char*)(src + (size_t)c * ld_src * 8), dst + (size_t)c * rows * 4, (size_t)rows * 8, nullptr});
    staged_copy(ws, segs, true, st, true);
    return 4;
  }
  if (is_pinned(src) || small) {
    // pinned: straight to the copy engine; small: the driver's own staging beats spinning up threads
    CU_TRY(cudaMemcpy2DAsync(dst, rows * elem, src, ld_src * elem, rows * elem, cols, cudaMemcpyHostToDevice,
                             st));
    return elem;
  }
  std::vector<Seg> segs;
  for (int c = 0; c < cols; ++c)
    segs.push_back({(char*)(src + (size_t)c * ld_src * elem), dst + (size_t)c * rows * elem,
                    (size_t)rows * elem, nullptr});
  staged_copy(ws, segs, true, st);
  return elem;
}

// Device -> host of contiguous runs (each optionally behind an event).  Pinned destinations:
// plain async copies; pageable ones: staged_copy.
void d2h_segs(DeviceWs& ws, const std::vector<Seg>& segs, cudaStream_t st) {
  if (segs.empty()) return;
  size_t total = 0;
  for (const Seg& g : segs) total += g.bytes;
  if (is_pinned(segs[0].host) || total <= kSmallCopyBytes) {
    for (const Seg& g : segs) {
      if (g.wait_before) CU_TRY(cudaStreamWaitEvent(st, g.wait_before, 0));
      if (g.bytes) CU_TRY(cudaMemcpyAsync(g.host, g.dev, g.bytes, cudaMemcpyDeviceToHost, st));
    }
    return;
  }
  staged_copy(ws, segs, false, st);
}

struct SlabResult {
  unsigned flags = 0;
  long long n_written = -1;
  float ms_h2d = 0, ms_k0 = 0, ms_k1 = 0, ms_d2h = 0, ms_gather = 0;
  int launches = 0;
  double d2h_bytes = 0;       // bytes that crossed PCIe towards the host
  double h2d_bytes = 0;       // ... and towards the device
  int out_mode = kOutDma;     // how the output columns were produced (OutMode)
  double host_items = 0;      // share of the output pieces written by host threads
  bool counts_ready = false;  // phase 1 left fast-kernel counts in ws.counts
  Err err;
};

struct Slab {
  int rank, ndev, k, kp, mode;
  int dev;                    // CUDA device ordinal (== rank inside one process)
  ncclComm_t comm = nullptr;  // communicator of this rank when ndev > 1
  long long n, rows_per, lo, hi, rows, E, slab_e;
  const void* h_idx;
  int elem = 8;  // bytes per element of the caller's matrix: 8 = double, 4 = int32
  int out_mode = kOutDma;  // resolved OutMode of this call (never kOutAuto)
  double* h_out;
  Slab(int rank_, int ndev_, const void* h_idx_, long long n_, int k_, long long rows_per_,
       double* h_out_, int mode_)
      : rank(rank_), ndev(ndev_), k(k_), kp(row_stride(k_)), mode(mode_), dev(rank_), n(n_),
        rows_per(rows_per_), h_idx(h_idx_), h_out(h_out_) {
    lo = std::min<long long>(n, rank * rows_per);
    hi = std::min<long long>(n, lo + rows_per);
    rows = hi - lo;
    E = n * (long long)k;
    slab_e = rows * (long long)k;
  }
};

void read_small(DeviceWs& ws, SlabResult* res) {
  CU_TRY(cudaMemcpyAsync(ws.h_small, ws.small.p, 16, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaStreamSynchronize(ws.s_comp));
  res->flags |= ws.h_small[0];
}

void d2h_slab(DeviceWs& ws, const Slab& s, SlabResult* res) {
  double* d_from = (double*)ws.out.p;
  double* d_to = d_from + s.slab_e;
  double* d_w = d_to + s.slab_e;
  CU_TRY(cudaEventRecord(ws.ev[4], ws.s_copy));
  const size_t bytes = (size_t)s.slab_e * sizeof(double);
  d2h_segs(ws,
           {{(char*)(s.h_out + s.lo * s.k), (char*)d_from, bytes, nullptr},
            {(char*)(s.h_out + s.E + s.lo * s.k), (char*)d_to, bytes, nullptr},
            {(char*)(s.h_out + 2 * s.E + s.lo * s.k), (char*)d_w, bytes, nullptr}},
           ws.s_copy);
  CU_TRY(cudaEventRecord(ws.ev[5], ws.s_copy));
  CU_TRY(cudaStreamSynchronize(ws.s_copy));
  float ms = 0;
  CU_TRY(cudaEventElapsedTime(&ms, ws.ev[4], ws.ev[5]));
  res->ms_d2h += ms;
}

// Counts-over-PCIe output of the parallel export (modes host / hybrid, see OutMode).
// On entry: ws.counts holds the slab's 1-byte counts and their D2H into ws.h_counts is in flight on
// s_copy (ev_cnt_done behind it); with use_dma, ws.out holds the expanded doubles (ev_exp on s_comp).
// The slab's output is cut into (column, row-chunk) pieces kept in ONE list ordered by what the host
// threads do cheapest: from (no input read), weight (table lookup), to (transposed read of the
// caller's matrix).  Host threads claim from the front, the copy engine from the back; the call is
// over when the two ends meet -- the split adapts to whatever the host's memory system and the
// PCIe link deliver, nothing is calibrated.
void counts_output_phase(DeviceWs& ws, const Slab& s, SlabResult* res, bool use_dma) {
  const int k = s.k;
  const long long rows_per_piece = std::max<long long>(256, (6ll << 20) / (8ll * k));
  const long long nc = (s.rows + rows_per_piece - 1) / rows_per_piece;
  const long long nitems = 3 * nc;
  static const int kCpuOrder[3] = {0, 2, 1};
  std::atomic<unsigned long long> ends((unsigned long long)nitems);  // front in the high 32 bits, back in the low
  auto claim = [&](bool front, long long* item) {
    unsigned long long v = ends.load();
    for (;;) {
      const unsigned long long lo = v >> 32, hi = v & 0xffffffffull;
      if (lo >= hi) return false;
      const unsigned long long nv = front ? (((lo + 1) << 32) | hi) : ((lo << 32) | (hi - 1));
      if (ends.compare_exchange_weak(v, nv)) {
        *item = (long long)(front ? lo : hi - 1);
        return true;
      }
    }
  };
  double lut[256];
  gficf_host::fill_weight_table(k, lut);
  gficf_host::ExpandJob job{s.h_idx, s.elem, s.n, k, (const uint8_t*)ws.h_counts.p, s.lo, s.h_out, s.E, lut};
  CU_TRY(cudaEventSynchronize(ws.ev_cnt_done));  // the counts are on the host
  const int nthreads = (int)std::min<long long>(expand_threads(), nitems);
  std::vector<std::thread> pool;
  std::atomic<long long> cpu_items(0);
  for (int t = 0; t < nthreads; ++t)
    pool.emplace_back([&] {
      long long it;
      while (claim(true, &it)) {
        const int col = kCpuOrder[it / nc];
        const long long a = (it % nc) * rows_per_piece, b = std::min(s.rows, a + rows_per_piece);
        gficf_host::expand_column(job, col, s.lo + a, s.lo + b);
        cpu_items.fetch_add(1);
      }
    });
  cudaError_t err = cudaSuccess;
  long long dma_items = 0;
  if (use_dma) {
    const double* d_out = (const double*)ws.out.p;
    err = cudaStreamWaitEvent(ws.s_copy, ws.ev_exp, 0);
    long long it;
    // at most 3 copies queued: the copy engine never idles, and it never claims far ahead of what it moves
    while (err == cudaSuccess && claim(false, &it)) {
      const int col = kCpuOrder[it / nc];
      const long long a = (it % nc) * rows_per_piece, b = std::min(s.rows, a + rows_per_piece);
      const size_t bytes = (size_t)(b - a) * k * sizeof(double);
      if (dma_items >= 3) err = cudaEventSynchronize(ws.ev_dma[(dma_items - 3) & 3]);
      if (err == cudaSuccess)
        err = cudaMemcpyAsync(s.h_out + (size_t)col * s.E + (size_t)(s.lo + a) * k,
                              d_out + (size_t)col * s.slab_e + (size_t)a * k, bytes, cudaMemcpyDeviceToHost,
                              ws.s_copy);
      if (err == cudaSuccess) err = cudaEventRecord(ws.ev_dma[dma_items & 3], ws.s_copy);
      res->d2h_bytes += (double)bytes;
      ++dma_items;
    }
  }
  for (auto& t : pool) t.join();
  if (err == cudaSuccess) err = cudaStreamSynchronize(ws.s_copy);
  if (err != cudaSuccess) throw Err{GFICF_E_CUDA, fmt("output copy failed: %s", cudaGetErrorString(err))};
  res->out_mode = use_dma ? kOutHybrid : kOutHost;
  res->host_items = (double)cpu_items.load() / (double)std::max<long long>(1, nitems);
}

// Phase 1 of one device's share (rows [lo,hi) of n): H2D of its rows, layout pre-pass, exchange
// of the int32 index slabs (in-place NCCL all-gather when ndev>1), then the fast kernel:
//   parallel export, k<=128: fused kernel in row chunks, the D2H of chunk c overlapping the
//     kernel of chunk c+1 (the result stands unless some device raises a dup/hash flag);
//   serial export, k<=128:   fast count kernel (the compaction happens in phase 2).
// Phase 0: everything that can fail locally -- workspaces, H2D of the device's rows, layout
// pre-pass.  No collective in here: if any device fails, the call ends before anybody enters the
// all-gather (a collective that one participant never joins would hang the others' GPUs).
void device_phase0(Slab s, SlabResult* res) {
  try {
    DeviceWs& ws = g_ws[s.dev];
    CU_TRY(cudaSetDevice(s.dev));
    ws.ensure(s.dev);
    const int k = s.k;
    const int cbytes = k <= 255 ? 1 : 2;
    ws.in_raw.need(std::max<size_t>(16, (size_t)s.rows * k * s.elem));
    ws.idx.need(std::max<size_t>(16, (size_t)s.rows_per * s.ndev * s.kp * sizeof(int)));
    if (s.out_mode != kOutHost) ws.out.need(std::max<size_t>(16, (size_t)s.slab_e * 3 * sizeof(double)));
    if (s.mode == GFICF_MODE_SERIAL || k > kLargeMaxK || s.out_mode != kOutDma) {
      ws.counts.need(std::max<size_t>(16, (size_t)s.slab_e * cbytes));
      ws.scratch.need(expand_scratch_bytes(s.slab_e));
    }
    if (s.out_mode != kOutDma) ws.h_counts.need(std::max<size_t>(16, (size_t)s.slab_e));
    if (s.out_mode == kOutHost) ws.out.need(16);  // grown on demand should the exact path be needed
    unsigned* d_flags = (unsigned*)ws.small.p;
    CU_TRY(cudaMemsetAsync(ws.small.p, 0, 64, ws.s_comp));
    CU_TRY(cudaEventRecord(ws.ev[0], ws.s_comp));
    const size_t dev_elem = h2d_block(ws, (const char*)s.h_idx + (size_t)s.lo * s.elem, s.n, ws.in_raw.p,
                                      s.rows, k, s.elem, ws.s_comp);
    res->h2d_bytes = (double)s.rows * k * dev_elem;
    CU_TRY(cudaEventRecord(ws.ev[1], ws.s_comp));
    if (dev_elem == 8)
      launch_layout(jac_ctx(ws.s_comp), (const double*)ws.in_raw.p, s.rows, s.lo, s.n, k, s.lo, s.hi,
                    (int*)ws.idx.p, d_flags);
    else
      launch_layout(jac_ctx(ws.s_comp), (const int*)ws.in_raw.p, s.rows, s.lo, s.n, k, s.lo, s.hi, (int*)ws.idx.p,
                    d_flags);
    res->launches += s.rows > 0;
    CU_TRY(cudaEventRecord(ws.ev[2], ws.s_comp));
  } catch (const Err& e) {
    res->err = e;
  }
}

void device_phase1(Slab s, SlabResult* res) {
  try {
    DeviceWs& ws = g_ws[s.dev];
    CU_TRY(cudaSetDevice(s.dev));
    const int k = s.k;
    const int cbytes = k <= 255 ? 1 : 2;
    unsigned* d_flags = (unsigned*)ws.small.p;
    if (s.ndev > 1) {
      const size_t cnt = (size_t)s.rows_per * s.kp;
      NCCL_TRY(nccl_dyn::get().AllGather((const char*)ws.idx.p + (size_t)s.rank * cnt * sizeof(int),
                                         ws.idx.p, cnt, ncclInt32, s.comm, ws.s_comp));
    }
    CU_TRY(cudaEventRecord(ws.ev[3], ws.s_comp));

    const int* d_idx = (const int*)ws.idx.p;
    const bool fast_ok = k <= kLargeMaxK;
    double* d_from = (double*)ws.out.p;
    double* d_to = d_from + s.slab_e;
    double* d_w = d_to + s.slab_e;
    int used = 0;
    if (fast_ok && s.mode == GFICF_MODE_PARALLEL && s.out_mode != kOutDma && s.slab_e > 0) {
      // counts-over-PCIe: count kernel in row chunks, the D2H of chunk c's counts overlapping the
      // kernel of chunk c+1; then the output phase (host threads [+ copy engine])
      const bool use_dma = s.out_mode == kOutHybrid;
      const int nch = (int)std::min<long long>(8, std::max<long long>(1, s.slab_e / (8ll << 20)));
      const long long rpc = (s.rows + nch - 1) / nch;
      uint8_t* d_cnt = (uint8_t*)ws.counts.p;
      CU_TRY(cudaStreamWaitEvent(ws.s_copy, ws.ev[3], 0));
      for (int c = 0; c < nch; ++c) {
        const long long clo = s.lo + c * rpc, chi = std::min(s.hi, clo + rpc);
        if (clo >= chi) break;
        const long long eo = (clo - s.lo) * k;
        CU_TRY(cudaEventRecord(ws.ev_k0[c], ws.s_comp));
        launch_fast<1>(jac_ctx(ws.s_comp), d_idx, k, clo, chi, nullptr, nullptr, nullptr, d_cnt + eo, d_flags);
        CU_TRY(cudaEventRecord(ws.ev_k1[c], ws.s_comp));
        CU_TRY(cudaEventRecord(ws.ev_chunk[c], ws.s_comp));
        CU_TRY(cudaStreamWaitEvent(ws.s_copy, ws.ev_chunk[c], 0));
        CU_TRY(cudaMemcpyAsync((char*)ws.h_counts.p + eo, d_cnt + eo, (size_t)(chi - clo) * k,
                               cudaMemcpyDeviceToHost, ws.s_copy));
        res->launches++;
        used = c + 1;
      }
      CU_TRY(cudaEventRecord(ws.ev_cnt_done, ws.s_copy));
      res->d2h_bytes += (double)s.slab_e;
      if (use_dma) {
        launch_expand(jac_ctx(ws.s_comp), d_idx, k, s.lo, s.hi, d_cnt, false, d_from, d_to, d_w, nullptr, nullptr);
        res->launches++;
      }
      CU_TRY(cudaEventRecord(ws.ev_exp, ws.s_comp));
      read_small(ws, res);  // flags of the count kernels (waits for s_comp)
      res->counts_ready = true;
      const auto t_out0 = std::chrono::steady_clock::now();
      if (!(res->flags & (kFlagBadId | kFlagDupId | kFlagHashFail)))
        counts_output_phase(ws, s, res, use_dma);  // else: the exact path rewrites everything
      res->ms_d2h = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_out0).count();
      CU_TRY(cudaStreamSynchronize(ws.s_copy));
      CU_TRY(cudaEventElapsedTime(&res->ms_h2d, ws.ev[0], ws.ev[1]));
      CU_TRY(cudaEventElapsedTime(&res->ms_k0, ws.ev[1], ws.ev[2]));
      CU_TRY(cudaEventElapsedTime(&res->ms_gather, ws.ev[2], ws.ev[3]));
      for (int c = 0; c < used; ++c) {
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, ws.ev_k0[c], ws.ev_k1[c]));
        res->ms_k1 += ms;
      }
      return;
    }
    if (fast_ok && s.mode == GFICF_MODE_PARALLEL) {
      const int nch =
          (int)std::min<long long>(kMaxChunks, std::max<long long>(1, s.slab_e * 24 / (48ll << 20)));
      const long long rpc = (s.rows + nch - 1) / nch;
      for (int c = 0; c < nch; ++c) {
        const long long clo = s.lo + c * rpc, chi = std::min(s.hi, clo + rpc);
        if (clo >= chi) break;
        const long long eo = (clo - s.lo) * k;
        CU_TRY(cudaEventRecord(ws.ev_k0[c], ws.s_comp));
        launch_fast<0>(jac_ctx(ws.s_comp), d_idx, k, clo, chi, d_from + eo, d_to + eo, d_w + eo, nullptr, d_flags);
        CU_TRY(cudaEventRecord(ws.ev_k1[c], ws.s_comp));
        CU_TRY(cudaEventRecord(ws.ev_chunk[c], ws.s_comp));
        res->launches++;
        used = c + 1;
      }
      CU_TRY(cudaStreamWaitEvent(ws.s_copy, ws.ev[3], 0));
      CU_TRY(cudaEventRecord(ws.ev[4], ws.s_copy));
      std::vector<Seg> segs;
      for (int c = 0; c < used; ++c) {
        const long long clo = s.lo + c * rpc, chi = std::min(s.hi, clo + rpc);
        const long long eo = (clo - s.lo) * k;
        const size_t cb = (size_t)(chi - clo) * k * sizeof(double);
        segs.push_back({(char*)(s.h_out + s.lo * k + eo), (char*)(d_from + eo), cb, ws.ev_chunk[c]});
        segs.push_back({(char*)(s.h_out + s.E + s.lo * k + eo), (char*)(d_to + eo), cb, nullptr});
        segs.push_back({(char*)(s.h_out + 2 * s.E + s.lo * k + eo), (char*)(d_w + eo), cb, nullptr});
      }
      d2h_segs(ws, segs, ws.s_copy);
      res->d2h_bytes += 24.0 * (double)s.slab_e;
      CU_TRY(cudaEventRecord(ws.ev[5], ws.s_copy));
    } else if (fast_ok && s.slab_e > 0) {
      ws.counts.need(std::max<size_t>(16, (size_t)s.slab_e * cbytes));
      CU_TRY(cudaEventRecord(ws.ev_k0[0], ws.s_comp));
      launch_fast<1>(jac_ctx(ws.s_comp), d_idx, k, s.lo, s.hi, nullptr, nullptr, nullptr, ws.counts.p, d_flags);
      CU_TRY(cudaEventRecord(ws.ev_k1[0], ws.s_comp));
      res->launches++;
      res->counts_ready = true;
    }
    read_small(ws, res);
    CU_TRY(cudaStreamSynchronize(ws.s_copy));
    CU_TRY(cudaEventElapsedTime(&res->ms_h2d, ws.ev[0], ws.ev[1]));
    CU_TRY(cudaEventElapsedTime(&res->ms_k0, ws.ev[1], ws.ev[2]));
    CU_TRY(cudaEventElapsedTime(&res->ms_gather, ws.ev[2], ws.ev[3]));
    for (int c = 0; c < std::max(used, res->counts_ready ? 1 : 0); ++c) {
      float ms = 0;
      CU_TRY(cudaEventElapsedTime(&ms, ws.ev_k0[c], ws.ev_k1[c]));
      res->ms_k1 += ms;
    }
    if (used) CU_TRY(cudaEventElapsedTime(&res->ms_d2h, ws.ev[4], ws.ev[5]));
  } catch (const Err& e) {
    res->err = e;
  }
}

// Phase 2 (only when needed): counts -> expand -> D2H.  `exact` is decided from the flags of
// ALL devices: a row with a repeated id invalidates the fast count of every edge that targets
// it, whichever device owns that edge.
void device_phase2(Slab s, bool exact, SlabResult* res) {
  try {
    DeviceWs& ws = g_ws[s.dev];
    CU_TRY(cudaSetDevice(s.dev));
    if (s.slab_e <= 0) return;
    const int k = s.k;
    const int cbytes = k <= 255 ? 1 : 2;
    const int* d_idx = (const int*)ws.idx.p;
    ws.out.need(std::max<size_t>(16, (size_t)s.slab_e * 3 * sizeof(double)));  // host mode kept it empty
    double* d_from = (double*)ws.out.p;
    double* d_to = d_from + s.slab_e;
    double* d_w = d_to + s.slab_e;
    long long* d_nw = (long long*)((char*)ws.small.p + 8);
    ws.counts.need(std::max<size_t>(16, (size_t)s.slab_e * cbytes));
    ws.scratch.need(expand_scratch_bytes(s.slab_e));
    CU_TRY(cudaEventRecord(ws.ev[6], ws.s_comp));
    if (exact || !res->counts_ready) {
      launch_exact(jac_ctx(ws.s_comp), d_idx, k, s.lo, s.hi, s.mode == GFICF_MODE_SERIAL ? 1 : 0, ws.counts.p);
      res->launches++;
    }
    launch_expand(jac_ctx(ws.s_comp), d_idx, k, s.lo, s.hi, ws.counts.p, s.mode == GFICF_MODE_SERIAL, d_from, d_to,
                  d_w, ws.scratch.p, d_nw);
    res->launches += s.mode == GFICF_MODE_SERIAL ? 4 : 1;
    CU_TRY(cudaEventRecord(ws.ev[7], ws.s_comp));
    read_small(ws, res);
    if (s.mode == GFICF_MODE_SERIAL) res->n_written = *(long long*)((char*)ws.h_small + 8);
    float ms = 0;
    CU_TRY(cudaEventElapsedTime(&ms, ws.ev[6], ws.ev[7]));
    res->ms_k1 += ms;
    d2h_slab(ws, s, res);
  } catch (const Err& e) {
    res->err = e;
  }
}

// OutMode of a host-buffer call (never kOutAuto): the counts-over-PCIe modes need 1-byte counts and
// the fixed-slot export; the copy engine can only take part when the output buffer is page-locked
int resolve_out_mode(const double* out, int k, int mode) {
  if (mode != GFICF_MODE_PARALLEL || k > 255) return kOutDma;
  OutMode m = out_mode_env();
  if (m == kOutDma) return kOutDma;
  const bool pinned = is_pinned(out);
  if (m == kOutAuto) return pinned ? kOutHybrid : kOutHost;
  if (m == kOutHybrid && !pinned) return kOutHost;
  return m;
}

int visible_devices() {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return c;
}

int default_devices() {
  if (g_default_devices < 0) {
    const char* e = getenv("GFICF_CUDA_DEVICES");
    int v = e ? atoi(e) : 1;
    g_default_devices = v >= 1 ? v : 1;
  }
  return g_default_devices;
}

}  // namespace

// ============================================================================
// C ABI
// ============================================================================
#define API_BEGIN try {
#define API_END                                \
  }                                            \
  catch (const Err& e) {                       \
    set_err(err, errlen, e.msg);               \
    return e.code;                             \
  }                                            \
  catch (const std::exception& e) {            \
    set_err(err, errlen, e.what());            \
    return GFICF_E_CUDA;                       \
  }                                            \
  catch (...) {                                \
    set_err(err, errlen, "unknown failure");   \
    return GFICF_E_CUDA;                       \
  }

extern "C" {

const char* gficf_cuda_version(void) { return "gficf_cuda 0.1 (sm_100a; CUDA " __DATE__ ")"; }

int32_t gficf_cuda_row_stride(int32_t k) { return k < 1 ? 0 : row_stride(k); }

int gficf_cuda_device_count(void) { return visible_devices(); }

int gficf_cuda_set_devices(int32_t n_devices) {
  if (n_devices < 1 || n_devices > kMaxDevices) return GFICF_E_ARG;
  g_default_devices = n_devices;
  return GFICF_OK;
}

int gficf_cuda_get_devices(void) { return default_devices(); }

int gficf_cuda_host_alloc(void** p, size_t bytes) {
  if (!p) return GFICF_E_ARG;
  *p = nullptr;
  if (cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_host_free(void* p) {
  if (!p) return GFICF_OK;
  if (cudaFreeHost(p) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_host_register(void* p, size_t bytes) {
  if (!p || !bytes) return GFICF_E_ARG;
  if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_host_unregister(void* p) {
  if (!p) return GFICF_OK;
  if (cudaHostUnregister(p) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_release(void) {
  std::lock_guard<std::mutex> lk(g_call_mu);
  nccl_release();
  mp_release();
  for (auto& w : g_ws) w.release();
  return GFICF_OK;
}

int gficf_cuda_last_timings(double* ms8) {
  if (!ms8) return GFICF_E_ARG;
  memcpy(ms8, tl_timings, sizeof tl_timings);
  return GFICF_OK;
}

int gficf_cuda_last_output(int32_t* out_mode, double* host_share, double* d2h_bytes, double* h2d_bytes) {
  if (out_mode) *out_mode = tl_output.mode;
  if (host_share) *host_share = tl_output.host_share;
  if (d2h_bytes) *d2h_bytes = tl_timings[7];
  if (h2d_bytes) *h2d_bytes = tl_output.h2d_bytes;
  return GFICF_OK;
}

int gficf_cuda_expand_host(const void* idx_colmajor, int32_t elem_bytes, int64_t n, int32_t k,
                           const uint8_t* counts, int64_t row_lo, int64_t row_hi, double* out_colmajor,
                           int32_t n_threads) {
  if (!idx_colmajor || !counts || !out_colmajor || (elem_bytes != 8 && elem_bytes != 4) || n < 0 || k < 1 ||
      k > 255 || row_lo < 0 || row_hi > n || row_hi < row_lo)
    return GFICF_E_ARG;
  double lut[256];
  gficf_host::fill_weight_table(k, lut);
  const gficf_host::ExpandJob job{idx_colmajor, elem_bytes, (long long)n, k, counts, (long long)row_lo,
                                  out_colmajor, (long long)n * k, lut};
  const long long rows = row_hi - row_lo;
  const int nt = (int)std::max<long long>(1, std::min<long long>(n_threads > 0 ? n_threads : expand_threads(),
                                                                 (rows + 4095) / 4096));
  if (nt == 1) {
    gficf_host::expand_rows(job, row_lo, row_hi);
    return GFICF_OK;
  }
  std::atomic<long long> next(row_lo);
  std::vector<std::thread> pool;
  for (int t = 0; t < nt; ++t)
    pool.emplace_back([&] {
      for (;;) {
        const long long a = next.fetch_add(4096);
        if (a >= row_hi) return;
        gficf_host::expand_rows(job, a, std::min<long long>(row_hi, a + 4096));
      }
    });
  for (auto& t : pool) t.join();
  return GFICF_OK;
}

int gficf_cuda_set_launch_ctas_per_sm(int32_t ctas_per_sm) {
  if (ctas_per_sm < 0) return GFICF_E_ARG;
  tl_cta_cap = ctas_per_sm;
  return GFICF_OK;
}

int gficf_cuda_last_launch(int32_t* grid, int32_t* block, int32_t* smem_bytes, int32_t* variant) {
  if (grid) *grid = tl_launch.grid;
  if (block) *block = tl_launch.block;
  if (smem_bytes) *smem_bytes = tl_launch.smem;
  if (variant) *variant = tl_launch.variant;
  return GFICF_OK;
}

}  // extern "C"

namespace {
// The caller's current device, made current again when a host-level call ends, whichever way it ends.
struct DeviceRestore {
  int dev = -1;
  DeviceRestore() {
    if (cudaGetDevice(&dev) != cudaSuccess) {
      cudaGetLastError();
      dev = -1;
    }
  }
  ~DeviceRestore() {
    if (dev >= 0) cudaSetDevice(dev);
  }
};

float event_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0;
  CU_TRY(cudaEventElapsedTime(&ms, a, b));
  return ms;
}

// One single-device host-buffer call: a device must be visible; the call holds g_call_mu and runs on device 0
// with its workspace ready, and the caller's device is current again when it ends.
struct SingleDeviceCall {
  std::unique_lock<std::mutex> lk;
  DeviceRestore restore;
  DeviceWs& ws = g_ws[0];
  std::chrono::steady_clock::time_point t0;
  SingleDeviceCall() {
    if (visible_devices() < 1) throw Err{GFICF_E_CUDA, "no CUDA device is visible (this path has no CPU fallback)"};
    lk = std::unique_lock<std::mutex>(g_call_mu);
    t0 = std::chrono::steady_clock::now();
    CU_TRY(cudaSetDevice(0));
    ws.ensure(0);
    g_active_devices.store(1);
  }
  // gficf_cuda_last_timings: the four phase times, the wall time of the call, launches and bytes copied back
  void timings(double h2d_ms, double k0_ms, double k1_ms, double d2h_ms, double launches, double d2h_bytes) {
    const double wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    const double tm[8] = {h2d_ms, k0_ms, k1_ms, d2h_ms, wall, 0, launches, d2h_bytes};
    memcpy(tl_timings, tm, sizeof tm);
  }
};

int jaccard_host_call(const void* idx, int elem, int64_t n, int32_t k, double* out, int32_t n_devices,
                      int32_t mode, int64_t* n_written, char* err, size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  if (n < 0 || k < 0) throw Err{GFICF_E_ARG, "negative matrix dimension"};
  if (mode != GFICF_MODE_PARALLEL && mode != GFICF_MODE_SERIAL)
    throw Err{GFICF_E_ARG, "mode must be 0 (parallel, fixed slots) or 1 (serial, compacted)"};
  if (n_written) *n_written = 0;
  if (n == 0 || k == 0) return GFICF_OK;
  if (!idx || !out) throw Err{GFICF_E_ARG, "null matrix pointer"};
  // the reference holds rows and nrow*ncol in `int` (rcpp_parallel_jaccard_coeff.cpp:28,67)
  if (n >= 0x7fffffffLL - 2 || (long double)n * k >= 2147483647.0L)
    throw Err{GFICF_E_LIMIT, "n*k must stay below 2^31 (the reference's int row index)"};
  if (k > 65535) throw Err{GFICF_E_LIMIT, "k above 65535 is not supported"};
  int ndev = n_devices > 0 ? n_devices : default_devices();
  const int vis = visible_devices();
  if (vis < 1) throw Err{GFICF_E_CUDA, "no CUDA device is visible (this path has no CPU fallback)"};
  if (ndev > vis)
    throw Err{GFICF_E_ARG, fmt("%d devices requested but only %d visible", ndev, vis)};
  if (ndev > kMaxDevices) throw Err{GFICF_E_ARG, "too many devices"};
  if (mode == GFICF_MODE_SERIAL) ndev = 1;  // global row compaction: one device
  if ((long long)ndev > n) ndev = 1;

  std::lock_guard<std::mutex> lk(g_call_mu);
  DeviceRestore restore;
  const auto t0 = std::chrono::steady_clock::now();
  const long long rows_per = (n + ndev - 1) / ndev;
  g_active_devices.store(ndev);
  std::vector<SlabResult> res(ndev);
  std::vector<Slab> slabs;
  const int out_mode = resolve_out_mode(out, (int)k, (int)mode);
  for (int r = 0; r < ndev; ++r) {
    slabs.emplace_back(r, ndev, idx, (long long)n, (int)k, rows_per, out, (int)mode);
    slabs.back().elem = elem;
    slabs.back().out_mode = out_mode;
  }
  auto first_error = [&]() {
    for (auto& r : res)
      if (r.err.code != GFICF_OK) throw r.err;
  };
  if (ndev == 1) {
    device_phase0(slabs[0], &res[0]);
    first_error();
    device_phase1(slabs[0], &res[0]);
  } else {
    nccl_ensure(ndev);
    for (int r = 0; r < ndev; ++r) slabs[r].comm = g_nccl.comms[r];
    {
      std::vector<std::thread> th;
      for (int r = 0; r < ndev; ++r) th.emplace_back(device_phase0, slabs[r], &res[r]);
      for (auto& t : th) t.join();
    }
    first_error();  // nobody has entered a collective yet
    std::vector<std::thread> th;
    for (int r = 0; r < ndev; ++r) th.emplace_back(device_phase1, slabs[r], &res[r]);
    for (auto& t : th) t.join();
  }
  unsigned all_flags = 0;
  for (auto& r : res) all_flags |= r.flags;
  bool bad_id = (all_flags & kFlagBadId) != 0;
  if (!bad_id) {
    first_error();
    const bool exact = k > kLargeMaxK || (all_flags & (kFlagDupId | kFlagHashFail));
    if (exact || mode == GFICF_MODE_SERIAL) {
      if (ndev == 1) {
        device_phase2(slabs[0], exact, &res[0]);
      } else {
        std::vector<std::thread> th;
        for (int r = 0; r < ndev; ++r) th.emplace_back(device_phase2, slabs[r], exact, &res[r]);
        for (auto& t : th) t.join();
      }
    }
  }
  const auto t1 = std::chrono::steady_clock::now();
  unsigned flags = 0;
  double tm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (auto& r : res) {
    if (!bad_id && r.err.code != GFICF_OK) throw r.err;
    flags |= r.flags;
    tm[0] = std::max<double>(tm[0], r.ms_h2d);
    tm[1] = std::max<double>(tm[1], r.ms_k0);
    tm[2] = std::max<double>(tm[2], r.ms_k1);
    tm[3] = std::max<double>(tm[3], r.ms_d2h);
    tm[5] = std::max<double>(tm[5], r.ms_gather);
    tm[6] += r.launches;
    tm[7] += r.d2h_bytes;
  }
  double h2d_total = 0;
  for (auto& r : res) h2d_total += r.h2d_bytes;
  tl_output = {res[0].out_mode, res[0].host_items, h2d_total};
  tm[4] = std::chrono::duration<double, std::milli>(t1 - t0).count();
  memcpy(tl_timings, tm, sizeof tm);
  if (flags & kFlagBadId)
    throw Err{GFICF_E_RANGE,
              "neighbour ids must be integers in [1, nrow] (NaN, fractional or out-of-range id found)"};
  if (n_written) *n_written = res[0].n_written;
  return GFICF_OK;
  API_END
}
}  // namespace

extern "C" {

int gficf_cuda_jaccard(const double* idx, int64_t n, int32_t k, double* out, int32_t n_devices,
                       int32_t mode, int64_t* n_written, char* err, size_t errlen) {
  return jaccard_host_call(idx, 8, n, k, out, n_devices, mode, n_written, err, errlen);
}

int gficf_cuda_jaccard_i32(const int32_t* idx, int64_t n, int32_t k, double* out, int32_t n_devices,
                           int32_t mode, int64_t* n_written, char* err, size_t errlen) {
  return jaccard_host_call(idx, 4, n, k, out, n_devices, mode, n_written, err, errlen);
}

// ---------------------------------------------------------------- one process per GPU
int gficf_cuda_comm_unique_id(void* id128) {
  char* err = nullptr;
  size_t errlen = 0;
  API_BEGIN
  if (!id128) return GFICF_E_ARG;
  if (!nccl_dyn::get().ok) return GFICF_E_NCCL;
  static_assert(sizeof(ncclUniqueId) == GFICF_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  NCCL_TRY(nccl_dyn::get().GetUniqueId(&id));
  memcpy(id128, &id, sizeof id);
  return GFICF_OK;
  API_END
}

int gficf_cuda_comm_init_rank(const void* id128, int32_t nranks, int32_t rank, int32_t device,
                              char* err, size_t errlen) {
  API_BEGIN
  if (!id128 || nranks < 1 || rank < 0 || rank >= nranks || device < 0 || device >= kMaxDevices)
    throw Err{GFICF_E_ARG, "bad communicator arguments"};
  if (!nccl_dyn::get().ok) throw Err{GFICF_E_NCCL, "cannot load libnccl.so.2: " + nccl_dyn::get().why};
  std::lock_guard<std::mutex> lk(g_call_mu);
  mp_release();
  CU_TRY(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  NCCL_TRY(nccl_dyn::get().CommInitRank(&g_mp.comm, nranks, id, rank));
  g_mp.nranks = nranks;
  g_mp.rank = rank;
  g_mp.dev = device;
  g_sharers.store(nranks);  // one node: the ranks share the host's cores
  return GFICF_OK;
  API_END
}

int gficf_cuda_comm_destroy(void) {
  std::lock_guard<std::mutex> lk(g_call_mu);
  mp_release();
  return GFICF_OK;
}

int gficf_cuda_jaccard_rank(const double* idx, int64_t n, int32_t k, double* out, char* err,
                            size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  if (!g_mp.comm) throw Err{GFICF_E_ARG, "gficf_cuda_comm_init_rank has not been called"};
  if (n < 0 || k < 0) throw Err{GFICF_E_ARG, "negative matrix dimension"};
  if (n == 0 || k == 0) return GFICF_OK;
  if (!idx || !out) throw Err{GFICF_E_ARG, "null matrix pointer"};
  if (n >= 0x7fffffffLL - 2 || (long double)n * k >= 2147483647.0L)
    throw Err{GFICF_E_LIMIT, "n*k must stay below 2^31 (the reference's int row index)"};
  if (k > 65535) throw Err{GFICF_E_LIMIT, "k above 65535 is not supported"};
  std::lock_guard<std::mutex> lk(g_call_mu);
  DeviceRestore restore;
  const auto t0 = std::chrono::steady_clock::now();
  const int nr = g_mp.nranks;
  const long long rows_per = (n + nr - 1) / nr;
  Slab s(g_mp.rank, nr, idx, (long long)n, (int)k, rows_per, out, GFICF_MODE_PARALLEL);
  s.dev = g_mp.dev;
  s.comm = g_mp.comm;
  s.out_mode = resolve_out_mode(out, (int)k, GFICF_MODE_PARALLEL);
  SlabResult res;
  device_phase0(s, &res);
  DeviceWs& ws = g_ws[s.dev];
  {
    // agree that every rank got through its local phase BEFORE the index all-gather: a rank that
    // failed (out of memory ...) still takes part in this tiny all-reduce, then everybody leaves
    CU_TRY(cudaSetDevice(s.dev));
    ws.ensure(s.dev);
    int* okbit = (int*)((char*)ws.small.p + 48);
    int h = res.err.code != GFICF_OK;
    CU_TRY(cudaMemcpyAsync(okbit, &h, sizeof h, cudaMemcpyHostToDevice, ws.s_comp));
    NCCL_TRY(nccl_dyn::get().AllReduce(okbit, okbit, 1, ncclInt32, ncclMax, s.comm, ws.s_comp));
    CU_TRY(cudaMemcpyAsync(&h, okbit, sizeof h, cudaMemcpyDeviceToHost, ws.s_comp));
    CU_TRY(cudaStreamSynchronize(ws.s_comp));
    if (res.err.code != GFICF_OK) throw res.err;
    if (h) throw Err{GFICF_E_CUDA, "another rank failed before the index exchange"};
  }
  device_phase1(s, &res);
  // flags of all ranks (every rank must reach this collective, error or not)
  unsigned all_flags = res.flags;
  {
    CU_TRY(cudaSetDevice(s.dev));
    int* bits = (int*)((char*)ws.small.p + 32);
    int h[4] = {(int)(res.flags & 1u), (int)((res.flags >> 1) & 1u), (int)((res.flags >> 2) & 1u),
                res.err.code != GFICF_OK};
    CU_TRY(cudaMemcpyAsync(bits, h, sizeof h, cudaMemcpyHostToDevice, ws.s_comp));
    NCCL_TRY(nccl_dyn::get().AllReduce(bits, bits, 4, ncclInt32, ncclMax, s.comm, ws.s_comp));
    CU_TRY(cudaMemcpyAsync(h, bits, sizeof h, cudaMemcpyDeviceToHost, ws.s_comp));
    CU_TRY(cudaStreamSynchronize(ws.s_comp));
    all_flags = (unsigned)h[0] | ((unsigned)h[1] << 1) | ((unsigned)h[2] << 2);
    if (res.err.code != GFICF_OK) throw res.err;
    if (h[3]) throw Err{GFICF_E_CUDA, "another rank failed"};
  }
  if (all_flags & kFlagBadId)
    throw Err{GFICF_E_RANGE,
              "neighbour ids must be integers in [1, nrow] (NaN, fractional or out-of-range id found)"};
  if (k > kLargeMaxK || (all_flags & (kFlagDupId | kFlagHashFail))) {
    device_phase2(s, true, &res);
    if (res.err.code != GFICF_OK) throw res.err;
  }
  const auto t1 = std::chrono::steady_clock::now();
  double tm[8] = {res.ms_h2d, res.ms_k0, res.ms_k1, res.ms_d2h,
                  std::chrono::duration<double, std::milli>(t1 - t0).count(), res.ms_gather,
                  (double)res.launches, res.d2h_bytes};
  memcpy(tl_timings, tm, sizeof tm);
  tl_output = {res.out_mode, res.host_items, res.h2d_bytes};
  return GFICF_OK;
  API_END
}

// ---------------------------------------------------------------- peer-memory gather
int gficf_cuda_ipc_alloc(size_t bytes, void** dptr, void* handle64) {
  char* err = nullptr;
  size_t errlen = 0;
  API_BEGIN
  if (!dptr || !handle64 || !bytes) return GFICF_E_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == GFICF_IPC_HANDLE_BYTES, "ipc handle size");
  void* p = nullptr;
  CU_TRY(cudaMalloc(&p, bytes));
  CU_TRY(cudaMemset(p, 0, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    CU_TRY(e);
  }
  memcpy(handle64, &h, sizeof h);
  *dptr = p;
  return GFICF_OK;
  API_END
}

int gficf_cuda_ipc_open(const void* handle64, void** dptr) {
  char* err = nullptr;
  size_t errlen = 0;
  API_BEGIN
  if (!dptr || !handle64) return GFICF_E_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof h);
  CU_TRY(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
  return GFICF_OK;
  API_END
}

int gficf_cuda_ipc_close(void* dptr) {
  if (dptr && cudaIpcCloseMemHandle(dptr) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_ipc_free(void* dptr) {
  if (dptr && cudaFree(dptr) != cudaSuccess) {
    cudaGetLastError();
    return GFICF_E_CUDA;
  }
  return GFICF_OK;
}

int gficf_cuda_signal_dev(uint32_t* d_flag, uint32_t value, void* stream) {
  char* err = nullptr;
  size_t errlen = 0;
  API_BEGIN
  if (!d_flag) return GFICF_E_ARG;
  signal_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(d_flag, value);
  CU_TRY(cudaGetLastError());
  return GFICF_OK;
  API_END
}

int gficf_cuda_wait_dev(const uint32_t* d_flag, uint32_t expected, uint32_t* d_flags, void* stream) {
  char* err = nullptr;
  size_t errlen = 0;
  API_BEGIN
  if (!d_flag || !d_flags) return GFICF_E_ARG;
  wait_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(d_flag, expected, d_flags, peer_spin_clocks(0));
  CU_TRY(cudaGetLastError());
  return GFICF_OK;
  API_END
}

// ---------------------------------------------------------------- device-buffer entries
#define DEV_BEGIN      \
  char* err = nullptr; \
  size_t errlen = 0;   \
  API_BEGIN
#define DEV_END API_END

int gficf_cuda_layout_dev(const double* d_idx_f64, int64_t ld_rows, int64_t ld_row0, int64_t n,
                          int32_t k, int64_t row_lo, int64_t row_hi, int32_t* d_idx_i32,
                          uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_f64 || !d_idx_i32 || !d_flags || k < 1 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  launch_layout(jac_ctx((cudaStream_t)stream), d_idx_f64, ld_rows, ld_row0, n, k, row_lo, row_hi, d_idx_i32, d_flags);
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_pad_dev(const int32_t* d_idx_dense, int64_t n, int32_t k, int64_t row_lo,
                       int64_t row_hi, int32_t* d_idx_i32, uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_dense || !d_idx_i32 || !d_flags || k < 1 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  launch_pad(jac_ctx((cudaStream_t)stream), d_idx_dense, n, k, row_lo, row_hi, d_idx_i32, d_flags);
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_jaccard_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                           int64_t row_hi, double* d_from, double* d_to, double* d_w,
                           uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_from || !d_to || !d_w || !d_flags || k < 1 || row_lo < 0 || row_hi > n)
    return GFICF_E_ARG;
  if (!launch_fast<0>(jac_ctx((cudaStream_t)stream), d_idx_i32, k, row_lo, row_hi, d_from, d_to, d_w, nullptr,
                      d_flags))
    return GFICF_E_LIMIT;
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_jaccard_counts_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                  int64_t row_hi, uint8_t* d_u, uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_u || !d_flags || k < 1 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  if (!launch_fast<1>(jac_ctx((cudaStream_t)stream), d_idx_i32, k, row_lo, row_hi, nullptr, nullptr, nullptr,
                      (void*)d_u, d_flags))
    return GFICF_E_LIMIT;
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_jaccard_counts_tagged_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                         int64_t row_hi, uint8_t* d_u, uint32_t tag, uint32_t* d_flags,
                                         void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_u || !d_flags || k < 1 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  if ((tag & ~0x180u) || k > 127) return GFICF_E_LIMIT;
  const bool by_rows = (tag & 0x100u) != 0;  // GFICF_TAG_ROW_STORES
  tag &= 0x80u;
  // k <= 32: grouped rows, 16-byte vector stores (d_u is typically a peer GPU's memory)
  const bool grouped = k <= 32 && !by_rows;
  const JacCtx cx = jac_ctx((cudaStream_t)stream);
  const bool ok = grouped ? launch_fast<3>(cx, d_idx_i32, k, row_lo, row_hi, nullptr, nullptr, nullptr, (void*)d_u,
                                           d_flags, tag)
                          : launch_fast<1>(cx, d_idx_i32, k, row_lo, row_hi, nullptr, nullptr, nullptr, (void*)d_u,
                                           d_flags, tag);
  if (!ok) return GFICF_E_LIMIT;
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_expand_stream_dev(const int32_t* d_idx_i32, int32_t k, const int64_t* seg_lo,
                                 const int64_t* seg_hi, int32_t n_seg, const uint8_t* d_u, double* d_from,
                                 double* d_to, double* d_w, uint32_t tag, int64_t timeout_ms,
                                 uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_u || !d_from || !d_to || !d_w || !d_flags || !seg_lo || !seg_hi) return GFICF_E_ARG;
  if (k < 1 || k > 127 || (tag & ~0x80u) || n_seg < 0 || n_seg > kMaxStreamSegs) return GFICF_E_LIMIT;
  if (!launch_expand_stream(jac_ctx((cudaStream_t)stream), d_idx_i32, k, seg_lo, seg_hi, n_seg, d_u, d_from, d_to,
                            d_w, tag, peer_spin_clocks(timeout_ms), d_flags))
    return GFICF_E_ARG;
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_jaccard_exact_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                 int64_t row_hi, int32_t set_semantics, void* d_u, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_u || k < 1 || k > 65535 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  launch_exact(jac_ctx((cudaStream_t)stream), d_idx_i32, k, row_lo, row_hi, set_semantics, d_u);
  return GFICF_OK;
  DEV_END
}

size_t gficf_cuda_expand_scratch_bytes(int64_t slab_edges) {
  return expand_scratch_bytes(slab_edges < 0 ? 0 : slab_edges);
}

int gficf_cuda_expand_dev(const int32_t* d_idx_i32, int32_t k, int64_t row_lo, int64_t row_hi,
                          const void* d_u, int32_t mode, double* d_from, double* d_to, double* d_w,
                          void* d_scratch, int64_t* d_n_written, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_u || !d_from || !d_to || !d_w || k < 1 || k > 65535 || row_lo < 0)
    return GFICF_E_ARG;
  if (mode == GFICF_MODE_SERIAL && (!d_scratch || !d_n_written)) return GFICF_E_ARG;
  if (mode != GFICF_MODE_SERIAL && mode != GFICF_MODE_PARALLEL) return GFICF_E_ARG;
  launch_expand(jac_ctx((cudaStream_t)stream), d_idx_i32, k, row_lo, row_hi, d_u, mode == GFICF_MODE_SERIAL, d_from,
                d_to, d_w, d_scratch, (long long*)d_n_written);
  return GFICF_OK;
  DEV_END
}

// ---------------------------------------------------------------- SNN graph (next row after the path)
int gficf_cuda_jaccard_counts_mutual_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, int64_t row_lo,
                                         int64_t row_hi, uint8_t* d_um, uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_um || !d_flags || k < 1 || row_lo < 0 || row_hi > n) return GFICF_E_ARG;
  if (!launch_fast<2>(jac_ctx((cudaStream_t)stream), d_idx_i32, k, row_lo, row_hi, nullptr, nullptr, nullptr,
                      (void*)d_um, d_flags))
    return GFICF_E_LIMIT;
  return GFICF_OK;
  DEV_END
}

size_t gficf_cuda_snn_scratch_bytes(int64_t n, int64_t cap) {
  if (n < 0 || cap < 0) return 0;
  return snn_scratch_layout(nullptr, n, cap).bytes;
}

int gficf_cuda_snn_lower_dev(const int32_t* d_idx_i32, int64_t n, int32_t k, const uint8_t* d_um,
                             int64_t* d_colptr, int32_t* d_row, double* d_w, int64_t cap,
                             int32_t* d_vertex_cell, int64_t* d_n_vertices, void* d_scratch,
                             uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  if (!d_idx_i32 || !d_um || !d_colptr || !d_row || !d_w || !d_scratch || !d_flags || n < 1 || k < 1)
    return GFICF_E_ARG;
  if (k > 127 || n >= 0x7fffffffLL || n * (long long)k >= 0xffffffffLL) return GFICF_E_LIMIT;
  if (cap < n * (int64_t)k) return GFICF_E_ARG;
  net_max_dynamic_smem(snn_sort_big_kernel, kSnnSmemSortMax * 12);
  snn_lower((cudaStream_t)stream, snn_scratch_layout((char*)d_scratch, n, cap), sm_count() * 8, sm_count() * 2,
            d_idx_i32, n, k, row_stride(k), d_um, (long long*)d_colptr, d_row, d_w, d_vertex_cell,
            (long long*)d_n_vertices, d_flags);
  CU_TRY(cudaGetLastError());
  return GFICF_OK;
  DEV_END
}

int gficf_cuda_snn_lower(const void* idx_colmajor, int32_t elem_bytes, int64_t n, int32_t k,
                         int64_t* colptr, int32_t* row, double* w, int64_t cap, int32_t* vertex_cell,
                         int64_t* n_vertices, int64_t* nnz, char* err, size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  if (nnz) *nnz = 0;
  if (n_vertices) *n_vertices = 0;
  if (n < 0 || k < 0 || (elem_bytes != 8 && elem_bytes != 4)) throw Err{GFICF_E_ARG, "bad matrix description"};
  if (n == 0 || k == 0) return GFICF_OK;
  if (!idx_colmajor || !colptr || !row || !w || cap < 0) throw Err{GFICF_E_ARG, "null output pointer"};
  if (k > 127) throw Err{GFICF_E_LIMIT, "the graph build carries the mutual flag in bit 7 of the count byte: k <= 127"};
  if (n >= 0x7fffffffLL - 2 || (long double)n * k >= 2147483647.0L)
    throw Err{GFICF_E_LIMIT, "n*k must stay below 2^31 (the reference's int row index)"};
  SingleDeviceCall call;
  DeviceWs& ws = call.ws;
  const long long E = (long long)n * k;
  const int kp = row_stride(k);
  ws.in_raw.need((size_t)E * elem_bytes);
  ws.idx.need((size_t)n * kp * sizeof(int));
  ws.counts.need((size_t)E);
  ws.scratch.need(gficf_cuda_snn_scratch_bytes(n, E));
  // results on the device: colptr | w | row | vertex map
  int64_t* d_colptr;
  double* d_w;
  int *d_row, *d_vc;
  auto results = [&](char* base) {
    ScratchCarver c{base};
    d_colptr = c.take<int64_t>(n + 1);
    d_w = c.take<double>(E);
    d_row = c.take<int>(E);
    d_vc = c.take<int>(n);
    return c.bytes;
  };
  ws.out.need(results(nullptr));
  results((char*)ws.out.p);
  unsigned* d_flags = (unsigned*)ws.small.p;
  int64_t* d_nv = (int64_t*)((char*)ws.small.p + 16);
  CU_TRY(cudaMemsetAsync(ws.small.p, 0, 64, ws.s_comp));
  CU_TRY(cudaEventRecord(ws.ev[0], ws.s_comp));
  const size_t dev_elem = h2d_block(ws, idx_colmajor, n, ws.in_raw.p, n, k, (size_t)elem_bytes, ws.s_comp);
  CU_TRY(cudaEventRecord(ws.ev[1], ws.s_comp));
  if (dev_elem == 8)
    launch_layout(jac_ctx(ws.s_comp), (const double*)ws.in_raw.p, n, 0, n, k, 0, n, (int*)ws.idx.p, d_flags);
  else
    launch_layout(jac_ctx(ws.s_comp), (const int*)ws.in_raw.p, n, 0, n, k, 0, n, (int*)ws.idx.p, d_flags);
  CU_TRY(cudaEventRecord(ws.ev[2], ws.s_comp));
  if (!launch_fast<2>(jac_ctx(ws.s_comp), (const int*)ws.idx.p, k, 0, n, nullptr, nullptr, nullptr, ws.counts.p,
                      d_flags))
    throw Err{GFICF_E_LIMIT, "k outside the range of the mutual-bit count kernel"};
  const int rc = gficf_cuda_snn_lower_dev((const int32_t*)ws.idx.p, n, k, (const uint8_t*)ws.counts.p, d_colptr, d_row,
                                          d_w, E, d_vc, d_nv, ws.scratch.p, d_flags, ws.s_comp);
  if (rc != GFICF_OK) throw Err{rc, "graph kernels could not be launched"};
  CU_TRY(cudaEventRecord(ws.ev[3], ws.s_comp));
  // flags, vertex count and entry count decide what is copied back
  CU_TRY(cudaMemcpyAsync(ws.h_small, ws.small.p, 32, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaMemcpyAsync((char*)ws.h_small + 32, d_colptr + n, 8, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaStreamSynchronize(ws.s_comp));
  const unsigned flags = ws.h_small[0];
  const long long nv = *(long long*)((char*)ws.h_small + 16), total = *(long long*)((char*)ws.h_small + 32);
  if (flags & kFlagBadId)
    throw Err{GFICF_E_RANGE,
              "neighbour ids must be integers in [1, nrow] (NaN, fractional or out-of-range id found)"};
  if (flags & (kFlagDupId | kFlagHashFail))
    throw Err{GFICF_E_LIMIT, "a row lists an id twice: the device graph build needs distinct ids per row"};
  if (nnz) *nnz = total;
  if (n_vertices) *n_vertices = nv;
  if (total > cap) throw Err{GFICF_E_ARG, fmt("row / w capacity %lld is below the %lld entries of the graph", (long long)cap, total)};
  std::vector<Seg> segs;
  segs.push_back({(char*)colptr, (char*)d_colptr, (size_t)(n + 1) * 8, nullptr});
  if (total) {
    segs.push_back({(char*)row, (char*)d_row, (size_t)total * 4, nullptr});
    segs.push_back({(char*)w, (char*)d_w, (size_t)total * 8, nullptr});
  }
  if (vertex_cell && nv) segs.push_back({(char*)vertex_cell, (char*)d_vc, (size_t)nv * 4, nullptr});
  CU_TRY(cudaEventRecord(ws.ev[4], ws.s_copy));
  d2h_segs(ws, segs, ws.s_copy);
  CU_TRY(cudaEventRecord(ws.ev[5], ws.s_copy));
  CU_TRY(cudaStreamSynchronize(ws.s_copy));
  call.timings(event_ms(ws.ev[0], ws.ev[1]), event_ms(ws.ev[1], ws.ev[2]), event_ms(ws.ev[2], ws.ev[3]),
               event_ms(ws.ev[4], ws.ev[5]), 22,
               (double)(n + 1) * 8 + (double)total * 12 + (vertex_cell ? (double)nv * 4 : 0.0));
  return GFICF_OK;
  API_END
}

}  // extern "C"

namespace {
// Argument checks shared by both markers entries: sizes and cluster cap, then every id and every cluster's
// size (each cluster needs cells).
void markers_check_sizes(int64_t n_genes, int64_t n_cells, int32_t n_clusters) {
  if (n_genes < 0 || n_cells < 0) throw Err{GFICF_E_ARG, "negative matrix dimension"};
  if (n_clusters < 2) throw Err{GFICF_E_ARG, "one-vs-rest needs at least two clusters"};
  if (n_clusters > kWmuMaxClusters)
    throw Err{GFICF_E_LIMIT, fmt("more than %d clusters (the per-CTA rank-sum accumulators)", kWmuMaxClusters)};
  if (n_cells >= 0x7fffffffLL) throw Err{GFICF_E_LIMIT, "more than 2^31 cells per gene"};
}

std::vector<long long> markers_cluster_sizes(const int32_t* cluster, int64_t n_cells, int32_t n_clusters) {
  std::vector<long long> size((size_t)n_clusters, 0);
  for (int64_t i = 0; i < n_cells; ++i) {
    const int32_t c = cluster[i];
    if (c < 0 || c >= n_clusters)
      throw Err{GFICF_E_ARG, fmt("cluster id %d of cell %lld is outside [0, %d)", c, (long long)i, n_clusters)};
    ++size[(size_t)c];
  }
  for (int32_t c = 0; c < n_clusters; ++c)
    if (!size[(size_t)c]) throw Err{GFICF_E_ARG, fmt("cluster %d has no cells", c)};
  return size;
}

// The end shared by the Mann-Whitney entries: launches checked, ev[2] recorded, z | ratio (n_clusters blocks of
// n_genes) and the per-gene single flags read back and finished into out (wmu_finish).
void wmu_read_and_finish(DeviceWs& ws, const double* d_z, const int* d_single, int64_t n_genes, int32_t n_clusters,
                         double* out) {
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaEventRecord(ws.ev[2], ws.s_comp));
  const size_t zc = (size_t)n_genes * n_clusters;
  std::vector<double> h(zc * 2);
  std::vector<int> hs((size_t)n_genes);
  CU_TRY(cudaMemcpyAsync(h.data(), d_z, zc * 16, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaMemcpyAsync(hs.data(), d_single, (size_t)n_genes * 4, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaStreamSynchronize(ws.s_comp));
  wmu_finish(h.data(), hs.data(), n_genes, n_clusters, out);
}
}  // namespace

extern "C" {

// ---------------------------------------------------------------- Mann-Whitney U per gene (next row 4)
int gficf_cuda_wmu_test(const double* mat_x, const double* mat_y, int64_t n_genes, int64_t n1, int64_t n2,
                        double* out, char* err, size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  if (n_genes < 0 || n1 < 0 || n2 < 0) throw Err{GFICF_E_ARG, "negative matrix dimension"};
  if (n_genes == 0) return GFICF_OK;
  if (!mat_x || !mat_y || !out) throw Err{GFICF_E_ARG, "null matrix pointer"};
  if (n1 < 1 || n2 < 1) throw Err{GFICF_E_ARG, "both groups need at least one cell"};
  if (n1 + n2 >= 0x7fffffffLL) throw Err{GFICF_E_LIMIT, "more than 2^31 cells per gene"};
  SingleDeviceCall call;
  DeviceWs& ws = call.ws;
  const long long N = n1 + n2;
  int per_sm = 0;
  CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wmu_rank_kernel, kWmuThreads, 0));
  const int grid = (int)std::min<long long>(n_genes, (long long)std::max(1, per_sm) * sm_count());
  // device buffers: X | Y in in_raw; per-CTA sort scratch in scratch (keys) and counts (payload);
  // z, ratio, single flags in out
  const size_t bx = (size_t)n_genes * n1 * 8, by = (size_t)n_genes * n2 * 8;
  ws.in_raw.need(bx + by);
  ws.scratch.need((size_t)grid * 2 * N * sizeof(unsigned long long));
  ws.counts.need((size_t)grid * (3 * N + 2) * sizeof(unsigned));
  ws.out.need((size_t)n_genes * (8 + 8 + 4) + 64);
  double* d_x = (double*)ws.in_raw.p;
  double* d_y = (double*)((char*)ws.in_raw.p + bx);
  double* d_z = (double*)ws.out.p;
  double* d_ratio = d_z + n_genes;
  int* d_single = (int*)(d_ratio + n_genes);
  CU_TRY(cudaEventRecord(ws.ev[0], ws.s_comp));
  h2d_block(ws, mat_x, n_genes * n1, d_x, n_genes * n1, 1, 8, ws.s_comp, /*ids=*/false);
  h2d_block(ws, mat_y, n_genes * n2, d_y, n_genes * n2, 1, 8, ws.s_comp, /*ids=*/false);
  CU_TRY(cudaEventRecord(ws.ev[1], ws.s_comp));
  wmu_test_launch(ws.s_comp, grid, d_x, d_y, n_genes, n1, n2, (unsigned long long*)ws.scratch.p, (unsigned*)ws.counts.p,
                  d_z, d_ratio, d_single);
  wmu_read_and_finish(ws, d_z, d_single, n_genes, 1, out);
  call.timings(event_ms(ws.ev[0], ws.ev[1]), 0, event_ms(ws.ev[1], ws.ev[2]), 0, 2, (double)n_genes * 20);
  return GFICF_OK;
  API_END
}

// One-vs-rest Mann-Whitney U for every cluster in one call: one upload, one sort per gene
int gficf_cuda_wmu_markers(const double* mat, int64_t n_genes, int64_t n_cells, const int32_t* cluster,
                           int32_t n_clusters, double* out, char* err, size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  markers_check_sizes(n_genes, n_cells, n_clusters);
  if (n_genes == 0) return GFICF_OK;
  if (!mat || !cluster || !out) throw Err{GFICF_E_ARG, "null matrix pointer"};
  const std::vector<long long> size = markers_cluster_sizes(cluster, n_cells, n_clusters);
  SingleDeviceCall call;
  DeviceWs& ws = call.ws;
  const long long N = n_cells, C = n_clusters;
  CU_TRY(cudaFuncSetAttribute(wmu_markers_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              kWmuMaxClusters * kWmuClusterSmemBytes));
  int per_sm = 0;
  CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wmu_markers_rank_kernel, kWmuThreads,
                                                       (size_t)C * kWmuClusterSmemBytes));
  const int grid = (int)std::min<long long>(n_genes, (long long)std::max(1, per_sm) * sm_count());
  // device buffers: the matrix in in_raw; cluster ids | cluster sizes in idx; per-CTA sort scratch in
  // scratch (keys) and counts (payload); z | ratio per (gene, cluster) and the per-gene single flags in out
  const size_t bm = (size_t)n_genes * N * 8;
  int* d_cl;
  long long* d_size;
  auto ids = [&](char* base) {
    ScratchCarver c{base};
    d_cl = c.take<int>(N);
    d_size = c.take<long long>(C);
    return c.bytes;
  };
  ws.in_raw.need(bm);
  ws.idx.need(ids(nullptr));
  ids((char*)ws.idx.p);
  ws.scratch.need((size_t)grid * 2 * N * sizeof(unsigned long long));
  ws.counts.need((size_t)grid * (3 * N + 2) * sizeof(unsigned));
  const size_t zc = (size_t)n_genes * C;
  ws.out.need(zc * 16 + (size_t)n_genes * 4 + 64);
  double* d_mat = (double*)ws.in_raw.p;
  double* d_z = (double*)ws.out.p;
  double* d_ratio = d_z + zc;
  int* d_single = (int*)(d_ratio + zc);
  CU_TRY(cudaEventRecord(ws.ev[0], ws.s_comp));
  h2d_block(ws, mat, n_genes * N, d_mat, n_genes * N, 1, 8, ws.s_comp, /*ids=*/false);
  h2d_block(ws, cluster, N, d_cl, N, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, size.data(), C, d_size, C, 1, 8, ws.s_comp, /*ids=*/false);
  CU_TRY(cudaEventRecord(ws.ev[1], ws.s_comp));
  wmu_markers_launch(ws.s_comp, grid, d_mat, n_genes, N, d_cl, d_size, n_clusters, (unsigned long long*)ws.scratch.p,
                     (unsigned*)ws.counts.p, d_z, d_ratio, d_single);
  wmu_read_and_finish(ws, d_z, d_single, n_genes, n_clusters, out);
  call.timings(event_ms(ws.ev[0], ws.ev[1]), 0, event_ms(ws.ev[1], ws.ev[2]), 0, 2, (double)zc * 16 + (double)n_genes * 4);
  return GFICF_OK;
  API_END
}

}  // extern "C"

// ---------------------------------------------------------------- network pieces of the community detection (next row 3)

extern "C" {

size_t gficf_cuda_network_scratch_bytes(int64_t n_nodes, int64_t n_items) {
  if (n_nodes < 0 || n_items < 0) return 0;
  return net_scratch_layout(nullptr, n_nodes, n_items).bytes;
}

int gficf_cuda_network_dev(const int64_t* d_colptr, const int32_t* d_row, const double* d_w, int64_t n_vertices,
                           int64_t nnz, int64_t* d_first, int32_t* d_neighbor, double* d_edge_w, double* d_node_w,
                           double* d_total_w, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                           void* stream) {
  DEV_BEGIN
  return net_entry_network(d_colptr, d_row, d_w, n_vertices, nnz, d_first, d_neighbor, d_edge_w, d_node_w, d_total_w,
                           d_scratch, scratch_bytes, d_flags, (cudaStream_t)stream, sm_count() * 8);
  DEV_END
}

int gficf_cuda_network_quality_dev(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                                   const double* d_node_w, int64_t n_nodes, int64_t n_edges,
                                   const int32_t* d_cluster, int32_t n_clusters, double resolution,
                                   double self_links, const double* d_total_w, double* d_cluster_w,
                                   double* d_quality, void* d_scratch, size_t scratch_bytes, uint32_t* d_flags,
                                   void* stream) {
  DEV_BEGIN
  return net_entry_quality(d_first, d_neighbor, d_edge_w, d_node_w, n_nodes, n_edges, d_cluster, n_clusters,
                           resolution, self_links, d_total_w, d_cluster_w, d_quality, d_scratch, scratch_bytes,
                           d_flags, (cudaStream_t)stream, sm_count() * 8);
  DEV_END
}

int gficf_cuda_network_reduce_dev(const int64_t* d_first, const int32_t* d_neighbor, const double* d_edge_w,
                                  const double* d_node_w, int64_t n_nodes, int64_t n_edges,
                                  const int32_t* d_cluster, int32_t n_clusters, double self_links,
                                  int64_t* d_r_first, int32_t* d_r_neighbor, double* d_r_edge_w, int64_t r_cap,
                                  double* d_r_node_w, double* d_r_self_links, double* d_r_total_w,
                                  int64_t* n_reduced_edges, void* d_scratch, size_t scratch_bytes,
                                  uint32_t* d_flags, void* stream) {
  DEV_BEGIN
  return net_entry_reduce(d_first, d_neighbor, d_edge_w, d_node_w, n_nodes, n_edges, d_cluster, n_clusters, self_links,
                          d_r_first, d_r_neighbor, d_r_edge_w, r_cap, d_r_node_w, d_r_self_links, d_r_total_w,
                          n_reduced_edges, d_scratch, scratch_bytes, d_flags, (cudaStream_t)stream, sm_count() * 8);
  DEV_END
}

}  // extern "C"

// ---------------------------------------------------------------- Mann-Whitney markers from a sparse matrix

extern "C" {

// gficf_cuda_wmu_markers on a compressed-column matrix: the stored values are uploaded, made gene-major on
// the device (wmu_csc_to_genes) and only they are read by the rank and means kernels.
int gficf_cuda_wmu_markers_csc(const int32_t* colptr, const int32_t* row, const double* x, int64_t n_genes,
                               int64_t n_cells, const int32_t* cluster, int32_t n_clusters, double* out, char* err,
                               size_t errlen) {
  API_BEGIN
  if (err && errlen) err[0] = 0;
  markers_check_sizes(n_genes, n_cells, n_clusters);
  if (n_genes == 0) return GFICF_OK;
  if (n_genes >= 0x7fffffffLL) throw Err{GFICF_E_LIMIT, "more than 2^31 genes (R's int row ids)"};
  if (!colptr || !cluster || !out) throw Err{GFICF_E_ARG, "null matrix pointer"};
  if (colptr[0] != 0) throw Err{GFICF_E_ARG, fmt("colptr[0] is %d, not 0", colptr[0])};
  for (int64_t j = 0; j < n_cells; ++j)
    if (colptr[j + 1] < colptr[j])
      throw Err{GFICF_E_ARG, fmt("colptr decreases at column %lld (%d after %d)", (long long)j, colptr[j + 1], colptr[j])};
  const long long nnz = colptr[n_cells];
  if (nnz > 0 && (!row || !x)) throw Err{GFICF_E_ARG, "null matrix pointer"};
  const std::vector<long long> size = markers_cluster_sizes(cluster, n_cells, n_clusters);
  SingleDeviceCall call;
  DeviceWs& ws = call.ws;
  const long long N = n_cells, C = n_clusters;
  const WmuClusterLists cl = wmu_cluster_lists(cluster, N, n_clusters);
  // device buffers: colptr | row | x in in_raw; cluster ids | crank | members | cluster sizes | cptr in idx;
  // the transpose's scratch in scratch (the gene-major values end up there); per-CTA sort scratch of the
  // rank kernel in counts; z | ratio per (gene, cluster) and the per-gene single flags in out
  int *d_colptr, *d_row, *d_cl, *d_crank, *d_members;
  double* d_x;
  long long *d_size, *d_cptr;
  auto matrix = [&](char* base) {
    ScratchCarver c{base};
    d_colptr = c.take<int>(N + 1);
    d_row = c.take<int>(nnz);
    d_x = c.take<double>(nnz + 1);
    return c.bytes;
  };
  auto lists = [&](char* base) {
    ScratchCarver c{base};
    d_cl = c.take<int>(N);
    d_crank = c.take<int>(N);
    d_members = c.take<int>(N);
    d_size = c.take<long long>(C);
    d_cptr = c.take<long long>(C + 1);
    return c.bytes;
  };
  ws.in_raw.need(matrix(nullptr));
  matrix((char*)ws.in_raw.p);
  ws.idx.need(lists(nullptr));
  lists((char*)ws.idx.p);
  ws.scratch.need(wmu_csc_layout(nullptr, n_genes, nnz).bytes);
  const WmuCscScratch sc = wmu_csc_layout((char*)ws.scratch.p, n_genes, nnz);
  const size_t zc = (size_t)n_genes * C;
  ws.out.need(zc * 16 + (size_t)n_genes * 4 + 64);
  double* d_z = (double*)ws.out.p;
  double* d_ratio = d_z + zc;
  int* d_single = (int*)(d_ratio + zc);
  CU_TRY(cudaEventRecord(ws.ev[0], ws.s_comp));
  h2d_block(ws, colptr, N + 1, d_colptr, N + 1, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, row, nnz, d_row, nnz, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, x, nnz, d_x, nnz, 1, 8, ws.s_comp, /*ids=*/false);
  h2d_block(ws, cluster, N, d_cl, N, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, cl.crank.data(), N, d_crank, N, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, cl.members.data(), N, d_members, N, 1, 4, ws.s_comp, /*ids=*/false);
  h2d_block(ws, size.data(), C, d_size, C, 1, 8, ws.s_comp, /*ids=*/false);
  h2d_block(ws, cl.cptr.data(), C + 1, d_cptr, C + 1, 1, 8, ws.s_comp, /*ids=*/false);
  CU_TRY(cudaEventRecord(ws.ev[1], ws.s_comp));
  const WmuGeneMajor gm = wmu_csc_to_genes(ws.s_comp, sc, sm_count() * 8, d_colptr, d_row, d_x, n_genes, N, nnz);
  CU_TRY(cudaGetLastError());
  // the row-id flag and the gene pointers (they size the rank kernel's scratch) before anything reads them
  unsigned flags = 0;
  std::vector<long long> gptr((size_t)n_genes + 1);
  CU_TRY(cudaMemcpyAsync(&flags, sc.flags, 4, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaMemcpyAsync(gptr.data(), sc.gene_ptr, gptr.size() * 8, cudaMemcpyDeviceToHost, ws.s_comp));
  CU_TRY(cudaStreamSynchronize(ws.s_comp));
  if (flags & kFlagCscRow)
    throw Err{GFICF_E_ARG, "a row id is outside [0, n_genes) or row ids are not strictly increasing in a column"};
  const long long cap = wmu_gene_cap(gptr.data(), n_genes);
  CU_TRY(cudaFuncSetAttribute(wmu_markers_csr_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              kWmuMaxClusters * kWmuClusterSmemBytes));
  int per_sm = 0;
  CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wmu_markers_csr_rank_kernel, kWmuThreads,
                                                       (size_t)C * kWmuClusterSmemBytes));
  const int grid = (int)std::min<long long>(n_genes, (long long)std::max(1, per_sm) * sm_count());
  ws.counts.need((size_t)grid * 2 * cap * (sizeof(unsigned long long) + sizeof(unsigned)));
  unsigned long long* d_keys = (unsigned long long*)ws.counts.p;
  unsigned* d_pay = (unsigned*)(d_keys + (size_t)grid * 2 * cap);
  wmu_markers_csc_launch(ws.s_comp, grid, gm, sc.gene_ptr, n_genes, N, d_cl, d_crank, d_members, d_size, d_cptr,
                         n_clusters, cap, d_keys, d_pay, d_z, d_ratio, d_single);
  wmu_read_and_finish(ws, d_z, d_single, n_genes, n_clusters, out);
  call.timings(event_ms(ws.ev[0], ws.ev[1]), 0, event_ms(ws.ev[1], ws.ev[2]), 0,
               (double)(7 + 5 * ((bits_for(n_genes - 1) + 7) / 8)),
               (double)zc * 16 + (double)n_genes * 4 + 4 + (double)gptr.size() * 8);
  return GFICF_OK;
  API_END
}

}  // extern "C"
