// plan_common.h -- what the launch plans (jaccard_plan.h, network_plan.h, snn_plan.h, wmu_csc_plan.h) are written
// in: a stream, launches, fills and copies, occupancy, one way to carve scratch, and the error of a size the
// path does not support.  In the product (gficf_cuda.cu, which includes the plans after its error helpers) they
// are CUDA calls; with GFICF_CUDA_EMU (tests/cuda_emu) they run on the CPU emulation, so the CPU test suite runs
// the same launch sequences as the B200.
#pragma once
#include <stddef.h>
#include <string.h>

#ifdef GFICF_CUDA_EMU
#include "cuda_emu.h"
typedef int net_stream_t;
#define GFICF_LAUNCH(st, kernel, grid, block, ...) \
  cuda_emu::launch((unsigned)(grid), (unsigned)(block), [=] { kernel(__VA_ARGS__); })
// 2-D grid (grid_x, grid_y) and `smem` bytes of dynamic shared memory
#define GFICF_LAUNCH_EX(st, kernel, grid_x, grid_y, block, smem, ...)                                    \
  cuda_emu::launch((unsigned)(grid_x), (unsigned)(block), [=] { kernel(__VA_ARGS__); }, (size_t)(smem), \
                   (unsigned)(grid_y))
inline void net_fill(net_stream_t, void* p, int byte, size_t bytes) { memset(p, byte, bytes); }
inline void net_copy(net_stream_t, void* dst, const void* src, size_t bytes) { memcpy(dst, src, bytes); }
inline void net_read(net_stream_t, void* host, const void* dev, size_t bytes) { memcpy(host, dev, bytes); }
inline void net_check_launches() {}
// the emulation runs one CTA at a time: one resident CTA per SM, so a persistent grid is the emulated SM count
template <class K>
inline int net_occupancy(K, int, size_t) { return 1; }
template <class K>
inline void net_max_dynamic_smem(K, size_t) {}
[[noreturn]] inline void net_limit(const char* msg) { cuda_emu::die(msg); }
#else
typedef cudaStream_t net_stream_t;
#define GFICF_LAUNCH(st, kernel, grid, block, ...) kernel<<<(unsigned)(grid), (unsigned)(block), 0, (st)>>>(__VA_ARGS__)
#define GFICF_LAUNCH_EX(st, kernel, grid_x, grid_y, block, smem, ...) \
  kernel<<<dim3((unsigned)(grid_x), (unsigned)(grid_y)), (unsigned)(block), (size_t)(smem), (st)>>>(__VA_ARGS__)
inline void net_fill(net_stream_t st, void* p, int byte, size_t bytes) { CU_TRY(cudaMemsetAsync(p, byte, bytes, st)); }
inline void net_copy(net_stream_t st, void* dst, const void* src, size_t bytes) {
  CU_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st));
}
// the few scalars the host needs to size the next launches (entry counts): one small synchronous read
inline void net_read(net_stream_t st, void* host, const void* dev, size_t bytes) {
  CU_TRY(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
}
inline void net_check_launches() { CU_TRY(cudaGetLastError()); }
// resident CTAs per SM of `kernel` at `block` threads and `smem` bytes of dynamic shared memory
template <class K>
inline int net_occupancy(K kernel, int block, size_t smem) {
  int per_sm = 0;
  CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
  return per_sm;
}
// lets `kernel` launch with `bytes` of dynamic shared memory (above the default 48 KiB)
template <class K>
inline void net_max_dynamic_smem(K kernel, size_t bytes) { set_max_dynamic_smem((const void*)kernel, bytes); }
// a size beyond what the path supports: GFICF_E_LIMIT
[[noreturn]] inline void net_limit(const char* msg) { throw Err{GFICF_E_LIMIT, msg}; }
#endif
inline void net_zero(net_stream_t st, void* p, size_t bytes) { net_fill(st, p, 0, bytes); }

// Test builds only (tests/cuda_emu, AddressSanitizer): every scratch piece is followed by a red zone and
// only the pieces themselves are addressable, so a kernel that runs past its piece is reported.
#ifdef GFICF_NET_ASAN
#include <sanitizer/asan_interface.h>
#define GFICF_NET_REDZONE 256
#else
#define GFICF_NET_REDZONE 0
#endif

namespace gficf {

inline size_t align256(size_t bytes) { return (bytes + 255) / 256 * 256; }

// Carves pieces out of one buffer in order, each starting 256-byte aligned; with base == nullptr it only
// counts: `bytes` is then the size the buffer needs.
struct ScratchCarver {
  char* base;
  size_t bytes = 0;
  template <class T>
  T* take(size_t count) {
    char* p = base + bytes;
    bytes += align256(count * sizeof(T) + GFICF_NET_REDZONE);
#ifdef GFICF_NET_ASAN
    if (base) __asan_unpoison_memory_region(p, count * sizeof(T));
#endif
    return reinterpret_cast<T*>(p);
  }
};

}  // namespace gficf
