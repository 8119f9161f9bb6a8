// nccl_dyn.h -- NCCL bound at run time (dlopen), so the library loads on a
// single-GPU host without libnccl and never conflicts with the NCCL a host
// process (e.g. PyTorch) already carries.  Only the entry points the multi-GPU
// paths need: communicator setup for the GPUs of one process, all-gather of the
// int32 index slabs, broadcast, and the point-to-point exchange of the sparse
// markers call's gene blocks.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stddef.h>

// The handful of NCCL declarations this file needs, restated from NCCL's public, ABI-stable C
// interface (nccl.h of NCCL 2.x) so that building the library needs no NCCL headers: NCCL is a
// RUN-time dependency of the multi-GPU calls only.  -DGFICF_USE_NCCL_HEADER takes them from <nccl.h>.
#ifdef GFICF_USE_NCCL_HEADER
#include <nccl.h>
#else
extern "C" {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;  // every other value is an error; text from ncclGetErrorString
typedef enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclUint32 = 3, ncclInt64 = 4, ncclUint64 = 5,
               ncclFloat16 = 6, ncclFloat32 = 7, ncclFloat64 = 8 } ncclDataType_t;
typedef enum { ncclSum = 0, ncclProd = 1, ncclMax = 2, ncclMin = 3, ncclAvg = 4 } ncclRedOp_t;
}
#endif

#include <string>

namespace nccl_dyn {

struct Api {
  bool ok = false;
  std::string why;
  void* handle = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;

  Api() {
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) {
      const char* e = dlerror();
      why = e ? e : "dlopen failed";
      return;
    }
#define GFICF_NCCL_SYM(field, sym)                           \
  field = reinterpret_cast<decltype(field)>(dlsym(handle, sym)); \
  if (!field) {                                              \
    why = std::string("missing symbol ") + sym;              \
    return;                                                  \
  }
    GFICF_NCCL_SYM(CommInitAll, "ncclCommInitAll")
    GFICF_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    GFICF_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    GFICF_NCCL_SYM(AllReduce, "ncclAllReduce")
    GFICF_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    GFICF_NCCL_SYM(AllGather, "ncclAllGather")
    GFICF_NCCL_SYM(Broadcast, "ncclBroadcast")
    GFICF_NCCL_SYM(Send, "ncclSend")
    GFICF_NCCL_SYM(Recv, "ncclRecv")
    GFICF_NCCL_SYM(GroupStart, "ncclGroupStart")
    GFICF_NCCL_SYM(GroupEnd, "ncclGroupEnd")
    GFICF_NCCL_SYM(GetErrorString, "ncclGetErrorString")
    GFICF_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef GFICF_NCCL_SYM
    ok = true;
  }
};

inline Api& get() {
  static Api api;
  return api;
}

}  // namespace nccl_dyn
