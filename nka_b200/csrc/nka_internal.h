// nka_internal.h -- declarations shared by the translation units of libnka_b200.so.
#pragma once

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

// NVTX ranges (header-only NVTX3: no link dependency, a no-op unless a profiler is attached):
// "nka:accel_update" around an update, "nka:pass_a", "nka:state", "nka:pass_b", "nka:h2d/d2h" inside.
#include <nvtx3/nvToolsExt.h>
struct NkaRange {
  explicit NkaRange(const char* name) { nvtxRangePushA(name); }
  ~NkaRange() { nvtxRangePop(); }
  NkaRange(const NkaRange&) = delete;
  NkaRange& operator=(const NkaRange&) = delete;
};

[[noreturn]] void nka_fail(const char* file, int line, const char* msg);

#define NKA_REQUIRE(cond, msg) do { if (!(cond)) nka_fail(__FILE__, __LINE__, msg); } while (0)
#define CUDA_CHECK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) {                 \
    char b_[256]; snprintf(b_, sizeof b_, "%s failed: %s", #call, cudaGetErrorString(e_));      \
    nka_fail(__FILE__, __LINE__, b_); } } while (0)

// CUDA graphs (nka_capi.cu).  nka_capture_status: 1 while `stream` captures (an invalidated capture
// counts: it has not ended yet), 0 when not, -1 when `stream` is the legacy default stream while a
// blocking stream captures.  nka_refuse_capture aborts with a message naming `call` unless it is 0.
int nka_capture_status(cudaStream_t stream);
[[noreturn]] void nka_capture_fail(const char* call, const char* why);
void nka_refuse_capture(cudaStream_t stream, const char* call, const char* why);

// The device state as include/nka_b200.h shows it (nka_get_state, nka_batch_get_state).
struct NkaDevState;
struct nka_state_view;
void nka_state_view_from(const NkaDevState& h, nka_state_view* out);

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    CUDA_CHECK(cudaGetDevice(&prev));
    if (prev != dev) CUDA_CHECK(cudaSetDevice(dev)); else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// NCCL, resolved at run time (dlopen) so single-GPU users need no NCCL at all.
struct NkaId128 { char bytes[128]; };
struct NkaNcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NkaId128, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
extern NkaNcclApi g_nccl;
bool nka_nccl_load();
static const int kNcclFloat64 = 8;   // ncclDouble
static const int kNcclSum = 0;       // ncclSum
static const int kNcclMin = 3;       // ncclMin
static const int kNcclChar = 0;      // ncclInt8
static const int kNcclInt32 = 2;     // ncclInt32

// A reference-counted communicator shared by vectors cloned from one another and by the
// accelerator created from them.
struct NkaComm {
  void* comm = nullptr;
  bool owned = false;
  int nranks = 1, rank = 0;
  int refs = 1;
};
struct nka_state;
// an accelerator joins an existing communicator (a vector's, a slab system's): nka_capi.cu
void nka_attach_shared_comm(nka_state* st, NkaComm* c);
NkaComm* nka_comm_retain(NkaComm* c);
void nka_comm_release(NkaComm* c);

// Collective over the communicator: every rank offers one device allocation (cudaMalloc'ed, a
// multiple of 2 MiB of its own) and receives, in mapped[r] for each r with want[r], rank r's
// allocation mapped into this process (CUDA IPC; mapped[rank] = local).  The outcome is
// unanimous: returns false on EVERY rank (nothing left mapped) if any rank could not export or
// open what it wanted.  Unmap with nka_ipc_unmap.
bool nka_ipc_exchange(NkaComm* c, cudaStream_t stream, void* local, void** mapped, const bool* want);
void nka_ipc_unmap(NkaComm* c, void** mapped);
