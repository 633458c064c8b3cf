// nka_capi.cu -- the C-ABI of libnka_b200.so: handle management, kernel
// dispatch, host<->device staging, the optional NCCL reduction of the partial
// dot products, and introspection.  Declarations: include/*.h.
//
// There is deliberately no CPU implementation of accel_update in this library:
// without a CUDA device every entry point that computes aborts with a message.

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/nka_b200.h"
#include "nka_internal.h"
#include "nka_dispatch.h"
#include "nka_aux_kernels.cuh"
#include "nka_hostcopy.h"

#define NKA_VERSION "nka_b200 0.1 (sm_100a)"

[[noreturn]] void nka_fail(const char* file, int line, const char* msg)
{
  // the reference's convention: "Assertion failed at file:line" then stop
  // (src-F08/f90_assert.F90:37-47); we abort so the failure cannot be ignored.
  fprintf(stderr, "nka_b200: %s:%d: %s\n", file, line, msg);
  fflush(stderr);
  abort();
}

// ---------------------------------------------------------------------------
// kernel dispatch (tables live in nka_pass_a.cu / nka_pass_b.cu)
// ---------------------------------------------------------------------------
#ifndef NKA_WAVES
#define NKA_WAVES 8          // CTAs per SM = resident CTAs x NKA_WAVES
#endif
static bool g_tables_ready = false;
static int g_grid_per_sm_a = 0, g_grid_per_sm_b = 0;   // 0 = occupancy-derived; env overrides for tuning
#ifdef NKA_EXPERIMENT_PDL
static bool g_pdl = true;                              // tuning builds only (nka_kernels.cuh: not kept); NKA_PDL=0 turns it off
#else
static const bool g_pdl = false;
#endif
static bool g_pass_b_tma = false;                      // NKA_PASS_B_TMA=1: the cp.async.bulk staging experiment
static void ensure_tables()
{
  if (!g_tables_ready) {
    if (const char* e = getenv("NKA_GRID_PER_SM_A")) g_grid_per_sm_a = atoi(e);
    if (const char* e = getenv("NKA_GRID_PER_SM_B")) g_grid_per_sm_b = atoi(e);
#ifdef NKA_EXPERIMENT_PDL
    if (const char* e = getenv("NKA_PDL")) g_pdl = atoi(e) != 0;
#endif
    if (const char* e = getenv("NKA_PASS_B_TMA")) g_pass_b_tma = atoi(e) != 0;
    g_tables_ready = true;
  }
}

// Plain stream-ordered launch.  (Tuning builds with -DNKA_EXPERIMENT_PDL add the programmatic stream
// serialization attribute: see nka_kernels.cuh, an experiment that was not kept.)
template <typename... KArgs, typename... Args>
static void launch_chained_smem(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t stream, Args... args)
{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_pdl ? 1 : 0;
  CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...));
}

template <typename... KArgs, typename... Args>
static void launch_chained(void (*kernel)(KArgs...), int grid, int block, cudaStream_t stream, Args... args)
{
  launch_chained_smem(kernel, grid, block, 0, stream, args...);
}

// ---------------------------------------------------------------------------
// NCCL, resolved at run time so single-GPU users need no NCCL at all
// ---------------------------------------------------------------------------
NkaNcclApi g_nccl;

bool nka_nccl_load()
{
  if (g_nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) return false;
  g_nccl.GetUniqueId = (int (*)(void*))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(void**, int, NkaId128, int))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
  g_nccl.Send = (int (*)(const void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclSend");
  g_nccl.Recv = (int (*)(void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclRecv");
  g_nccl.GroupStart = (int (*)())dlsym(g_nccl.lib, "ncclGroupStart");
  g_nccl.GroupEnd = (int (*)())dlsym(g_nccl.lib, "ncclGroupEnd");
  g_nccl.CommDestroy = (int (*)(void*))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
  return g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllReduce && g_nccl.CommDestroy;
}

NkaComm* nka_comm_retain(NkaComm* c) { if (c) c->refs += 1; return c; }
void nka_comm_release(NkaComm* c)
{
  if (!c) return;
  if (--c->refs == 0) {
    if (c->comm && c->owned && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    delete c;
  }
}

// ---------------------------------------------------------------------------
// the handle
// ---------------------------------------------------------------------------
enum { T_PASS_A = 0, T_STATE = 1, T_MAT = 2, T_PASS_B = 3, T_COMM = 4, T_NKIND = 5 };

struct TimedSpan { cudaEvent_t beg, end; int kind; };

struct nka_state {
  size_t vlen = 0, ld = 0;
  int mvec = 0;
  double vtol = 0.01;
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  double* W = nullptr;          // (mvec+1) columns of ld doubles: raw cached inputs / differences
  double* Z = nullptr;          // (mvec+1) columns of ld doubles: corrections
  NkaDevState* S = nullptr;     // device
  double* dots = nullptr;       // device, 2*NKA_MAXSLOT
  double* partials = nullptr;   // device, max_grid * 2*NKA_MAXSLOT
  unsigned* ticket = nullptr;   // device
  double* fstage = nullptr;     // device staging for host callers, vlen doubles (lazy)
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   // host callers: PCIe copies overlapped with the sweeps (lazy)
  cudaEvent_t chunk_ev[16] = {};
  cudaEvent_t order_ev = nullptr;
  size_t host_chunk_bytes = 0;
  // pageable host callers: pinned staging slots the host threads copy through (lazy)
  double* hslot[3] = {nullptr, nullptr, nullptr};
  size_t hslot_bytes = 0;
  cudaEvent_t hslot_ev[3] = {};
  int max_grid = 0;
  // host-side knowledge of the device list: exact `pending`, upper bound on its length
  bool pending = false;
  int ub_len = 0;
  bool lazy = true;             // skip the doomed oldest column in pass A (single GPU only)
  bool poison = false;          // NKA_POISON_ALLOC=1 (tests): data buffers start as NaN bytes, see poison_fill
  // the reference's dp hook: global sum of each partial dot product through a host callback
  double (*dp)(int, double*, double*) = nullptr;
  double (*dp_ctx)(int, double*, double*, void*) = nullptr;
  void* dp_user = nullptr;
  double* dots_host = nullptr;  // pinned, 2*NKA_MAXSLOT
  // distributed
  NkaComm* comm = nullptr;
  // peer-memory reduction fused into pass A (all ranks on one NVLink domain); else NCCL
  NkaPeerCtx* peer = nullptr;   // device copy of the context; nullptr = not in use
  void* peer_box = nullptr;     // this rank's exchange box (device memory, IPC-exported)
  void* peer_mapped[NKA_MAX_RANKS] = {};   // the peers' boxes as opened here
  int peer_n = 0;
  // accounting
  unsigned long long launches = 0;
  bool timing = false;
  std::vector<TimedSpan> spans;
  std::vector<cudaEvent_t> free_events;
  double t_ms[T_NKIND] = {0, 0, 0, 0, 0};
  unsigned long long t_cnt[T_NKIND] = {0, 0, 0, 0, 0};
  int occ_a[NKA_MAXSLOT + 1][3];
  int occ_b[NKA_MAXSLOT + 1][3];
};

static cudaEvent_t get_event(NKA st)
{
  if (!st->free_events.empty()) { cudaEvent_t e = st->free_events.back(); st->free_events.pop_back(); return e; }
  cudaEvent_t e;
  CUDA_CHECK(cudaEventCreate(&e));
  return e;
}

static void fold_timing(NKA st)
{
  if (st->spans.empty()) return;
  CUDA_CHECK(cudaStreamSynchronize(st->stream));
  for (const TimedSpan& sp : st->spans) {
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, sp.beg, sp.end));
    st->t_ms[sp.kind] += ms;
    st->t_cnt[sp.kind] += 1;
    st->free_events.push_back(sp.beg);
    st->free_events.push_back(sp.end);
  }
  st->spans.clear();
}

struct SpanScope {
  NKA st; int kind; cudaEvent_t beg = nullptr;
  SpanScope(NKA s, int k) : st(s), kind(k) {
    if (st->timing) { beg = get_event(st); CUDA_CHECK(cudaEventRecord(beg, st->stream)); }
  }
  ~SpanScope() {
    if (beg) {
      cudaEvent_t end = get_event(st);
      CUDA_CHECK(cudaEventRecord(end, st->stream));
      st->spans.push_back({beg, end, kind});
      if (st->spans.size() >= 8192) fold_timing(st);
    }
  }
};

static int grid_for(NKA st, int per_sm, size_t n, int V, int threads = NKA_THREADS)
{
  const size_t nv = n / V;
  size_t need = (nv + threads - 1) / threads;
  if (need < 1) need = 1;
  size_t full = (size_t)st->num_sms * (per_sm > 0 ? per_sm : 1);
  size_t g = need < full ? need : full;
  if (g > (size_t)st->max_grid) g = st->max_grid;
  return (int)g;
}

// CTAs per SM for a sweep over n elements = resident CTAs x waves.  Several waves even out the
// tail of a long grid-stride sweep (+1 % at n = 2^28 with 8 waves), but every wave costs each SM one
// more prologue / reduction epilogue and the last CTA one more partial row to fold: at n = 2^25
// one wave is 2.6 % faster than eight, at 2^24 5.5 % (profiles/r1i_waves_sweep.txt).  So: one
// wave per ~2^17 double2 per SM.
static int waves_for(NKA st, size_t n, int V)
{
  const size_t per_wave = (size_t)st->num_sms * 113000u;
  size_t w = (n / V) / per_wave;
  if (w < 1) w = 1;
  if (w > NKA_WAVES) w = NKA_WAVES;
  return (int)w;
}

static int resident_a(NKA st, int nc, int V)
{
  if (st->occ_a[nc][V] < 0) {
    int nb = 0;
    NKA_REQUIRE(nka_get_pass_a(nc, V) != nullptr, "pass A is not instantiated for this subspace size in this build");
    CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, nka_get_pass_a(nc, V), NKA_THREADS_A, 0));
    st->occ_a[nc][V] = nb > 0 ? nb : 1;
  }
  return st->occ_a[nc][V];
}

static int resident_b(NKA st, int nz, int V)
{
  if (st->occ_b[nz][V] < 0) {
    int nb = 0;
    NKA_REQUIRE(nka_get_pass_b(nz, V) != nullptr, "pass B is not instantiated for this subspace size in this build");
    CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, nka_get_pass_b(nz, V), nka_threads_b(nz), 0));
    st->occ_b[nz][V] = nb > 0 ? nb : 1;
  }
  return st->occ_b[nz][V];
}

static int per_sm_a(NKA st, int nc, int V, size_t len)
{
  return g_grid_per_sm_a > 0 ? g_grid_per_sm_a : resident_a(st, nc, V) * waves_for(st, len, V);
}

static int per_sm_b(NKA st, int nz, int V, size_t len)
{
  return g_grid_per_sm_b > 0 ? g_grid_per_sm_b : resident_b(st, nz, V) * waves_for(st, len, V);
}

// How many pairs are expected on the list at entry (pass B streams their Z columns): exact
// unless a vtol drop fired earlier on the device (pass B copes with any actual count).
static int nz_expected(NKA st)
{
  const int nz = st->pending ? st->ub_len - 1 : st->ub_len;
  return nz < 0 ? 0 : (nz > st->mvec ? st->mvec : nz);
}

// ---------------------------------------------------------------------------
// peer-memory exchange boxes (multi-GPU, one process per GPU, one NVLink domain)
// ---------------------------------------------------------------------------
static const size_t kPeerBoxBytes = 2u << 20;    // a whole 2 MiB allocation of its own: what CUDA IPC exports

static void peer_teardown(NKA st)
{
  if (!st->peer && !st->peer_box) return;
  DeviceGuard guard(st->device);
  cudaStreamSynchronize(st->stream);
  for (int r = 0; r < st->peer_n; ++r)
    if (st->peer_mapped[r]) { cudaIpcCloseMemHandle(st->peer_mapped[r]); st->peer_mapped[r] = nullptr; }
  cudaFree(st->peer); st->peer = nullptr;
  cudaFree(st->peer_box); st->peer_box = nullptr;
  st->peer_n = 0;
  cudaGetLastError();
}

void nka_ipc_unmap(NkaComm* c, void** mapped)
{
  for (int r = 0; r < c->nranks; ++r)
    if (r != c->rank && mapped[r]) { cudaIpcCloseMemHandle(mapped[r]); mapped[r] = nullptr; }
  cudaGetLastError();
}

bool nka_ipc_exchange(NkaComm* c, cudaStream_t stream, void* local, void** mapped, const bool* want)
{
  const int R = c->nranks, me = c->rank;
  struct Card { cudaIpcMemHandle_t h; int ok; int pad; };
  Card mine;
  memset(&mine, 0, sizeof mine);
  mine.ok = (local != nullptr && g_nccl.AllGather != nullptr) ? 1 : 0;
  if (mine.ok && cudaIpcGetMemHandle(&mine.h, local) != cudaSuccess) { cudaGetLastError(); mine.ok = 0; }
  for (int r = 0; r < R; ++r) mapped[r] = nullptr;
  if (!g_nccl.AllGather) return false;             // same library on every rank: unanimous
  Card* d_cards = nullptr;
  int* d_flag = nullptr;
  CUDA_CHECK(cudaMalloc(&d_cards, sizeof(Card) * (R + 1)));
  CUDA_CHECK(cudaMalloc(&d_flag, sizeof(int)));
  CUDA_CHECK(cudaMemcpyAsync(d_cards + R, &mine, sizeof mine, cudaMemcpyHostToDevice, stream));
  int rc = g_nccl.AllGather(d_cards + R, d_cards, sizeof(Card), kNcclChar, c->comm, stream);
  if (rc != 0) nka_fail(__FILE__, __LINE__, "ncclAllGather (IPC handles) failed");
  std::vector<Card> cards(R);
  CUDA_CHECK(cudaMemcpyAsync(cards.data(), d_cards, sizeof(Card) * R, cudaMemcpyDeviceToHost, stream));
  CUDA_CHECK(cudaStreamSynchronize(stream));
  int ok = 1;
  for (int r = 0; r < R; ++r) ok &= cards[r].ok;
  if (ok) {
    mapped[me] = local;
    for (int r = 0; r < R; ++r) {
      if (r == me || !want[r]) continue;
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, cards[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        ok = 0;
        break;
      }
      mapped[r] = p;
    }
  }
  CUDA_CHECK(cudaMemcpyAsync(d_flag, &ok, sizeof ok, cudaMemcpyHostToDevice, stream));
  rc = g_nccl.AllReduce(d_flag, d_flag, 1, kNcclInt32, kNcclMin, c->comm, stream);
  if (rc != 0) nka_fail(__FILE__, __LINE__, "ncclAllReduce (IPC agreement) failed");
  CUDA_CHECK(cudaMemcpyAsync(&ok, d_flag, sizeof ok, cudaMemcpyDeviceToHost, stream));
  CUDA_CHECK(cudaStreamSynchronize(stream));
  cudaFree(d_cards);
  cudaFree(d_flag);
  if (!ok) { nka_ipc_unmap(c, mapped); mapped[me] = nullptr; return false; }
  return true;
}

// Collective over the communicator.  Every rank allocates a box, the IPC handles are
// all-gathered with NCCL, every rank opens every peer's box, and an all-reduce(min) makes the
// outcome unanimous: either every rank reduces through peer memory or every rank stays on NCCL.
static bool peer_setup(NKA st)
{
  static_assert(sizeof(uint4) * NKA_PEER_BOX_WORDS16 <= kPeerBoxBytes, "exchange box does not fit its allocation");
  NkaComm* c = st->comm;
  if (!c || !g_nccl.AllGather) return false;
  if (const char* e = getenv("NKA_PEER_REDUCE")) if (atoi(e) == 0) return false;    // ablation: NCCL all-reduce
  if (c->nranks < 2 || c->nranks > NKA_MAX_RANKS) return false;
  const int R = c->nranks, me = c->rank;
  if (cudaMalloc(&st->peer_box, kPeerBoxBytes) != cudaSuccess) { cudaGetLastError(); st->peer_box = nullptr; }
  if (st->peer_box) {
    CUDA_CHECK(cudaMemsetAsync(st->peer_box, 0, kPeerBoxBytes, st->stream));
    CUDA_CHECK(cudaStreamSynchronize(st->stream));
  }
  bool want[NKA_MAX_RANKS];
  for (int r = 0; r < NKA_MAX_RANKS; ++r) want[r] = true;
  st->peer_n = R;
  if (!nka_ipc_exchange(c, st->stream, st->peer_box, st->peer_mapped, want)) {
    st->peer_mapped[me] = nullptr;
    peer_teardown(st);
    return false;
  }
  NkaPeerCtx ctx;
  memset(&ctx, 0, sizeof ctx);
  ctx.nranks = R; ctx.rank = me; ctx.epoch = 0; ctx.timed_out = 0;
  double timeout_s = 120.0;                       // NKA_PEER_TIMEOUT_S: how long to wait for a peer before trapping
  if (const char* e = getenv("NKA_PEER_TIMEOUT_S")) if (atof(e) > 0.0) timeout_s = atof(e);
  ctx.timeout_ns = (unsigned long long)(timeout_s * 1e9);
  for (int r = 0; r < R; ++r) ctx.box[r] = st->peer_mapped[r];
  st->peer_mapped[me] = nullptr;                  // own box: freed, not unmapped
  CUDA_CHECK(cudaMalloc(&st->peer, sizeof(NkaPeerCtx)));
  CUDA_CHECK(cudaMemcpyAsync(st->peer, &ctx, sizeof ctx, cudaMemcpyHostToDevice, st->stream));
  CUDA_CHECK(cudaStreamSynchronize(st->stream));
  return true;
}

// ---------------------------------------------------------------------------
// construction / destruction
// ---------------------------------------------------------------------------
// Test switch NKA_POISON_ALLOC=1: fill a freshly allocated data buffer with 0xFF bytes (a NaN for
// fp64) instead of leaving it as cudaMalloc returns it, which usually reads as zero.  A kernel that
// reads a value it has not written then yields NaN in place of a silent zero.  Only buffers of
// values are filled: never the state, the ticket or anything else read as an index or a counter.
static void poison_fill(NKA st, void* p, size_t bytes)
{
  if (st->poison) CUDA_CHECK(cudaMemsetAsync(p, 0xFF, bytes, st->stream));
}

extern "C" NKA nka_init_ex(size_t vlen, int mvec, double vtol, int device, void* stream)
{
  // preconditions: src-C/...c:217-219 ; src-F08/nka_type.F90:190-191,205
  NKA_REQUIRE(mvec > 0, "nka_init: mvec must be > 0");
  NKA_REQUIRE(mvec <= NKA_B200_MAX_MVEC, "nka_init: mvec > 32 is not supported by this build");
  NKA_REQUIRE(vtol > 0.0, "nka_init: vtol must be > 0");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    nka_fail(__FILE__, __LINE__, "no CUDA device: libnka_b200 has no CPU compute path");
  ensure_tables();

  NKA st = new nka_state();
  if (device < 0) CUDA_CHECK(cudaGetDevice(&device));
  st->device = device;
  DeviceGuard guard(device);
  CUDA_CHECK(cudaDeviceGetAttribute(&st->num_sms, cudaDevAttrMultiProcessorCount, device));
  st->vlen = vlen;
  st->mvec = mvec;
  st->vtol = vtol;
  st->ld = ((vlen + 15) / 16) * 16;                 // 128-byte aligned columns
  if (st->ld == 0) st->ld = 16;
  // NULL = the legacy default stream: ordered after everything the caller queued on it
  // (and on other blocking streams), like the synchronous CPU interface it replaces
  st->stream = (cudaStream_t)stream;
  st->own_stream = false;
  for (int i = 0; i <= NKA_MAXSLOT; ++i)
    for (int v = 0; v < 3; ++v) { st->occ_a[i][v] = -1; st->occ_b[i][v] = -1; }
  if (const char* e = getenv("NKA_LAZY_LAST")) st->lazy = atoi(e) != 0;      // ablation switch
  if (const char* e = getenv("NKA_POISON_ALLOC")) st->poison = atoi(e) != 0;

  const size_t colbytes = st->ld * sizeof(double);
  const size_t poolbytes = colbytes * (size_t)(mvec + 1);
  e = cudaMalloc(&st->W, poolbytes);
  if (e == cudaSuccess) e = cudaMalloc(&st->Z, poolbytes);
  if (e != cudaSuccess) {
    char b[200];
    snprintf(b, sizeof b, "nka_init: cannot allocate 2 x %zu bytes of device memory for the subspace: %s",
             poolbytes, cudaGetErrorString(e));
    nka_fail(__FILE__, __LINE__, b);
  }
  st->max_grid = st->num_sms * 32;
  CUDA_CHECK(cudaMalloc(&st->S, sizeof(NkaDevState)));
  CUDA_CHECK(cudaMalloc(&st->dots, 2 * NKA_MAXSLOT * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&st->partials, (size_t)st->max_grid * 2 * NKA_MAXSLOT * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&st->ticket, sizeof(unsigned)));
  CUDA_CHECK(cudaMemsetAsync(st->ticket, 0, sizeof(unsigned), st->stream));
  CUDA_CHECK(cudaMemsetAsync(st->dots, 0, 2 * NKA_MAXSLOT * sizeof(double), st->stream));
  poison_fill(st, st->W, poolbytes);
  poison_fill(st, st->Z, poolbytes);
  poison_fill(st, st->partials, (size_t)st->max_grid * 2 * NKA_MAXSLOT * sizeof(double));
  poison_fill(st, st->dots, 2 * NKA_MAXSLOT * sizeof(double));
  nka_init_kernel<<<1, 32, 0, st->stream>>>(st->S, mvec, vtol, st->lazy ? 1 : 0);
  CUDA_CHECK(cudaGetLastError());
  st->launches += 1;
  st->pending = false;
  st->ub_len = 0;
  return st;
}

static void set_lazy(NKA st, bool on)
{
  st->lazy = on;
  nka_set_lazy_kernel<<<1, 32, 0, st->stream>>>(st->S, on ? 1 : 0);
  CUDA_CHECK(cudaGetLastError());
  st->launches += 1;
}

static void install_dp(NKA st, double (*dp)(int, double*, double*), double (*dp_ctx)(int, double*, double*, void*), void* user)
{
  NKA_REQUIRE(st->comm == nullptr || (!dp && !dp_ctx),
              "nka_set_dot_prod: the handle already sums over ranks through nka_comm_init; use one or the other");
  DeviceGuard guard(st->device);
  st->dp = dp; st->dp_ctx = dp_ctx; st->dp_user = user;
  // the lazily skipped oldest column would need a second, conditional reduction: not with a host callback
  bool lazy = !(dp || dp_ctx);
  if (lazy) if (const char* e = getenv("NKA_LAZY_LAST")) lazy = atoi(e) != 0;
  set_lazy(st, lazy);
}

extern "C" void nka_set_dot_prod(NKA st, double (*dp)(int, double*, double*))
{
  NKA_REQUIRE(st != NULL, "nka_set_dot_prod: null handle");
  install_dp(st, dp, nullptr, nullptr);
}

extern "C" void nka_set_dot_prod_ctx(NKA st, double (*dp)(int, double*, double*, void*), void* ctx)
{
  NKA_REQUIRE(st != NULL, "nka_set_dot_prod_ctx: null handle");
  install_dp(st, nullptr, dp, ctx);
}

extern "C" NKA nka_init(int vlen, int mvec, double vtol, double (*dp)(int, double*, double*))
{
  // src-C/nonlinear_krylov_accelerator.c:211-258; dp: :227-231 (NULL selects the built-in reductions)
  NKA_REQUIRE(vlen >= 0, "nka_init: vlen must be >= 0");
  NKA st = nka_init_ex((size_t)vlen, mvec, vtol, -1, NULL);
  if (dp) install_dp(st, dp, nullptr, nullptr);
  return st;
}

extern "C" void nka_delete(NKA st)
{
  if (!st) return;
  DeviceGuard guard(st->device);
  cudaStreamSynchronize(st->stream);
  for (const TimedSpan& sp : st->spans) { cudaEventDestroy(sp.beg); cudaEventDestroy(sp.end); }
  for (cudaEvent_t ev : st->free_events) cudaEventDestroy(ev);
  peer_teardown(st);
  nka_comm_release(st->comm);
  cudaFree(st->W); cudaFree(st->Z); cudaFree(st->S); cudaFree(st->dots);
  cudaFree(st->partials); cudaFree(st->ticket); cudaFree(st->fstage);
  if (st->dots_host) cudaFreeHost(st->dots_host);
  for (int i = 0; i < 3; ++i) {
    if (st->hslot[i]) cudaFreeHost(st->hslot[i]);
    if (st->hslot_ev[i]) cudaEventDestroy(st->hslot_ev[i]);
  }
  if (st->copy_in) {
    cudaStreamDestroy(st->copy_in); cudaStreamDestroy(st->copy_out);
    for (cudaEvent_t ev : st->chunk_ev) cudaEventDestroy(ev);
    cudaEventDestroy(st->order_ev);
  }
  if (st->own_stream) cudaStreamDestroy(st->stream);
  delete st;
}

// ---------------------------------------------------------------------------
// the hot path
// ---------------------------------------------------------------------------
// One update = pass A (+ exchange + state step), [fix-up], pass B.  Both sweeps are element-wise,
// so either may be cut into chunks [off, off+len) of the vector launched one after the other on
// the handle's stream: the host-pointer path does that to overlap them with the PCIe copies.
struct UpdateShape {
  int V, L, NC, nz;
  bool fused, may_skip;
};

static UpdateShape update_shape(NKA st, const double* f)
{
  UpdateShape u;
  u.V = (((uintptr_t)f) % 16 == 0) ? 2 : 1;
  u.L = st->ub_len;                               // upper bound on the list length at entry
  // fused = the dot products are complete when pass A's last CTA has them (single GPU, or
  // summed over the ranks through peer memory inside pass A): state step in place, lazy last column
  u.fused = ((st->comm == nullptr) || (st->peer != nullptr)) && !st->dp && !st->dp_ctx;
  u.may_skip = u.fused && st->lazy && st->pending && u.L == st->mvec + 1;
  u.NC = u.may_skip ? st->mvec : u.L;             // columns pass A can be asked to stream
  u.nz = nz_expected(st);
  return u;
}

// Pass A over elements [off, off+len).  row0 = partial rows written by earlier chunks of this
// sweep; final: this launch folds all rows and carries on to the exchange / state step.
static int launch_pass_a(NKA st, const UpdateShape& u, double* f, size_t off, size_t len, int grid_cap, int row0, bool final)
{
  int grid = grid_for(st, per_sm_a(st, u.NC, u.V, len), len, u.V, NKA_THREADS_A);
  if (grid_cap > 0 && grid > grid_cap) grid = grid_cap;
  NKA_REQUIRE(row0 + grid <= st->max_grid, "pass A: too many partial rows");
  double* rows = st->partials + (size_t)row0 * 2 * u.NC;
  NkaRange nvtx("nka:pass_a");
  SpanScope t(st, T_PASS_A);
  launch_chained(nka_get_pass_a(u.NC, u.V), grid, NKA_THREADS_A, st->stream,
                 f + off, st->W + off, st->ld, len, st->S, rows, st->ticket, st->dots, u.fused ? 1 : 0, st->peer,
                 st->partials, final ? (unsigned)(row0 + grid) : 0u);
  st->launches += 1;
  return grid;
}

// What sits between the sweeps: the cross-rank sum and the scalar step when they are not fused
// into pass A, the fix-up for the lazily skipped column, or the bare state step of a first call.
static void launch_mid(NKA st, const UpdateShape& u, double* f)
{
  NkaRange nvtx("nka:state");
  const size_t n = st->vlen;
  if (u.L > 0) {
    if (!u.fused && (st->dp || st->dp_ctx)) {
      // the caller's reduction: every partial dot product becomes global through dp(1, &p, &1.0)
      {
        SpanScope t(st, T_COMM);
        const size_t bytes = 2 * NKA_MAXSLOT * sizeof(double);
        if (!st->dots_host) CUDA_CHECK(cudaMallocHost(&st->dots_host, bytes));
        CUDA_CHECK(cudaMemcpyAsync(st->dots_host, st->dots, bytes, cudaMemcpyDeviceToHost, st->stream));
        CUDA_CHECK(cudaStreamSynchronize(st->stream));
        double one = 1.0;
        for (int half = 0; half < 2; ++half)
          for (int j = 0; j < u.L; ++j) {
            double* p = st->dots_host + half * NKA_MAXSLOT + j;
            double part = *p;
            *p = st->dp ? st->dp(1, &part, &one) : st->dp_ctx(1, &part, &one, st->dp_user);
          }
        CUDA_CHECK(cudaMemcpyAsync(st->dots, st->dots_host, bytes, cudaMemcpyHostToDevice, st->stream));
      }
      SpanScope t(st, T_STATE);
      launch_chained(nka_state_kernel, 1, NKA_STATE_THREADS, st->stream, st->S, st->dots, 1);
      st->launches += 1;
    } else if (!u.fused) {
      {
        SpanScope t(st, T_COMM);
        const int rc = g_nccl.AllReduce(st->dots, st->dots, 2 * NKA_MAXSLOT, kNcclFloat64, kNcclSum, st->comm->comm, st->stream);
        if (rc != 0) nka_fail(__FILE__, __LINE__, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "ncclAllReduce failed");
      }
      SpanScope t(st, T_STATE);
      launch_chained(nka_state_kernel, 1, NKA_STATE_THREADS, st->stream, st->S, st->dots, 1);
      st->launches += 1;
    } else if (u.may_skip) {
      // the oldest column was left out of pass A; this exits at once unless a vtol drop
      // (or the s == 0 guard) means it is needed after all
      SpanScope t(st, T_STATE);
      launch_chained(nka_fixup_kernel, grid_for(st, 4, n, 1), NKA_THREADS, st->stream, f, st->W, st->ld, n, st->S,
                     st->partials, st->ticket, st->dots, st->peer);
      st->launches += 1;
    }
  } else {
    SpanScope t(st, T_STATE);
    launch_chained(nka_state_kernel, 1, NKA_STATE_THREADS, st->stream, st->S, st->dots, 1);
    st->launches += 1;
  }
}

static void launch_pass_b(NKA st, const UpdateShape& u, double* f, size_t off, size_t len)
{
  NkaRange nvtx("nka:pass_b");
  SpanScope t(st, T_PASS_B);
  if (g_pass_b_tma && u.V == 2 && len % 2 == 0 && len > 0) {
    int threads = 0, smem = 0;
    if (PassBFn k = nka_get_pass_b_tma(u.nz, &threads, &smem)) {
      const size_t ntiles = (len + 511) / 512;
      const int grid = (int)(ntiles < (size_t)st->num_sms ? ntiles : (size_t)st->num_sms);
      launch_chained_smem(k, grid, threads, (size_t)smem, st->stream, f + off, st->W + off, st->Z + off, st->ld, len, st->S);
      st->launches += 1;
      return;
    }
  }
  const int grid = grid_for(st, per_sm_b(st, u.nz, u.V, len), len, u.V, nka_threads_b(u.nz));
  launch_chained(nka_get_pass_b(u.nz, u.V), grid, nka_threads_b(u.nz), st->stream, f + off, st->W + off, st->Z + off,
                 st->ld, len, st->S);
  st->launches += 1;
}

static void update_done(NKA st, const UpdateShape& u)
{
  // list length: the pending slot (if any) became a pair, capacity mvec pairs, plus the new pending slot
  if (st->pending) st->ub_len = u.L + 1 < st->mvec + 1 ? u.L + 1 : st->mvec + 1;
  else st->ub_len = u.L + 1;
  st->pending = true;
}

extern "C" void nka_accel_update_dev(NKA st, double* f)
{
  NKA_REQUIRE(st != NULL, "nka_accel_update: null handle");
  NKA_REQUIRE(f != NULL || st->vlen == 0, "nka_accel_update: null vector");
  DeviceGuard guard(st->device);
  NkaRange nvtx("nka:accel_update");
  const UpdateShape u = update_shape(st, f);
  if (u.L > 0) launch_pass_a(st, u, f, 0, st->vlen, 0, 0, true);
  launch_mid(st, u, f);
  launch_pass_b(st, u, f, 0, st->vlen);
  update_done(st, u);
}

// Host f: the same two sweeps, cut into chunks and software-pipelined with the PCIe copies.
//   copy-in stream :  H2D c0 | H2D c1 | H2D c2 | ...
//   handle's stream:          passA c0| passA c1| ... passA c_last (+ exchange + state) | passB c0 | passB c1 | ...
//   copy-out stream:                                                                              | D2H c0  | D2H c1 ...
// The coefficients need every element of f (global reduction), so no byte can return before the
// last byte has arrived: the floor is (H2D + D2H) of the vector; the sweeps themselves hide
// behind the copies except for one chunk at each end.
#ifndef NKA_HOST_CHUNK_BYTES
#define NKA_HOST_CHUNK_BYTES (64u << 20)
#endif
#define NKA_HOST_MAX_CHUNKS 16

// Host threads for pageable callers (nka_hostcopy.h).  NKA_HOST_THREADS: helpers besides the calling
// thread (default 3: the copies are bound by host memory bandwidth, 7 / 11 / 15 helpers were no faster on the
// 16-core bench box, profiles/r2z_host_threads_sweep.txt; 0 = leave pageable memory to the driver's own staging).
static NkaHostCopier* host_copier()
{
  // (function-local static: initialised once, thread-safe)
  static NkaHostCopier* const c = [] () -> NkaHostCopier* {
    int nt = (int)std::thread::hardware_concurrency() - 1;
    if (nt > 3) nt = 3;
    if (nt < 0) nt = 0;
    if (const char* e = getenv("NKA_HOST_THREADS")) nt = atoi(e);
    return nt > 0 ? new NkaHostCopier(nt) : nullptr;     // lives until the process ends
  }();
  return c;
}

static bool host_pointer_is_pageable(const void* p)
{
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return attr.type == cudaMemoryTypeUnregistered;
}

extern "C" void nka_accel_update_host(NKA st, double* f)
{
  NKA_REQUIRE(st != NULL, "nka_accel_update: null handle");
  NKA_REQUIRE(f != NULL || st->vlen == 0, "nka_accel_update: null vector");
  DeviceGuard guard(st->device);
  NkaRange nvtx("nka:accel_update(host f: h2d | sweeps | d2h, pipelined)");
  const size_t n = st->vlen;
  const size_t bytes = n * sizeof(double);
  if (!st->fstage) {
    CUDA_CHECK(cudaMalloc(&st->fstage, bytes ? bytes : 16));
    poison_fill(st, st->fstage, bytes ? bytes : 16);
  }
  if (st->host_chunk_bytes == 0) {
    st->host_chunk_bytes = NKA_HOST_CHUNK_BYTES;
    if (const char* e = getenv("NKA_HOST_CHUNK_BYTES")) if (atoll(e) >= 128) st->host_chunk_bytes = (size_t)atoll(e);   // tests
  }
  size_t nchunk = (bytes + st->host_chunk_bytes - 1) / st->host_chunk_bytes;
  if (nchunk > NKA_HOST_MAX_CHUNKS) nchunk = NKA_HOST_MAX_CHUNKS;
  if (nchunk <= 1) {
    CUDA_CHECK(cudaMemcpyAsync(st->fstage, f, bytes, cudaMemcpyHostToDevice, st->stream));
    nka_accel_update_dev(st, st->fstage);
    CUDA_CHECK(cudaMemcpyAsync(f, st->fstage, bytes, cudaMemcpyDeviceToHost, st->stream));
    CUDA_CHECK(cudaStreamSynchronize(st->stream));
    return;
  }
  if (!st->copy_in) {
    CUDA_CHECK(cudaStreamCreateWithFlags(&st->copy_in, cudaStreamNonBlocking));
    CUDA_CHECK(cudaStreamCreateWithFlags(&st->copy_out, cudaStreamNonBlocking));
    for (int c = 0; c < NKA_HOST_MAX_CHUNKS; ++c) CUDA_CHECK(cudaEventCreateWithFlags(&st->chunk_ev[c], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&st->order_ev, cudaEventDisableTiming));
  }
  // chunk boundaries: multiples of 16 doubles, so every chunk keeps the columns' 128-byte alignment
  size_t per = ((n + nchunk - 1) / nchunk + 15) / 16 * 16;
  size_t off[NKA_HOST_MAX_CHUNKS + 1];
  int nc = 0;
  for (size_t o = 0; o < n; o += per) off[nc++] = o;
  off[nc] = n;

  double* d = st->fstage;
  const UpdateShape u = update_shape(st, d);
  // Pageable caller memory: the host threads copy each chunk into / out of a pinned slot (three slots,
  // so a slot is refilled while the previous two are on the bus); page-locked memory goes straight to the DMA engines.
  NkaHostCopier* hc = host_pointer_is_pageable(f) ? host_copier() : nullptr;
  // one process per GPU on a shared box: the ranks' copy threads compete for the same cores and the same host
  // memory bus and lose against the driver's own staging (8 ranks: 91 ms per update against 72 ms on 16- and
  // 32-core boxes, profiles/r2ab_*, r2am vs r2k_*): the host threads are for the single-process caller
  if (hc && st->comm && st->comm->nranks > 1) hc = nullptr;
  constexpr int NS = 3;
  if (hc) {
    const size_t need = per * sizeof(double);
    if (st->hslot_bytes < need) {
      for (int i = 0; i < NS; ++i) {
        if (st->hslot[i]) CUDA_CHECK(cudaFreeHost(st->hslot[i]));
        CUDA_CHECK(cudaMallocHost(&st->hslot[i], need));
        if (!st->hslot_ev[i]) CUDA_CHECK(cudaEventCreateWithFlags(&st->hslot_ev[i], cudaEventDisableTiming));
      }
      st->hslot_bytes = need;
    }
  }
  // the staging buffer is free once everything queued on the handle's stream has run
  CUDA_CHECK(cudaEventRecord(st->order_ev, st->stream));
  CUDA_CHECK(cudaStreamWaitEvent(st->copy_in, st->order_ev, 0));
  const int grid_cap = st->max_grid / nc;
  int row0 = 0;
  for (int c = 0; c < nc; ++c) {
    const size_t len = off[c + 1] - off[c];
    const double* src = f + off[c];
    if (hc) {
      const int sl = c % NS;
      if (c >= NS) CUDA_CHECK(cudaEventSynchronize(st->hslot_ev[sl]));      // the slot's previous copy has left it
      hc->copy(st->hslot[sl], src, len * sizeof(double));
      src = st->hslot[sl];
    }
    CUDA_CHECK(cudaMemcpyAsync(d + off[c], src, len * sizeof(double), cudaMemcpyHostToDevice, st->copy_in));
    if (hc) CUDA_CHECK(cudaEventRecord(st->hslot_ev[c % NS], st->copy_in));
    CUDA_CHECK(cudaEventRecord(st->chunk_ev[c], st->copy_in));
    CUDA_CHECK(cudaStreamWaitEvent(st->stream, st->chunk_ev[c], 0));
    if (u.L > 0) row0 += launch_pass_a(st, u, d, off[c], len, grid_cap, row0, c == nc - 1);
  }
  launch_mid(st, u, d);
  // (every copy-in has completed on the device timeline before the first pass B chunk: the slots are free again)
  auto drain = [&](int c) {                            // chunk c has arrived in its slot: hand it to the caller
    CUDA_CHECK(cudaEventSynchronize(st->hslot_ev[c % NS]));
    hc->copy(f + off[c], st->hslot[c % NS], (off[c + 1] - off[c]) * sizeof(double));
  };
  for (int c = 0; c < nc; ++c) {
    const size_t len = off[c + 1] - off[c];
    launch_pass_b(st, u, d, off[c], len);
    CUDA_CHECK(cudaEventRecord(st->chunk_ev[c], st->stream));
    CUDA_CHECK(cudaStreamWaitEvent(st->copy_out, st->chunk_ev[c], 0));
    if (hc) {
      if (c >= NS) drain(c - NS);                     // frees the slot chunk c is about to use
      CUDA_CHECK(cudaMemcpyAsync(st->hslot[c % NS], d + off[c], len * sizeof(double), cudaMemcpyDeviceToHost, st->copy_out));
      CUDA_CHECK(cudaEventRecord(st->hslot_ev[c % NS], st->copy_out));
    } else {
      CUDA_CHECK(cudaMemcpyAsync(f + off[c], d + off[c], len * sizeof(double), cudaMemcpyDeviceToHost, st->copy_out));
    }
  }
  if (hc) for (int c = nc > NS ? nc - NS : 0; c < nc; ++c) drain(c);
  update_done(st, u);
  // later work on the handle's stream must not overtake the copy-out (it may reuse the staging buffer)
  CUDA_CHECK(cudaEventRecord(st->order_ev, st->copy_out));
  CUDA_CHECK(cudaStreamWaitEvent(st->stream, st->order_ev, 0));
  CUDA_CHECK(cudaStreamSynchronize(st->copy_out));
}

extern "C" void nka_accel_update(NKA st, double* f)
{
  NKA_REQUIRE(st != NULL, "nka_accel_update: null handle");
  cudaPointerAttributes attr;
  cudaError_t e = cudaPointerGetAttributes(&attr, f);
  if (e != cudaSuccess) { cudaGetLastError(); attr.type = cudaMemoryTypeUnregistered; }
  if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) nka_accel_update_dev(st, f);
  else nka_accel_update_host(st, f);
}

extern "C" void nka_restart(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_restart: null handle");
  DeviceGuard guard(st->device);
  nka_restart_kernel<<<1, NKA_STATE_THREADS, 0, st->stream>>>(st->S);
  CUDA_CHECK(cudaGetLastError());
  st->launches += 1;
  st->pending = false;
  st->ub_len = 0;
}

extern "C" void nka_relax(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_relax: null handle");
  if (!st->pending) return;                       // src-C/...c:470: nothing pending, nothing to do
  DeviceGuard guard(st->device);
  nka_relax_kernel<<<1, NKA_STATE_THREADS, 0, st->stream>>>(st->S);
  CUDA_CHECK(cudaGetLastError());
  st->launches += 1;
  if (st->ub_len >= 2) {
    const int grid = grid_for(st, 4, st->vlen, 1);
    launch_chained(nka_materialise, grid, NKA_THREADS, st->stream, st->W, st->ld, st->vlen, st->S);
    st->launches += 1;
  }
  st->pending = false;
  st->ub_len -= 1;
}

// ---------------------------------------------------------------------------
// queries
// ---------------------------------------------------------------------------
static void fetch_state(NKA st, NkaDevState* h)
{
  DeviceGuard guard(st->device);
  CUDA_CHECK(cudaMemcpyAsync(h, st->S, sizeof(NkaDevState), cudaMemcpyDeviceToHost, st->stream));
  CUDA_CHECK(cudaStreamSynchronize(st->stream));
}

extern "C" int nka_num_vec(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_num_vec: null handle");
  static thread_local NkaDevState h;
  fetch_state(st, &h);
  int n = 0;
  for (int k = h.first; k != NKA_NIL; k = h.next[k]) ++n;
  return h.pending ? n - 1 : n;
}

extern "C" int nka_max_vec(NKA st) { NKA_REQUIRE(st != NULL, "nka_max_vec: null handle"); return st->mvec; }
extern "C" int nka_vec_len(NKA st) { NKA_REQUIRE(st != NULL, "nka_vec_len: null handle"); return (int)st->vlen; }
extern "C" size_t nka_vec_len64(NKA st) { NKA_REQUIRE(st != NULL, "nka_vec_len64: null handle"); return st->vlen; }
extern "C" double nka_vec_tol(NKA st) { NKA_REQUIRE(st != NULL, "nka_vec_tol: null handle"); return st->vtol; }

extern "C" void nka_set_vec_tol(NKA st, double vtol)
{
  NKA_REQUIRE(st != NULL, "nka_set_vec_tol: null handle");
  NKA_REQUIRE(vtol > 0.0, "nka_set_vec_tol: vtol must be > 0");
  DeviceGuard guard(st->device);
  st->vtol = vtol;
  nka_set_vtol_kernel<<<1, 32, 0, st->stream>>>(st->S, vtol);
  CUDA_CHECK(cudaGetLastError());
  st->launches += 1;
}

extern "C" int nka_defined(NKA st)
{
  if (!st || !st->W || !st->Z || !st->S) return 0;
  static thread_local NkaDevState h;
  fetch_state(st, &h);
  if (h.mvec != st->mvec) return 0;
  return nka_state_defined(h);
}

extern "C" void nka_get_state(NKA st, nka_state_view* out)
{
  NKA_REQUIRE(st != NULL && out != NULL, "nka_get_state: null argument");
  static thread_local NkaDevState h;
  fetch_state(st, &h);
  memset(out, 0, sizeof *out);
  const int n = h.mvec + 1;
  out->mvec = h.mvec; out->subspace = h.subspace; out->pending = h.pending;
  out->first = h.first; out->last = h.last; out->free_slot = h.free_;
  for (int k = 0; k < n; ++k) {
    out->next[k] = h.next[k]; out->prev[k] = h.prev[k]; out->chained[k] = h.chained[k];
    out->c[k] = h.c[k]; out->s[k] = h.s[k];
    for (int j = 0; j < n; ++j) out->h[k * n + j] = h.h[k * NKA_MAXSLOT + j];
  }
  out->ndrop_last = h.ndrop_last; out->evicted_last = h.evicted_last; out->relaxed_last = h.relaxed_last;
  out->error = h.error; out->vtol = h.vtol; out->min_margin = h.min_margin; out->s_last = h.s_last;
  out->ncalls = h.ncalls;
}

extern "C" void nka_set_stream(NKA st, void* stream)
{
  NKA_REQUIRE(st != NULL, "nka_set_stream: null handle");
  DeviceGuard guard(st->device);
  fold_timing(st);
  CUDA_CHECK(cudaStreamSynchronize(st->stream));
  st->stream = (cudaStream_t)stream;
}

extern "C" void* nka_get_stream(NKA st) { NKA_REQUIRE(st != NULL, "nka_get_stream: null handle"); return (void*)st->stream; }

extern "C" void nka_synchronize(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_synchronize: null handle");
  DeviceGuard guard(st->device);
  CUDA_CHECK(cudaStreamSynchronize(st->stream));
}

extern "C" unsigned long long nka_launch_count(NKA st) { NKA_REQUIRE(st != NULL, "nka_launch_count: null handle"); return st->launches; }

extern "C" void nka_timing_enable(NKA st, int on)
{
  NKA_REQUIRE(st != NULL, "nka_timing_enable: null handle");
  DeviceGuard guard(st->device);
  if (!on) fold_timing(st);
  st->timing = on != 0;
}

extern "C" void nka_timing_reset(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_timing_reset: null handle");
  DeviceGuard guard(st->device);
  fold_timing(st);
  for (int k = 0; k < T_NKIND; ++k) { st->t_ms[k] = 0.0; st->t_cnt[k] = 0; }
}

extern "C" void nka_timing_read(NKA st, double ms[5], unsigned long long count[5])
{
  NKA_REQUIRE(st != NULL, "nka_timing_read: null handle");
  DeviceGuard guard(st->device);
  fold_timing(st);
  for (int k = 0; k < T_NKIND; ++k) { ms[k] = st->t_ms[k]; count[k] = st->t_cnt[k]; }
}

extern "C" void nka_launch_geometry(NKA st, int* grid_a, int* grid_b, int* threads)
{
  NKA_REQUIRE(st != NULL, "nka_launch_geometry: null handle");
  DeviceGuard guard(st->device);
  const int L = st->ub_len;
  const bool may_skip = (st->comm == nullptr || st->peer != nullptr) && st->lazy && st->pending && L == st->mvec + 1;
  const int NC = may_skip ? st->mvec : L;
  if (grid_a) *grid_a = L > 0 ? grid_for(st, per_sm_a(st, NC, 2, st->vlen), st->vlen, 2, NKA_THREADS_A) : 0;
  const int nz = nz_expected(st);
  if (grid_b) *grid_b = grid_for(st, per_sm_b(st, nz, 2, st->vlen), st->vlen, 2, nka_threads_b(nz));
  if (threads) *threads = NKA_THREADS_A * 10000 + nka_threads_b(nz);
}

extern "C" const char* nka_b200_version(void) { return NKA_VERSION; }

// ---------------------------------------------------------------------------
// multi-GPU
// ---------------------------------------------------------------------------
extern "C" int nka_comm_unique_id(void* id128)
{
  if (!nka_nccl_load()) return -1;
  return g_nccl.GetUniqueId(id128);
}

static void attach_comm(NKA st, NkaComm* c)
{
  NKA_REQUIRE(!st->dp && !st->dp_ctx, "nka_comm_init: the handle already reduces through a dp callback; use one or the other");
  peer_teardown(st);
  nka_comm_release(st->comm);
  st->comm = c;
  // On one NVLink domain the reduction is fused into pass A (peer memory).  Otherwise NCCL
  // reduces between pass A and the state kernel, and the lazy column is off: its conditional
  // second all-reduce is not worth it, every rank streams all columns.
  if (!peer_setup(st)) set_lazy(st, false);
}

extern "C" int nka_comm_mode(NKA st)
{
  NKA_REQUIRE(st != NULL, "nka_comm_mode: null handle");
  return st->comm == nullptr ? 0 : (st->peer ? 2 : 1);
}

extern "C" int nka_comm_init(NKA st, int nranks, int rank, const void* id128)
{
  NKA_REQUIRE(st != NULL && id128 != NULL, "nka_comm_init: null argument");
  NKA_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "nka_comm_init: bad rank/nranks");
  if (!nka_nccl_load()) return -1;
  DeviceGuard guard(st->device);
  NkaId128 id;
  memcpy(id.bytes, id128, sizeof id.bytes);
  void* comm = nullptr;
  const int rc = g_nccl.CommInitRank(&comm, nranks, id, rank);
  if (rc != 0) return rc;
  NkaComm* c = new NkaComm();
  c->comm = comm; c->owned = true; c->nranks = nranks; c->rank = rank;
  attach_comm(st, c);
  return 0;
}

extern "C" void nka_comm_adopt(NKA st, void* nccl_comm, int nranks, int rank)
{
  NKA_REQUIRE(st != NULL, "nka_comm_adopt: null handle");
  NKA_REQUIRE(nka_nccl_load(), "nka_comm_adopt: libnccl.so.2 not found");
  DeviceGuard guard(st->device);
  NkaComm* c = new NkaComm();
  c->comm = nccl_comm; c->owned = false; c->nranks = nranks; c->rank = rank;
  attach_comm(st, c);
}

// used by nka_vec.cu: an accelerator shaped like a vector shares that vector's communicator
void nka_attach_shared_comm(NKA st, NkaComm* c)
{
  DeviceGuard guard(st->device);
  attach_comm(st, nka_comm_retain(c));
}
