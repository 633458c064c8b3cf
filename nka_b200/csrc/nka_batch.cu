// nka_batch.cu -- the batched accelerator: nbatch independent same-length NKA instances in one handle,
// updated by a fixed number of launches whatever nbatch is (include/nka_b200.h, DESIGN.md section 12).
//
// Every member runs in the capacity shape of a single handle (nka_capi.cu, update_shape): pass A
// `mvec` columns wide with the lazy oldest column (`mvec + 1` without), the fix-up always queued where
// the lazy column applies, pass B at `mvec` pairs.  The bits a member gets are those of a single
// capacity-shape handle fed its calls:
//   - pass A's fold order depends only on its CTA count, taken from the single handle's rule
//     (nka_grid_for / nka_per_sm_a with the single kernels' occupancy), likewise the fix-up's;
//   - nka_state_step gives the same bits on any number of lanes, and a warp runs it here as there;
//   - pass B is element-wise.
//
// Memory, member-major: member b's slot k is W + (b*(mvec+1) + k)*ld (likewise Z); its state S[b],
// dots[b*2*NKA_MAXSLOT ...], partial rows at partials + b*prow and ticket tickets[b].

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/nka_b200.h"
#include "nka_internal.h"
#include "nka_batch.h"
#include "nka_kernels.cuh"

#define NKA_BATCH_MAX 65535            // members ride on blockIdx.y
// Members per CTA of the batched state kernel: one warp each, each staging ~13 KB of state in shared
// memory.  Three stay under the 48 KB a kernel gets without opting in; an SM then holds five such CTAs
// (15 members) in its 228 KB, about what one member per CTA would reach (17).
#define NKA_BATCH_STATE_MEMBERS 3
static_assert(NKA_BATCH_STATE_MEMBERS * sizeof(NkaStateStage) <= 48 * 1024,
              "the batched state kernel's staging must fit 48 KB of static shared memory");

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool nka_member_on(const unsigned char* active, size_t b) { return !active || active[b]; }

// The state step of NKA_BATCH_STATE_MEMBERS members, one warp each.  The staging goes through the
// single handle's nka_stage_in / nka_stage_out with the whole CTA; the step, on the staged copy, is
// committed unless it needs the lazily skipped column: then only need_fixup is published (the fix-up
// kernel runs the step again with both missing dots), as nka_run_state_step does.
__global__ void __launch_bounds__(32 * NKA_BATCH_STATE_MEMBERS)
nka_batch_state_kernel(NkaDevState* Sall, const double* dots_all, int nbatch, const unsigned char* active)
{
  __shared__ NkaStateStage sm[NKA_BATCH_STATE_MEMBERS];
  __shared__ int need[NKA_BATCH_STATE_MEMBERS];
  const int b0 = blockIdx.x * NKA_BATCH_STATE_MEMBERS;
  // (whether member b0 + w takes part is the same in every thread: stage_in's barrier is safe)
  for (int w = 0; w < NKA_BATCH_STATE_MEMBERS; ++w)
    if (b0 + w < nbatch && nka_member_on(active, b0 + w))
      nka_stage_in(sm[w], Sall + b0 + w, dots_all + (size_t)(b0 + w) * (2 * NKA_MAXSLOT));
  const int warp = threadIdx.x >> 5;
  if (b0 + warp < nbatch && nka_member_on(active, b0 + warp)) {
    const int r = nka_state_step_dev(&sm[warp].st, &sm[warp].x, sm[warp].dots, /*have_last=*/0);
    if ((threadIdx.x & 31) == 0) need[warp] = r;
  }
  __syncthreads();
  for (int w = 0; w < NKA_BATCH_STATE_MEMBERS; ++w) {
    if (b0 + w >= nbatch || !nka_member_on(active, b0 + w)) continue;
    NkaDevState* S = Sall + b0 + w;
    if (need[w]) {
      if (threadIdx.x == 0) S->need_fixup = 1;
    } else {
      nka_stage_out(sm[w], S);
    }
  }
}

// nka_fixup_kernel per member (blockIdx.y), with the single handle's CTA count in x.
__global__ void __launch_bounds__(NKA_THREADS)
nka_batch_fixup_kernel(const double* __restrict__ F, size_t ldf, const double* __restrict__ Wall, size_t wstride,
                       size_t ld, size_t n, NkaDevState* __restrict__ Sall, double* __restrict__ partials_all, size_t prow,
                       unsigned* __restrict__ tickets, double* __restrict__ dots_all, const unsigned char* __restrict__ active)
{
  const size_t b = blockIdx.y;
  if (!nka_member_on(active, b)) return;
  NkaDevState* S = Sall + b;
  if (!S->need_fixup) return;
  const double* f = F + b * ldf;
  const double* W = Wall + b * wstride;
  double* partials = partials_all + b * prow;
  double* dots = dots_all + b * (2 * NKA_MAXSLOT);
  const NkaPlanA& A = S->planA;
  const int jl = A.ncol - 1;
  const double* w0 = W + (size_t)A.col[0] * ld;
  const double* wl = W + (size_t)A.col[jl] * ld;
  const double* wp = W + (size_t)A.col[jl - 1] * ld;
  const bool sub = (A.submask >> jl) & 1ull;
  double acc[2] = {0.0, 0.0};
  const size_t stride = (size_t)gridDim.x * NKA_THREADS;
  for (size_t i = (size_t)blockIdx.x * NKA_THREADS + threadIdx.x; i < n; i += stride) {
    const double x0 = f[i];
    const double d0 = w0[i] - x0;
    const double dl = sub ? wl[i] - wp[i] : wl[i];
    acc[0] = fma(d0, dl, acc[0]);
    acc[1] = fma(x0, dl, acc[1]);
  }
  __shared__ NkaStateStage sm;
  __shared__ double xv[2];
  const bool last = nka_grid_reduce<2, NKA_THREADS>(acc, partials, tickets + b, partials, gridDim.x,
                                                  [&](int j, double v) { xv[j] = v; });
  if (last) {
    if (threadIdx.x < 2) dots[(threadIdx.x == 0 ? 0 : NKA_MAXSLOT) + jl] = xv[threadIdx.x];
    __threadfence();
    __syncthreads();
    nka_stage_in(sm, S, dots);
    nka_run_state_step(sm, S, /*have_last=*/1);
  }
}

// relax() of the selected members, one CTA each
__global__ void __launch_bounds__(NKA_STATE_THREADS) nka_batch_relax_kernel(NkaDevState* Sall, const unsigned char* mask)
{
  if (!nka_member_on(mask, blockIdx.x)) return;
  NkaDevState* S = Sall + blockIdx.x;
  __shared__ NkaStateStage sm;
  nka_stage_in(sm, S, nullptr);
  if (threadIdx.x == 0) nka_state_relax(sm.st);
  __syncthreads();
  nka_stage_out(sm, S);
}

__global__ void __launch_bounds__(NKA_STATE_THREADS) nka_batch_restart_kernel(NkaDevState* Sall, const unsigned char* mask)
{
  if (!nka_member_on(mask, blockIdx.x)) return;
  NkaDevState* S = Sall + blockIdx.x;
  __shared__ NkaStateStage sm;
  nka_stage_in(sm, S, nullptr);
  if (threadIdx.x == 0) nka_state_restart(sm.st);
  __syncthreads();
  nka_stage_out(sm, S);
}

// nka_materialise per selected member (blockIdx.y): the conversions the relax kernel planned
__global__ void __launch_bounds__(NKA_THREADS)
nka_batch_materialise(double* Wall, size_t wstride, size_t ld, size_t n, const NkaDevState* __restrict__ Sall,
                      const unsigned char* __restrict__ mask)
{
  const size_t b = blockIdx.y;
  if (!nka_member_on(mask, b)) return;
  const NkaDevState* S = Sall + b;
  double* W = Wall + b * wstride;
  const int m = S->planM.n;
  if (m == 0) return;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS;
  for (size_t i = (size_t)blockIdx.x * NKA_THREADS + threadIdx.x; i < n; i += stride) {
    for (int e = 0; e < m; ++e) {
      double* dst = W + (size_t)S->planM.dst[e] * ld;
      const double* sub = W + (size_t)S->planM.sub[e] * ld;
      dst[i] = dst[i] - sub[i];
    }
  }
}

__global__ void nka_batch_init_kernel(NkaDevState* Sall, int mvec, double vtol, int lazy_last)
{
  if (threadIdx.x == 0) {
    NkaDevState& S = Sall[blockIdx.x];
    nka_state_init(S, mvec, vtol);
    S.lazy_last = lazy_last;
    nka_build_plan_a(S);
  }
}

__global__ void nka_batch_set_vtol_kernel(NkaDevState* Sall, int nbatch, double vtol)
{
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < nbatch; b += gridDim.x * blockDim.x) Sall[b].vtol = vtol;
}

// per member: num_vec, and whether nka_state_defined holds with the handle's mvec
__global__ void nka_batch_query_kernel(const NkaDevState* Sall, int nbatch, int mvec, int* num, int* ok)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nbatch) return;
  const NkaDevState& S = Sall[b];
  const int good = S.mvec == mvec && nka_state_defined(S);
  int n = 0;
  if (good)
    for (int k = S.first; k != NKA_NIL; k = S.next[k]) ++n;
  num[b] = good ? (S.pending ? n - 1 : n) : -1;
  ok[b] = good;
}

// ---------------------------------------------------------------------------
// the handle
// ---------------------------------------------------------------------------
static void batch_poison(NKABATCH bt, void* p, size_t bytes)
{
  if (bt->poison) CUDA_CHECK(cudaMemsetAsync(p, 0xFF, bytes, bt->stream));
}

// A capturable call: aborts on the legacy default stream during another stream's capture (nothing can
// be queued), and returns whether this call is being captured (then nothing counts as launched).
static bool batch_capturing(NKABATCH bt, const char* call)
{
  const int c = nka_capture_status(bt->stream);
  if (c < 0)
    nka_capture_fail(call, "the handle is on the legacy default stream while another stream captures; "
                           "nka_batch_set_stream to the capture stream before the capture begins");
  return c > 0;
}

static void batch_launched(NKABATCH bt, bool capturing, int n)
{
  CUDA_CHECK(cudaGetLastError());
  if (!capturing) bt->launches += (unsigned long long)n;
}

// CTAs of one member's pass A, fix-up and pass B: the single handle's rule for the same length
static int batch_grid_a(NKABATCH bt, int V)
{
  return nka_grid_for(bt->geom, nka_per_sm_a(bt->geom, bt->nc, V, bt->vlen), bt->vlen, V, NKA_THREADS_A);
}
static int batch_grid_fixup(NKABATCH bt) { return nka_grid_for(bt->geom, 4, bt->vlen, 1, NKA_THREADS); }
static int batch_grid_b(NKABATCH bt, int V)
{
  return nka_grid_for(bt->geom, nka_per_sm_b(bt->geom, bt->mvec, V, bt->vlen), bt->vlen, V, nka_threads_b(bt->mvec));
}

extern "C" NKABATCH nka_batch_init(int nbatch, size_t vlen, int mvec, double vtol, int device, void* stream)
{
  NKA_REQUIRE(nbatch >= 1 && nbatch <= NKA_BATCH_MAX, "nka_batch_init: nbatch must be in 1..65535");
  NKA_REQUIRE(vlen >= 1, "nka_batch_init: vlen must be >= 1");
  NKA_REQUIRE(mvec > 0, "nka_batch_init: mvec must be > 0");
  NKA_REQUIRE(mvec <= NKA_B200_MAX_MVEC, "nka_batch_init: mvec > 32 is not supported by this build");
  NKA_REQUIRE(vtol > 0.0, "nka_batch_init: vtol must be > 0");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    nka_fail(__FILE__, __LINE__, "no CUDA device: libnka_b200 has no CPU compute path");
  NKABATCH bt = new nka_batch();
  if (device < 0) CUDA_CHECK(cudaGetDevice(&device));
  bt->device = device;
  DeviceGuard guard(device);
  bt->nbatch = nbatch;
  bt->vlen = vlen;
  bt->mvec = mvec;
  bt->vtol = vtol;
  bt->ld = ((vlen + 15) / 16) * 16;                 // 128-byte aligned columns, as a single handle's
  bt->wstride = bt->ld * (size_t)(mvec + 1);
  bt->stream = (cudaStream_t)stream;
  if (const char* s = getenv("NKA_LAZY_LAST")) bt->lazy = atoi(s) != 0;
  if (const char* s = getenv("NKA_POISON_ALLOC")) bt->poison = atoi(s) != 0;
  bt->nc = bt->lazy ? mvec : mvec + 1;
  nka_geom_init(bt->geom, device, mvec);
  NKA_REQUIRE(nka_get_batch_pass_a(bt->nc, 1) && nka_get_batch_pass_a(bt->nc, 2) && nka_get_batch_pass_b(mvec, 1) &&
              nka_get_batch_pass_b(mvec, 2), "nka_batch_init: the batched sweeps are not instantiated for this mvec");

  // partial rows per member: the widest of pass A (either access width) and the fix-up
  size_t rows_a = 0;
  for (int V = 1; V <= 2; ++V) {
    const size_t g = (size_t)batch_grid_a(bt, V);
    if (g > rows_a) rows_a = g;
  }
  bt->prow = rows_a * 2 * bt->nc;
  if ((size_t)batch_grid_fixup(bt) * 2 > bt->prow) bt->prow = (size_t)batch_grid_fixup(bt) * 2;

  const size_t nb = (size_t)nbatch;
  const size_t poolbytes = nb * bt->wstride * sizeof(double);
  e = cudaMalloc(&bt->W, poolbytes);
  if (e == cudaSuccess) e = cudaMalloc(&bt->Z, poolbytes);
  if (e != cudaSuccess) {
    char b[200];
    snprintf(b, sizeof b, "nka_batch_init: cannot allocate 2 x %zu bytes of device memory for the subspaces: %s",
             poolbytes, cudaGetErrorString(e));
    nka_fail(__FILE__, __LINE__, b);
  }
  const size_t dotbytes = nb * 2 * NKA_MAXSLOT * sizeof(double);
  const size_t rowbytes = nb * bt->prow * sizeof(double);
  CUDA_CHECK(cudaMalloc(&bt->S, nb * sizeof(NkaDevState)));
  CUDA_CHECK(cudaMalloc(&bt->dots, dotbytes));
  CUDA_CHECK(cudaMalloc(&bt->partials, rowbytes));
  CUDA_CHECK(cudaMalloc(&bt->tickets, nb * sizeof(unsigned)));
  CUDA_CHECK(cudaMalloc(&bt->query, 2 * nb * sizeof(int)));
  CUDA_CHECK(cudaMemsetAsync(bt->tickets, 0, nb * sizeof(unsigned), bt->stream));
  CUDA_CHECK(cudaMemsetAsync(bt->dots, 0, dotbytes, bt->stream));
  batch_poison(bt, bt->W, poolbytes);
  batch_poison(bt, bt->Z, poolbytes);
  batch_poison(bt, bt->partials, rowbytes);
  batch_poison(bt, bt->dots, dotbytes);
  nka_batch_init_kernel<<<nbatch, 32, 0, bt->stream>>>(bt->S, mvec, vtol, bt->lazy ? 1 : 0);
  batch_launched(bt, false, 1);
  return bt;
}

extern "C" void nka_batch_delete(NKABATCH bt)
{
  if (!bt) return;
  DeviceGuard guard(bt->device);
  cudaStreamSynchronize(bt->stream);
  cudaFree(bt->W); cudaFree(bt->Z); cudaFree(bt->S); cudaFree(bt->dots);
  cudaFree(bt->partials); cudaFree(bt->tickets); cudaFree(bt->query);
  delete bt;
}

// One batched update: pass A, state step, [fix-up], pass B, each one launch over every member, queued
// on `stream`; a captured update (cap) counts no launches.
static void batch_update(NKABATCH bt, double* f, size_t ldf, const unsigned char* active, cudaStream_t stream, bool cap)
{
  // the 16-byte path needs every row 16-byte aligned: f itself and an even row stride
  const int V = ((uintptr_t)f % 16 == 0 && ldf % 2 == 0) ? 2 : 1;
  const unsigned nb = (unsigned)bt->nbatch;
  const size_t n = bt->vlen;
  nka_get_batch_pass_a(bt->nc, V)<<<dim3((unsigned)batch_grid_a(bt, V), nb), NKA_THREADS_A, 0, stream>>>(
      f, ldf, bt->W, bt->wstride, bt->ld, n, bt->S, bt->partials, bt->prow, bt->tickets, bt->dots, active);
  batch_launched(bt, cap, 1);
  const unsigned nstate = (nb + NKA_BATCH_STATE_MEMBERS - 1) / NKA_BATCH_STATE_MEMBERS;
  nka_batch_state_kernel<<<nstate, 32 * NKA_BATCH_STATE_MEMBERS, 0, stream>>>(bt->S, bt->dots, bt->nbatch, active);
  batch_launched(bt, cap, 1);
  if (bt->lazy) {
    // exits at once for every member whose step did not ask for the skipped column
    nka_batch_fixup_kernel<<<dim3((unsigned)batch_grid_fixup(bt), nb), NKA_THREADS, 0, stream>>>(
        f, ldf, bt->W, bt->wstride, bt->ld, n, bt->S, bt->partials, bt->prow, bt->tickets, bt->dots, active);
    batch_launched(bt, cap, 1);
  }
  nka_get_batch_pass_b(bt->mvec, V)<<<dim3((unsigned)batch_grid_b(bt, V), nb), nka_threads_b(bt->mvec), 0, stream>>>(
      f, ldf, bt->W, bt->Z, bt->wstride, bt->ld, n, bt->S, active);
  batch_launched(bt, cap, 1);
}

extern "C" void nka_batch_accel_update(NKABATCH bt, double* f, size_t ldf, const unsigned char* active)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_accel_update: null handle");
  NKA_REQUIRE(f != NULL, "nka_batch_accel_update: null f");
  NKA_REQUIRE(ldf >= bt->vlen, "nka_batch_accel_update: ldf must be >= vlen");
  DeviceGuard guard(bt->device);
  const bool cap = batch_capturing(bt, "nka_batch_accel_update");
  NkaRange nvtx("nka:batch_accel_update");
  batch_update(bt, f, ldf, active, bt->stream, cap);
}

void nka_batch_update_captured(NKABATCH bt, double* f, size_t ldf, const unsigned char* active, cudaStream_t stream)
{
  batch_update(bt, f, ldf, active, stream, true);
}

extern "C" void nka_batch_relax(NKABATCH bt, const unsigned char* mask)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_relax: null handle");
  DeviceGuard guard(bt->device);
  const bool cap = batch_capturing(bt, "nka_batch_relax");
  // as a captured single handle: both kernels always; a member with nothing pending plans no conversion
  nka_batch_relax_kernel<<<bt->nbatch, NKA_STATE_THREADS, 0, bt->stream>>>(bt->S, mask);
  batch_launched(bt, cap, 1);
  nka_batch_materialise<<<dim3((unsigned)batch_grid_fixup(bt), (unsigned)bt->nbatch), NKA_THREADS, 0, bt->stream>>>(
      bt->W, bt->wstride, bt->ld, bt->vlen, bt->S, mask);
  batch_launched(bt, cap, 1);
}

extern "C" void nka_batch_restart(NKABATCH bt, const unsigned char* mask)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_restart: null handle");
  DeviceGuard guard(bt->device);
  const bool cap = batch_capturing(bt, "nka_batch_restart");
  nka_batch_restart_kernel<<<bt->nbatch, NKA_STATE_THREADS, 0, bt->stream>>>(bt->S, mask);
  batch_launched(bt, cap, 1);
}

void nka_batch_restart_captured(NKABATCH bt, const unsigned char* mask, cudaStream_t stream)
{
  nka_batch_restart_kernel<<<bt->nbatch, NKA_STATE_THREADS, 0, stream>>>(bt->S, mask);
  batch_launched(bt, true, 1);
}

extern "C" void nka_batch_set_vec_tol(NKABATCH bt, double vtol)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_set_vec_tol: null handle");
  NKA_REQUIRE(vtol > 0.0, "nka_batch_set_vec_tol: vtol must be > 0");
  DeviceGuard guard(bt->device);
  const bool cap = batch_capturing(bt, "nka_batch_set_vec_tol");
  if (!cap) bt->vtol = vtol;
  const int grid = (bt->nbatch + 255) / 256;
  nka_batch_set_vtol_kernel<<<grid, 256, 0, bt->stream>>>(bt->S, bt->nbatch, vtol);
  batch_launched(bt, cap, 1);
}

// ---------------------------------------------------------------------------
// queries (never captured)
// ---------------------------------------------------------------------------
static void batch_query(NKABATCH bt, std::vector<int>& num, std::vector<int>& ok, const char* call)
{
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, call, "it copies the device state to the host and synchronises");
  const int nb = bt->nbatch;
  nka_batch_query_kernel<<<(nb + 127) / 128, 128, 0, bt->stream>>>(bt->S, nb, bt->mvec, bt->query, bt->query + nb);
  CUDA_CHECK(cudaGetLastError());
  num.resize(nb);
  ok.resize(nb);
  CUDA_CHECK(cudaMemcpyAsync(num.data(), bt->query, nb * sizeof(int), cudaMemcpyDeviceToHost, bt->stream));
  CUDA_CHECK(cudaMemcpyAsync(ok.data(), bt->query + nb, nb * sizeof(int), cudaMemcpyDeviceToHost, bt->stream));
  CUDA_CHECK(cudaStreamSynchronize(bt->stream));
}

extern "C" void nka_batch_num_vec(NKABATCH bt, int* out)
{
  NKA_REQUIRE(bt != NULL && out != NULL, "nka_batch_num_vec: null argument");
  std::vector<int> num, ok;
  batch_query(bt, num, ok, "nka_batch_num_vec");
  memcpy(out, num.data(), num.size() * sizeof(int));
}

extern "C" int nka_batch_defined(NKABATCH bt)
{
  if (!bt || !bt->W || !bt->Z || !bt->S) return 0;
  std::vector<int> num, ok;
  batch_query(bt, num, ok, "nka_batch_defined");
  for (int v : ok)
    if (!v) return 0;
  return 1;
}

extern "C" void nka_batch_get_state(NKABATCH bt, int member, nka_state_view* out)
{
  NKA_REQUIRE(bt != NULL && out != NULL, "nka_batch_get_state: null argument");
  NKA_REQUIRE(member >= 0 && member < bt->nbatch, "nka_batch_get_state: member out of range");
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, "nka_batch_get_state", "it copies the device state to the host and synchronises");
  static thread_local NkaDevState h;
  CUDA_CHECK(cudaMemcpyAsync(&h, bt->S + member, sizeof(NkaDevState), cudaMemcpyDeviceToHost, bt->stream));
  CUDA_CHECK(cudaStreamSynchronize(bt->stream));
  nka_state_view_from(h, out);
}

extern "C" void nka_batch_set_stream(NKABATCH bt, void* stream)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_set_stream: null handle");
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, "nka_batch_set_stream",
                     "it synchronises the handle's stream; set the capture stream before the capture begins");
  CUDA_CHECK(cudaStreamSynchronize(bt->stream));
  bt->stream = (cudaStream_t)stream;
}

extern "C" void nka_batch_synchronize(NKABATCH bt)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_synchronize: null handle");
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, "nka_batch_synchronize", "it synchronises the handle's stream");
  CUDA_CHECK(cudaStreamSynchronize(bt->stream));
}

extern "C" int nka_batch_stream_capturing(NKABATCH bt)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_stream_capturing: null handle");
  DeviceGuard guard(bt->device);
  return nka_capture_status(bt->stream);
}

extern "C" unsigned long long nka_batch_launch_count(NKABATCH bt)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_launch_count: null handle");
  return bt->launches;
}
