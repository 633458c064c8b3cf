// nka_batch_loop.cu -- device-side fixed-point loops over a batched accelerator (include/nka_b200.h,
// INTEGRATION.md section 8, DESIGN.md section 13).  One graph launch runs a whole solve:
//
//   reset -> WHILE (any member running) { residual graph -> check -> decide -> batched update -> step }
//
// check reduces each running member's ||F_b||_2 (or a scaled ||s_b . F_b||_2) with the batch's
// fixed-order grid reduction, records it and decides the member's status by its stop test; decide sets
// the WHILE node's condition; the update and step touch only members still running.  A member's bits are those of a host-driven loop making the same calls:
//   - check's CTA count per member follows vlen only (nka_grid_for, as the batch's fix-up), and
//     nka_grid_reduce folds its partial rows in a fixed order, so a norm depends on the row alone;
//   - the update is nka_batch_accel_update's own launch sequence, with check's mask;
//   - step is X_b + F_b element by element, as X[b] += F[b] computes it.
// The host side is the solve core the work queues share (nka_batch.h: NkaSolve, nka_solve_create): the
// per-slot state, the create steps, the check and step launchers and the entry points' common parts.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/nka_b200.h"
#include "nka_internal.h"
#include "nka_batch.h"
#include "nka_kernels.cuh"

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// Every member running at step 0, the history NaN.  (r0 needs no reset: check 0 writes it.)
__global__ void __launch_bounds__(NKA_THREADS)
nka_loop_reset(int* __restrict__ iters, int* __restrict__ status, unsigned char* __restrict__ active,
               double* __restrict__ rlast, double* __restrict__ hist, size_t nhist, int nbatch)
{
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nhist; i += stride) {
    hist[i] = nan;
    if (i < (size_t)nbatch) {
      iters[i] = 0;
      status[i] = NKA_LOOP_RUNNING;
      active[i] = 1;
      rlast[i] = nan;
    }
  }
}

// ||s_b . F_b|| of every running member (blockIdx.y), recorded as check k = iters[b], and its status by
// member (or, with `index`, problem) p = index[b]'s rule in `stop` (include/nka_b200.h: nka_stop_test).
// Without a scale the sweep is ||F_b||'s; with one, t = s_i * f_i enters the same fma in the same order
// on the same CTAs, F at width V as without, the scale 16 bytes at a time when scale16 (V = 2 only).
template <int V>
__global__ void __launch_bounds__(NKA_THREADS)
nka_loop_check(const double* __restrict__ F, size_t ldf, size_t n, int nbatch, const int* __restrict__ iters,
               int* __restrict__ status, unsigned char* __restrict__ active, double* __restrict__ r0,
               double* __restrict__ rlast, double* __restrict__ hist, double* __restrict__ partials_all, size_t prow,
               unsigned* __restrict__ tickets, const nka_stop_test stop, const int* __restrict__ index, int scale16)
{
  const size_t b = blockIdx.y;
  // every CTA of a member sees the same status: only the member's last CTA writes it, after all took tickets
  if (status[b] != NKA_LOOP_RUNNING) return;
  const double* f = F + b * ldf;
  double acc[1] = {0.0};
  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS;
  const size_t start = (size_t)blockIdx.x * NKA_THREADS + threadIdx.x;
  const double* sc = stop.scale_dev;
  if (!sc) {
    for (size_t i = start; i < nv; i += stride) {
      const Vec<V> x = Vec<V>::ld(f, i);
      x.dot_into(x, acc[0]);
    }
    if (V == 2 && (n & 1) && start == 0) acc[0] = fma(f[n - 1], f[n - 1], acc[0]);
  } else {
    sc += b * stop.ldscale;
    if constexpr (V == 2) {
      if (scale16) {
        for (size_t i = start; i < nv; i += stride) {
          const Vec<2> x = Vec<2>::ld(f, i), s = Vec<2>::ld(sc, i);
          const Vec<2> t = {s.x * x.x, s.y * x.y};
          t.dot_into(t, acc[0]);
        }
      } else {
        for (size_t i = start; i < nv; i += stride) {
          const Vec<2> x = Vec<2>::ld(f, i);
          const Vec<2> t = {__ldg(sc + 2 * i) * x.x, __ldg(sc + 2 * i + 1) * x.y};
          t.dot_into(t, acc[0]);
        }
      }
    } else {
      for (size_t i = start; i < nv; i += stride) {
        const double t = __ldg(sc + i) * Vec<1>::ld(f, i).x;
        acc[0] = fma(t, t, acc[0]);
      }
    }
    if (V == 2 && (n & 1) && start == 0) {
      const double t = __ldg(sc + n - 1) * f[n - 1];
      acc[0] = fma(t, t, acc[0]);
    }
  }
  __shared__ double ss;
  double* partials = partials_all + b * prow;
  const bool last = nka_grid_reduce<1, NKA_THREADS>(acc, partials, tickets + b, partials, gridDim.x,
                                                    [&](int, double v) { ss = v; });
  if (last && threadIdx.x == 0) {
    const double r = sqrt(ss);
    const int k = iters[b];
    hist[(size_t)k * nbatch + b] = r;
    rlast[b] = r;
    if (k == 0) r0[b] = r;
    const size_t p = index ? (size_t)index[b] : b;
    const double atol = stop.atol_dev ? stop.atol_dev[p] : stop.atol;
    const double rtol = stop.rtol_dev ? stop.rtol_dev[p] : stop.rtol;
    const int maxit = stop.maxit_dev ? min(max(stop.maxit_dev[p], 0), stop.maxit) : stop.maxit;
    int st = NKA_LOOP_RUNNING;
    if (!isfinite(r)) st = NKA_LOOP_NONFINITE;
    else if (r < fmax(atol, rtol * r0[b])) st = NKA_LOOP_CONVERGED;
    else if (stop.dtol > 0.0 && r > stop.dtol * r0[b]) st = NKA_LOOP_DIVERGED;
    else if (k >= maxit) st = NKA_LOOP_MAXIT;
    status[b] = st;
    active[b] = st == NKA_LOOP_RUNNING;
  }
}

// The WHILE node's condition: whether any member is still running.
__global__ void __launch_bounds__(1024)
nka_loop_decide(const unsigned char* __restrict__ active, int nbatch, cudaGraphConditionalHandle cond)
{
  int any = 0;
  for (int b = threadIdx.x; b < nbatch; b += blockDim.x) any |= active[b];
  any = __syncthreads_or(any);
  if (threadIdx.x == 0) cudaGraphSetConditional(cond, any ? 1u : 0u);
}

// X_b += F_b and one more step for every running member (blockIdx.y).
template <int V>
__global__ void __launch_bounds__(NKA_THREADS)
nka_loop_step(double* __restrict__ X, size_t ldx, const double* __restrict__ F, size_t ldf, size_t n,
              const unsigned char* __restrict__ active, int* __restrict__ iters)
{
  const size_t b = blockIdx.y;
  if (!active[b]) return;
  double* x = X + b * ldx;
  const double* f = F + b * ldf;
  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS;
  const size_t start = (size_t)blockIdx.x * NKA_THREADS + threadIdx.x;
  for (size_t i = start; i < nv; i += stride) (Vec<V>::ld_plain(x, i) + Vec<V>::ld(f, i)).st(x, i);
  if (V == 2 && (n & 1) && start == 0) x[n - 1] = x[n - 1] + f[n - 1];
  if (start == 0) iters[b] += 1;
}

// ---------------------------------------------------------------------------
// the solve core, shared with the work queues (nka_batch_queue.cu)
// ---------------------------------------------------------------------------
NkaSolve::~NkaSolve()
{
  if (exec) cudaGraphExecDestroy(exec);
  cudaFree(iters); cudaFree(status); cudaFree(active); cudaFree(r0); cudaFree(rlast); cudaFree(hist);
  cudaFree(partials); cudaFree(tickets); cudaFree(rprev); cudaFree(nrst); cudaFree(rmask);
}

int nka_loop_grid(NKABATCH bt, int V) { return nka_grid_for(bt->geom, 4, bt->vlen, V, NKA_THREADS); }

unsigned nka_grid_clamp(size_t n)
{
  const size_t g = (n + NKA_THREADS - 1) / NKA_THREADS;
  return (unsigned)(g < 1024 ? (g < 1 ? 1 : g) : 1024);
}

// Aborts (file:line, under `call`) unless `stop` is a valid nka_stop_test for members of length vlen and
// gamma a valid restart_growth.
static void solve_require(const char* call, const nka_stop_test* stop, size_t vlen, double gamma)
{
  char msg[160];
  const auto require = [&](bool ok, const char* what) {
    if (ok) return;
    snprintf(msg, sizeof msg, "%s: %s", call, what);
    nka_fail(__FILE__, __LINE__, msg);
  };
  require(stop != NULL, "null stop test");
  require(stop->atol >= 0.0 && stop->rtol >= 0.0, "atol and rtol must be >= 0");
  require(stop->maxit >= 0, "maxit must be >= 0");
  require(stop->dtol == 0.0 || stop->dtol >= 1.0, "dtol must be 0 (off) or >= 1");
  require(!stop->scale_dev || stop->ldscale >= vlen, "ldscale must be >= vlen");
  require(gamma >= 0.0 && isfinite(gamma), "restart_growth must be 0 (off) or a finite number > 0");
}

// 0 if the driver has conditional graph nodes (12.4); otherwise prints why `call` cannot build its graph.
static int driver_refused(const char* call)
{
  int driver = 0;
  CUDA_CHECK(cudaDriverGetVersion(&driver));
  if (driver >= 12040) return 0;
  fprintf(stderr, "nka_b200: %s: conditional graph nodes need a CUDA 12.4 driver, this one is %d.%d: %s\n", call,
          driver / 1000, (driver % 1000) / 10, cudaGetErrorString(cudaErrorInsufficientDriver));
  fflush(stderr);
  return 1;
}

// CUDA refused the graph: the caller's residual graph or the driver.  Not a library fault: print CUDA's
// reason, clear the (non-sticky) error and let the caller decide.
static cudaGraphExec_t graph_refused(const char* call, cudaGraph_t g, const char* what, cudaError_t e)
{
  fprintf(stderr, "nka_b200: %s: %s: %s\n", call, what, cudaGetErrorString(e));
  fflush(stderr);
  cudaGetLastError();
  if (g) cudaGraphDestroy(g);
  return nullptr;
}

// The graph  prologue -> WHILE (cond) { residual graph, cloned as a child -> body }, instantiated and
// uploaded on `s`.  A graph CUDA refuses gives nullptr, after printing CUDA's reason under `call`, with no
// error left behind.
static cudaGraphExec_t nka_while_graph(const char* call, cudaStream_t s, cudaGraph_t residual,
                                       const NkaCaptureFn& prologue, const NkaCaptureFn& body_fn)
{
  cudaGraph_t g = nullptr;
  CUDA_CHECK(cudaGraphCreate(&g, 0));
  cudaGraphConditionalHandle cond;
  cudaError_t e = cudaGraphConditionalHandleCreate(&cond, g, 1, cudaGraphCondAssignDefault);
  if (e != cudaSuccess) return graph_refused(call, g, "cudaGraphConditionalHandleCreate", e);
  CUDA_CHECK(cudaStreamBeginCaptureToGraph(s, g, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
  prologue(s, cond);
  CUDA_CHECK(cudaStreamEndCapture(s, &g));
  // the prologue is a chain: the WHILE node follows its one node without a dependent
  size_t nnodes = 0, nedges = 0;
  CUDA_CHECK(cudaGraphGetNodes(g, nullptr, &nnodes));
  CUDA_CHECK(cudaGraphGetEdges(g, nullptr, nullptr, &nedges));
  std::vector<cudaGraphNode_t> nodes(nnodes), from(nedges), to(nedges);
  CUDA_CHECK(cudaGraphGetNodes(g, nodes.data(), &nnodes));
  if (nedges) CUDA_CHECK(cudaGraphGetEdges(g, from.data(), to.data(), &nedges));
  cudaGraphNode_t tail = nullptr;
  int ntails = 0;
  for (cudaGraphNode_t nd : nodes)
    if (std::find(from.begin(), from.end(), nd) == from.end()) {
      tail = nd;
      ++ntails;
    }
  NKA_REQUIRE(ntails == 1, "nka_while_graph: the prologue must end in exactly one node (a chain)");
  cudaGraphNodeParams cp = {};
  cp.type = cudaGraphNodeTypeConditional;
  cp.conditional.handle = cond;
  cp.conditional.type = cudaGraphCondTypeWhile;
  cp.conditional.size = 1;
  cudaGraphNode_t wnode = nullptr;
  e = cudaGraphAddNode(&wnode, g, &tail, 1, &cp);
  if (e != cudaSuccess) return graph_refused(call, g, "cudaGraphAddNode (WHILE)", e);
  cudaGraph_t body = cp.conditional.phGraph_out[0];

  // the body: the caller's residual (cloned), then the body's kernels, captured after it
  cudaGraphNode_t child = nullptr;
  e = cudaGraphAddChildGraphNode(&child, body, nullptr, 0, residual);
  if (e != cudaSuccess) return graph_refused(call, g, "the residual graph cannot be a conditional body's child graph", e);
  CUDA_CHECK(cudaStreamBeginCaptureToGraph(s, body, &child, nullptr, 1, cudaStreamCaptureModeThreadLocal));
  body_fn(s, cond);
  CUDA_CHECK(cudaStreamEndCapture(s, &body));

  cudaGraphExec_t exec = nullptr;
  e = cudaGraphInstantiate(&exec, g, 0);
  if (e != cudaSuccess) return graph_refused(call, g, "cudaGraphInstantiate", e);
  CUDA_CHECK(cudaGraphUpload(exec, s));
  CUDA_CHECK(cudaGraphDestroy(g));
  return exec;
}

NkaSolve* nka_solve_create(const char* call, NkaSolve* H, void* residual, double* x, size_t ldx, const double* f,
                           size_t ldf, const nka_stop_test* stop, double gamma, bool history,
                           const std::function<void(cudaStream_t)>& init, const NkaCaptureFn& prologue,
                           const NkaCaptureFn& body)
{
  NKABATCH bt = H->bt;
  solve_require(call, stop, bt->vlen, gamma);
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, call, "it builds and uploads a graph and synchronises");
  if (driver_refused(call)) {
    delete H;
    return nullptr;
  }
  const size_t nb = (size_t)bt->nbatch;
  H->x = x, H->ldx = ldx, H->f = f, H->ldf = ldf;
  H->stop = *stop;
  H->gamma = gamma;
  H->hstride = history ? bt->nbatch : 0;
  H->nhist = history ? (size_t)(stop->maxit + 1) * nb : nb;
  // the 16-byte paths need every row 16-byte aligned
  H->Vc = nka_aligned16(f, ldf) ? 2 : 1;
  H->Vs = H->Vc == 2 && nka_aligned16(x, ldx) ? 2 : 1;
  H->gc = (unsigned)nka_loop_grid(bt, H->Vc);
  H->gs = (unsigned)nka_loop_grid(bt, H->Vs);
  H->prow = H->gc;
  CUDA_CHECK(cudaMalloc(&H->iters, nb * sizeof(int)));
  CUDA_CHECK(cudaMalloc(&H->status, nb * sizeof(int)));
  CUDA_CHECK(cudaMalloc(&H->active, nb));
  CUDA_CHECK(cudaMalloc(&H->r0, nb * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&H->rlast, nb * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&H->hist, H->nhist * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&H->partials, nb * H->prow * sizeof(double)));
  CUDA_CHECK(cudaMalloc(&H->tickets, nb * sizeof(unsigned)));
  if (gamma > 0.0) {
    CUDA_CHECK(cudaMalloc(&H->rprev, nb * sizeof(double)));
    CUDA_CHECK(cudaMalloc(&H->nrst, nb * sizeof(int)));
    CUDA_CHECK(cudaMalloc(&H->rmask, nb));
  }

  cudaStream_t s = nullptr;               // private: the batch's own stream may be the legacy default
  CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  CUDA_CHECK(cudaMemsetAsync(H->tickets, 0, nb * sizeof(unsigned), s));
  if (bt->poison) {
    CUDA_CHECK(cudaMemsetAsync(H->partials, 0xFF, nb * H->prow * sizeof(double), s));
    CUDA_CHECK(cudaMemsetAsync(H->r0, 0xFF, nb * sizeof(double), s));
    CUDA_CHECK(cudaMemsetAsync(H->rlast, 0xFF, nb * sizeof(double), s));
    CUDA_CHECK(cudaMemsetAsync(H->hist, 0xFF, H->nhist * sizeof(double), s));
    if (gamma > 0.0) CUDA_CHECK(cudaMemsetAsync(H->rprev, 0xFF, nb * sizeof(double), s));
  }
  init(s);
  H->exec = nka_while_graph(call, s, (cudaGraph_t)residual, prologue, body);
  if (!H->exec) {
    cudaStreamDestroy(s);
    delete H;
    return nullptr;
  }
  CUDA_CHECK(cudaStreamSynchronize(s));
  CUDA_CHECK(cudaStreamDestroy(s));
  return H;
}

void nka_solve_check(const NkaSolve& H, cudaStream_t s, const int* index)
{
  const dim3 g(H.gc, (unsigned)H.bt->nbatch);
  // the scale's load width follows its own rows' alignment; Vc and gc follow F's alone
  const int scale16 = H.stop.scale_dev && nka_aligned16(H.stop.scale_dev, H.stop.ldscale);
  if (H.Vc == 2)
    nka_loop_check<2><<<g, NKA_THREADS, 0, s>>>(H.f, H.ldf, H.bt->vlen, H.hstride, H.iters, H.status, H.active, H.r0,
                                                H.rlast, H.hist, H.partials, H.prow, H.tickets, H.stop, index, scale16);
  else
    nka_loop_check<1><<<g, NKA_THREADS, 0, s>>>(H.f, H.ldf, H.bt->vlen, H.hstride, H.iters, H.status, H.active, H.r0,
                                                H.rlast, H.hist, H.partials, H.prow, H.tickets, H.stop, index, scale16);
  CUDA_CHECK(cudaGetLastError());
}

void nka_solve_step(const NkaSolve& H, cudaStream_t s)
{
  const dim3 g(H.gs, (unsigned)H.bt->nbatch);
  if (H.Vs == 2)
    nka_loop_step<2><<<g, NKA_THREADS, 0, s>>>(H.x, H.ldx, H.f, H.ldf, H.bt->vlen, H.active, H.iters);
  else
    nka_loop_step<1><<<g, NKA_THREADS, 0, s>>>(H.x, H.ldx, H.f, H.ldf, H.bt->vlen, H.active, H.iters);
  CUDA_CHECK(cudaGetLastError());
}

void nka_solve_launch(const NkaSolve* H, const char* call)
{
  DeviceGuard guard(H->bt->device);
  if (nka_capture_status(H->bt->stream) != 0)
    nka_capture_fail(call, "a graph with conditional nodes cannot become a child of another graph");
  CUDA_CHECK(cudaGraphLaunch(H->exec, H->bt->stream));
}

void nka_solve_copy_out(const NkaSolve* H, const char* call, const char* why, std::initializer_list<NkaCopy> copies)
{
  NKABATCH bt = H->bt;
  DeviceGuard guard(bt->device);
  nka_refuse_capture(bt->stream, call, why);
  bool queued = false;
  for (const NkaCopy& c : copies) {
    if (!c.src) {
      memset(c.dst, 0, c.bytes);
      continue;
    }
    CUDA_CHECK(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, bt->stream));
    queued = true;
  }
  if (queued) CUDA_CHECK(cudaStreamSynchronize(bt->stream));
}

void nka_solve_destroy(NkaSolve* H)
{
  if (!H) return;
  DeviceGuard guard(H->bt->device);
  cudaStreamSynchronize(H->bt->stream);
  delete H;
}

// ---------------------------------------------------------------------------
// the handle and its entry points
// ---------------------------------------------------------------------------
struct nka_batch_loop : NkaSolve {};

extern "C" NKABATCHLOOP nka_batch_loop_create(NKABATCH bt, void* residual_graph, double* x, size_t ldx, double* f,
                                             size_t ldf, double atol, double rtol, int maxit)
{
  const nka_stop_test stop = {atol, rtol, 0.0, maxit, NULL, NULL, NULL, NULL, 0};
  return nka_batch_loop_create_stop(bt, residual_graph, x, ldx, f, ldf, &stop);
}

extern "C" NKABATCHLOOP nka_batch_loop_create_stop(NKABATCH bt, void* residual_graph, double* x, size_t ldx, double* f,
                                                  size_t ldf, const nka_stop_test* stop_in)
{
  return nka_batch_loop_create_restart(bt, residual_graph, x, ldx, f, ldf, stop_in, 0.0);
}

extern "C" NKABATCHLOOP nka_batch_loop_create_restart(NKABATCH bt, void* residual_graph, double* x, size_t ldx,
                                                     double* f, size_t ldf, const nka_stop_test* stop_in,
                                                     double restart_growth)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_loop_create: null handle");
  NKA_REQUIRE(residual_graph != NULL, "nka_batch_loop_create: null residual graph");
  NKA_REQUIRE(x != NULL && f != NULL, "nka_batch_loop_create: null x or f");
  NKA_REQUIRE(ldx >= bt->vlen && ldf >= bt->vlen, "nka_batch_loop_create: ldx and ldf must be >= vlen");
  NKABATCHLOOP L = new nka_batch_loop();
  L->bt = bt;
  // reset [, guard reset]; at create time too: every member RUNNING at 0 steps, as the results of a loop
  // never launched read
  const auto reset = [&](cudaStream_t cs) {
    nka_loop_reset<<<nka_grid_clamp(L->nhist), NKA_THREADS, 0, cs>>>(L->iters, L->status, L->active, L->rlast, L->hist,
                                                                     L->nhist, bt->nbatch);
    CUDA_CHECK(cudaGetLastError());
    if (L->gamma > 0.0) nka_solve_guard_reset(*L, cs, nullptr, 0);
  };
  // then the WHILE node: { residual, check, decide, [guard, restart,] update, step }
  const auto body = [&](cudaStream_t cs, cudaGraphConditionalHandle cond) {
    nka_solve_check(*L, cs, /*index=*/nullptr);
    nka_loop_decide<<<1, 1024, 0, cs>>>(L->active, bt->nbatch, cond);
    CUDA_CHECK(cudaGetLastError());
    if (L->gamma > 0.0) nka_solve_guard_restart(*L, cs, nullptr, nullptr, nullptr);
    nka_batch_update_captured(bt, f, ldf, L->active, cs);
    nka_solve_step(*L, cs);
  };
  return static_cast<NKABATCHLOOP>(nka_solve_create("nka_batch_loop_create", L, residual_graph, x, ldx, f, ldf, stop_in,
                                                    restart_growth, /*history=*/true, reset,
                                                    [&](cudaStream_t cs, cudaGraphConditionalHandle) { reset(cs); },
                                                    body));
}

extern "C" void nka_batch_loop_launch(NKABATCHLOOP L)
{
  NKA_REQUIRE(L != NULL, "nka_batch_loop_launch: null loop");
  nka_solve_launch(L, "nka_batch_loop_launch");
}

extern "C" void nka_batch_loop_results(NKABATCHLOOP L, int* iters, int* status, double* norm)
{
  NKA_REQUIRE(L != NULL && iters != NULL && status != NULL && norm != NULL, "nka_batch_loop_results: null argument");
  const size_t nb = (size_t)L->bt->nbatch;
  nka_solve_copy_out(L, "nka_batch_loop_results", "it copies the loop's results to the host and synchronises",
                     {{iters, L->iters, nb * sizeof(int)}, {status, L->status, nb * sizeof(int)},
                      {norm, L->rlast, nb * sizeof(double)}});
}

extern "C" void nka_batch_loop_history(NKABATCHLOOP L, double* norms)
{
  NKA_REQUIRE(L != NULL && norms != NULL, "nka_batch_loop_history: null argument");
  nka_solve_copy_out(L, "nka_batch_loop_history", "it copies the loop's history to the host and synchronises",
                     {{norms, L->hist, L->nhist * sizeof(double)}});
}

extern "C" void nka_batch_loop_restarts(NKABATCHLOOP L, int* restarts)
{
  NKA_REQUIRE(L != NULL && restarts != NULL, "nka_batch_loop_restarts: null argument");
  nka_solve_copy_out(L, "nka_batch_loop_restarts", "it copies the loop's restart counts to the host and synchronises",
                     {{restarts, L->nrst, (size_t)L->bt->nbatch * sizeof(int)}});
}

extern "C" void nka_batch_loop_destroy(NKABATCHLOOP L) { nka_solve_destroy(L); }
