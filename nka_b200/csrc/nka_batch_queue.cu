// nka_batch_queue.cu -- device-side work queues over a batched accelerator (include/nka_b200.h,
// INTEGRATION.md section 9, DESIGN.md section 14).  nproblems fixed-point problems run through the
// batch's nbatch members, used as slots, in one graph launch:
//
//   reset -> claim -> rows -> restart
//   WHILE (any slot holds a problem) { residual graph -> check -> claim -> rows -> restart -> update -> step }
//
// check and step are the loop's kernels (nka_batch_loop.cu); check reads each slot's problem from
// slot_problem for the per-problem parts of the stop test.  claim (one CTA) retires every
// slot whose problem stopped, writing that problem's steps, status and norm, and hands the free slots
// the next problem ids in slot order; rows copies a retired slot's X row out and a claimed problem's
// initial guess in; restart restarts the claimed slots' accelerators.  A claimed slot is not checked
// until the next body, whose check sees the residual at its initial guess and sets r0 there, as the
// loop's first check does.  Every kernel is per slot or element-wise, so a problem's bits are those
// of the loop on a just-restarted member, whatever slot it lands in and whatever surrounds it.  The
// queue is built on the loop's solve core (nka_batch.h: NkaSolve, nka_solve_create); this file keeps
// the queue's own arguments and per-problem arrays, its kernels, and its prologue and body.
#include <cuda_runtime.h>
#include <limits.h>
#include <math.h>
#include <stdio.h>

#include "../../include/nka_b200.h"
#include "nka_internal.h"
#include "nka_batch.h"
#include "nka_kernels.cuh"

#define NKA_QUEUE_IDLE (-1)             // a slot's status while it holds no problem: check skips it
#define NKA_QUEUE_CLAIM_THREADS 1024    // claim's one CTA: 32 warps, a two-level scan

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// Every problem RUNNING at 0 steps with a NaN norm; every slot idle; no problem handed out yet.
__global__ void __launch_bounds__(NKA_THREADS)
nka_queue_reset(int* __restrict__ p_iters, int* __restrict__ p_status, double* __restrict__ p_norm, size_t nproblems,
                int* __restrict__ slot_problem, int* __restrict__ status, unsigned char* __restrict__ active, int nbatch,
                long long* __restrict__ next)
{
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t n = nproblems > (size_t)nbatch ? nproblems : (size_t)nbatch;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (i < nproblems) {
      p_iters[i] = 0;
      p_status[i] = NKA_LOOP_RUNNING;
      p_norm[i] = nan;
    }
    if (i < (size_t)nbatch) {
      slot_problem[i] = -1;
      status[i] = NKA_QUEUE_IDLE;
      active[i] = 0;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *next = 0;
}

// Retire the slots whose problem stopped, then give the free slots the next problem ids in slot order
// (an exclusive scan of free slots over contiguous per-thread ranges), and set the WHILE condition.
// move_out[b] / move_in[b]: the problem whose row leaves / enters slot b's X row, or -1.
__global__ void __launch_bounds__(NKA_QUEUE_CLAIM_THREADS)
nka_queue_claim(int* __restrict__ slot_problem, int nbatch, long long* __restrict__ next, long long nproblems,
                int* __restrict__ iters, int* __restrict__ status, unsigned char* __restrict__ active,
                const double* __restrict__ rlast, int* __restrict__ p_iters, int* __restrict__ p_status,
                double* __restrict__ p_norm, int* __restrict__ move_out, int* __restrict__ move_in,
                unsigned char* __restrict__ claimed, cudaGraphConditionalHandle cond)
{
  __shared__ int wsum[NKA_QUEUE_CLAIM_THREADS / 32];
  const int per = (nbatch + NKA_QUEUE_CLAIM_THREADS - 1) / NKA_QUEUE_CLAIM_THREADS;
  const int b0 = threadIdx.x * per;
  const int b1 = b0 + per < nbatch ? b0 + per : nbatch;
  int nfree = 0;
  for (int b = b0; b < b1; ++b) {
    int p = slot_problem[b];
    int out = -1;
    if (p >= 0 && status[b] != NKA_LOOP_RUNNING) {
      p_iters[p] = iters[b];
      p_status[p] = status[b];
      p_norm[p] = rlast[b];
      out = p;
      p = -1;
      slot_problem[b] = -1;
    }
    move_out[b] = out;
    nfree += p < 0;
  }
  // inclusive scan of nfree over the CTA: within each warp, then over the warp totals
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int v = nfree;
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  if (lane == 31) wsum[warp] = v;
  __syncthreads();
  if (warp == 0) {
    int w = wsum[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += u;
    }
    wsum[lane] = w;
  }
  __syncthreads();
  const long long base = *next;
  long long k = base + (warp ? wsum[warp - 1] : 0) + v - nfree;
  int busy = 0;
  for (int b = b0; b < b1; ++b) {
    int p = slot_problem[b];
    int in = -1;
    if (p < 0) {
      if (k < nproblems) {
        p = in = (int)k;
        slot_problem[b] = p;
        iters[b] = 0;
        status[b] = NKA_LOOP_RUNNING;
        active[b] = 0;                  // not updated or stepped before its first check
      } else {
        status[b] = NKA_QUEUE_IDLE;
        active[b] = 0;
      }
      ++k;
    }
    move_in[b] = in;
    claimed[b] = in >= 0;
    busy |= p >= 0;
  }
  busy = __syncthreads_or(busy);          // also orders every read of *next before its update
  if (threadIdx.x == 0) {
    const long long taken = base + wsum[NKA_QUEUE_CLAIM_THREADS / 32 - 1];
    *next = taken < nproblems ? taken : nproblems;
    cudaGraphSetConditional(cond, busy ? 1u : 0u);
  }
}

// Per slot (blockIdx.y): a retired problem's final iterate X_b -> Xout[move_out[b]], then a claimed
// problem's initial guess X0[move_in[b]] -> X_b.  The two rows are different problems', so Xout == X0
// is safe; each element is read before it is overwritten by the same thread.
template <int V>
__global__ void __launch_bounds__(NKA_THREADS)
nka_queue_rows(double* __restrict__ X, size_t ldx, const double* X0, size_t ldx0, double* Xout, size_t ldxout, size_t n,
               const int* __restrict__ move_out, const int* __restrict__ move_in)
{
  const size_t b = blockIdx.y;
  const int po = move_out[b], pi = move_in[b];
  if (po < 0 && pi < 0) return;
  double* x = X + b * ldx;
  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS;
  const size_t start = (size_t)blockIdx.x * NKA_THREADS + threadIdx.x;
  if (po >= 0) {
    double* xo = Xout + (size_t)po * ldxout;
    for (size_t i = start; i < nv; i += stride) Vec<V>::ld_plain(x, i).st(xo, i);
    if (V == 2 && (n & 1) && start == 0) xo[n - 1] = x[n - 1];
  }
  if (pi >= 0) {
    const double* x0 = X0 + (size_t)pi * ldx0;
    for (size_t i = start; i < nv; i += stride) Vec<V>::ld_plain(x0, i).st(x, i);
    if (V == 2 && (n & 1) && start == 0) x[n - 1] = x0[n - 1];
  }
}

// ---------------------------------------------------------------------------
// the handle: the solve core's slot state (nka_batch.h) and the queue's own arrays
// ---------------------------------------------------------------------------
struct nka_batch_queue : NkaSolve {
  size_t nproblems = 0;
  unsigned char* claimed = nullptr;       // device, nbatch: the restart's mask
  int* move_out = nullptr;                // device, nbatch
  int* move_in = nullptr;                 // device, nbatch
  long long* next = nullptr;              // device: the next problem id to hand out
  int* p_iters = nullptr;                 // device, nproblems
  int* p_status = nullptr;                // device, nproblems
  double* p_norm = nullptr;               // device, nproblems
  int* p_restarts = nullptr;              // device, nproblems (restart_growth > 0 only)
  ~nka_batch_queue() override
  {
    cudaFree(claimed); cudaFree(move_out); cudaFree(move_in); cudaFree(next); cudaFree(p_iters); cudaFree(p_status);
    cudaFree(p_norm); cudaFree(p_restarts);
  }
};

extern "C" NKABATCHQUEUE nka_batch_queue_create(NKABATCH bt, void* residual_graph, double* x, size_t ldx, double* f,
                                               size_t ldf, int* slot_problem, const double* x0, size_t ldx0,
                                               double* xout, size_t ldxout, size_t nproblems, double atol, double rtol,
                                               int maxit)
{
  const nka_stop_test stop = {atol, rtol, 0.0, maxit, NULL, NULL, NULL, NULL, 0};
  return nka_batch_queue_create_stop(bt, residual_graph, x, ldx, f, ldf, slot_problem, x0, ldx0, xout, ldxout, nproblems,
                                     &stop);
}

extern "C" NKABATCHQUEUE nka_batch_queue_create_stop(NKABATCH bt, void* residual_graph, double* x, size_t ldx, double* f,
                                                    size_t ldf, int* slot_problem, const double* x0, size_t ldx0,
                                                    double* xout, size_t ldxout, size_t nproblems,
                                                    const nka_stop_test* stop_in)
{
  return nka_batch_queue_create_restart(bt, residual_graph, x, ldx, f, ldf, slot_problem, x0, ldx0, xout, ldxout,
                                        nproblems, stop_in, 0.0);
}

extern "C" NKABATCHQUEUE nka_batch_queue_create_restart(NKABATCH bt, void* residual_graph, double* x, size_t ldx,
                                                       double* f, size_t ldf, int* slot_problem, const double* x0,
                                                       size_t ldx0, double* xout, size_t ldxout, size_t nproblems,
                                                       const nka_stop_test* stop_in, double restart_growth)
{
  NKA_REQUIRE(bt != NULL, "nka_batch_queue_create: null handle");
  NKA_REQUIRE(residual_graph != NULL, "nka_batch_queue_create: null residual graph");
  NKA_REQUIRE(x != NULL && f != NULL && slot_problem != NULL && x0 != NULL && xout != NULL,
              "nka_batch_queue_create: null x, f, slot_problem, x0 or xout");
  NKA_REQUIRE(ldx >= bt->vlen && ldf >= bt->vlen && ldx0 >= bt->vlen && ldxout >= bt->vlen,
              "nka_batch_queue_create: ldx, ldf, ldx0 and ldxout must be >= vlen");
  NKA_REQUIRE(nproblems >= 1 && nproblems <= (size_t)INT_MAX, "nka_batch_queue_create: nproblems must be in 1..INT_MAX");
  NKABATCHQUEUE Q = new nka_batch_queue();
  Q->bt = bt;
  Q->nproblems = nproblems;
  const size_t nb = (size_t)bt->nbatch;
  const int Vr = nka_aligned16(x, ldx) && nka_aligned16(x0, ldx0) && nka_aligned16(xout, ldxout) ? 2 : 1;
  const dim3 grows((unsigned)nka_loop_grid(bt, Vr), (unsigned)nb);
  const unsigned greset = nka_grid_clamp(nproblems > nb ? nproblems : nb);
  const auto reset = [&](cudaStream_t cs, int nslots) {
    nka_queue_reset<<<greset, NKA_THREADS, 0, cs>>>(Q->p_iters, Q->p_status, Q->p_norm, nproblems, slot_problem, Q->status,
                                                   Q->active, nslots, Q->next);
    CUDA_CHECK(cudaGetLastError());
    if (Q->gamma > 0.0) nka_solve_guard_reset(*Q, cs, Q->p_restarts, nproblems);
  };
  const auto init = [&](cudaStream_t s) {
    CUDA_CHECK(cudaMalloc(&Q->claimed, nb));
    CUDA_CHECK(cudaMalloc(&Q->move_out, nb * sizeof(int)));
    CUDA_CHECK(cudaMalloc(&Q->move_in, nb * sizeof(int)));
    CUDA_CHECK(cudaMalloc(&Q->next, sizeof(long long)));
    CUDA_CHECK(cudaMalloc(&Q->p_iters, nproblems * sizeof(int)));
    CUDA_CHECK(cudaMalloc(&Q->p_status, nproblems * sizeof(int)));
    CUDA_CHECK(cudaMalloc(&Q->p_norm, nproblems * sizeof(double)));
    if (Q->gamma > 0.0) CUDA_CHECK(cudaMalloc(&Q->p_restarts, nproblems * sizeof(int)));
    // before any launch: every problem RUNNING at 0 steps (slot_problem is the caller's until a launch)
    reset(s, 0);
  };
  auto claim_rows_restart = [&](cudaStream_t cs, cudaGraphConditionalHandle cond) {
    nka_queue_claim<<<1, NKA_QUEUE_CLAIM_THREADS, 0, cs>>>(slot_problem, bt->nbatch, Q->next, (long long)nproblems, Q->iters,
                                                          Q->status, Q->active, Q->rlast, Q->p_iters, Q->p_status,
                                                          Q->p_norm, Q->move_out, Q->move_in, Q->claimed, cond);
    CUDA_CHECK(cudaGetLastError());
    if (Vr == 2)
      nka_queue_rows<2><<<grows, NKA_THREADS, 0, cs>>>(x, ldx, x0, ldx0, xout, ldxout, bt->vlen, Q->move_out, Q->move_in);
    else
      nka_queue_rows<1><<<grows, NKA_THREADS, 0, cs>>>(x, ldx, x0, ldx0, xout, ldxout, bt->vlen, Q->move_out, Q->move_in);
    CUDA_CHECK(cudaGetLastError());
    if (Q->gamma > 0.0)   // restart the claimed slots and the running ones the rule picks: rmask = claimed | rule
      nka_solve_guard_restart(*Q, cs, Q->claimed, Q->move_out, Q->p_restarts);
    else
      nka_batch_restart_captured(bt, Q->claimed, cs);
  };
  // reset [, guard reset], claim, rows, [guard,] restart; then the WHILE node:
  //   { residual, check, claim, rows, [guard,] restart, update, step }
  auto prologue = [&](cudaStream_t cs, cudaGraphConditionalHandle cond) {
    reset(cs, bt->nbatch);
    claim_rows_restart(cs, cond);
  };
  auto body = [&](cudaStream_t cs, cudaGraphConditionalHandle cond) {
    // check's history stride is 0: every check of slot b writes hist[b], which nothing reads.  It runs after
    // the residual and before claim, so slot_problem[b] is still the problem whose F it checks.
    nka_solve_check(*Q, cs, /*index=*/slot_problem);
    claim_rows_restart(cs, cond);
    nka_batch_update_captured(bt, f, ldf, Q->active, cs);
    nka_solve_step(*Q, cs);
  };
  return static_cast<NKABATCHQUEUE>(nka_solve_create("nka_batch_queue_create", Q, residual_graph, x, ldx, f, ldf, stop_in,
                                                     restart_growth, /*history=*/false, init, prologue, body));
}

extern "C" void nka_batch_queue_launch(NKABATCHQUEUE Q)
{
  NKA_REQUIRE(Q != NULL, "nka_batch_queue_launch: null queue");
  nka_solve_launch(Q, "nka_batch_queue_launch");
}

extern "C" void nka_batch_queue_results(NKABATCHQUEUE Q, int* iters, int* status, double* norm)
{
  NKA_REQUIRE(Q != NULL && iters != NULL && status != NULL && norm != NULL, "nka_batch_queue_results: null argument");
  const size_t np = Q->nproblems;
  nka_solve_copy_out(Q, "nka_batch_queue_results", "it copies the queue's results to the host and synchronises",
                     {{iters, Q->p_iters, np * sizeof(int)}, {status, Q->p_status, np * sizeof(int)},
                      {norm, Q->p_norm, np * sizeof(double)}});
}

extern "C" void nka_batch_queue_restarts(NKABATCHQUEUE Q, int* restarts)
{
  NKA_REQUIRE(Q != NULL && restarts != NULL, "nka_batch_queue_restarts: null argument");
  nka_solve_copy_out(Q, "nka_batch_queue_restarts", "it copies the queue's restart counts to the host and synchronises",
                     {{restarts, Q->p_restarts, Q->nproblems * sizeof(int)}});
}

extern "C" void nka_batch_queue_destroy(NKABATCHQUEUE Q) { nka_solve_destroy(Q); }
