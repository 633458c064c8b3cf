// nka_batch_guard.cu -- the residual-growth restart of device-side loops and queues (include/nka_b200.h,
// INTEGRATION.md section 9b, DESIGN.md section 16).  With restart_growth = gamma > 0 the loop's and the
// queue's graph bodies gain two nodes after check (and, in a queue, after claim and rows):
//
//   guard -> batched restart(rmask)
//
// guard writes the restart mask: a member (slot) that check k >= 1 left RUNNING with r_k > gamma * r_{k-1}
// is restarted before this body's update, so that update sees an empty subspace, returns F_b unchanged and
// the step is a plain one; in a queue a slot that claim just filled is restarted too (the mask the queue
// restarted before), so the queue still makes one restart launch per body.  r_k and r_{k-1} are the norms
// check recorded (rlast), kept per slot in rprev.  rprev is read only when k >= 1 and written at every
// check of a running member, so r_{k-1} is always this launch's (loop) or this problem's (queue).  The
// guard is per slot and reads only the slot's own values, so a problem's bits do not depend on its slot.
// Its launchers take the solve core's handle (nka_batch.h: NkaSolve), whose rprev, nrst and rmask it uses.
#include <cuda_runtime.h>

#include "nka_internal.h"
#include "nka_batch.h"
#include "nka_kernels.cuh"

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// The prologue's: no restarts yet in this launch (loop) or for any problem (queue).
__global__ void __launch_bounds__(NKA_THREADS)
nka_loop_guard_reset(int* __restrict__ nrst, int nbatch, int* __restrict__ p_restarts, size_t nproblems)
{
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t n = nproblems > (size_t)nbatch ? nproblems : (size_t)nbatch;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (i < (size_t)nbatch) nrst[i] = 0;
    if (i < nproblems) p_restarts[i] = 0;
  }
}

// One thread per slot.  claimed / move_out / p_restarts: NULL in a loop.  A retiring slot's count goes
// to its problem first; a claimed slot is restarted with its count zeroed (that restart is not counted);
// a running slot is restarted by the rule and remembers r_k; any other slot is left alone.
__global__ void __launch_bounds__(NKA_THREADS)
nka_loop_guard(const unsigned char* __restrict__ active, const int* __restrict__ iters,
               const double* __restrict__ rlast, const unsigned char* __restrict__ claimed,
               const int* __restrict__ move_out, double gamma, double* __restrict__ rprev, int* __restrict__ nrst,
               int* __restrict__ p_restarts, unsigned char* __restrict__ rmask, int nbatch)
{
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < nbatch; b += gridDim.x * blockDim.x) {
    unsigned char m = 0;
    if (move_out) {
      const int po = move_out[b];
      if (po >= 0) p_restarts[po] = nrst[b];
    }
    if (claimed && claimed[b]) {
      m = 1;
      nrst[b] = 0;
    } else if (active[b]) {
      const double r = rlast[b];
      if (iters[b] >= 1 && r > gamma * rprev[b]) {
        m = 1;
        nrst[b] += 1;
      }
      rprev[b] = r;
    }
    rmask[b] = m;
  }
}

// ---------------------------------------------------------------------------
// launchers (nka_batch.h)
// ---------------------------------------------------------------------------
void nka_solve_guard_reset(const NkaSolve& H, cudaStream_t s, int* p_restarts, size_t nproblems)
{
  const int nbatch = H.bt->nbatch;
  const size_t n = nproblems > (size_t)nbatch ? nproblems : (size_t)nbatch;
  nka_loop_guard_reset<<<nka_grid_clamp(n), NKA_THREADS, 0, s>>>(H.nrst, nbatch, p_restarts, nproblems);
  CUDA_CHECK(cudaGetLastError());
}

void nka_solve_guard_restart(const NkaSolve& H, cudaStream_t s, const unsigned char* claimed, const int* move_out,
                             int* p_restarts)
{
  nka_loop_guard<<<nka_grid_clamp((size_t)H.bt->nbatch), NKA_THREADS, 0, s>>>(H.active, H.iters, H.rlast, claimed, move_out,
                                                                            H.gamma, H.rprev, H.nrst, p_restarts, H.rmask,
                                                                            H.bt->nbatch);
  CUDA_CHECK(cudaGetLastError());
  nka_batch_restart_captured(H.bt, H.rmask, s);
}
