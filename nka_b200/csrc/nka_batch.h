// nka_batch.h -- the batched accelerator's handle and kernel tables (nka_batch.cu, nka_batch_pass_a.cu,
// nka_batch_pass_b.cu), shared with its device-side fixed-point loops (nka_batch_loop.cu) and work
// queues (nka_batch_queue.cu); and the solve core both build on (NkaSolve: nka_batch_loop.cu, whose
// guard launchers are in nka_batch_guard.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <initializer_list>
#include "nka_dispatch.h"
#include "../../include/nka_b200.h"

struct nka_batch {
  int nbatch = 0, mvec = 0;
  size_t vlen = 0, ld = 0, wstride = 0;   // wstride = (mvec+1)*ld: one member's W (or Z) block
  double vtol = 0.01;
  int device = 0;
  cudaStream_t stream = nullptr;
  NkaSweepGeom geom;
  bool lazy = true;                       // NKA_LAZY_LAST, as nka_init_ex reads it
  bool poison = false;                    // NKA_POISON_ALLOC
  int nc = 0;                             // pass A's columns: mvec (lazy) or mvec + 1
  double* W = nullptr;
  double* Z = nullptr;
  NkaDevState* S = nullptr;
  double* dots = nullptr;                 // nbatch x 2*NKA_MAXSLOT
  double* partials = nullptr;             // nbatch x prow
  size_t prow = 0;                        // doubles of partial rows per member
  unsigned* tickets = nullptr;            // nbatch
  int* query = nullptr;                   // device, 2*nbatch ints (nka_batch_query_kernel)
  unsigned long long launches = 0;
};

// One batched update queued on `stream` while that stream captures (a loop's body graph): the update
// nka_batch_accel_update queues, counted as no launch, whatever stream the handle itself uses.
void nka_batch_update_captured(nka_batch* bt, double* f, size_t ldf, const unsigned char* active, cudaStream_t stream);
// nka_batch_restart of the masked members, queued on a capturing `stream` likewise.
void nka_batch_restart_captured(nka_batch* bt, const unsigned char* mask, cudaStream_t stream);

// ---- the solve core shared by the device-side loops and queues (nka_batch_loop.cu, nka_batch_guard.cu) ----
// A device-side solve over a batch: its graph, the per-slot state (slot b is member b) and what every body
// launch needs.  nka_batch_loop and nka_batch_queue derive from it; deleting one frees everything.
struct NkaSolve {
  NKABATCH bt = nullptr;
  cudaGraphExec_t exec = nullptr;
  int* iters = nullptr;                   // device, nbatch: the slot's steps
  int* status = nullptr;                  // device, nbatch: NKA_LOOP_* (or a queue's NKA_QUEUE_IDLE)
  unsigned char* active = nullptr;        // device, nbatch: status == RUNNING, the update's and step's mask
  double* r0 = nullptr;                   // device, nbatch: each slot's norm at check 0
  double* rlast = nullptr;                // device, nbatch: each slot's latest norm
  double* hist = nullptr;                 // device, nhist: check k of slot b at hist[k * hstride + b]
  double* partials = nullptr;             // device, nbatch x prow
  unsigned* tickets = nullptr;            // device, nbatch
  double* rprev = nullptr;                // device, nbatch: the previous check's norm (gamma > 0 only)
  int* nrst = nullptr;                    // device, nbatch: restarts (gamma > 0 only)
  unsigned char* rmask = nullptr;         // device, nbatch: the guard's restart mask (gamma > 0 only)
  double* x = nullptr;                    // the caller's X and F rows
  const double* f = nullptr;
  size_t ldx = 0, ldf = 0;
  size_t nhist = 0, prow = 0;
  int hstride = 0;                        // a loop's nbatch (maxit+1 rows of history); a queue's 0 (one scratch row)
  int Vc = 1, Vs = 1;                     // access widths of check (F) and step (X, F)
  unsigned gc = 0, gs = 0;                // their CTAs per slot
  nka_stop_test stop = {};
  double gamma = 0.0;                     // restart_growth; 0: no guard
  virtual ~NkaSolve();
};

// The graph's prologue or body: its kernels queued on the capturing stream.
typedef std::function<void(cudaStream_t, cudaGraphConditionalHandle)> NkaCaptureFn;
// The create steps loops and queues share, under `call`, for H (a new handle with bt set): the stop test's
// and gamma's checks, the capture refusal, the driver check, the slot state for x, f and a history of
// maxit+1 rows (history) or one scratch row, a private stream on which the tickets are zeroed, the state
// poisoned (NKA_POISON_ALLOC), then `init` allocates and resets the rest, and the graph
//   prologue -> WHILE (cond) { residual graph, cloned as a child -> body },
// instantiated, uploaded and synchronised.  A driver or graph CUDA refuses deletes H and gives nullptr,
// after printing why on stderr.
NkaSolve* nka_solve_create(const char* call, NkaSolve* H, void* residual, double* x, size_t ldx, const double* f,
                           size_t ldf, const nka_stop_test* stop, double gamma, bool history,
                           const std::function<void(cudaStream_t)>& init, const NkaCaptureFn& prologue,
                           const NkaCaptureFn& body);
// The body's nka_loop_check<Vc> over dim3(gc, nbatch) on the capturing `s`; it applies the stop test with
// the per-problem entries of row b at index[b] (index NULL: at b).
void nka_solve_check(const NkaSolve& H, cudaStream_t s, const int* index);
// The body's nka_loop_step<Vs> over dim3(gs, nbatch): X_b += F_b of the active slots.
void nka_solve_step(const NkaSolve& H, cudaStream_t s);
// The residual-growth restart (nka_batch_guard.cu): the reset of the restart counts nrst and, in a queue,
// p_restarts (nproblems; NULL and 0 in a loop); and the body's guard followed by the batch's restart of
// its mask rmask.  claimed, move_out and p_restarts are the queue's (NULL in a loop).
void nka_solve_guard_reset(const NkaSolve& H, cudaStream_t s, int* p_restarts, size_t nproblems);
void nka_solve_guard_restart(const NkaSolve& H, cudaStream_t s, const unsigned char* claimed, const int* move_out,
                             int* p_restarts);
// The graph launch on the batch's stream, refused (under `call`) while that stream captures.
void nka_solve_launch(const NkaSolve* H, const char* call);
// The device-to-host copies of a results query on the batch's stream, refused (call, why) while it captures,
// then a synchronise.  A copy from NULL zeroes dst instead; with no copy left nothing is synchronised.
struct NkaCopy { void* dst; const void* src; size_t bytes; };
void nka_solve_copy_out(const NkaSolve* H, const char* call, const char* why, std::initializer_list<NkaCopy> copies);
// Waits for the batch's stream and deletes H (NULL: nothing).
void nka_solve_destroy(NkaSolve* H);
// CTAs per member of the loop's check and step kernels at access width V (vlen only, as the batch's fix-up)
int nka_loop_grid(nka_batch* bt, int V);
// ceil(n / NKA_THREADS) CTAs, clamped to 1..1024: the grid of the solves' element-wise reset kernels
unsigned nka_grid_clamp(size_t n);
// Whether rows at p with stride ld are all 16-byte aligned: the base address and an even row stride.
inline bool nka_aligned16(const void* p, size_t ld) { return (uintptr_t)p % 16 == 0 && ld % 2 == 0; }

// (F, ldf, W, wstride, ld, n, S, partials, prow, tickets, dots, active)
typedef void (*NkaBatchPassAFn)(const double*, size_t, const double*, size_t, size_t, size_t, const NkaDevState*, double*,
                                size_t, unsigned*, double*, const unsigned char*);
// (F, ldf, W, Z, wstride, ld, n, S, active)
typedef void (*NkaBatchPassBFn)(double*, size_t, double*, double*, size_t, size_t, size_t, const NkaDevState*,
                                const unsigned char*);

// nc in 1..NKA_MAXSLOT, nz in 0..NKA_MAXSLOT-1, v in {1,2}; nullptr if not instantiated in this build
NkaBatchPassAFn nka_get_batch_pass_a(int nc, int v);
NkaBatchPassBFn nka_get_batch_pass_b(int nz, int v);
