// nka_batch.h -- the batched accelerator's handle and kernel tables (nka_batch.cu, nka_batch_pass_a.cu,
// nka_batch_pass_b.cu), shared with its device-side fixed-point loops (nka_batch_loop.cu) and work
// queues (nka_batch_queue.cu).
#pragma once
#include <cuda_runtime.h>
#include <functional>
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

// ---- shared by the device-side loops and queues (nka_batch_loop.cu) ----
// 0 if the driver has conditional graph nodes (12.4); otherwise prints why `call` cannot build its graph.
int nka_loop_driver_refused(const char* call);
// CTAs per member of the loop's check and step kernels at access width V (vlen only, as the batch's fix-up)
int nka_loop_grid(nka_batch* bt, int V);
// nka_loop_check<V> / nka_loop_step<V> queued on `s` over dim3(grid, nbatch) (nka_batch_loop.cu documents
// them); check k of member b is recorded at hist[k * hstride + b].  check applies `stop` with the per-problem
// entries of row b at index[b] (index NULL: at b).
void nka_loop_queue_check(int V, unsigned grid, int nbatch, cudaStream_t s, const double* F, size_t ldf, size_t n,
                          int hstride, const int* iters, int* status, unsigned char* active, double* r0, double* rlast,
                          double* hist, double* partials, size_t prow, unsigned* tickets, const nka_stop_test& stop,
                          const int* index);
// Aborts (file:line, under `call`) unless `stop` is a valid nka_stop_test for members of length vlen.
void nka_stop_test_require(const char* call, const nka_stop_test* stop, size_t vlen);
void nka_loop_queue_step(int V, unsigned grid, cudaStream_t s, double* X, size_t ldx, const double* F, size_t ldf,
                         size_t n, int nbatch, const unsigned char* active, int* iters);
// The residual-growth restart (nka_batch_guard.cu): the prologue's reset of the restart counts nrst (nbatch)
// and, in a queue, p_restarts (nproblems; NULL and 0 in a loop); and the body's guard followed by the
// batch's restart of its mask rmask, queued on the capturing `s`.  claimed, move_out and p_restarts are
// the queue's (NULL in a loop).
void nka_loop_guard_reset_launch(cudaStream_t s, int* nrst, int nbatch, int* p_restarts, size_t nproblems);
void nka_loop_guard_restart(nka_batch* bt, cudaStream_t s, double gamma, const unsigned char* active, const int* iters,
                            const double* rlast, const unsigned char* claimed, const int* move_out, double* rprev,
                            int* nrst, int* p_restarts, unsigned char* rmask);
// The graph  prologue -> WHILE (cond) { residual graph, cloned as a child -> body }, instantiated and
// uploaded on `s`.  prologue and body queue their kernels on `s` while it captures.  A graph CUDA
// refuses gives nullptr, after printing CUDA's reason under `call`, with no error left behind.
typedef std::function<void(cudaStream_t, cudaGraphConditionalHandle)> NkaCaptureFn;
cudaGraphExec_t nka_while_graph(const char* call, cudaStream_t s, cudaGraph_t residual, const NkaCaptureFn& prologue,
                                const NkaCaptureFn& body);

// (F, ldf, W, wstride, ld, n, S, partials, prow, tickets, dots, active)
typedef void (*NkaBatchPassAFn)(const double*, size_t, const double*, size_t, size_t, size_t, const NkaDevState*, double*,
                                size_t, unsigned*, double*, const unsigned char*);
// (F, ldf, W, Z, wstride, ld, n, S, active)
typedef void (*NkaBatchPassBFn)(double*, size_t, double*, double*, size_t, size_t, size_t, const NkaDevState*,
                                const unsigned char*);

// nc in 1..NKA_MAXSLOT, nz in 0..NKA_MAXSLOT-1, v in {1,2}; nullptr if not instantiated in this build
NkaBatchPassAFn nka_get_batch_pass_a(int nc, int v);
NkaBatchPassBFn nka_get_batch_pass_b(int nz, int v);
