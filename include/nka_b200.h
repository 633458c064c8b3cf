/* nka_b200.h -- additive C-ABI entry points of libnka_b200.so.
 *
 * Everything a host language needs beyond the reference's nine C functions
 * (include/nonlinear_krylov_accelerator.h): the parts of the Fortran API the C
 * header lacks, 64-bit lengths, device pointers and streams, the built-in
 * multi-GPU dot-product reduction, and read-only introspection for parity
 * tests and benchmarks.  Plain pointers and sizes only; no C++/torch types.
 *
 * These are the symbols the Fortran modules in nka_b200/fortran/ bind with
 * ISO_C_BINDING (see INTEGRATION.md for the interface blocks).
 */
#ifndef NKA_B200_H
#define NKA_B200_H

#include <stddef.h>

#include "nonlinear_krylov_accelerator.h"

#ifdef __cplusplus
extern "C" {
#endif

#define NKA_B200_MAX_MVEC 32

/* ---- construction ------------------------------------------------------ */

/* nka_init with a 64-bit length (the reference's int arithmetic overflows at
 * (mvec+1)*vlen >= 2^31, src-C/nonlinear_krylov_accelerator.c:235,241).
 * device < 0: the current CUDA device.  stream: a cudaStream_t, or NULL for the
 * legacy default stream (work is then ordered after whatever the caller queued
 * there, as with the synchronous CPU interface this replaces).  Fortran: init, src-F08/nka_type.F90:185-200
 * (vtol defaults to 0.01 there, :160). */
NKA nka_init_ex (size_t vlen, int mvec, double vtol, int device, void *stream);

/* src-F08/nka_type.F90:202-207 (set_vec_tol), src-F95/nka_type.F90:227-232 */
void nka_set_vec_tol (NKA, double vtol);

/* src-F08/nka_type.F90:460-524 (defined), src-F95/nka_type.F90:511-578.
 * Copies the small device state to the host and checks every list invariant. */
int nka_defined (NKA);

size_t nka_vec_len64 (NKA);

/* src-F08/nka_type.F90:209-219 (set_dot_prod), and the per-call `dp` of src-F95/nka_type.F90:284-291:
 * install (or with dp == NULL remove) the global-sum callback after construction; see
 * nonlinear_krylov_accelerator.h for how dp is used.  The _ctx form passes a caller context
 * through (what a Fortran trampoline needs to find its procedure pointer). */
void nka_set_dot_prod (NKA, double (*dp)(int, double *, double *));
void nka_set_dot_prod_ctx (NKA, double (*dp)(int, double *, double *, void *), void *ctx);

/* ---- the hot path with explicit memory spaces -------------------------- */

/* f is a device pointer on the handle's device; asynchronous on the handle's
 * stream (kernels only, no host synchronisation). */
void nka_accel_update_dev (NKA, double *f_dev);
/* f is a host pointer; copies in, updates, copies out, returns when f holds
 * the result. */
void nka_accel_update_host (NKA, double *f_host);

void nka_set_stream (NKA, void *stream);
void *nka_get_stream (NKA);
/* Block until everything queued on the handle's stream has finished. */
void nka_synchronize (NKA);

/* ---- CUDA graphs -------------------------------------------------------- */
/* nka_accel_update_dev (and nka_accel_update with a device pointer,
 * nka_accel_update_vec), nka_relax, nka_restart and nka_set_vec_tol can be
 * captured in a stream capture (cudaStreamBeginCapture, torch.cuda.graph) of
 * the handle's stream, which must be set with nka_set_stream before the
 * capture begins (not the legacy default stream).  The graph holds f's device
 * address.  A capture does not run anything: it leaves nka_launch_count and the
 * timing unchanged.  The first capture switches the handle for good to the
 * capacity shape, a launch shape valid for any list state (pass A at full width,
 * the fix-up kernel always queued, pass B at mvec pairs), for eager calls too;
 * in steady state it is the shape an eager call uses anyway.  Calls that
 * synchronise or stage through the host abort with a message while the
 * handle's stream captures: nka_accel_update_host (and a host pointer), an
 * update on a handle with a dot-product callback, nka_num_vec, nka_defined,
 * nka_get_state, nka_timing_*, nka_set_stream, nka_synchronize,
 * nka_set_dot_prod*, nka_comm_init / nka_comm_adopt.  With several ranks,
 * every rank captures and replays the same graphs in the same order.
 * Returns 1 while the handle's stream is capturing, 0 when it is not, -1 when
 * the handle is on the legacy default stream while a blocking stream captures
 * (nothing can be queued on the handle then). */
int nka_stream_capturing (NKA);

/* ---- multi-GPU: one process per GPU, each holding a row slab ------------ */
/* The only exchange in accel_update is one fp64 sum-allreduce of the
 * 2*(mvec+1) partial dot products (the reference's `dp` hook contract:
 * src-C/...c:61-68, src-F08-vector/README.md:16-22).  vlen passed to
 * nka_init_ex is the LOCAL slab length.
 *   nka_comm_unique_id: rank 0 fills a 128-byte NCCL id; ship it to the other
 *   ranks with whatever the application has (MPI, torch.distributed, files).
 *   nka_comm_init: collective over all ranks.  Returns 0 on success. */
int nka_comm_unique_id (void *id128);
int nka_comm_init (NKA, int nranks, int rank, const void *id128);
/* Alternatively adopt an existing ncclComm_t (not owned). */
void nka_comm_adopt (NKA, void *nccl_comm, int nranks, int rank);
/* How the partial dot products are summed: 0 = single GPU (no exchange); 1 = one NCCL
 * all-reduce between pass A and the state kernel; 2 = fused into pass A through peer memory
 * (every rank maps every peer's exchange box with CUDA IPC; chosen automatically by
 * nka_comm_init / nka_comm_adopt when all ranks share one NVLink domain, unanimous across
 * ranks; NKA_PEER_REDUCE=0 in the environment of every rank forces 1). */
int nka_comm_mode (NKA);

/* ---- device vectors: the operations of the reference's abstract `vector` ---- */
/* What a concrete gpu_vector extension of src-F08-vector/vector_class.F90:90-109
 * needs.  Expression order follows grid_vector (grid_vector_type.F90:108-197).
 * dot/norm2 return the value to the host (they synchronise the vector's stream)
 * and, with a communicator, sum over all ranks' slabs. */
typedef struct nka_vec *NKAVEC;
NKAVEC nka_vec_create (size_t n, int device, void *stream);   /* contents undefined, like allocate() */
NKAVEC nka_vec_clone (NKAVEC src);                            /* allocate(clone, source=src): :86-97 */
void nka_vec_destroy (NKAVEC);
size_t nka_vec_size (NKAVEC);
double *nka_vec_data (NKAVEC);                                /* device pointer */
void nka_vec_set_host (NKAVEC, const double *host);           /* host -> device, synchronous */
void nka_vec_get_host (NKAVEC, double *host);                 /* device -> host, synchronous */
void nka_vec_copy (NKAVEC dst, NKAVEC src);                   /* copy_   :99-106 */
void nka_vec_setval (NKAVEC, double val);                     /* setval  :108-112 */
void nka_vec_scale (NKAVEC, double a);                        /* scale   :114-118 */
void nka_vec_update1 (NKAVEC y, double a, NKAVEC x);                       /* y = a*x + y        :121-129 */
void nka_vec_update2 (NKAVEC y, double a, NKAVEC x, double b);             /* y = a*x + b*y      :132-140 */
void nka_vec_update3 (NKAVEC z, double a, NKAVEC x, double b, NKAVEC y);   /* z = a*x + b*y + z  :143-154 */
void nka_vec_update4 (NKAVEC z, double a, NKAVEC x, double b, NKAVEC y, double c); /* z = a*x+b*y+c*z :157-168 */
double nka_vec_dot (NKAVEC x, NKAVEC y);                      /* dot_    :170-184 */
double nka_vec_norm2 (NKAVEC x);                              /* norm2   :186-197 */
int nka_vec_comm_init (NKAVEC, int nranks, int rank, const void *id128); /* clones share it */
/* The vector flavour's init(vec, mvec) and accel_update(f):
 * src-F08-vector/nka_type.F90:175-188, :219-222. */
NKA nka_init_like (NKAVEC proto, int mvec, double vtol);
void nka_accel_update_vec (NKA, NKAVEC f);

/* ---- introspection (tests, benchmarks; never on the hot path) ---------- */

typedef struct nka_state_view {
  int mvec, subspace, pending, first, last, free_slot;
  int next[NKA_B200_MAX_MVEC + 1], prev[NKA_B200_MAX_MVEC + 1];
  int chained[NKA_B200_MAX_MVEC + 1];
  int ndrop_last, evicted_last, relaxed_last, error;
  double vtol, min_margin, s_last;
  double c[NKA_B200_MAX_MVEC + 1];
  double s[NKA_B200_MAX_MVEC + 1];
  double h[(NKA_B200_MAX_MVEC + 1) * (NKA_B200_MAX_MVEC + 1)]; /* h[r*(mvec+1)+c], compacted */
  unsigned long long ncalls;
} nka_state_view;

void nka_get_state (NKA, nka_state_view *out);

/* Kernel launches issued by this handle so far (all of them ours); kernels
 * captured into a CUDA graph are not launches and are not counted. */
unsigned long long nka_launch_count (NKA);

/* Per-kernel device timing with CUDA events on the handle's stream.
 * which: 0 = pass A, 1 = state, 2 = materialise, 3 = pass B, 4 = allreduce.
 * nka_timing_read synchronises the stream and returns accumulated ms and
 * launch counts since the last nka_timing_reset (eager calls only: a graph
 * replay records no events). */
void nka_timing_enable (NKA, int on);
void nka_timing_reset (NKA);
void nka_timing_read (NKA, double ms[5], unsigned long long count[5]);

/* Grid/block geometry of the two streaming kernels for the next update;
 * *threads = 10000 * (pass A block size) + (pass B block size). */
void nka_launch_geometry (NKA, int *grid_a, int *grid_b, int *threads);

const char *nka_b200_version (void);

/* ---- batched accelerators: many independent same-length instances ------- */
/* One handle holds nbatch (1..65535) independent accelerators that share vlen,
 * mvec and vtol.  Each member has its own subspace, list, Gram factor, vtol
 * decisions, relax and restart, and gives bit for bit what a single handle in
 * the capacity shape (see "CUDA graphs" above) gives when fed that member's
 * calls, whatever nbatch, the member's index and the other members hold.
 * Device-only and single-GPU.  One update is four kernel launches whatever
 * nbatch is (three with NKA_LAZY_LAST=0).
 *
 * f_dev holds nbatch rows of vlen doubles, row b at f_dev + b*ldf (ldf >= vlen).
 * active_dev / mask_dev: NULL (every member) or nbatch device bytes, nonzero =
 * selected, read by the kernels on the device.  An unselected member's update
 * is exactly no call: its row of f is neither read nor written and its state is
 * untouched.  Update, relax, restart and set_vec_tol can be captured in a CUDA
 * graph (the handle keeps no host-side shape state); the queries, set_stream
 * and synchronize abort while the handle's stream captures.
 *
 * The prototypes spell the handle as `struct nka_batch *`, which NKABATCH is. */
typedef struct nka_batch *NKABATCH;
struct nka_batch *nka_batch_init (int nbatch, size_t vlen, int mvec, double vtol, int device, void *stream);
void nka_batch_delete (struct nka_batch *b);
void nka_batch_accel_update (struct nka_batch *b, double *f_dev, size_t ldf, const unsigned char *active_dev);
void nka_batch_relax (struct nka_batch *b, const unsigned char *mask_dev);
void nka_batch_restart (struct nka_batch *b, const unsigned char *mask_dev);
void nka_batch_set_vec_tol (struct nka_batch *b, double vtol);
/* nbatch ints on the host; synchronises */
void nka_batch_num_vec (struct nka_batch *b, int *out);
/* 1 if every member passes the invariant check of nka_defined; synchronises */
int nka_batch_defined (struct nka_batch *b);
void nka_batch_get_state (struct nka_batch *b, int member, nka_state_view *out);
void nka_batch_set_stream (struct nka_batch *b, void *stream);
void nka_batch_synchronize (struct nka_batch *b);
/* as nka_stream_capturing */
int nka_batch_stream_capturing (struct nka_batch *b);
/* kernel launches run eagerly so far; captured kernels are not counted */
unsigned long long nka_batch_launch_count (struct nka_batch *b);

/* ---- device-side fixed-point loops over a batched accelerator ----------- */
/* One graph launch runs a whole solve of x_b = G(x_b) for every member b: a
 * WHILE graph node repeats { residual graph; record r = ||F_b||_2 of each
 * running member and stop it when r is not finite (NONFINITE), when
 * r < max(atol, rtol * r0_b) (CONVERGED, r0_b = its norm at the launch's first
 * check) or after maxit steps (MAXIT); nka_batch_accel_update(F, ldf, running);
 * X_b += F_b for the running members } until no member runs.
 *
 * residual_graph is a cudaGraph_t that reads X and writes F = G(X) - X for
 * every row.  It is cloned: the caller may destroy it, but keeps alive the
 * memory it addresses.  It may hold only node types a conditional body can
 * (kernels, memsets, memcopies, child graphs): a graph CUDA refuses, or a
 * driver older than 12.4, makes create print CUDA's reason and return NULL.
 * x_dev, f_dev: nbatch rows of vlen doubles at row strides ldx, ldf >= vlen.
 *
 * Each member's X, F, step count, status, history and state are bit for bit
 * those of a host-driven loop making the same residual, accel_update (same
 * masks) and X_b += F_b calls.  The accelerator is not restarted by a launch.
 * launch is queued on the batch's stream and aborts while that stream
 * captures; results and history synchronise (refused while it captures).
 * A launch is not counted by nka_batch_launch_count.
 *
 * The prototypes spell the handle as `struct nka_batch_loop *`, which
 * NKABATCHLOOP is. */
typedef struct nka_batch_loop *NKABATCHLOOP;
#define NKA_LOOP_RUNNING   0     /* never launched, or the launch has not finished */
#define NKA_LOOP_CONVERGED 1
#define NKA_LOOP_MAXIT     2
#define NKA_LOOP_NONFINITE 3
struct nka_batch_loop *nka_batch_loop_create (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                              double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                              double atol, double rtol, int maxit);
/* async on the batch's stream */
void nka_batch_loop_launch (struct nka_batch_loop *L);
/* nbatch each: steps taken, NKA_LOOP_* status, latest norm; synchronises */
void nka_batch_loop_results (struct nka_batch_loop *L, int *iters, int *status, double *norm);
/* (maxit+1) x nbatch, row k = check k, NaN where a member made no check k; synchronises */
void nka_batch_loop_history (struct nka_batch_loop *L, double *norms);
void nka_batch_loop_destroy (struct nka_batch_loop *L);

/* ---- device-side work queues: more fixed-point problems than members ---- */
/* One graph launch solves nproblems independent problems x_p = G_p(x_p) on the
 * batch's nbatch members, used as slots: when a slot's problem stops, the same
 * launch writes that problem's final iterate out, loads the next problem into
 * the slot and restarts the slot's accelerator, with no host round trip.
 *
 * x0_dev holds nproblems rows of vlen doubles (row stride ldx0): each problem's
 * initial guess, read when the problem is claimed.  xout_dev receives each
 * problem's final iterate (row stride ldxout) when it retires; xout_dev ==
 * x0_dev solves in place.  x_dev, f_dev are the slots' rows (nbatch rows, as
 * for nka_batch_loop_create).  slot_problem_dev is nbatch device ints the
 * queue keeps: the problem slot b solves, or -1 while it is idle.  The
 * residual graph reads it to find each row's parameters; it runs over every
 * row, idle ones included, so it must accept -1 (its output there is ignored).
 *
 * Each problem stops by fixed_point_loop's rule: NONFINITE, CONVERGED when
 * r < max(atol, rtol * r0_p), MAXIT after maxit steps.  Its final iterate,
 * steps, status and norm are bit for bit what nka_batch_loop_create's loop
 * gives it on a member just restarted with X row = its x0 row, whichever slot
 * it lands in, whatever nbatch, that slot's earlier problems and the other
 * slots hold.  Free slots take the next problem ids in slot order, so two
 * launches on the same inputs assign slots alike.  A launch starts from
 * problem 0 and the current x0 rows, and leaves every slot idle (-1).
 *
 * launch is queued on the batch's stream, aborts while that stream captures
 * and is not counted by nka_batch_launch_count; results synchronise (refused
 * while it captures).  create returns NULL, after printing CUDA's reason, on a
 * residual graph CUDA refuses or a driver older than 12.4.
 *
 * The prototypes spell the handle as `struct nka_batch_queue *`, which
 * NKABATCHQUEUE is. */
typedef struct nka_batch_queue *NKABATCHQUEUE;
struct nka_batch_queue *nka_batch_queue_create (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                                double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                                int *slot_problem_dev, const double *x0_dev, size_t ldx0,
                                                double *xout_dev, size_t ldxout, size_t nproblems,
                                                double atol, double rtol, int maxit);
/* async on the batch's stream */
void nka_batch_queue_launch (struct nka_batch_queue *Q);
/* nproblems each: steps taken, NKA_LOOP_* status, final norm; synchronises */
void nka_batch_queue_results (struct nka_batch_queue *Q, int *iters, int *status, double *norm);
void nka_batch_queue_destroy (struct nka_batch_queue *Q);

/* ---- per-problem stopping tests for device-side loops and queues -------- */
/* The _stop creates take the stopping rule as a struct.  For member p of a loop,
 * or problem p of a queue, at check k, with r0_p its norm at check 0:
 *
 *   r = || s_b . F_b ||_2      (s_b = row b of scale_dev; no scale: ||F_b||_2)
 *   NONFINITE  if r is not finite
 *   CONVERGED  else if r < fmax(atol_p, rtol_p * r0_p)
 *   DIVERGED   else if dtol > 0 and r > dtol * r0_p
 *   MAXIT      else if k >= maxit_p,  maxit_p = min(max(maxit_dev[p], 0), maxit)
 *
 * evaluated as written, in IEEE double (fmax included: a NaN atol_p or rtol_p
 * term drops out of it).  atol_p is atol_dev[p] when atol_dev is given, else
 * atol; rtol_p and maxit_p likewise.  In a loop p = b; in a queue p =
 * slot_problem[b], the problem slot b holds.  The arrays are device memory,
 * read at every launch (the caller may change them between launches).
 *
 * scale_dev: NULL, or nbatch rows (slots, shaped like f_dev) of vlen doubles at
 * row stride ldscale >= vlen, read after the residual graph in every
 * iteration: the residual graph may write it, e.g. weights 1/(atol_i +
 * rtol*|x_i|) from X.  Per element t = s_i * f_i; r^2 accumulates fma(t, t, .)
 * in the order and on the CTAs of the unscaled norm, so a scale of 1.0 gives
 * the unscaled bits, and the bits never depend on where the scale rows sit.
 * The iteration itself (the accelerator, X_b += F_b) always uses F unscaled.
 *
 * create aborts (file:line) on a NULL stop, atol or rtol < 0 (or NaN),
 * maxit < 0, dtol neither 0 nor >= 1, or a scale with ldscale < vlen.  The
 * scalar maxit also sizes a loop's history: (maxit+1) x nbatch.
 * nka_batch_loop_create / nka_batch_queue_create are the _stop creates with
 * {atol, rtol, 0, maxit, NULL, NULL, NULL, NULL, 0}. */
#define NKA_LOOP_DIVERGED  4     /* r > dtol * r0: its X row keeps its last finite iterate */
typedef struct nka_stop_test {
  double atol, rtol, dtol;           /* dtol = 0: off; else >= 1 */
  int maxit;                         /* >= 0; bounds maxit_dev entries and the loop's history */
  const double *atol_dev, *rtol_dev; /* NULL, or one per member (loop) / per problem (queue), device */
  const int *maxit_dev;              /* likewise */
  const double *scale_dev;           /* NULL, or nbatch rows of vlen doubles at stride ldscale, device */
  size_t ldscale;
} nka_stop_test;
struct nka_batch_loop *nka_batch_loop_create_stop (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                                   double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                                   const nka_stop_test *stop);
struct nka_batch_queue *nka_batch_queue_create_stop (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                                     double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                                     int *slot_problem_dev, const double *x0_dev, size_t ldx0,
                                                     double *xout_dev, size_t ldxout, size_t nproblems,
                                                     const nka_stop_test *stop);

/* ---- residual-growth restarts in device-side loops and queues ----------- */
/* The _restart creates are the _stop creates with one more rule,
 * restart_growth = gamma (0: off; else finite and > 0).  For member b of a
 * loop, or the problem in slot b of a queue: when check k >= 1 leaves it
 * RUNNING and r_k > gamma * r_{k-1} (the norms that check recorded: scaled when
 * the stop test has a scale), its accelerator is restarted before this
 * iteration's update, as nka_batch_restart with only b in the mask does.  That
 * update then returns F_b unchanged and starts a new subspace from it, and
 * X_b += F_b is a plain step.  gamma >= 1 restarts on growth, gamma < 1 when
 * the decrease is too small.  A member that check stops (DIVERGED included) is
 * never restarted; r0, the stop test and the step are unchanged; a loop launch
 * still does not restart members at its start.  r_{k-1} is always the same
 * launch's (loop) or the same problem's (queue), never a slot's previous
 * problem's.
 *
 * Each member's bits are those of a host-driven loop that, after each
 * residual, calls nka_batch_restart with the members the rule picks, then the
 * masked accel_update and X_b += F_b; each queue problem's are those of the
 * loop with the same gamma on a just-restarted member, whatever its slot.  A
 * rule that never fires gives the _stop creates' bits.  Memory: per slot one
 * double, one int and one byte; in a queue 4 bytes per problem more.
 *
 * create aborts (file:line) when restart_growth is negative or not finite, as
 * it does on a bad stop test.  The _stop creates are these with gamma = 0,
 * which build exactly the graphs they built before.
 *
 * _restarts copy the restarts the rule made: per member in the last launch
 * (loop, nbatch ints), or per problem (queue, nproblems ints; the restart a
 * queue makes when a slot takes a problem is not counted).  Zeros when
 * restart_growth was 0.  They synchronise and abort while the batch's stream
 * captures. */
struct nka_batch_loop *nka_batch_loop_create_restart (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                                      double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                                      const nka_stop_test *stop, double restart_growth);
struct nka_batch_queue *nka_batch_queue_create_restart (struct nka_batch *b, void *residual_graph /* cudaGraph_t */,
                                                        double *x_dev, size_t ldx, double *f_dev, size_t ldf,
                                                        int *slot_problem_dev, const double *x0_dev, size_t ldx0,
                                                        double *xout_dev, size_t ldxout, size_t nproblems,
                                                        const nka_stop_test *stop, double restart_growth);
/* nbatch ints on the host; synchronises */
void nka_batch_loop_restarts (struct nka_batch_loop *L, int *restarts);
/* nproblems ints on the host; synchronises */
void nka_batch_queue_restarts (struct nka_batch_queue *Q, int *restarts);

/* ---- interleaved batched accelerators: one thread per member ------------ */
/* One handle holds nbatch (1..2^31-1, limited only by memory) independent
 * accelerators that share vlen, mvec (1..32) and vtol, stored component-major:
 * element i of member b is at f_dev[i*ldf + b] (ldf >= nbatch), the layout of a
 * Fortran array f(ncell, nvar) with one member per cell.  One update is one
 * kernel launch whatever nbatch is; each member runs on its own thread.
 *
 * Member b's correction vectors, num_vec, lists, Gram factor entries among
 * list slots, coefficients c, min_margin, ndrop_last, evicted_last and
 * relaxed_last are bit for bit what the reference's C nka_accel_update /
 * nka_relax / nka_restart give when fed that member's calls: its dot products
 * are the reference's serial sums, and no multiply-add is contracted.  They do
 * not depend on nbatch, the member's index, the other members' data or masks,
 * ldf, or f_dev's alignment.
 *
 * active_dev / mask_dev: NULL (every member) or nbatch device bytes, nonzero =
 * selected; an unselected member's column of f is neither read nor written and
 * its state is untouched.  Update, relax, restart and set_vec_tol can be
 * captured in a CUDA graph (the handle keeps no host-side shape state; vtol
 * lives on the device); the queries, set_stream and synchronize abort while the
 * handle's stream captures.  Device-only, single-GPU, no dot-product callback.
 *
 * nka_ibatch_get_state fills mvec, subspace, pending, first, last, free_slot,
 * next, prev, c, h (h[r*(mvec+1)+c]), vtol, min_margin, ndrop_last,
 * evicted_last and relaxed_last; every other field is zero.
 *
 * The prototypes spell the handle as `struct nka_ibatch *`, which NKAIBATCH is. */
typedef struct nka_ibatch *NKAIBATCH;
struct nka_ibatch *nka_ibatch_init (int nbatch, size_t vlen, int mvec, double vtol, int device, void *stream);
void nka_ibatch_delete (struct nka_ibatch *b);
void nka_ibatch_accel_update (struct nka_ibatch *b, double *f_dev, size_t ldf, const unsigned char *active_dev);
void nka_ibatch_relax (struct nka_ibatch *b, const unsigned char *mask_dev);
void nka_ibatch_restart (struct nka_ibatch *b, const unsigned char *mask_dev);
void nka_ibatch_set_vec_tol (struct nka_ibatch *b, double vtol);
/* nbatch ints on the host; synchronises */
void nka_ibatch_num_vec (struct nka_ibatch *b, int *out);
/* 1 if every member passes the invariant check of nka_defined; synchronises */
int nka_ibatch_defined (struct nka_ibatch *b);
void nka_ibatch_get_state (struct nka_ibatch *b, int member, nka_state_view *out);
void nka_ibatch_set_stream (struct nka_ibatch *b, void *stream);
void nka_ibatch_synchronize (struct nka_ibatch *b);
/* as nka_stream_capturing */
int nka_ibatch_stream_capturing (struct nka_ibatch *b);
/* kernel launches run eagerly so far; captured kernels are not counted */
unsigned long long nka_ibatch_launch_count (struct nka_ibatch *b);

#ifdef __cplusplus
}
#endif

#endif
