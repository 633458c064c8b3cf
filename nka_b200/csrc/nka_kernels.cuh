// nka_kernels.cuh -- the sm_100a kernels of accel_update.
//
//   nka_pass_a        one read-only sweep: every difference d_j of the subspace is
//                     formed in registers from the raw cached inputs and reduced
//                     against d_0 and f (2*ncol dot products); deterministic
//                     two-stage reduction; the last CTA folds the per-CTA partials
//                     and (single GPU) runs the scalar state step in place.
//                     Replaces src-C/nonlinear_krylov_accelerator.c:299-301,
//                     :323-324, the dp() calls of :406, and :333-417.
//   nka_state_kernel  the scalar state step alone (multi-GPU: after the all-reduce).
//   nka_fixup_kernel  rare: the two dot products of the lazily skipped oldest
//                     column, then the state step again.  Exits at once otherwise.
//   nka_materialise   rare, relax() only: W[dst] -= W[sub] after a chain break.
//   nka_pass_b        one sweep: rebuild the pending correction, form the new
//                     pair's Z column, the accelerated correction, cache the raw
//                     f.  Replaces :316-320, :397-398, :419-430.
//
// All streaming kernels are HBM-bandwidth bound (0.2-0.4 flop/byte, fp64);
// tensor cores do not apply.  Loads/stores are 16-byte (double2), coalesced,
// with streaming cache hints; grids are multiples of the SM count.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "nka_state.h"

// Tunables.  Defaults picked by the sweeps recorded in profiles/r1*_tune_sweep.jsonl
// (n = 2^28, mvec = 10 on B200): plain ld.global.nc / st.global beat the .cs streaming
// hints by 10 % in pass B; 256 threads suit the register-heavy pass A, 512 pass B.
#ifndef NKA_THREADS
#define NKA_THREADS 256      // fix-up / materialise kernels and the default for both passes
#endif
#ifndef NKA_THREADS_A
#define NKA_THREADS_A NKA_THREADS
#endif
#ifndef NKA_THREADS_B
#define NKA_THREADS_B 512
#endif
#ifndef NKA_MINB_A
#define NKA_MINB_A 1      // __launch_bounds__ min CTAs/SM for pass A
#endif
#ifndef NKA_MINB_B
#define NKA_MINB_B 1
#endif
#ifndef NKA_STORE_STREAM
#define NKA_STORE_STREAM 0   // 1: st.global.cs for the cached columns, 0: default write-back policy
#endif
#ifndef NKA_LOAD_STREAM
#define NKA_LOAD_STREAM 0    // 0: ld.global.nc, 1: ld.global.cs (evict-first), 2/3: L1::no_allocate variants
#endif
#define NKA_STATE_THREADS 128
// Pass B holds NZ column values (double2) and 2 NZ coefficients per thread: beyond 12 columns the
// 128 registers a 512-thread CTA allows spill (388 B at NZ = 20: 5.9 instead of 7.0 TB/s).  From
// NKA_COEF_SMEM_FROM columns on, the 2 NZ coefficients live in shared memory (one broadcast LDS.64
// per use: the sweep is HBM bound, the issue slots are free) so that the column values alone fill the
// registers and the CTA keeps its 512 threads; beyond NKA_THREADS_B_WIDE_FROM columns even those
// do not fit and the CTA drops to 256 threads with up to 255 registers.
#ifndef NKA_COEF_SMEM_FROM
#define NKA_COEF_SMEM_FROM 13
#endif
#ifndef NKA_THREADS_B_WIDE_FROM
#define NKA_THREADS_B_WIDE_FROM 24
#endif
__host__ __device__ constexpr int nka_threads_b(int nz) { return nz >= NKA_THREADS_B_WIDE_FROM ? 256 : NKA_THREADS_B; }

// ---------------------------------------------------------------------------
// 16-byte / 8-byte element access with streaming cache hints.  V = 2 uses
// double2 (LDG.E.128 / STG.E.128), V = 1 is the fallback for a caller's f that
// is not 16-byte aligned, and handles the odd tail element.
// ---------------------------------------------------------------------------
template <int V> struct Vec;
template <> struct Vec<2> {
  double x, y;
  static __device__ __forceinline__ Vec ld(const double* p, size_t i) {
#if NKA_LOAD_STREAM == 1
    const double2 t = __ldcs(reinterpret_cast<const double2*>(p) + i);
    return {t.x, t.y};
#elif NKA_LOAD_STREAM == 2
    double a, b;
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v2.f64 {%0,%1}, [%2];"
                 : "=d"(a), "=d"(b) : "l"(reinterpret_cast<const double2*>(p) + i));
    return {a, b};
#elif NKA_LOAD_STREAM == 3
    double a, b;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                 : "=d"(a), "=d"(b) : "l"(reinterpret_cast<const double2*>(p) + i));
    return {a, b};
#else
    const double2 t = __ldg(reinterpret_cast<const double2*>(p) + i);
    return {t.x, t.y};
#endif
  }
  static __device__ __forceinline__ Vec ld_keep(const double* p, size_t i) {
    const double2 t = __ldg(reinterpret_cast<const double2*>(p) + i);
    return {t.x, t.y};
  }
  static __device__ __forceinline__ Vec ld_plain(const double* p, size_t i) {
    const double2 t = reinterpret_cast<const double2*>(p)[i];
    return {t.x, t.y};
  }
  __device__ __forceinline__ void st_stream(double* p, size_t i) const {
#if NKA_STORE_STREAM
    __stcs(reinterpret_cast<double2*>(p) + i, make_double2(x, y));
#else
    reinterpret_cast<double2*>(p)[i] = make_double2(x, y);
#endif
  }
  __device__ __forceinline__ void st(double* p, size_t i) const {
    reinterpret_cast<double2*>(p)[i] = make_double2(x, y);
  }
  static __device__ __forceinline__ Vec zero() { return {0.0, 0.0}; }
  __device__ __forceinline__ Vec operator-(const Vec& o) const { return {x - o.x, y - o.y}; }
  __device__ __forceinline__ Vec operator+(const Vec& o) const { return {x + o.x, y + o.y}; }
  __device__ __forceinline__ void fma_into(double a, Vec& acc) const { acc.x = fma(a, x, acc.x); acc.y = fma(a, y, acc.y); }
  __device__ __forceinline__ void dot_into(const Vec& o, double& acc) const { acc = fma(x, o.x, acc); acc = fma(y, o.y, acc); }
};
template <> struct Vec<1> {
  double x;
  static __device__ __forceinline__ Vec ld(const double* p, size_t i) {
#if NKA_LOAD_STREAM == 1
    return {__ldcs(p + i)};
#else
    return {__ldg(p + i)};
#endif
  }
  static __device__ __forceinline__ Vec ld_keep(const double* p, size_t i) { return {__ldg(p + i)}; }
  static __device__ __forceinline__ Vec ld_plain(const double* p, size_t i) { return {p[i]}; }
  __device__ __forceinline__ void st_stream(double* p, size_t i) const {
#if NKA_STORE_STREAM
    __stcs(p + i, x);
#else
    p[i] = x;
#endif
  }
  __device__ __forceinline__ void st(double* p, size_t i) const { p[i] = x; }
  static __device__ __forceinline__ Vec zero() { return {0.0}; }
  __device__ __forceinline__ Vec operator-(const Vec& o) const { return {x - o.x}; }
  __device__ __forceinline__ Vec operator+(const Vec& o) const { return {x + o.x}; }
  __device__ __forceinline__ void fma_into(double a, Vec& acc) const { acc.x = fma(a, x, acc.x); }
  __device__ __forceinline__ void dot_into(const Vec& o, double& acc) const { acc = fma(x, o.x, acc); }
};

__device__ __forceinline__ double nka_warp_sum(double v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Programmatic dependent launch (sm_90+) -- EXPERIMENT, compiled in only with -DNKA_EXPERIMENT_PDL
// and never in the product build.  The kernels of the update chain (pass A -> fix-up -> pass B)
// were launched with the programmatic-stream-serialization attribute and began with
// `griddepcontrol.wait`; pass A issued `launch_dependents` when its streaming loop was done, so
// the next kernel's CTAs were scheduled onto the idle SMs during pass A's serial tail (ticket,
// fold, exchange, state step: ~24 us on one CTA).  Measured: -6 us per update (0.320 -> 0.314 ms
// at n = 2^24, mvec = 5; 0.978 -> 0.972 ms at n = 2^25, mvec = 10; profiles/r2d_pdl_ab.jsonl).
// Triggering at the start of every kernel instead cost 4-6 % (parked CTAs beside the streaming
// ones, profiles/r2b_pdl_ab_early_trigger.jsonl).  NOT KEPT: with the attribute set, 19 parity
// tests failed in one full-suite run on small vectors and passed in the next
// (gpurun_out/pytest_gpu_r2e.log vs bisect_parity_r2f.txt) -- the overlap removes the kernel
// boundary that the L1-cached (ld.global.nc) loads of W, Z and the device state rely on for
// coherence, and the loads that avoid L1 cost 10 % of pass B (profiles/r1a_tune_sweep.jsonl).
#ifdef NKA_EXPERIMENT_PDL
__device__ __forceinline__ void nka_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void nka_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#else
__device__ __forceinline__ void nka_pdl_wait() {}
__device__ __forceinline__ void nka_pdl_trigger() {}
#endif

__device__ __forceinline__ unsigned long long nka_globaltimer()
{
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---------------------------------------------------------------------------
// Tuning aid, compiled in only with -DNKA_TRACE (tools/pass_a_trace.py): globaltimer stamps of
// pass A's phases.  [0] first CTA start (min) [1] last CTA's loop end (max) [2] ticket won
// [3] partial rows folded [4] exchange done [5] state step committed.
// ---------------------------------------------------------------------------
#ifdef NKA_TRACE
static __device__ unsigned long long g_nka_trace[8];
#define NKA_STAMP_MIN(i) do { if (threadIdx.x == 0) atomicMin(&g_nka_trace[i], nka_globaltimer()); } while (0)
#define NKA_STAMP_MAX(i) do { if (threadIdx.x == 0) atomicMax(&g_nka_trace[i], nka_globaltimer()); } while (0)
#define NKA_STAMP(i) do { if (threadIdx.x == 0) g_nka_trace[i] = nka_globaltimer(); } while (0)
#else
#define NKA_STAMP_MIN(i) do { } while (0)
#define NKA_STAMP_MAX(i) do { } while (0)
#define NKA_STAMP(i) do { } while (0)
#endif

// ---------------------------------------------------------------------------
// Deterministic grid reduction of K per-thread accumulators: shuffle tree inside
// each warp, fixed-order sum across warps, one partial row per CTA, and the last
// CTA to take a ticket folds the rows in a fixed order (run-to-run bit-stable for
// a given grid).  Returns true in every thread of that last CTA, after out(j, v)
// has been called for each j.  Atomic-free except for the ticket.
// ---------------------------------------------------------------------------
//
// A sweep may be cut into several launches over consecutive chunks of the vector (the
// host-pointer path overlaps them with the PCIe copy of the next chunk): each launch writes its
// rows at `partials`, and only the final one (fold_rows > 0) takes tickets and folds all
// fold_rows rows starting at fold_base, earlier launches' rows included (same stream: complete).
template <int K, int THREADS, typename Out>
__device__ __forceinline__ bool nka_grid_reduce(const double (&acc)[K], double* __restrict__ partials,
                                                unsigned* __restrict__ ticket, const double* __restrict__ fold_base,
                                                unsigned fold_rows, Out out)
{
  __shared__ double red[THREADS / 32][K];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const double v = nka_warp_sum(acc[j]);
    if (lane == 0) red[warp][j] = v;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) v += red[w][threadIdx.x];
    partials[(size_t)blockIdx.x * K + threadIdx.x] = v;
  }
  if (fold_rows == 0) return false;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return false;
  NKA_STAMP(2);
  __threadfence();
  for (int j = warp; j < K; j += THREADS / 32) {
    double v = 0.0;
    // the same left-to-right sum as a plain loop, with the (independent) loads of eight rows in
    // flight at once: at 1184 rows the plain loop paid 37 L2 round trips per value (16 us)
    unsigned b = lane;
#ifndef NKA_FOLD_PLAIN
    for (; b + 7 * 32 < fold_rows; b += 8 * 32) {
      double t[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = __ldcg(&fold_base[(size_t)(b + 32 * u) * K + j]);
#pragma unroll
      for (int u = 0; u < 8; ++u) v += t[u];
    }
#endif
    for (; b < fold_rows; b += 32) v += __ldcg(&fold_base[(size_t)b * K + j]);
    v = nka_warp_sum(v);
    if (lane == 0) out(j, v);
  }
  if (threadIdx.x == 0) *ticket = 0u;
  __syncthreads();
  return true;
}

// ---------------------------------------------------------------------------
// Cross-GPU sum of K doubles held in shared memory, executed by one CTA per rank
// (the last CTA of pass A / of the fix-up sweep), fused into that kernel: every
// rank stores its values straight into every peer's exchange box over NVLink and
// then folds the R contributions it received in rank order, so all ranks hold
// bit-identical sums and take identical drop decisions.  One NVLink store
// latency end to end; no fence, no separate collective launch.
//   slot = {lo32(v), tag, hi32(v), tag}: each 8-byte half carries the tag, the
//   receiver spins until both halves show this exchange's tag.
//   Two parities: a rank can run at most one exchange ahead of a peer (it needs
//   that peer's contribution to finish the current one), so the slot written
//   for exchange e+2 has been consumed by everyone.
// ---------------------------------------------------------------------------

__device__ __forceinline__ void nka_peer_allreduce(NkaPeerCtx* __restrict__ P, double* vals, int K)
{
  __shared__ unsigned ep_s;
  if (threadIdx.x == 0) ep_s = *reinterpret_cast<volatile unsigned*>(&P->epoch) + 1u;
  __syncthreads();
  const unsigned ep = ep_s;
  const int R = P->nranks, me = P->rank;
  const unsigned long long timeout_ns = P->timeout_ns;
  const size_t par = (size_t)(ep & 1u) * NKA_MAX_RANKS * NKA_PEER_K;
  for (int i = threadIdx.x; i < R * K; i += blockDim.x) {
    const int r = i / K, t = i - r * K;
    const double v = vals[t];
    uint4* dst = reinterpret_cast<uint4*>(P->box[r]) + par + (size_t)me * NKA_PEER_K + t;
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};"
                 :: "l"(dst), "r"((unsigned)__double2loint(v)), "r"(ep), "r"((unsigned)__double2hiint(v)), "r"(ep)
                 : "memory");
  }
  __syncthreads();                                   // every value has been read before it is replaced
  const uint4* mine = reinterpret_cast<const uint4*>(P->box[me]) + par;
  for (int t = threadIdx.x; t < K; t += blockDim.x) {
    double sum = 0.0;
    for (int r = 0; r < R; ++r) {
      const uint4* src = mine + (size_t)r * NKA_PEER_K + t;
      unsigned lo, t0, hi, t1;
      unsigned long long t_start = 0;
      for (unsigned spins = 0;; ++spins) {
        asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(src) : "memory");
        if (t0 == ep && t1 == ep) break;
        if ((spins & 0xfffu) == 0xfffu) {
          const unsigned long long now = nka_globaltimer();
          if (t_start == 0) t_start = now;
          else if (now - t_start > timeout_ns) { P->timed_out = 1; __threadfence_system(); __trap(); }
        }
      }
      const double v = __hiloint2double((int)hi, (int)lo);
      sum = (r == 0) ? v : sum + v;
    }
    vals[t] = sum;
  }
  __syncthreads();
  if (threadIdx.x == 0) *reinterpret_cast<volatile unsigned*>(&P->epoch) = ep;
}

// ---------------------------------------------------------------------------
// State staging.  The ~11 KB state is worked on in shared memory: the scalar
// algorithm is a chain of dependent loads, and from global memory every one of
// them paid an L2 round trip (43 us at mvec = 10 on B200; profiles/r1a_*).
// ---------------------------------------------------------------------------
struct NkaStateStage {
  NkaDevState st;
  double dots[2 * NKA_MAXSLOT];
  NkaStepScratch x;
};

// The step is run by the 32 lanes of one warp (nka_state.h: lane-parallel over entries, the
// reference's operation order within each entry).
struct NkaWarpPar {
  int l;
  __device__ __forceinline__ int lane() const { return l; }
  __device__ __forceinline__ int nlanes() const { return 32; }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
};

__device__ __forceinline__ void nka_stage_in(NkaStateStage& sm, const NkaDevState* S, const double* dots)
{
  static_assert(sizeof(NkaDevState) % 4 == 0, "state is copied in 4-byte words");
  const uint32_t* src = reinterpret_cast<const uint32_t*>(S);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&sm.st);
  for (unsigned i = threadIdx.x; i < sizeof(NkaDevState) / 4; i += blockDim.x) dst[i] = __ldcg(src + i);
  if (dots)
    for (unsigned i = threadIdx.x; i < 2 * NKA_MAXSLOT; i += blockDim.x) sm.dots[i] = __ldcg(dots + i);
  __syncthreads();
}

__device__ __forceinline__ void nka_stage_out(const NkaStateStage& sm, NkaDevState* S)
{
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&sm.st);
  uint32_t* dst = reinterpret_cast<uint32_t*>(S);
  for (unsigned i = threadIdx.x; i < sizeof(NkaDevState) / 4; i += blockDim.x) dst[i] = src[i];
}

// One copy of the scalar step per translation unit (it is inlined nowhere: pass A is
// instantiated 66 times and would otherwise carry 66 copies of it).
static __device__ __noinline__ int nka_state_step_dev(NkaDevState* st, NkaStepScratch* x, const double* dots, int have_last)
{
  const NkaWarpPar par = {(int)(threadIdx.x & 31)};
  return nka_state_step(*st, *x, dots, NKA_MAXSLOT, have_last, par);
}

// Runs the step on the staged copy (dots already in sm.dots) and commits it,
// unless it needs the lazily skipped column: then only the flag is published.
__device__ __forceinline__ void nka_run_state_step(NkaStateStage& sm, NkaDevState* S, int have_last)
{
  __shared__ int need_more;
  if (threadIdx.x < 32) {                         // warp 0, all lanes
    const int r = nka_state_step_dev(&sm.st, &sm.x, sm.dots, have_last);
    if (threadIdx.x == 0) need_more = r;
  }
  __syncthreads();
  if (need_more) {
    if (threadIdx.x == 0) S->need_fixup = 1;
  } else {
    nka_stage_out(sm, S);
  }
}

// ---------------------------------------------------------------------------
// Pass A.
//   acc[j]      += d_0 . d_j      acc[NC + j] += f . d_j       (j < ncol_eff <= NC)
// FULL = the plan streams exactly NC chained columns: no predicates at all.
// ---------------------------------------------------------------------------
template <int NC, int V, bool FULL>
__device__ __forceinline__ void nka_pass_a_elem(const double* __restrict__ f, const double* const (&wcol)[NC],
                                                size_t i, int ncol, unsigned long long submask, double (&acc)[2 * NC])
{
  using T = Vec<V>;
  const T x0 = T::ld_keep(f, i);          // f is read again by pass B: leave it in L2 if it fits
  T xs[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    if (FULL || j < ncol) xs[j] = T::ld(wcol[j], i);
    else xs[j] = T::zero();
  }
  T prev = x0;
  T d0 = T::zero();
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    T d;
    if (FULL) d = xs[j] - prev;
    else d = ((submask >> j) & 1ull) ? (xs[j] - prev) : xs[j];
    if (j == 0) d0 = d;
    d0.dot_into(d, acc[j]);
    x0.dot_into(d, acc[NC + j]);
    prev = xs[j];
  }
}

template <int NC, int V>
__global__ void __launch_bounds__(NKA_THREADS_A, NKA_MINB_A)
nka_pass_a(const double* __restrict__ f, const double* __restrict__ W, size_t ld, size_t n,
           NkaDevState* __restrict__ S, double* __restrict__ partials, unsigned* __restrict__ ticket,
           double* __restrict__ dots, int fuse_state, NkaPeerCtx* __restrict__ peer,
           const double* __restrict__ fold_base, unsigned fold_rows)
{
  nka_pdl_wait();
  NKA_STAMP_MIN(0);
  const int ncol = S->planA.ncol - S->planA.skip_last;      // columns actually streamed
  const unsigned long long submask = S->planA.submask;
  // Columns j >= ncol are never loaded.  Their address is column 0 rather than planA.col[0]: with
  // an empty list (the capacity shape of a captured handle runs pass A on the first call) that
  // entry has never been written.
  const double* wcol[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) wcol[j] = W + (size_t)(j < ncol ? S->planA.col[j] : 0) * ld;

  double acc[2 * NC];
#pragma unroll
  for (int j = 0; j < 2 * NC; ++j) acc[j] = 0.0;

  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS_A;
  const size_t start = (size_t)blockIdx.x * NKA_THREADS_A + threadIdx.x;
  const unsigned long long allbits = (1ull << NC) - 1ull;          // NC <= NKA_MAXSLOT = 33
  const bool full = (ncol == NC) && ((submask & allbits) == allbits);
  if (full) {
    for (size_t i = start; i < nv; i += stride) nka_pass_a_elem<NC, V, true>(f, wcol, i, ncol, submask, acc);
  } else {
    for (size_t i = start; i < nv; i += stride) nka_pass_a_elem<NC, V, false>(f, wcol, i, ncol, submask, acc);
  }
  if (V == 2 && (n & 1) && start == 0) nka_pass_a_elem<NC, 1, false>(f, wcol, n - 1, ncol, submask, acc);

  NKA_STAMP_MAX(1);
  if (fuse_state) nka_pdl_trigger();   // the next kernel (fix-up / pass B: both wait) may be scheduled during the tail
  __shared__ NkaStateStage sm;     // used by the last CTA only
  __shared__ double xv[2 * NC];
  const bool last = nka_grid_reduce<2 * NC, NKA_THREADS_A>(acc, partials, ticket, fold_base, fold_rows,
                                                         [&](int j, double v) { xv[j] = v; });
  if (!last) return;
  NKA_STAMP(3);
  // multi-GPU on one NVLink domain: sum over the ranks right here, through peer memory
  if (peer) nka_peer_allreduce(peer, xv, 2 * NC);
  NKA_STAMP(4);
  for (int j = threadIdx.x; j < 2 * NC; j += NKA_THREADS_A) {
    const int at = (j < NC) ? j : (NKA_MAXSLOT + (j - NC));
    dots[at] = xv[j];
    sm.dots[at] = xv[j];
  }
  __syncthreads();
  if (fuse_state) {
    // the scalar step runs right here, no extra launch
    const uint32_t* src = reinterpret_cast<const uint32_t*>(S);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&sm.st);
    for (unsigned i = threadIdx.x; i < sizeof(NkaDevState) / 4; i += blockDim.x) dst[i] = __ldcg(src + i);
    __syncthreads();
    nka_run_state_step(sm, S, /*have_last=*/0);
    __syncthreads();
    NKA_STAMP(5);
  }
}

// ---------------------------------------------------------------------------
// Pass B.  NZ is the host's expectation of how many pairs were on the list at
// entry (exact unless a vtol drop fired earlier); the FULL body is predicate-free.
// Any other plan goes through the general body, which handles nz != NZ, a missing
// pair, and the chain-break conversions W[dst] -= W[sub] (same thread, same
// element, before W[newslot] is overwritten, so no cross-thread hazard exists).
// ---------------------------------------------------------------------------
// In the FULL body f, W[newslot], Z[pslot] and the streamed Z columns are distinct arrays: the no-alias promise
// is true there and lets the compiler lift the next element's loads above this element's stores (worth 8 %
// at mvec = 2, where an element has only three loads in flight).  The general body reads columns of W that
// it also writes (the chain-break conversions): no promise.
template <bool FULL> struct NkaOutPtr { typedef double* type; };
template <> struct NkaOutPtr<true> { typedef double* __restrict__ type; };

template <int NZ, int V, bool FULL>
__device__ __forceinline__ void nka_pass_b_elem(const Vec<V> x0, typename NkaOutPtr<FULL>::type f,
                                                typename NkaOutPtr<FULL>::type wnew, typename NkaOutPtr<FULL>::type zp,
                                                const double* const (&zcol)[NZ > 0 ? NZ : 1],
                                                const double (&coefN)[NZ > 0 ? NZ : 1],
                                                const double (&coefY)[NZ > 0 ? NZ : 1], double coef_p,
                                                int has_pair, int nz, int write_f, size_t i,
                                                double* W, const double* Z, size_t ld, const NkaDevState* S)
{
  using T = Vec<V>;
  // x0 = f[i], loaded by the caller with a plain load: f is stored to below, and PTX defines the read-only
  // (ld.global.nc) path only for data that no thread writes during the kernel
  T zs[NZ > 0 ? NZ : 1];
#pragma unroll
  for (int k = 0; k < NZ; ++k) {
    if (FULL || k < nz) zs[k] = T::ld(zcol[k], i);
    else zs[k] = T::zero();
  }
  if (!FULL) {
    const int m = S->planM.n;
    for (int e = 0; e < m; ++e) {
      double* dst = W + (size_t)S->planM.dst[e] * ld;
      const double* sub = W + (size_t)S->planM.sub[e] * ld;
      (T::ld_plain(dst, i) - T::ld_plain(sub, i)).st(dst, i);
    }
    // W[newslot] may be one of the `sub` columns: keep its overwrite below after these reads
    if (m > 0) asm volatile("" ::: "memory");
  }
  T y = T::zero();
  if (FULL || has_pair) {
    T yprev = T::zero();                     // the previous call's correction, same fma order as then
#pragma unroll
    for (int k = 0; k < NZ; ++k) zs[k].fma_into(coefY[k], yprev);
    if (!FULL)
      for (int k = NZ; k < nz; ++k) T::ld(Z + (size_t)S->planB.zcol[k] * ld, i).fma_into(S->planB.coefY[k], yprev);
    const T zpv = yprev + x0;                // Z'_p = Y_p + f
    zpv.st_stream(zp, i);
    zpv.fma_into(coef_p, y);
  }
#pragma unroll
  for (int k = 0; k < NZ; ++k) zs[k].fma_into(coefN[k], y);
  if (!FULL)
    for (int k = NZ; k < nz; ++k) T::ld(Z + (size_t)S->planB.zcol[k] * ld, i).fma_into(S->planB.coefN[k], y);
  x0.st_stream(wnew, i);
  if (FULL || write_f) (x0 + y).st(f, i);
}

template <int NZ, int V>
__global__ void __launch_bounds__(nka_threads_b(NZ), NKA_MINB_B)
nka_pass_b(double* f, double* W, double* Z, size_t ld, size_t n, const NkaDevState* __restrict__ S)
{
  constexpr int NZA = NZ > 0 ? NZ : 1;
  nka_pdl_wait();
  const NkaPlanB* B = &S->planB;
  const int nz = B->nz, has_pair = B->has_pair, write_f = B->write_f;
  double* wnew = W + (size_t)B->newslot * ld;
  double* zp = Z + (size_t)B->pslot * ld;
  const double coef_p = B->coef_p;
  constexpr bool kCoefSmem = NZ >= NKA_COEF_SMEM_FROM;    // coefficients and column addresses in shared memory
  __shared__ double s_coefN[kCoefSmem ? NZA : 1], s_coefY[kCoefSmem ? NZA : 1];
  __shared__ const double* s_zcol[kCoefSmem ? NZA : 1];
  double r_coefN[kCoefSmem ? 1 : NZA], r_coefY[kCoefSmem ? 1 : NZA];
  const double* r_zcol[kCoefSmem ? 1 : NZA];
  double (&coefN)[NZA] = *reinterpret_cast<double (*)[NZA]>(kCoefSmem ? s_coefN : r_coefN);
  double (&coefY)[NZA] = *reinterpret_cast<double (*)[NZA]>(kCoefSmem ? s_coefY : r_coefY);
  const double* (&zcol)[NZA] = *reinterpret_cast<const double* (*)[NZA]>(kCoefSmem ? s_zcol : r_zcol);
  if (!kCoefSmem) {
#pragma unroll
    for (int k = 0; k < NZA; ++k) {
      const bool on = (k < nz) && (k < NZ);
      zcol[k] = Z + (size_t)(on ? B->zcol[k] : B->newslot) * ld;
      coefN[k] = on ? B->coefN[k] : 0.0;
      coefY[k] = on ? B->coefY[k] : 0.0;
    }
  } else {
    for (int k = threadIdx.x; k < NZA; k += blockDim.x) {
      const bool on = (k < nz) && (k < NZ);
      s_zcol[k] = Z + (size_t)(on ? B->zcol[k] : B->newslot) * ld;
      s_coefN[k] = on ? B->coefN[k] : 0.0;
      s_coefY[k] = on ? B->coefY[k] : 0.0;
    }
    __syncthreads();
  }
  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * nka_threads_b(NZ);
  const size_t start = (size_t)blockIdx.x * nka_threads_b(NZ) + threadIdx.x;
  const bool full = (nz == NZ) && has_pair && write_f && (S->planM.n == 0);
  if (full) {
    // f of the next element is fetched before this element's stores are issued: the compiler cannot lift a
    // plain load of f above stores to f by itself (it cannot prove i + stride != i), and at small NZ the
    // loads in flight per thread are what the bandwidth hangs on
    Vec<V> x0 = start < nv ? Vec<V>::ld_plain(f, start) : Vec<V>::zero();
    for (size_t i = start; i < nv; i += stride) {
      const size_t inext = i + stride;
      const Vec<V> x0n = inext < nv ? Vec<V>::ld_plain(f, inext) : Vec<V>::zero();
      nka_pass_b_elem<NZ, V, true>(x0, f, wnew, zp, zcol, coefN, coefY, coef_p, has_pair, nz, write_f, i, W, Z, ld, S);
      x0 = x0n;
    }
  } else {
    for (size_t i = start; i < nv; i += stride)
      nka_pass_b_elem<NZ, V, false>(Vec<V>::ld_plain(f, i), f, wnew, zp, zcol, coefN, coefY, coef_p, has_pair, nz, write_f,
                                    i, W, Z, ld, S);
  }
  if (V == 2 && (n & 1) && start == 0)
    nka_pass_b_elem<NZ, 1, false>(Vec<1>::ld_plain(f, n - 1), f, wnew, zp, zcol, coefN, coefY, coef_p, has_pair, nz, write_f,
                                  n - 1, W, Z, ld, S);
}
