// nka_ibatch.cu -- interleaved batched accelerators: nbatch independent same-length NKA instances whose
// vectors are stored component-major (element i of member b at f[i*ldf + b]), one thread per member
// (include/nka_b200.h, DESIGN.md section 17).
//
// Each thread runs its member's update as a statement-by-statement port of the C reference's
// nka_accel_update (oracle/nka_oracle.c:198-301, flavour 0): every dot product is the reference's serial
// j-ascending sum, and every multiply, add and subtract is written with __dmul_rn / __dadd_rn / __dsub_rn,
// so no contraction into an FMA can change a rounding.  Double division and sqrt are IEEE-rounded on the
// device.  A member's bits are therefore the reference's, whatever nbatch, its index, ldf, f's alignment
// or the other members hold.
//
// The vector loops are fused into three sweeps over the member's elements:
//   1. step A: the norm of w_p - f (w_p, the pending slot's cached f; the difference is not stored);
//   2. step B's normalisation (w_p = (w_p - f)/s, v_p = v_p/s, written), every Gram dot H(p,k) over the
//      pre-drop list and every step-D dot f.w_k, accumulated per list position in registers;
//   3. step C's raw copy of f into w_nw, the correction f += c_k (v_k - w_k) in list order and step E's
//      copy into v_nw.
// A column that step B frees is read in sweep 2 only, before sweep 3 may overwrite it as w_nw / v_nw.
// Steady-state traffic with a full list (mvec+1 slots on entry, mvec after the eviction) is
// 2 + (5 + mvec) + (4 + 2*mvec) = 11 + 3*mvec vectors of vlen doubles per member.
//
// Memory, all interleaved with member stride ldb = nbatch rounded up to 16 (128-byte aligned rows):
//   V, W: slot k, element i at ((size_t)k*vlen + i)*ldb + b;
//   D:    h(r,c) at (r*nslot + c)*ldb + b, then c[k] at (nslot*nslot + k)*ldb + b, then min_margin;
//   I:    the IB_* rows below, next[k] at (IB_NEXT + k)*ldb + b, prev[k] at (IB_NEXT + nslot + k)*ldb + b;
//   vtol: one device double, written by a kernel (set_vec_tol is capturable).

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <utility>

#include "../../include/nka_b200.h"
#include "nka_internal.h"

#define IB_THREADS 64
#define IB_NIL (-1)

enum { IB_SUBSPACE = 0, IB_PENDING, IB_FIRST, IB_LAST, IB_FREE, IB_NDROP, IB_EVICTED, IB_RELAXED, IB_NEXT };

struct IbArrays {
  double* V;
  double* W;
  double* D;
  int* I;
  double* vtol;
  size_t vlen, ldb;
  int nbatch, nslot;
};

struct nka_ibatch {
  int nbatch = 0, mvec = 0, device = 0;
  bool poison = false;                  // NKA_POISON_ALLOC
  cudaStream_t stream = nullptr;
  IbArrays A{};
  int* query = nullptr;                 // device: nbatch ints of num_vec, then the defined flag
  nka_state_view* view = nullptr;       // device: get_state's gather target
  unsigned long long launches = 0;
};

// ---------------------------------------------------------------------------
// one member's storage, seen from its thread
// ---------------------------------------------------------------------------
struct IbMember {
  const IbArrays& A;
  size_t b;
  __device__ int& I(int r) const { return A.I[(size_t)r * A.ldb + b]; }
  __device__ int& next(int k) const { return I(IB_NEXT + k); }
  __device__ int& prev(int k) const { return I(IB_NEXT + A.nslot + k); }
  __device__ double& H(int r, int c) const { return A.D[((size_t)r * A.nslot + c) * A.ldb + b]; }
  __device__ double& C(int k) const { return A.D[((size_t)A.nslot * A.nslot + k) * A.ldb + b]; }
  __device__ double& margin() const { return A.D[((size_t)A.nslot * (A.nslot + 1)) * A.ldb + b]; }
  // element i of a column is at [i * ldb]
  __device__ double* vcol(int k) const { return A.V + (size_t)k * A.vlen * A.ldb + b; }
  __device__ double* wcol(int k) const { return A.W + (size_t)k * A.vlen * A.ldb + b; }
};

struct IbList {
  int subspace, pending, first, last, free_;
};

__device__ __forceinline__ IbList ib_load(const IbMember& m)
{
  return {m.I(IB_SUBSPACE), m.I(IB_PENDING), m.I(IB_FIRST), m.I(IB_LAST), m.I(IB_FREE)};
}

__device__ __forceinline__ void ib_store(const IbMember& m, const IbList& s)
{
  m.I(IB_SUBSPACE) = s.subspace; m.I(IB_PENDING) = s.pending;
  m.I(IB_FIRST) = s.first; m.I(IB_LAST) = s.last; m.I(IB_FREE) = s.free_;
}

__device__ __forceinline__ bool ib_selected(const unsigned char* mask, size_t b) { return !mask || mask[b]; }

// oracle/nka_oracle.c:153-163
__device__ __forceinline__ void ib_restart(const IbMember& m, IbList& s)
{
  s.subspace = 0; s.pending = 0; s.first = IB_NIL; s.last = IB_NIL; s.free_ = 0;
  for (int k = 0; k < m.A.nslot - 1; ++k) m.next(k) = k + 1;
  m.next(m.A.nslot - 1) = IB_NIL;
}

// oracle/nka_oracle.c:165-176
__device__ __forceinline__ void ib_relax(const IbMember& m, IbList& s)
{
  if (!s.pending) return;
  const int head = s.first;
  s.first = m.next(head);
  if (s.first == IB_NIL) s.last = IB_NIL;
  else m.prev(s.first) = IB_NIL;
  m.next(head) = s.free_;
  s.free_ = head;
  s.pending = 0;
}

// ---------------------------------------------------------------------------
// the update: oracle/nka_oracle.c:198-301 with the vector loops fused into three sweeps.  NS = mvec + 1,
// a compile-time bound so that the per-position accumulators and column indices live in registers.
// ---------------------------------------------------------------------------
template <int NS>
__global__ void __launch_bounds__(IB_THREADS, 1)
nka_ibatch_update(IbArrays A, double* __restrict__ f, size_t ldf, const unsigned char* __restrict__ active)
{
  const size_t b = (size_t)blockIdx.x * IB_THREADS + threadIdx.x;
  if (b >= (size_t)A.nbatch || !ib_selected(active, b)) return;
  const IbMember m{A, b};
  const size_t n = A.vlen, ldb = A.ldb;
  f += b;                                                   // element i at f[i * ldf]
  IbList s = ib_load(m);
  double sn = 0.0;
  double margin = __longlong_as_double(0x7ff0000000000000ll);   // HUGE_VAL
  int ndrop = 0, evicted = 0, relaxed = 0;

  // Step A (sweep 1): s = sqrt(dot(w1 - f, w1 - f)); s == 0 relaxes.
  if (s.pending) {
    const double* w1 = m.wcol(s.first);
    double ss = 0.0;
    for (size_t i = 0; i < n; ++i) {
      const double d = __dsub_rn(w1[i * ldb], f[i * ldf]);
      ss = __dadd_rn(ss, __dmul_rn(d, d));
    }
    sn = sqrt(ss);
    if (sn == 0.0) { ib_relax(m, s); relaxed = 1; }
  }
  const bool stepb = s.pending;

  // the list on entry to step B, by position (col[0] is p when step B runs)
  int col[NS];
  int ncol = 0;
  {
    int k = s.first;
#pragma unroll
    for (int q = 0; q < NS; ++q) {
      col[q] = k;
      if (k != IB_NIL) { ++ncol; k = m.next(k); }
    }
  }

  // Sweep 2: normalise (step B), H(p, col[q]) = w_p . w_q (step B), f . w_q (step D) for every position.
  double hd[NS], fd[NS];
#pragma unroll
  for (int q = 0; q < NS; ++q) { hd[q] = 0.0; fd[q] = 0.0; }
  if (ncol > 0 && (stepb || s.subspace)) {
    double* w1 = m.wcol(col[0]);
    double* v1 = m.vcol(col[0]);
    for (size_t i = 0; i < n; ++i) {
      const double fi = f[i * ldf];
      double w0;
      if (stepb) {
        w0 = __dsub_rn(w1[i * ldb], fi) / sn;
        const double v0 = v1[i * ldb] / sn;
        w1[i * ldb] = w0;
        v1[i * ldb] = v0;
      } else {
        w0 = w1[i * ldb];
      }
      fd[0] = __dadd_rn(fd[0], __dmul_rn(fi, w0));
#pragma unroll
      for (int q = 1; q < NS; ++q) {
        if (q < ncol) {
          const double wq = m.wcol(col[q])[i * ldb];
          if (stepb) hd[q] = __dadd_rn(hd[q], __dmul_rn(w0, wq));
          fd[q] = __dadd_rn(fd[q], __dmul_rn(fi, wq));
        }
      }
    }
  }

  // Step B, scalar part: Gram row, Cholesky refactor, capacity eviction, vtol drops.
  if (stepb) {
    const int p = s.first;
#pragma unroll
    for (int q = 1; q < NS; ++q)
      if (q < ncol) m.H(p, col[q]) = hd[q];
    int nvec = 1;
    m.H(p, p) = 1.0;
    const double vtol = *A.vtol;
    for (int k = m.next(p); k != IB_NIL; k = m.next(k)) {
      if (++nvec > NS - 1) {
        m.next(s.last) = s.free_;
        s.free_ = k;
        s.last = m.prev(k);
        m.next(s.last) = IB_NIL;
        evicted = 1;
        break;
      }
      double hkk = 1.0;
      for (int j = p; j != k; j = m.next(j)) {
        double hkj = m.H(j, k);
        for (int i = p; i != j; i = m.next(i)) hkj = __dsub_rn(hkj, __dmul_rn(m.H(k, i), m.H(j, i)));
        hkj = hkj / m.H(j, j);
        m.H(k, j) = hkj;
        hkk = __dsub_rn(hkk, __dmul_rn(hkj, hkj));
      }
      const double tol2 = __dmul_rn(vtol, vtol);
      if (__dsub_rn(hkk, tol2) < margin) margin = __dsub_rn(hkk, tol2);
      if (hkk > tol2) {
        m.H(k, k) = sqrt(hkk);
      } else {
        const int pk = m.prev(k), nk = m.next(k);
        m.next(pk) = nk;
        if (nk == IB_NIL) s.last = pk;
        else m.prev(nk) = pk;
        m.next(k) = s.free_;
        s.free_ = k;
        k = pk;
        nvec--;
        ndrop++;
      }
    }
    s.subspace = 1;
    s.pending = 0;
  }

  // Step C: take a free slot (sweep 3 caches the raw f there).
  const int nw = s.free_;
  s.free_ = m.next(nw);

  // Step D, scalar part: c_j starts as sweep 2's f . w_j for every slot left on the list, then the two
  // triangular solves.
  int col2[NS];
  double ck[NS];
  int n2 = 0;
  if (s.subspace) {
    unsigned long long alive = 0;
    for (int k = s.first; k != IB_NIL; k = m.next(k)) alive |= 1ull << k;
#pragma unroll
    for (int q = 0; q < NS; ++q)
      if (q < ncol && ((alive >> col[q]) & 1ull)) m.C(col[q]) = fd[q];
    for (int j = s.first; j != IB_NIL; j = m.next(j)) {
      double cj = m.C(j);
      for (int i = s.first; i != j; i = m.next(i)) cj = __dsub_rn(cj, __dmul_rn(m.H(j, i), m.C(i)));
      m.C(j) = cj / m.H(j, j);
    }
    for (int j = s.last; j != IB_NIL; j = m.prev(j)) {
      double cj = m.C(j);
      for (int i = s.last; i != j; i = m.prev(i)) cj = __dsub_rn(cj, __dmul_rn(m.H(i, j), m.C(i)));
      m.C(j) = cj / m.H(j, j);
    }
    int k = s.first;
#pragma unroll
    for (int q = 0; q < NS; ++q) {
      col2[q] = k;
      ck[q] = 0.0;
      if (k != IB_NIL) { ck[q] = m.C(k); ++n2; k = m.next(k); }
    }
  }

  // Sweep 3: w_nw = f; f += c_k (v_k - w_k) in list order; v_nw = f.
  {
    double* wn = m.wcol(nw);
    double* vn = m.vcol(nw);
    for (size_t i = 0; i < n; ++i) {
      double fi = f[i * ldf];
      wn[i * ldb] = fi;
#pragma unroll
      for (int q = 0; q < NS; ++q)
        if (q < n2) fi = __dadd_rn(fi, __dmul_rn(ck[q], __dsub_rn(m.vcol(col2[q])[i * ldb], m.wcol(col2[q])[i * ldb])));
      vn[i * ldb] = fi;
      if (n2 > 0) f[i * ldf] = fi;
    }
  }

  // Step E: push the new slot and mark it pending.
  m.prev(nw) = IB_NIL;
  m.next(nw) = s.first;
  if (s.first == IB_NIL) s.last = nw;
  else m.prev(s.first) = nw;
  s.first = nw;
  s.pending = 1;
  ib_store(m, s);
  m.margin() = margin;
  m.I(IB_NDROP) = ndrop;
  m.I(IB_EVICTED) = evicted;
  m.I(IB_RELAXED) = relaxed;
}

typedef void (*IbUpdateFn)(IbArrays, double*, size_t, const unsigned char*);

template <size_t... M>
static IbUpdateFn ib_update_fn(int mvec, std::index_sequence<M...>)
{
  static const IbUpdateFn table[] = {nka_ibatch_update<(int)M + 2>...};
  return table[mvec - 1];
}

// ---------------------------------------------------------------------------
// init, relax, restart, set_vec_tol and the queries: one thread per member
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(IB_THREADS) nka_ibatch_init_kernel(IbArrays A)
{
  const size_t b = (size_t)blockIdx.x * IB_THREADS + threadIdx.x;
  if (b >= (size_t)A.nbatch) return;
  const IbMember m{A, b};
  for (int k = 0; k < A.nslot; ++k) m.prev(k) = IB_NIL;   // oracle/nka_oracle.c:141
  IbList s;
  ib_restart(m, s);
  ib_store(m, s);
  m.I(IB_NDROP) = 0;
  m.I(IB_EVICTED) = 0;
  m.I(IB_RELAXED) = 0;
}

__global__ void __launch_bounds__(IB_THREADS) nka_ibatch_relax_kernel(IbArrays A, const unsigned char* mask)
{
  const size_t b = (size_t)blockIdx.x * IB_THREADS + threadIdx.x;
  if (b >= (size_t)A.nbatch || !ib_selected(mask, b)) return;
  const IbMember m{A, b};
  IbList s = ib_load(m);
  ib_relax(m, s);
  ib_store(m, s);
}

__global__ void __launch_bounds__(IB_THREADS) nka_ibatch_restart_kernel(IbArrays A, const unsigned char* mask)
{
  const size_t b = (size_t)blockIdx.x * IB_THREADS + threadIdx.x;
  if (b >= (size_t)A.nbatch || !ib_selected(mask, b)) return;
  const IbMember m{A, b};
  IbList s;
  ib_restart(m, s);
  ib_store(m, s);
}

__global__ void nka_ibatch_set_vtol_kernel(double* vtol_dev, double vtol) { *vtol_dev = vtol; }

// The invariant check of oracle/nka_oracle.c:337-375 (src-F08/nka_type.F90:460-524), with the slot tags in
// a bit mask.
__device__ bool ib_defined(const IbMember& m, const IbList& s)
{
  const int n = m.A.nslot;
  for (int k = 0; k < n; ++k)
    if (m.next(k) < IB_NIL || m.next(k) >= n) return false;
  if (s.first < IB_NIL || s.first >= n) return false;
  if (s.free_ < IB_NIL || s.free_ >= n) return false;
  unsigned long long tag = 0;
  if (s.first == IB_NIL) {
    if (s.last != IB_NIL) return false;
  } else {
    int k = s.first;
    if (m.prev(k) != IB_NIL) return false;
    tag |= 1ull << k;
    while (m.next(k) != IB_NIL) {
      if (m.prev(m.next(k)) != k) return false;
      k = m.next(k);
      if ((tag >> k) & 1ull) return false;
      tag |= 1ull << k;
    }
    if (s.last != k) return false;
  }
  for (int k = s.free_; k != IB_NIL; k = m.next(k)) {
    if ((tag >> k) & 1ull) return false;
    tag |= 1ull << k;
  }
  return tag == (1ull << n) - 1;
}

// num[b] = num_vec of member b (oracle/nka_oracle.c:184-190), -1 if its lists fail the check; *bad = 1 if
// any member fails it (the caller zeroes it first).
__global__ void __launch_bounds__(IB_THREADS) nka_ibatch_query_kernel(IbArrays A, int* num, int* bad)
{
  const size_t b = (size_t)blockIdx.x * IB_THREADS + threadIdx.x;
  if (b >= (size_t)A.nbatch) return;
  const IbMember m{A, b};
  const IbList s = ib_load(m);
  const bool good = *A.vtol > 0.0 && ib_defined(m, s);
  int cnt = 0;
  if (good)
    for (int k = s.first; k != IB_NIL; k = m.next(k)) ++cnt;
  num[b] = good ? (s.pending ? cnt - 1 : cnt) : -1;
  if (!good) *bad = 1;
}

// Member b's state into a zeroed nka_state_view: the reference's fields and the last update's diagnostics.
__global__ void nka_ibatch_state_kernel(IbArrays A, size_t b, int mvec, nka_state_view* out)
{
  const IbMember m{A, b};
  const int n = A.nslot;
  out->mvec = mvec;
  out->subspace = m.I(IB_SUBSPACE); out->pending = m.I(IB_PENDING);
  out->first = m.I(IB_FIRST); out->last = m.I(IB_LAST); out->free_slot = m.I(IB_FREE);
  out->ndrop_last = m.I(IB_NDROP); out->evicted_last = m.I(IB_EVICTED); out->relaxed_last = m.I(IB_RELAXED);
  out->vtol = *A.vtol;
  out->min_margin = m.margin();
  for (int k = 0; k < n; ++k) {
    out->next[k] = m.next(k);
    out->prev[k] = m.prev(k);
    out->c[k] = m.C(k);
    for (int j = 0; j < n; ++j) out->h[k * n + j] = m.H(k, j);
  }
}

// ---------------------------------------------------------------------------
// the handle
// ---------------------------------------------------------------------------
static unsigned ib_grid(const nka_ibatch* h) { return (unsigned)(((size_t)h->nbatch + IB_THREADS - 1) / IB_THREADS); }

// A capturable call: aborts on the legacy default stream during another stream's capture (nothing can
// be queued), and returns whether this call is being captured (then nothing counts as launched).
static bool ib_capturing(NKAIBATCH h, const char* call)
{
  const int c = nka_capture_status(h->stream);
  if (c < 0)
    nka_capture_fail(call, "the handle is on the legacy default stream while another stream captures; "
                           "nka_ibatch_set_stream to the capture stream before the capture begins");
  return c > 0;
}

static void ib_launched(NKAIBATCH h, bool capturing)
{
  CUDA_CHECK(cudaGetLastError());
  if (!capturing) ++h->launches;
}

static void* ib_alloc(size_t bytes, const char* what)
{
  void* p = nullptr;
  const cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    char b[200];
    snprintf(b, sizeof b, "nka_ibatch_init: cannot allocate %zu bytes of device memory for %s: %s", bytes, what,
             cudaGetErrorString(e));
    nka_fail(__FILE__, __LINE__, b);
  }
  return p;
}

extern "C" NKAIBATCH nka_ibatch_init(int nbatch, size_t vlen, int mvec, double vtol, int device, void* stream)
{
  NKA_REQUIRE(nbatch >= 1, "nka_ibatch_init: nbatch must be in 1..2^31-1");
  NKA_REQUIRE(vlen >= 1, "nka_ibatch_init: vlen must be >= 1");
  NKA_REQUIRE(mvec > 0, "nka_ibatch_init: mvec must be > 0");
  NKA_REQUIRE(mvec <= NKA_B200_MAX_MVEC, "nka_ibatch_init: mvec > 32 is not supported by this build");
  NKA_REQUIRE(vtol > 0.0, "nka_ibatch_init: vtol must be > 0");
  const size_t ldb = ((size_t)nbatch + 15) / 16 * 16;
  const size_t nslot = (size_t)mvec + 1;
  NKA_REQUIRE(vlen <= SIZE_MAX / sizeof(double) / nslot / ldb, "nka_ibatch_init: the subspace size overflows size_t");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    nka_fail(__FILE__, __LINE__, "no CUDA device: libnka_b200 has no CPU compute path");
  NKAIBATCH h = new nka_ibatch();
  if (device < 0) CUDA_CHECK(cudaGetDevice(&device));
  h->device = device;
  DeviceGuard guard(device);
  h->nbatch = nbatch;
  h->mvec = mvec;
  h->stream = (cudaStream_t)stream;
  if (const char* s = getenv("NKA_POISON_ALLOC")) h->poison = atoi(s) != 0;
  IbArrays& A = h->A;
  A.vlen = vlen;
  A.ldb = ldb;
  A.nbatch = nbatch;
  A.nslot = (int)nslot;
  const size_t colbytes = nslot * vlen * ldb * sizeof(double);
  const size_t dbytes = (nslot * nslot + nslot + 1) * ldb * sizeof(double);
  const size_t ibytes = (IB_NEXT + 2 * nslot) * ldb * sizeof(int);
  A.V = (double*)ib_alloc(colbytes, "the subspace (V)");
  A.W = (double*)ib_alloc(colbytes, "the subspace (W)");
  A.D = (double*)ib_alloc(dbytes, "the Gram factors");
  A.I = (int*)ib_alloc(ibytes, "the lists");
  A.vtol = (double*)ib_alloc(sizeof(double), "vtol");
  h->query = (int*)ib_alloc(((size_t)nbatch + 1) * sizeof(int), "the queries");
  h->view = (nka_state_view*)ib_alloc(sizeof(nka_state_view), "the state view");
  // NKA_POISON_ALLOC: 0xFF bytes (a NaN in every double) wherever the init kernel writes nothing
  const int fill = h->poison ? 0xFF : 0;
  if (h->poison) {
    CUDA_CHECK(cudaMemsetAsync(A.V, 0xFF, colbytes, h->stream));
    CUDA_CHECK(cudaMemsetAsync(A.W, 0xFF, colbytes, h->stream));
  }
  CUDA_CHECK(cudaMemsetAsync(A.D, fill, dbytes, h->stream));
  CUDA_CHECK(cudaMemsetAsync(A.I, fill, ibytes, h->stream));
  nka_ibatch_set_vtol_kernel<<<1, 1, 0, h->stream>>>(A.vtol, vtol);
  ib_launched(h, false);
  nka_ibatch_init_kernel<<<ib_grid(h), IB_THREADS, 0, h->stream>>>(A);
  ib_launched(h, false);
  return h;
}

extern "C" void nka_ibatch_delete(NKAIBATCH h)
{
  if (!h) return;
  DeviceGuard guard(h->device);
  cudaStreamSynchronize(h->stream);
  cudaFree(h->A.V); cudaFree(h->A.W); cudaFree(h->A.D); cudaFree(h->A.I); cudaFree(h->A.vtol);
  cudaFree(h->query); cudaFree(h->view);
  delete h;
}

extern "C" void nka_ibatch_accel_update(NKAIBATCH h, double* f_dev, size_t ldf, const unsigned char* active_dev)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_accel_update: null handle");
  NKA_REQUIRE(f_dev != NULL, "nka_ibatch_accel_update: null f");
  NKA_REQUIRE(ldf >= (size_t)h->nbatch, "nka_ibatch_accel_update: ldf must be >= nbatch");
  DeviceGuard guard(h->device);
  const bool cap = ib_capturing(h, "nka_ibatch_accel_update");
  NkaRange nvtx("nka:ibatch_accel_update");
  ib_update_fn(h->mvec, std::make_index_sequence<NKA_B200_MAX_MVEC>())<<<ib_grid(h), IB_THREADS, 0, h->stream>>>(
      h->A, f_dev, ldf, active_dev);
  ib_launched(h, cap);
}

extern "C" void nka_ibatch_relax(NKAIBATCH h, const unsigned char* mask_dev)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_relax: null handle");
  DeviceGuard guard(h->device);
  const bool cap = ib_capturing(h, "nka_ibatch_relax");
  nka_ibatch_relax_kernel<<<ib_grid(h), IB_THREADS, 0, h->stream>>>(h->A, mask_dev);
  ib_launched(h, cap);
}

extern "C" void nka_ibatch_restart(NKAIBATCH h, const unsigned char* mask_dev)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_restart: null handle");
  DeviceGuard guard(h->device);
  const bool cap = ib_capturing(h, "nka_ibatch_restart");
  nka_ibatch_restart_kernel<<<ib_grid(h), IB_THREADS, 0, h->stream>>>(h->A, mask_dev);
  ib_launched(h, cap);
}

extern "C" void nka_ibatch_set_vec_tol(NKAIBATCH h, double vtol)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_set_vec_tol: null handle");
  NKA_REQUIRE(vtol > 0.0, "nka_ibatch_set_vec_tol: vtol must be > 0");
  DeviceGuard guard(h->device);
  const bool cap = ib_capturing(h, "nka_ibatch_set_vec_tol");
  nka_ibatch_set_vtol_kernel<<<1, 1, 0, h->stream>>>(h->A.vtol, vtol);
  ib_launched(h, cap);
}

// ---------------------------------------------------------------------------
// queries (never captured)
// ---------------------------------------------------------------------------
// num_vec of every member into query[0..nbatch), 1 into query[nbatch] if any member fails the check
static void ib_query(NKAIBATCH h, const char* call)
{
  nka_refuse_capture(h->stream, call, "it copies the device state to the host and synchronises");
  CUDA_CHECK(cudaMemsetAsync(h->query + h->nbatch, 0, sizeof(int), h->stream));
  nka_ibatch_query_kernel<<<ib_grid(h), IB_THREADS, 0, h->stream>>>(h->A, h->query, h->query + h->nbatch);
  CUDA_CHECK(cudaGetLastError());
}

extern "C" void nka_ibatch_num_vec(NKAIBATCH h, int* out)
{
  NKA_REQUIRE(h != NULL && out != NULL, "nka_ibatch_num_vec: null argument");
  DeviceGuard guard(h->device);
  ib_query(h, "nka_ibatch_num_vec");
  CUDA_CHECK(cudaMemcpyAsync(out, h->query, (size_t)h->nbatch * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
}

extern "C" int nka_ibatch_defined(NKAIBATCH h)
{
  if (!h || !h->A.V || !h->A.W || !h->A.D || !h->A.I) return 0;
  DeviceGuard guard(h->device);
  ib_query(h, "nka_ibatch_defined");
  int bad = 1;
  CUDA_CHECK(cudaMemcpyAsync(&bad, h->query + h->nbatch, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return bad ? 0 : 1;
}

extern "C" void nka_ibatch_get_state(NKAIBATCH h, int member, nka_state_view* out)
{
  NKA_REQUIRE(h != NULL && out != NULL, "nka_ibatch_get_state: null argument");
  NKA_REQUIRE(member >= 0 && member < h->nbatch, "nka_ibatch_get_state: member out of range");
  DeviceGuard guard(h->device);
  nka_refuse_capture(h->stream, "nka_ibatch_get_state", "it copies the device state to the host and synchronises");
  CUDA_CHECK(cudaMemsetAsync(h->view, 0, sizeof(nka_state_view), h->stream));
  nka_ibatch_state_kernel<<<1, 1, 0, h->stream>>>(h->A, (size_t)member, h->mvec, h->view);
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaMemcpyAsync(out, h->view, sizeof(nka_state_view), cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
}

extern "C" void nka_ibatch_set_stream(NKAIBATCH h, void* stream)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_set_stream: null handle");
  DeviceGuard guard(h->device);
  nka_refuse_capture(h->stream, "nka_ibatch_set_stream",
                     "it synchronises the handle's stream; set the capture stream before the capture begins");
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->stream = (cudaStream_t)stream;
}

extern "C" void nka_ibatch_synchronize(NKAIBATCH h)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_synchronize: null handle");
  DeviceGuard guard(h->device);
  nka_refuse_capture(h->stream, "nka_ibatch_synchronize", "it synchronises the handle's stream");
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
}

extern "C" int nka_ibatch_stream_capturing(NKAIBATCH h)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_stream_capturing: null handle");
  DeviceGuard guard(h->device);
  return nka_capture_status(h->stream);
}

extern "C" unsigned long long nka_ibatch_launch_count(NKAIBATCH h)
{
  NKA_REQUIRE(h != NULL, "nka_ibatch_launch_count: null handle");
  return h->launches;
}
