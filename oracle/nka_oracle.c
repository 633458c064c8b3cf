/*
 * oracle/nka_oracle.c -- CPU restatement of the reference's accel_update path.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity checker for the CUDA
 * product in nka_b200/.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may build, load or call
 * it.  Nothing under nka_b200/ links, imports or executes anything here; the
 * product has no CPU compute path.
 *
 * What it restates (reference = /root/reference, nncarlson/nka):
 *   - the accelerator state and list bookkeeping
 *       src-C/nonlinear_krylov_accelerator.c:179-197 (state), :447-463
 *       (restart), :466-485 (relax), :488-506 (queries)
 *       src-F08/nka_type.F90:154-181, :422-457, :221-247
 *   - accel_update, statement by statement
 *       src-C/nonlinear_krylov_accelerator.c:285-444
 *       src-F08/nka_type.F90:249-419, src-F95/nka_type.F90:278-470
 *   - the structural invariant check `defined`
 *       src-F08/nka_type.F90:460-524
 *   - the example's discrete system (residual, update_system, SSOR) in both
 *     scalings: src-C/nka_example.c:176-333 (== src-F95/nka_example.F90) and
 *     src-F08/nka_example.F90:103-179
 *
 * Parity pinning: tests/test_oracle.py checks this port (a) bit-for-bit
 * against the reference's own C library compiled from /root/reference into
 * oracle/_ref/ (same inputs, every correction vector and num_vec), and
 * (b) against the reference's golden `reference_output` tables through the
 * example restated below (tests/golden/).
 *
 * Differences from the reference, all deliberate:
 *   - sizes are size_t (the reference's `n * vlen * sizeof(double)` overflows
 *     int for (mvec+1)*vlen >= 2^31, src-C/...c:235,241);
 *   - slots are 0-based with -1 as the end marker in every flavour;
 *   - the dot product is selectable: 0 = the reference's serial left-to-right
 *     sum (src-C/...c:200-208), 1 = long double accumulation (the arbiter for
 *     n > 2^18, SURVEY.md section 7 hard part 3); orc_nka_set_dp installs a
 *     caller's dp hook instead, as the reference's nka_init does;
 *   - `flavour` picks the correction statement: 0 = C  f += c*(v-w)
 *     (src-C/...c:423), 1 = Fortran  f = f - c*w + c*v (src-F08/...F90:397);
 *   - set_vec_tol/defined exist (Fortran API) although the C header lacks them.
 *
 * Build: oracle/build.py (gcc -O2 -ffp-contract=off -shared -fPIC).
 */

#include <math.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define NIL (-1)

typedef struct orc_nka {
  size_t vlen;
  int mvec, nslot;       /* nslot = mvec + 1 */
  double vtol;
  int dotmode;           /* 0 serial double, 1 long double */
  double (*dp)(int, double *, double *);   /* the reference's dp hook; NULL = dotmode */
  int flavour;           /* 0 C, 1 Fortran association in the correction */
  int subspace, pending;
  int first, last, free;
  int *next, *prev;
  double *v, *w;         /* nslot columns of length vlen, column-major */
  double *h;             /* nslot x nslot, row-major: h[r*nslot + c] */
  double *c;             /* work: projection coefficients */
  double min_margin;     /* min over Cholesky rows of (hkk - vtol^2), last update */
  int ndrop_last;        /* vtol drops taken in the last update */
  int evicted_last;      /* capacity eviction taken in the last update */
  int relaxed_last;      /* s == 0 guard fired in the last update */
} orc_nka;

#define COL(a, st, k) ((a) + (size_t)(k) * (st)->vlen)
#define H(st, r, c_) ((st)->h[(size_t)(r) * (st)->nslot + (c_)])

/* ---- dot products ------------------------------------------------------ */

static double dot_serial(size_t n, const double *a, const double *b)
{
  /* src-C/nonlinear_krylov_accelerator.c:200-208 */
  double s = 0.0;
  for (size_t j = 0; j < n; j++) s += a[j] * b[j];
  return s;
}

static double dot_ld(size_t n, const double *a, const double *b)
{
  long double s = 0.0L;
  for (size_t j = 0; j < n; j++) s += (long double)a[j] * (long double)b[j];
  return (double)s;
}

static double dot(const orc_nka *st, const double *a, const double *b)
{
  /* src-C/...c:227-231: a caller-supplied dp replaces every dot product */
  if (st->dp) return st->dp((int)st->vlen, (double *)a, (double *)b);
  return st->dotmode == 1 ? dot_ld(st->vlen, a, b) : dot_serial(st->vlen, a, b);
}

/* Exported with the signature of the reference's `dp` hook so tests can hand
 * it to the compiled reference (oracle/_ref) through nka_init's 4th argument:
 * src-C/nonlinear_krylov_accelerator.c:227-231. */
double orc_dp_long_double(int len, double *x, double *y)
{
  return dot_ld((size_t)len, x, y);
}

/* ---- life cycle -------------------------------------------------------- */

/* The reference's dp argument of nka_init (src-C/...c:227-231), set after init; NULL restores dotmode. */
void orc_nka_set_dp(orc_nka *st, double (*dp)(int, double *, double *))
{
  st->dp = dp;
}

void orc_nka_restart(orc_nka *st);

orc_nka *orc_nka_init(size_t vlen, int mvec, double vtol, int dotmode, int flavour)
{
  /* src-C/...c:211-258; src-F08/nka_type.F90:185-200 */
  if (mvec <= 0 || !(vtol > 0.0)) return NULL;
  orc_nka *st = (orc_nka *)calloc(1, sizeof *st);
  if (!st) return NULL;
  st->vlen = vlen;
  st->mvec = mvec;
  st->nslot = mvec + 1;
  st->vtol = vtol;
  st->dotmode = dotmode;
  st->flavour = flavour;
  size_t ncol = (size_t)st->nslot;
  st->v = (double *)malloc((ncol * vlen + 1) * sizeof(double));
  st->w = (double *)malloc((ncol * vlen + 1) * sizeof(double));
  st->h = (double *)calloc(ncol * ncol, sizeof(double));
  st->c = (double *)calloc(ncol, sizeof(double));
  st->next = (int *)malloc(ncol * sizeof(int));
  st->prev = (int *)malloc(ncol * sizeof(int));
  if (!st->v || !st->w || !st->h || !st->c || !st->next || !st->prev) {
    free(st->v); free(st->w); free(st->h); free(st->c); free(st->next); free(st->prev);
    free(st);
    return NULL;
  }
  for (int k = 0; k < st->nslot; k++) st->prev[k] = NIL;
  orc_nka_restart(st);
  return st;
}

void orc_nka_delete(orc_nka *st)
{
  if (!st) return;
  free(st->v); free(st->w); free(st->h); free(st->c); free(st->next); free(st->prev);
  free(st);
}

void orc_nka_restart(orc_nka *st)
{
  /* src-C/...c:447-463; src-F08/nka_type.F90:422-436 */
  st->subspace = 0;
  st->pending = 0;
  st->first = NIL;
  st->last = NIL;
  st->free = 0;
  for (int k = 0; k < st->mvec; k++) st->next[k] = k + 1;
  st->next[st->mvec] = NIL;
}

void orc_nka_relax(orc_nka *st)
{
  /* src-C/...c:466-485; src-F08/nka_type.F90:439-457 */
  if (!st->pending) return;
  int head = st->first;
  st->first = st->next[head];
  if (st->first == NIL) st->last = NIL;
  else st->prev[st->first] = NIL;
  st->next[head] = st->free;
  st->free = head;
  st->pending = 0;
}

void orc_nka_set_vec_tol(orc_nka *st, double vtol)
{
  /* src-F08/nka_type.F90:202-207 */
  if (vtol > 0.0) st->vtol = vtol;
}

int orc_nka_num_vec(const orc_nka *st)
{
  /* src-C/...c:488-499 */
  int n = 0;
  for (int k = st->first; k != NIL; k = st->next[k]) n++;
  return st->pending ? n - 1 : n;
}

int orc_nka_max_vec(const orc_nka *st) { return st->mvec; }
size_t orc_nka_vec_len(const orc_nka *st) { return st->vlen; }
double orc_nka_vec_tol(const orc_nka *st) { return st->vtol; }

/* ---- the hot path ------------------------------------------------------ */

void orc_nka_accel_update(orc_nka *st, double *f)
{
  const size_t n = st->vlen;
  double s = 0.0;
  st->min_margin = HUGE_VAL;
  st->ndrop_last = 0;
  st->evicted_last = 0;
  st->relaxed_last = 0;

  /* Step A: next function difference and its norm.  src-C/...c:295-311 */
  if (st->pending) {
    double *w1 = COL(st->w, st, st->first);
    for (size_t j = 0; j < n; j++) w1[j] -= f[j];
    s = sqrt(dot(st, w1, w1));
    if (s == 0.0) { orc_nka_relax(st); st->relaxed_last = 1; }
  }

  /* Step B: normalise, Gram row, refactor, capacity/vtol drops.  :313-385 */
  if (st->pending) {
    const int p = st->first;
    double *w1 = COL(st->w, st, p);
    double *v1 = COL(st->v, st, p);
    for (size_t j = 0; j < n; j++) { v1[j] /= s; w1[j] /= s; }

    for (int k = st->next[p]; k != NIL; k = st->next[k])
      H(st, p, k) = dot(st, w1, COL(st->w, st, k));

    int nvec = 1;
    H(st, p, p) = 1.0;
    for (int k = st->next[p]; k != NIL; k = st->next[k]) {
      if (++nvec > st->mvec) {              /* capacity: drop the oldest.  :339-347 */
        st->next[st->last] = st->free;
        st->free = k;
        st->last = st->prev[k];
        st->next[st->last] = NIL;
        st->evicted_last = 1;
        break;
      }
      double hkk = 1.0;                     /* one Cholesky row.  :350-360 */
      for (int j = p; j != k; j = st->next[j]) {
        double hkj = H(st, j, k);
        for (int i = p; i != j; i = st->next[i]) hkj -= H(st, k, i) * H(st, j, i);
        hkj /= H(st, j, j);
        H(st, k, j) = hkj;
        hkk -= hkj * hkj;
      }
      const double tol2 = st->vtol * st->vtol;   /* pow(vtol,2) :362; vtol**2 F08:326 */
      if (hkk - tol2 < st->min_margin) st->min_margin = hkk - tol2;
      if (hkk > tol2) {
        H(st, k, k) = sqrt(hkk);
      } else {                               /* vtol drop.  :364-379 */
        const int pk = st->prev[k], nk = st->next[k];
        st->next[pk] = nk;
        if (nk == NIL) st->last = pk;
        else st->prev[nk] = pk;
        st->next[k] = st->free;
        st->free = k;
        k = pk;
        nvec--;
        st->ndrop_last++;
      }
    }
    st->subspace = 1;
    st->pending = 0;                         /* F08:351 (C leaves it set; no observable difference) */
  }

  /* Step C: take a free slot, cache the raw f.  :391-398 */
  const int nw = st->free;
  st->free = st->next[nw];
  memcpy(COL(st->w, st, nw), f, n * sizeof(double));

  /* Step D: project and correct.  :400-426 */
  if (st->subspace) {
    double *c = st->c;
    for (int j = st->first; j != NIL; j = st->next[j]) {
      double cj = dot(st, f, COL(st->w, st, j));
      for (int i = st->first; i != j; i = st->next[i]) cj -= H(st, j, i) * c[i];
      c[j] = cj / H(st, j, j);
    }
    for (int j = st->last; j != NIL; j = st->prev[j]) {
      double cj = c[j];
      for (int i = st->last; i != j; i = st->prev[i]) cj -= H(st, i, j) * c[i];
      c[j] = cj / H(st, j, j);
    }
    for (int k = st->first; k != NIL; k = st->next[k]) {
      const double *wk = COL(st->w, st, k), *vk = COL(st->v, st, k);
      const double ck = c[k];
      if (st->flavour == 0) {
        for (size_t j = 0; j < n; j++) f[j] += ck * (vk[j] - wk[j]);
      } else {
        for (size_t j = 0; j < n; j++) f[j] = f[j] - ck * wk[j] + ck * vk[j];
      }
    }
  }

  /* Step E: cache the accelerated f, push the slot, mark pending.  :428-443 */
  memcpy(COL(st->v, st, nw), f, n * sizeof(double));
  st->prev[nw] = NIL;
  st->next[nw] = st->first;
  if (st->first == NIL) st->last = nw;
  else st->prev[st->first] = nw;
  st->first = nw;
  st->pending = 1;
}

/* ---- introspection for the parity tests -------------------------------- */

double orc_nka_min_margin(const orc_nka *st) { return st->min_margin; }
int orc_nka_ndrop_last(const orc_nka *st) { return st->ndrop_last; }
int orc_nka_evicted_last(const orc_nka *st) { return st->evicted_last; }
int orc_nka_relaxed_last(const orc_nka *st) { return st->relaxed_last; }

/* out[0..4] = subspace,pending,first,last,free ; next/prev have nslot entries */
void orc_nka_get_lists(const orc_nka *st, int *out, int *next, int *prev)
{
  out[0] = st->subspace; out[1] = st->pending;
  out[2] = st->first; out[3] = st->last; out[4] = st->free;
  memcpy(next, st->next, (size_t)st->nslot * sizeof(int));
  memcpy(prev, st->prev, (size_t)st->nslot * sizeof(int));
}

void orc_nka_get_h(const orc_nka *st, double *h)
{
  memcpy(h, st->h, (size_t)st->nslot * st->nslot * sizeof(double));
}

/* Projection coefficients of the last update, in list order (newest first).
 * Returns how many were written. */
int orc_nka_get_coeffs(const orc_nka *st, double *out)
{
  int m = 0;
  if (!st->subspace) return 0;
  /* list after the update: head is the new pending slot; skip it */
  int k = st->first;
  if (st->pending && k != NIL) k = st->next[k];
  for (; k != NIL; k = st->next[k]) out[m++] = st->c[k];
  return m;
}

int orc_nka_defined(const orc_nka *st)
{
  /* src-F08/nka_type.F90:460-524, 0-based */
  if (!st || st->mvec < 1 || !st->v || !st->w || !st->h || !st->next || !st->prev) return 0;
  if (!(st->vtol > 0.0)) return 0;
  const int n = st->nslot;
  for (int k = 0; k < n; k++)
    if (st->next[k] < NIL || st->next[k] >= n) return 0;
  if (st->first < NIL || st->first >= n) return 0;
  if (st->free < NIL || st->free >= n) return 0;
  char *tag = (char *)calloc((size_t)n, 1);
  int ok = 0;
  do {
    if (st->first == NIL) {
      if (st->last != NIL) break;
    } else {
      int k = st->first, bad = 0;
      if (st->prev[k] != NIL) break;
      tag[k] = 1;
      while (st->next[k] != NIL) {
        if (st->prev[st->next[k]] != k) { bad = 1; break; }
        k = st->next[k];
        if (tag[k]) { bad = 1; break; }
        tag[k] = 1;
      }
      if (bad || st->last != k) break;
    }
    int bad = 0;
    for (int k = st->free; k != NIL; k = st->next[k]) {
      if (tag[k]) { bad = 1; break; }
      tag[k] = 1;
    }
    if (bad) break;
    ok = 1;
    for (int k = 0; k < n; k++) if (!tag[k]) ok = 0;
  } while (0);
  free(tag);
  return ok;
}

/* ======================================================================= */
/* The example's discrete system: -div((a+u) grad u) = q on an nx x ny cell */
/* grid, zero boundary values, mimetic discretisation.                      */
/*   scaling 0: F95 / C   (q = hx*hy, face terms rx*t, ry*t)                */
/*              src-C/nka_example.c:209-267, src-F95/nka_example.F90:163-196*/
/*   scaling 1: F08       (q = 1, face terms t*hx^2, t*hy^2)                */
/*              src-F08/nka_example.F90:122-145                             */
/* Arrays use the reference's C layout: u padded (nx+2)x(ny+2) row-major in */
/* k (y) with x fastest; ax is (nx+1) x ny, ay is nx x (ny+1), ac nx x ny.  */
/* ======================================================================= */

typedef struct orc_system {
  int nx, ny, scaling;
  double a, hx, hy;
  double *ax, *ay, *ac, *q;
} orc_system;

orc_system *orc_system_init(int nx, int ny, double a, int scaling)
{
  orc_system *sy = (orc_system *)calloc(1, sizeof *sy);
  sy->nx = nx; sy->ny = ny; sy->a = a; sy->scaling = scaling;
  sy->hx = 1.0 / nx; sy->hy = 1.0 / ny;
  sy->ax = (double *)malloc((size_t)ny * (nx + 1) * sizeof(double));
  sy->ay = (double *)malloc((size_t)nx * (ny + 1) * sizeof(double));
  sy->ac = (double *)malloc((size_t)nx * ny * sizeof(double));
  sy->q  = (double *)malloc((size_t)nx * ny * sizeof(double));
  const double qv = scaling == 0 ? sy->hx * sy->hy : 1.0;  /* nka_example.c:97 ; F08:100 */
  for (size_t i = 0; i < (size_t)nx * ny; i++) sy->q[i] = qv;
  return sy;
}

void orc_system_delete(orc_system *sy)
{
  if (!sy) return;
  free(sy->ax); free(sy->ay); free(sy->ac); free(sy->q); free(sy);
}

#define UP(j, k) upad[(size_t)((k) + 1) * (nx + 2) + (j) + 1]   /* interior cell (j,k), 0-based */
#define AX(j, k) sy->ax[(size_t)(k) * (nx + 1) + (j)]           /* face left of cell (j,k); j in 0..nx */
#define AY(j, k) sy->ay[(size_t)(k) * nx + (j)]                 /* face below cell (j,k); k in 0..ny */
#define AC(j, k) sy->ac[(size_t)(k) * nx + (j)]

void orc_update_system(orc_system *sy, const double *upad)
{
  const int nx = sy->nx, ny = sy->ny;
  double fx, fy;
  if (sy->scaling == 0) { fx = sy->hx / sy->hy; fy = sy->hy / sy->hx; }
  else { fx = sy->hx * sy->hx; fy = sy->hy * sy->hy; }
  memset(sy->ax, 0, (size_t)ny * (nx + 1) * sizeof(double));
  memset(sy->ay, 0, (size_t)nx * (ny + 1) * sizeof(double));
  /* scatter-add in the reference's cell order so the sums round identically */
  for (int k = 0; k < ny; k++)
    for (int j = 0; j < nx; j++) {
      const double t = 1.0 / (sy->a + UP(j, k));
      /* C/F95: ax += rx*t ; F08: ax += (t*hx**2) -- same operands, product is commutative */
      const double tx = sy->scaling == 0 ? fx * t : t * fx;
      const double ty = sy->scaling == 0 ? fy * t : t * fy;
      AX(j, k) += tx; AX(j + 1, k) += tx;
      AY(j, k) += ty; AY(j, k + 1) += ty;
    }
  for (size_t i = 0; i < (size_t)ny * (nx + 1); i++) sy->ax[i] = 2.0 / sy->ax[i];
  for (size_t i = 0; i < (size_t)nx * (ny + 1); i++) sy->ay[i] = 2.0 / sy->ay[i];
  for (int k = 0; k < ny; k++)
    for (int j = 0; j < nx; j++)
      AC(j, k) = AX(j, k) + AX(j + 1, k) + AY(j, k) + AY(j, k + 1);
}

void orc_residual(orc_system *sy, const double *upad, double *r)
{
  /* src-C/nka_example.c:176-206 ; src-F08/nka_example.F90:103-120 */
  const int nx = sy->nx, ny = sy->ny;
  orc_update_system(sy, upad);
  for (int k = 0; k < ny; k++)
    for (int j = 0; j < nx; j++)
      r[(size_t)k * nx + j] = AC(j, k) * UP(j, k) - AX(j, k) * UP(j - 1, k) - AX(j + 1, k) * UP(j + 1, k)
                              - AY(j, k) * UP(j, k - 1) - AY(j, k + 1) * UP(j, k + 1)
                              - sy->q[(size_t)k * nx + j];
}

void orc_ssor(const orc_system *sy, int nsweep, double omega, double *r)
{
  /* src-C/nka_example.c:270-333 ; src-F08/nka_example.F90:147-179.
   * Lexicographic Gauss-Seidel order, forward then backward, z = 0 start. */
  const int nx = sy->nx, ny = sy->ny;
  double *zpad = (double *)calloc((size_t)(nx + 2) * (ny + 2), sizeof(double));
#define Z(j, k) zpad[(size_t)((k) + 1) * (nx + 2) + (j) + 1]
#define SSOR_CELL(j, k)                                                            \
  Z(j, k) = (1.0 - omega) * Z(j, k)                                                \
          + omega * (r[(size_t)(k) * nx + (j)] + AX(j, k) * Z(j - 1, k) + AX(j + 1, k) * Z(j + 1, k) \
                     + AY(j, k) * Z(j, k - 1) + AY(j, k + 1) * Z(j, k + 1)) / AC(j, k)
  for (int it = 0; it < nsweep; it++) {
    for (int k = 0; k < ny; k++)
      for (int j = 0; j < nx; j++) SSOR_CELL(j, k);
    for (int k = ny - 1; k >= 0; k--)
      for (int j = nx - 1; j >= 0; j--) SSOR_CELL(j, k);
  }
  for (int k = 0; k < ny; k++)
    for (int j = 0; j < nx; j++) r[(size_t)k * nx + j] = Z(j, k);
  free(zpad);
#undef Z
#undef SSOR_CELL
}

static double l2norm(const double *x, size_t n)
{
  /* src-C/nka_example.c:336-345 (serial sum of squares) */
  double a = 0.0;
  for (size_t i = 0; i < n; i++) a += x[i] * x[i];
  return sqrt(a);
}

double orc_l2norm(const double *x, size_t n) { return l2norm(x, n); }

/* Picard solve of the example (src-C/nka_example.c:109-173,
 * src-F08/nka_example.F90:226-256).  mvec == 0 means unaccelerated.
 * rnorm[0..] receives the residual norm after iteration 0,1,...; at most
 * maxitr+1 entries.  If fseq/gseq are non-NULL they receive, per iteration,
 * the vector handed to accel_update and the vector it returned (each nx*ny),
 * so the device path can be replayed on identical inputs.  Returns the number
 * of iterations taken.  upad ((nx+2)*(ny+2)) holds the solution on exit. */
int orc_example_solve(int nx, int ny, double a, int nsweep, double omega, int mvec,
                      double vtol, int scaling, int flavour, int maxitr, double tol,
                      double *rnorm, double *upad, double *fseq, double *gseq, int *nvec_seq)
{
  const size_t n = (size_t)nx * ny;
  orc_system *sy = orc_system_init(nx, ny, a, scaling);
  orc_nka *acc = mvec > 0 ? orc_nka_init(n, mvec, vtol, 0, flavour) : NULL;
  double *r = (double *)malloc(n * sizeof(double));
  memset(upad, 0, (size_t)(nx + 2) * (ny + 2) * sizeof(double));
  orc_residual(sy, upad, r);
  const double rnorm0 = l2norm(r, n);
  rnorm[0] = rnorm0;
  int itr;
  for (itr = 1; itr <= maxitr; itr++) {
    orc_ssor(sy, nsweep, omega, r);
    if (acc) {
      if (fseq) memcpy(fseq + (size_t)(itr - 1) * n, r, n * sizeof(double));
      orc_nka_accel_update(acc, r);
      if (gseq) memcpy(gseq + (size_t)(itr - 1) * n, r, n * sizeof(double));
      if (nvec_seq) nvec_seq[itr - 1] = orc_nka_num_vec(acc);
    }
    for (int k = 0; k < ny; k++)
      for (int j = 0; j < nx; j++) UP(j, k) -= r[(size_t)k * nx + j];
    orc_residual(sy, upad, r);
    rnorm[itr] = l2norm(r, n);
    if (rnorm[itr] < tol * rnorm0) break;
  }
  if (itr > maxitr) itr = maxitr;
  free(r);
  orc_nka_delete(acc);
  orc_system_delete(sy);
  return itr;
}

/* Format one line of the example's table exactly as the reference prints it
 * (src-C/nka_example.c:135,158): "%3d:%14.6E" / "%3d:%14.6E%13.3E%8.3f". */
int orc_format_line(char *buf, size_t cap, int itr, double rnorm, double rnorm0)
{
  if (itr == 0) return snprintf(buf, cap, "%3d:%14.6E", 0, rnorm);
  const double red = rnorm / rnorm0;
  const double rate = pow(red, 1.0 / itr);
  return snprintf(buf, cap, "%3d:%14.6E%13.3E%8.3f", itr, rnorm, red, rate);
}
