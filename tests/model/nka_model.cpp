// tests/model/nka_model.cpp -- TEST-ONLY host model of the device algorithm.
//
// The build container has no GPU.  This file lets the CPU test-suite exercise
// the exact state-machine code the device runs (nka_b200/csrc/nka_state.h is
// included verbatim) together with a plain-loop emulation of what the three
// streaming kernels do with the plans it emits, so that the raw-chain storage
// scheme, the materialisation rule and the host-side launch bookkeeping are
// checked against the oracle before any GPU time is spent.
//
// It is NOT part of the product: nothing under nka_b200/ builds, links or
// loads it, and libnka_b200.so contains no host compute path.
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../nka_b200/csrc/nka_state.h"

// How the state step is executed: by one thread here; tests/model/lanes_test.cpp runs it on
// several host threads instead, to check that the result does not depend on the lane count.
typedef int (*ModelStepFn)(NkaDevState& S, NkaStepScratch& X, const double* dots, int have_last);

static int serial_step(NkaDevState& S, NkaStepScratch& X, const double* dots, int have_last)
{
  return nka_state_step(S, X, dots, NKA_MAXSLOT, have_last, NkaSerial());
}

struct Model {
  size_t n, ld;
  int mvec;
  std::vector<double> W, Z;
  NkaDevState S;
  NkaStepScratch scratch;
  double dots[2 * NKA_MAXSLOT];
  // host-side bookkeeping mirrored from nka_capi.cu
  bool pending;
  int ub_len;
  int bound_violations;
  unsigned long long mat_entries;
  unsigned long long fixups;
  bool lazy;
  ModelStepFn step;
};

static void pass_a(Model* m, const double* f)
{
  const NkaPlanA& A = m->S.planA;
  const int ncol = A.ncol - A.skip_last;
  for (int j = 0; j < 2 * NKA_MAXSLOT; ++j) m->dots[j] = 0.0;
  // long double accumulation: the model checks logic, not summation order
  std::vector<long double> dd(ncol, 0.0L), fd(ncol, 0.0L);
  for (size_t i = 0; i < m->n; ++i) {
    double prev = f[i], d0 = 0.0;
    for (int j = 0; j < ncol; ++j) {
      const double x = m->W[(size_t)A.col[j] * m->ld + i];
      const double d = ((A.submask >> j) & 1ull) ? x - prev : x;
      if (j == 0) d0 = d;
      dd[j] += (long double)d0 * d;
      fd[j] += (long double)f[i] * d;
      prev = x;
    }
  }
  for (int j = 0; j < ncol; ++j) { m->dots[j] = (double)dd[j]; m->dots[NKA_MAXSLOT + j] = (double)fd[j]; }
}

// the two dot products of the skipped oldest column (nka_fixup_kernel)
static void fixup(Model* m, const double* f)
{
  const NkaPlanA& A = m->S.planA;
  const int jl = A.ncol - 1;
  long double dd = 0.0L, fd = 0.0L;
  for (size_t i = 0; i < m->n; ++i) {
    const double d0 = m->W[(size_t)A.col[0] * m->ld + i] - f[i];
    const double xl = m->W[(size_t)A.col[jl] * m->ld + i];
    const double dl = ((A.submask >> jl) & 1ull) ? xl - m->W[(size_t)A.col[jl - 1] * m->ld + i] : xl;
    dd += (long double)d0 * dl;
    fd += (long double)f[i] * dl;
  }
  m->dots[jl] = (double)dd;
  m->dots[NKA_MAXSLOT + jl] = (double)fd;
  m->fixups++;
}

static void materialise(Model* m)
{
  const NkaPlanM& P = m->S.planM;
  m->mat_entries += P.n;
  for (size_t i = 0; i < m->n; ++i)
    for (int e = 0; e < P.n; ++e)
      m->W[(size_t)P.dst[e] * m->ld + i] -= m->W[(size_t)P.sub[e] * m->ld + i];
}

static void pass_b(Model* m, double* f)
{
  const NkaPlanB& B = m->S.planB;
  const NkaPlanM& P = m->S.planM;
  m->mat_entries += P.n;
  for (size_t i = 0; i < m->n; ++i) {
    const double x0 = f[i];
    for (int e = 0; e < P.n; ++e)
      m->W[(size_t)P.dst[e] * m->ld + i] -= m->W[(size_t)P.sub[e] * m->ld + i];
    double y = 0.0;
    if (B.has_pair) {
      double yprev = 0.0;
      for (int k = 0; k < B.nz; ++k) yprev += B.coefY[k] * m->Z[(size_t)B.zcol[k] * m->ld + i];
      const double zp = yprev + x0;
      m->Z[(size_t)B.pslot * m->ld + i] = zp;
      y += B.coef_p * zp;
    }
    for (int k = 0; k < B.nz; ++k) y += B.coefN[k] * m->Z[(size_t)B.zcol[k] * m->ld + i];
    m->W[(size_t)B.newslot * m->ld + i] = x0;
    if (B.write_f) f[i] = x0 + y;
  }
}

extern "C" {

// poison = 1: the state and the step's scratch start as 0xFF bytes (NaN doubles, -1 ints), as
// uninitialised device memory may, so that init has to set everything the step reads.
Model* model_init_ex(size_t n, int mvec, double vtol, int poison)
{
  if (mvec < 1 || mvec + 1 > NKA_MAXSLOT || !(vtol > 0.0)) return nullptr;
  Model* m = new Model();
  m->n = n; m->ld = ((n + 15) / 16) * 16; if (m->ld == 0) m->ld = 16;
  m->mvec = mvec;
  m->W.assign(m->ld * (mvec + 1), 0.0);
  m->Z.assign(m->ld * (mvec + 1), 0.0);
  if (poison) {
    memset(&m->S, 0xFF, sizeof m->S);
    memset(&m->scratch, 0xFF, sizeof m->scratch);
  }
  nka_state_init(m->S, mvec, vtol);
  m->pending = false; m->ub_len = 0; m->bound_violations = 0; m->mat_entries = 0; m->fixups = 0; m->lazy = true;
  m->step = serial_step;
  return m;
}

Model* model_init(size_t n, int mvec, double vtol) { return model_init_ex(n, mvec, vtol, 0); }

void model_delete(Model* m) { delete m; }

void model_accel_update(Model* m, double* f)
{
  const int L = m->ub_len;
  const bool may_skip = m->lazy && m->pending && L == m->mvec + 1;
  const int NC = may_skip ? m->mvec : L;
  if (m->S.planA.ncol - m->S.planA.skip_last > NC) m->bound_violations++;
  if (m->S.planA.skip_last && !may_skip) m->bound_violations++;
  if (L > 0) {
    pass_a(m, f);
    NkaDevState copy = m->S;                       // the device works on a staged copy
    if (m->step(copy, m->scratch, m->dots, 0)) {
      if (!may_skip) m->bound_violations++;        // the host must have queued the fix-up kernel
      m->S.need_fixup = 1;
      fixup(m, f);
      copy = m->S;
      if (m->step(copy, m->scratch, m->dots, 1)) m->bound_violations++;
    }
    m->S = copy;
  } else {
    m->step(m->S, m->scratch, m->dots, 1);
  }
  pass_b(m, f);
  if (m->pending) m->ub_len = L + 1 < m->mvec + 1 ? L + 1 : m->mvec + 1;
  else m->ub_len = L + 1;
  m->pending = true;
}

void model_set_lazy(Model* m, int on) { m->lazy = on != 0; m->S.lazy_last = on; nka_build_plan_a(m->S); }
unsigned long long model_fixups(Model* m) { return m->fixups; }

void model_restart(Model* m) { nka_state_restart(m->S); m->pending = false; m->ub_len = 0; }

void model_relax(Model* m)
{
  if (!m->pending) return;
  nka_state_relax(m->S);
  if (m->ub_len >= 2) materialise(m);
  else if (m->S.planM.n != 0) m->bound_violations++;
  m->pending = false;
  m->ub_len -= 1;
}

int model_num_vec(Model* m)
{
  int n = 0;
  for (int k = m->S.first; k != NKA_NIL; k = m->S.next[k]) ++n;
  return m->S.pending ? n - 1 : n;
}

int model_defined(Model* m) { return nka_state_defined(m->S); }
int model_bound_violations(Model* m) { return m->bound_violations; }
unsigned long long model_mat_entries(Model* m) { return m->mat_entries; }
int model_error(Model* m) { return m->S.error; }
int model_ndrop_last(Model* m) { return m->S.ndrop_last; }
int model_relaxed_last(Model* m) { return m->S.relaxed_last; }
int model_evicted_last(Model* m) { return m->S.evicted_last; }
double model_min_margin(Model* m) { return m->S.min_margin; }
int model_host_pending(Model* m) { return m->pending ? 1 : 0; }
int model_dev_pending(Model* m) { return m->S.pending; }
int model_list_len(Model* m) { int n = 0; for (int k = m->S.first; k != NKA_NIL; k = m->S.next[k]) ++n; return n; }
int model_ub_len(Model* m) { return m->ub_len; }

// The plans, for tests that work out which kernel instantiation and body the device runs:
// plan A as pass A will read it on the next update, plans B and M as the last update left them.
int model_plan_a_ncol(Model* m) { return m->S.planA.ncol; }
int model_plan_a_skip_last(Model* m) { return m->S.planA.skip_last; }
unsigned long long model_plan_a_submask(Model* m) { return m->S.planA.submask; }
int model_plan_b_nz(Model* m) { return m->S.planB.nz; }
int model_plan_b_has_pair(Model* m) { return m->S.planB.has_pair; }
int model_plan_b_write_f(Model* m) { return m->S.planB.write_f; }
int model_plan_m_n(Model* m) { return m->S.planM.n; }

}  // extern "C"
