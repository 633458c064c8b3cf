// nka_batch_pass_b.cu -- pass B of the batched accelerator (nka_batch.cu): every member's sweep in one
// launch, blockIdx.y = member.  Each member follows its own plan (planB, planM); a member whose list is
// not full at entry takes the general body, as a single handle in the capacity shape does.  The sweep is
// element-wise, so its results do not depend on the CTA count.
#include "nka_batch.h"
#include "nka_kernels.cuh"

template <int NZ, int V>
__global__ void __launch_bounds__(nka_threads_b(NZ), NKA_MINB_B)
nka_batch_pass_b(double* F, size_t ldf, double* Wall, double* Zall, size_t wstride, size_t ld, size_t n,
                 const NkaDevState* __restrict__ Sall, const unsigned char* __restrict__ active)
{
  constexpr int NZA = NZ > 0 ? NZ : 1;
  const size_t b = blockIdx.y;
  if (active && !active[b]) return;                 // an inactive member: as if no call was made
  double* f = F + b * ldf;
  double* W = Wall + b * wstride;
  double* Z = Zall + b * wstride;
  const NkaDevState* S = Sall + b;

  const NkaPlanB* B = &S->planB;
  const int nz = B->nz, has_pair = B->has_pair, write_f = B->write_f;
  double* wnew = W + (size_t)B->newslot * ld;
  double* zp = Z + (size_t)B->pslot * ld;
  const double coef_p = B->coef_p;
  constexpr bool kCoefSmem = NZ >= NKA_COEF_SMEM_FROM;    // as nka_pass_b: coefficients in shared memory
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

static NkaBatchPassBFn g_batch_pass_b[NKA_MAXSLOT + 1][3];

template <int N> struct FillBatchB {
  static void run() {
    g_batch_pass_b[N - 1][1] = nka_batch_pass_b<N - 1, 1>;
    g_batch_pass_b[N - 1][2] = nka_batch_pass_b<N - 1, 2>;
    FillBatchB<N - 1>::run();
  }
};
template <> struct FillBatchB<0> { static void run() {} };

NkaBatchPassBFn nka_get_batch_pass_b(int nz, int v)
{
  static bool ready = false;
  if (!ready) { FillBatchB<NKA_INSTANTIATE_MAX>::run(); ready = true; }
  if (nz < 0 || nz >= NKA_MAXSLOT || v < 1 || v > 2) return nullptr;
  return g_batch_pass_b[nz][v];
}
