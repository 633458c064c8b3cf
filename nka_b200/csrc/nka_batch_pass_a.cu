// nka_batch_pass_a.cu -- pass A of the batched accelerator (nka_batch.cu): every member's sweep in one
// launch.  blockIdx.y is the member, blockIdx.x the CTA within it; gridDim.x is the CTA count a single
// handle of the same length uses, so nka_grid_reduce (whose blockIdx.x / gridDim.x are per member here)
// folds every member's partial rows in the single handle's order.  No state step: the last CTA of a
// member only publishes that member's dot products; nka_batch_state_kernel steps all members after.
#include "nka_batch.h"
#include "nka_kernels.cuh"

template <int NC, int V>
__global__ void __launch_bounds__(NKA_THREADS_A, NKA_MINB_A)
nka_batch_pass_a(const double* __restrict__ F, size_t ldf, const double* __restrict__ Wall, size_t wstride, size_t ld,
                 size_t n, const NkaDevState* __restrict__ Sall, double* __restrict__ partials_all, size_t prow,
                 unsigned* __restrict__ tickets, double* __restrict__ dots_all, const unsigned char* __restrict__ active)
{
  const size_t b = blockIdx.y;
  if (active && !active[b]) return;                 // an inactive member: as if no call was made
  const double* f = F + b * ldf;
  const double* W = Wall + b * wstride;
  const NkaDevState* S = Sall + b;
  double* partials = partials_all + b * prow;

  const int ncol = S->planA.ncol - S->planA.skip_last;
  const unsigned long long submask = S->planA.submask;
  const double* wcol[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) wcol[j] = W + (size_t)(j < ncol ? S->planA.col[j] : 0) * ld;

  double acc[2 * NC];
#pragma unroll
  for (int j = 0; j < 2 * NC; ++j) acc[j] = 0.0;

  const size_t nv = n / V;
  const size_t stride = (size_t)gridDim.x * NKA_THREADS_A;
  const size_t start = (size_t)blockIdx.x * NKA_THREADS_A + threadIdx.x;
  const unsigned long long allbits = (1ull << NC) - 1ull;
  const bool full = (ncol == NC) && ((submask & allbits) == allbits);
  if (full) {
    for (size_t i = start; i < nv; i += stride) nka_pass_a_elem<NC, V, true>(f, wcol, i, ncol, submask, acc);
  } else {
    for (size_t i = start; i < nv; i += stride) nka_pass_a_elem<NC, V, false>(f, wcol, i, ncol, submask, acc);
  }
  if (V == 2 && (n & 1) && start == 0) nka_pass_a_elem<NC, 1, false>(f, wcol, n - 1, ncol, submask, acc);

  double* dots = dots_all + b * (2 * NKA_MAXSLOT);
  nka_grid_reduce<2 * NC, NKA_THREADS_A>(acc, partials, tickets + b, partials, gridDim.x,
                                         [&](int j, double v) { dots[j < NC ? j : NKA_MAXSLOT + (j - NC)] = v; });
}

static NkaBatchPassAFn g_batch_pass_a[NKA_MAXSLOT + 1][3];

template <int N> struct FillBatchA {
  static void run() {
    g_batch_pass_a[N][1] = nka_batch_pass_a<N, 1>;
    g_batch_pass_a[N][2] = nka_batch_pass_a<N, 2>;
    FillBatchA<N - 1>::run();
  }
};
template <> struct FillBatchA<0> { static void run() {} };

NkaBatchPassAFn nka_get_batch_pass_a(int nc, int v)
{
  static bool ready = false;
  if (!ready) { FillBatchA<NKA_INSTANTIATE_MAX>::run(); ready = true; }
  if (nc < 1 || nc > NKA_MAXSLOT || v < 1 || v > 2) return nullptr;
  return g_batch_pass_a[nc][v];
}
