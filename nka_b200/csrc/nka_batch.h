// nka_batch.h -- kernel tables of the batched accelerator (nka_batch.cu, nka_batch_pass_a.cu,
// nka_batch_pass_b.cu).
#pragma once
#include "nka_dispatch.h"

// (F, ldf, W, wstride, ld, n, S, partials, prow, tickets, dots, active)
typedef void (*NkaBatchPassAFn)(const double*, size_t, const double*, size_t, size_t, size_t, const NkaDevState*, double*,
                                size_t, unsigned*, double*, const unsigned char*);
// (F, ldf, W, Z, wstride, ld, n, S, active)
typedef void (*NkaBatchPassBFn)(double*, size_t, double*, double*, size_t, size_t, size_t, const NkaDevState*,
                                const unsigned char*);

// nc in 1..NKA_MAXSLOT, nz in 0..NKA_MAXSLOT-1, v in {1,2}; nullptr if not instantiated in this build
NkaBatchPassAFn nka_get_batch_pass_a(int nc, int v);
NkaBatchPassBFn nka_get_batch_pass_b(int nz, int v);
