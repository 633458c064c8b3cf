// nka_dispatch.h -- kernel tables shared by the translation units of libnka_b200.so.
#pragma once
#include <stddef.h>
#include "nka_state.h"

typedef void (*PassAFn)(const double*, const double*, size_t, size_t, NkaDevState*, double*, unsigned*, double*, int, NkaPeerCtx*,
                        const double*, unsigned);
typedef void (*PassBFn)(double*, double*, double*, size_t, size_t, const NkaDevState*);

#ifndef NKA_INSTANTIATE_MAX
#define NKA_INSTANTIATE_MAX NKA_MAXSLOT     // tuning builds instantiate fewer sizes to compile faster
#endif

// nc in 1..NKA_MAXSLOT, nz in 0..NKA_MAXSLOT-1, v in {1,2}; nullptr if not instantiated in this build
PassAFn nka_get_pass_a(int nc, int v);
PassBFn nka_get_pass_b(int nz, int v);
// experimental (NKA_PASS_B_TMA=1): operand tiles staged by cp.async.bulk; nullptr if nz is not instantiated
PassBFn nka_get_pass_b_tma(int nz, int* threads, int* smem_bytes);

// How many CTAs a sweep over one vector gets on a device (nka_capi.cu).  Pass A's fold order depends
// on its CTA count, so the batched handle (nka_batch.cu) sizes every member's sweep with these same
// functions and the occupancy of the single handle's kernels: a member then reduces in exactly the
// order a single handle of the same length does.
struct NkaSweepGeom {
  int num_sms = 0;
  int max_grid = 0;                       // CTAs per sweep at most (= partial rows a handle allocates)
  int occ_a[NKA_MAXSLOT + 1][3];          // resident CTAs per SM of nka_pass_a<nc, V>, -1 = not queried yet
  int occ_b[NKA_MAXSLOT + 1][3];          // resident CTAs per SM of nka_pass_b<nz, V>
};
// num_sms, max_grid, and the occupancy of the capacity shape's kernels for mvec (queried now: never
// from inside a stream capture)
void nka_geom_init(NkaSweepGeom& g, int device, int mvec);
int nka_grid_for(const NkaSweepGeom& g, int per_sm, size_t n, int V, int threads);
int nka_per_sm_a(NkaSweepGeom& g, int nc, int V, size_t len);
int nka_per_sm_b(NkaSweepGeom& g, int nz, int V, size_t len);
