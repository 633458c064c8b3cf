"""Seeded f-sequences that drive every branch of accel_update.

A scenario is a list of ops: ("update", f) | ("relax",) | ("restart",).
Inputs come from numpy's PCG64 (bit-reproducible across machines), so the
GPU box regenerates exactly what tests/golden/make_golden.py fed to the
compiled reference.

Branches covered (reference lines: src-C/nonlinear_krylov_accelerator.c):
  first call / growth / steady-state eviction        :339-347, :391-443
  vtol drop mid-list and at the tail                  :362-379
  s == 0 guard (exact repeat, zero vectors)           :309
  relax() with and without a subspace, restart()      :447-485
  n smaller than the subspace (rank deficiency)
"""
from __future__ import annotations

import numpy as np


def _upd(f):
    return ("update", np.ascontiguousarray(f, dtype=np.float64))


def iid(n, ncall, seed):
    rng = np.random.default_rng(seed)
    return [_upd(rng.uniform(-0.5, 0.5, n)) for _ in range(ncall)]


def contraction(n, ncall, seed, rho=0.7, spread=0.5):
    """f_t = A^t f_0 for a diagonal contraction with clustered rates: the
    differences quickly become nearly dependent, forcing vtol drops."""
    rng = np.random.default_rng(seed)
    lam = rho * (1.0 - spread * rng.uniform(0, 1, n) ** 4)
    f = rng.uniform(-0.5, 0.5, n)
    ops = []
    for _ in range(ncall):
        ops.append(_upd(f.copy()))
        f = lam * f
    return ops


def collinear(n, ncall, seed, rho=0.9, eps=1e-3, delta=1e-6):
    """SURVEY.md 8(d) stress family: f_t = rho^t g (1 + eps phi_t) + delta noise."""
    rng = np.random.default_rng(seed)
    g = rng.uniform(-0.5, 0.5, n)
    ops = []
    for t in range(ncall):
        phi = rng.uniform(-1, 1, n)
        noise = rng.uniform(-1, 1, n)
        ops.append(_upd(rho ** t * g * (1 + eps * phi) + delta * noise))
    return ops


def with_repeats(n, ncall, seed, repeat_at=(3, 4, 9)):
    """Exact repeats of the previous input: s == 0 -> the relax guard."""
    rng = np.random.default_rng(seed)
    ops = []
    last = None
    for t in range(ncall):
        if t in repeat_at and last is not None:
            f = last.copy()
        else:
            f = rng.uniform(-0.5, 0.5, n)
        last = f.copy()
        ops.append(_upd(f))
    return ops


def zeros_then_iid(n, ncall, seed):
    rng = np.random.default_rng(seed)
    ops = [_upd(np.zeros(n)), _upd(np.zeros(n))]
    ops += [_upd(rng.uniform(-0.5, 0.5, n)) for _ in range(ncall - 3)]
    ops.append(_upd(np.zeros(n)))
    return ops


def relax_restart(n, ncall, seed, relax_at=(5, 6, 11), restart_at=(8,)):
    """relax() (also twice in a row and right after restart) and restart()
    between updates; the subspace is carried across relax()."""
    rng = np.random.default_rng(seed)
    ops = []
    for t in range(ncall):
        if t in relax_at:
            ops.append(("relax",))
            if t == relax_at[1]:
                ops.append(("relax",))
        if t in restart_at:
            ops.append(("restart",))
            ops.append(("relax",))
        ops.append(_upd(rng.uniform(-0.5, 0.5, n)))
    return ops


def picard_like(n, ncall, seed):
    """A nonlinear fixed-point map's update sequence, driven open-loop (the
    accelerator's output is not fed back), giving smoothly shrinking,
    strongly correlated f's: realistic conditioning with occasional drops."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.1, 1.0, n)
    b = rng.uniform(0.5, 1.5, n)
    ops = []
    for _ in range(ncall):
        g = b / (1.0 + 0.5 * np.roll(x, 1) + 0.3 * x * x)
        f = x - g
        ops.append(_upd(f))
        x = x - 0.8 * f
    return ops


def mixed_stress(n, ncall, seed):
    """Collinear drift + exact repeats + relax/restart in one sequence
    (BASELINE.json configs[4] in miniature)."""
    base = collinear(n, ncall, seed, rho=0.8, eps=5e-2, delta=1e-4)
    ops = []
    for t, op in enumerate(base):
        if t == 6:
            ops.append(_upd(base[5][1].copy()))   # exact repeat
        if t == 10:
            ops.append(("relax",))
        if t == 15:
            ops.append(("restart",))
        ops.append(op)
    return ops


def fill_then_collinear(n, nfill, ncol, seed, eps=2e-3):
    """nfill i.i.d. calls (fills the list: no drops), then ncol nearly collinear ones: vtol
    drops fire while the list is at capacity, so the lazily skipped oldest column is needed
    after all (the fix-up sweep) at the largest list position."""
    rng = np.random.default_rng(seed)
    ops = [_upd(rng.uniform(-0.5, 0.5, n)) for _ in range(nfill)]
    g = rng.uniform(-0.5, 0.5, n)
    for t in range(ncol):
        ops.append(_upd(0.9 ** t * g * (1 + eps * rng.uniform(-1, 1, n))))
    return ops


# name -> (n, mvec, vtol, ops builder)
SCENARIOS = {
    "iid_n64_m3":          (64, 3, 0.01, lambda: iid(64, 12, 1)),
    "iid_n1000_m10":       (1000, 10, 0.01, lambda: iid(1000, 25, 2)),
    "iid_n7_m5":           (7, 5, 0.01, lambda: iid(7, 14, 3)),
    "mvec1_n17":           (17, 1, 0.01, lambda: iid(17, 7, 4)),
    "n1_m3":               (1, 3, 0.01, lambda: iid(1, 8, 5)),
    "n2_m4":               (2, 4, 0.01, lambda: iid(2, 10, 6)),
    "n3_m5_rankdef":       (3, 5, 0.01, lambda: iid(3, 12, 7)),
    "contraction_n200_m5": (200, 5, 0.01, lambda: contraction(200, 20, 8)),
    "contraction_n50_m8":  (50, 8, 0.05, lambda: contraction(50, 24, 9, rho=0.5, spread=0.9)),
    "collinear_n300_m6":   (300, 6, 0.01, lambda: collinear(300, 20, 10)),
    "collinear_n300_m6_v3": (300, 6, 0.3, lambda: collinear(300, 20, 11, eps=0.3, delta=1e-2)),
    "repeats_n128_m4":     (128, 4, 0.01, lambda: with_repeats(128, 14, 12)),
    "zeros_n33_m3":        (33, 3, 0.01, lambda: zeros_then_iid(33, 10, 13)),
    "relax_restart_n96_m4": (96, 4, 0.01, lambda: relax_restart(96, 16, 14)),
    "picard_n500_m5":      (500, 5, 0.01, lambda: picard_like(500, 30, 15)),
    "picard_n500_m5_v2":   (500, 5, 0.2, lambda: picard_like(500, 30, 16)),
    "mixed_n257_m5":       (257, 5, 0.1, lambda: mixed_stress(257, 22, 17)),
    "odd_n1023_m7":        (1023, 7, 0.01, lambda: iid(1023, 12, 18)),
    "n4097_m2":            (4097, 2, 0.01, lambda: iid(4097, 8, 19)),
    # wide subspaces: the 256-thread instantiations of pass B (13 columns and more)
    "iid_n2000_m16":       (2000, 16, 0.01, lambda: iid(2000, 40, 20)),
    "collinear_n400_m20":  (400, 20, 0.05, lambda: collinear(400, 48, 21, rho=0.9, eps=2e-1, delta=1e-3)),
    "iid_n513_m32":        (513, 32, 0.01, lambda: iid(513, 70, 22)),
    # mvec = 32 with vtol drops at a full list: list position 32 (the 33rd) carries a chained bit
    "fullthendrop_n700_m32": (700, 32, 0.1, lambda: fill_then_collinear(700, 36, 14, 24)),
    "fullthendrop_n300_m4":  (300, 4, 0.1, lambda: fill_then_collinear(300, 8, 10, 25)),
}


def run_ops(acc, ops):
    """Drive any accelerator with the reference's call shapes; returns
    (list of output vectors, list of num_vec after each op)."""
    outs, nvecs = [], []
    for op in ops:
        if op[0] == "update":
            f = op[1].copy()
            acc.accel_update(f)
            outs.append(f)
        elif op[0] == "relax":
            acc.relax()
        elif op[0] == "restart":
            acc.restart()
        nvecs.append(acc.num_vec())
    return outs, nvecs


def tolerances(serial, arbiter, inputs, factor=4.0):
    """Per-call relative tolerance for comparing an implementation with the long-double
    arbiter: 1e-12, or `factor` times the reference's OWN sensitivity to summation order
    (its serial-sum run vs its long-double-sum run, same code) if that is larger.
    Factor 4: call by call the CUDA path is at most 2.6 times as far from the arbiter as the
    reference's serial run has been up to that call (contraction_n50_m8; 2.3 for
    contraction_n200_m5; 0.57 for collinear_n300_m6; every other scenario passes at the plain 1e-12) --
    `worst_ratio_to_reference_spread` in profiles/parity_errors.json, merged from the GPU run's table; a
    factor of 2 fails those two.  The
    sensitivity is carried forward as a running maximum because a perturbed stored
    vector keeps influencing later calls.  Returns (scales, rel_tols)."""
    scales, tols = [], []
    worst = 0.0
    for a, b, fin in zip(serial, arbiter, inputs):
        scale = max(np.linalg.norm(b), np.linalg.norm(fin), 1e-300)
        worst = max(worst, np.linalg.norm(a - b) / scale)
        scales.append(scale)
        tols.append(max(1e-12, factor * worst))
    return scales, tols
