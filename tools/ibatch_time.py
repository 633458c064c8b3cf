#!/usr/bin/env python3
"""Measure the interleaved batched accelerator (B200; one JSON line per case).

    python tools/ibatch_time.py [--reps R] [--out FILE] [--dry-run]

Every case runs updates at steady state with full lists: each member gets fresh seeded inputs
f_t = 0.9^t * U(-0.5, 0.5) per update, mvec + 3 warm-up updates first, then R timed updates (median, min,
max of CUDA events around each update; the inputs are written between the events).

(a) InterleavedBatchNKA against BatchNKA on the same members, alternating the two arms update by update, at
    (nbatch, vlen, mvec) = (4096, 16, 5), (65535, 16, 5), (65535, 64, 5), (4096, 256, 5), (65535, 256, 5).
    The inputs are written interleaved (torch.empty(vlen, nbatch).t()); the row batch gets a transposed copy,
    timed on its own (`transpose_ms`, one direction) and not included in its update time.  After the timed
    updates the two arms' corrections are compared (largest per-member relative difference; they sum in
    different orders) and num_vec must be identical.
(b) InterleavedBatchNKA alone at (2^20, 16, 5), (2^20, 16, 10), (2^22, 8, 5) (subspaces above the 126 MB L2)
    and (2^18, 16, 32) (the O(mvec^3) Cholesky per member).
(c) lockstep against warp-divergent lists at (65535, 16, 5): in the divergent arm member b is restarted
    during the warm-up at update b % 7, so neighbouring lanes hold their columns in different slots.
Bytes per update follow the interleaved kernel's model, (11 + 3*mvec) * vlen * 8 per member at steady state,
reported as bytes/s and as a share of the B200's 7.7 TB/s.  The card's name and power limit are read in the
same run.  Without a GPU the tool fails, except with --dry-run, which prints the cases and their byte models.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VERSUS = [(4096, 16, 5), (65535, 16, 5), (65535, 64, 5), (4096, 256, 5), (65535, 256, 5)]
ALONE = [(2**20, 16, 5), (2**20, 16, 10), (2**22, 8, 5), (2**18, 16, 32)]
DIVERGENT = (65535, 16, 5)
PEAK = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def model_bytes(nbatch, vlen, mvec):
    return (11 + 3 * mvec) * vlen * 8 * nbatch


def _stats(ts):
    return {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts))}


class Inputs:
    """Seeded inputs written into an interleaved F on the device."""

    def __init__(self, torch, nbatch, vlen, seed=11):
        self.torch, self.g = torch, torch.Generator(device="cuda").manual_seed(seed)
        self.X = torch.empty(nbatch, vlen, dtype=torch.float64, device="cuda")

    def next(self, t, Fi):
        self.X.uniform_(-0.5, 0.5, generator=self.g).mul_(0.9 ** t)
        Fi.copy_(self.X)


def _event_ms(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def interleaved(torch, nbatch, vlen):
    return torch.empty(vlen, nbatch, dtype=torch.float64, device="cuda").t()


def versus(torch, nbatch, vlen, mvec, reps):
    from nka_b200 import BatchNKA, InterleavedBatchNKA
    ib = InterleavedBatchNKA(nbatch, vlen, mvec, 0.01)
    rb = BatchNKA(nbatch, vlen, mvec, 0.01)
    inp = Inputs(torch, nbatch, vlen)
    Fi = interleaved(torch, nbatch, vlen)
    Fr = torch.empty(nbatch, vlen, dtype=torch.float64, device="cuda")
    t_ib, t_rb, t_tr = [], [], []
    warm = mvec + 3
    for t in range(warm + reps):
        inp.next(t, Fi)
        tr = _event_ms(torch, lambda: Fr.copy_(Fi))
        arms = [("ib", lambda: ib.accel_update(Fi)), ("rb", lambda: rb.accel_update(Fr))]
        if t % 2:
            arms.reverse()
        ms = {name: _event_ms(torch, fn) for name, fn in arms}
        if t >= warm:
            t_ib.append(ms["ib"])
            t_rb.append(ms["rb"])
            t_tr.append(tr)
    diff = torch.linalg.vector_norm(Fi - Fr, dim=1) / torch.linalg.vector_norm(Fr, dim=1).clamp_min(1e-300)
    nv_i, nv_r = ib.num_vec(), rb.num_vec()
    out = {"case": "versus_batch", "nbatch": nbatch, "vlen": vlen, "mvec": mvec, "reps": reps,
           "ibatch_ms": _stats(t_ib), "batch_ms": _stats(t_rb), "transpose_ms": _stats(t_tr),
           "speedup_median": float(np.median(t_rb) / np.median(t_ib)),
           "ibatch_bytes_per_s": model_bytes(nbatch, vlen, mvec) / (np.median(t_ib) * 1e-3),
           "max_rel_diff": float(diff.max()), "members_over_1e-12": int((diff > 1e-12).sum()),
           "num_vec_identical": bool(np.array_equal(nv_i, nv_r)), "num_vec_min": int(nv_i.min())}
    out["ibatch_share_of_7.7TBps"] = out["ibatch_bytes_per_s"] / PEAK
    ib.delete()
    rb.delete()
    return out


def alone(torch, nbatch, vlen, mvec, reps, divergent=False):
    from nka_b200 import InterleavedBatchNKA
    ib = InterleavedBatchNKA(nbatch, vlen, mvec, 0.01)
    inp = Inputs(torch, nbatch, vlen)
    Fi = interleaved(torch, nbatch, vlen)
    phase = torch.arange(nbatch, device="cuda") % 7
    ts = []
    warm = mvec + 3 + (7 if divergent else 0)
    for t in range(warm + reps):
        if divergent and t < 7:
            ib.restart(phase == t)
        inp.next(t, Fi)
        ms = _event_ms(torch, lambda: ib.accel_update(Fi))
        if t >= warm:
            ts.append(ms)
    nv = ib.num_vec()
    med = float(np.median(ts))
    out = {"case": "divergent" if divergent else "alone", "nbatch": nbatch, "vlen": vlen, "mvec": mvec, "reps": reps,
           "ibatch_ms": _stats(ts), "model_bytes": model_bytes(nbatch, vlen, mvec),
           "bytes_per_s": model_bytes(nbatch, vlen, mvec) / (med * 1e-3),
           "num_vec_min": int(nv.min()), "num_vec_max": int(nv.max())}
    out["share_of_7.7TBps"] = out["bytes_per_s"] / PEAK
    ib.delete()
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", help="append the JSON lines here as well")
    ap.add_argument("--dry-run", action="store_true")
    args = ap.parse_args()
    if args.dry_run:
        for shape in VERSUS + ALONE + [DIVERGENT]:
            print(json.dumps({"nbatch": shape[0], "vlen": shape[1], "mvec": shape[2], "model_bytes": model_bytes(*shape)}))
        return 0
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ibatch_time.py needs a CUDA device")
    info = card()
    lines = []
    for shape in VERSUS:
        lines.append(versus(torch, *shape, args.reps))
        print(json.dumps({**lines[-1], **info}), flush=True)
    for shape in ALONE:
        lines.append(alone(torch, *shape, args.reps))
        print(json.dumps({**lines[-1], **info}), flush=True)
    for div in (False, True):
        lines.append(alone(torch, *DIVERGENT, args.reps, divergent=div))
        print(json.dumps({**lines[-1], **info}), flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            for ln in lines:
                fh.write(json.dumps({**ln, **info}) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
