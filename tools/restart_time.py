#!/usr/bin/env python3
"""Measure the residual-growth restart of device-side loops and queues (B200; one JSON line per case).

    python tools/restart_time.py [--reps R] [--effect-reps R] [--out FILE] [--dry-run]

(a) cost of the guard: restart_growth = 0 against a rule that never fires (NEVER = 1e300), alternated in one
    process, R runs each (median, min, max):
      - loop: BatchNKA.fixed_point_loop solves of exactly K = 20 steps (atol = rtol = 0, maxit = 20) at
        tools/loop_time.py's four sizes and residual, from X = 0 after a restart;
      - queue: tools/queue_time.py's problems at (2^18 problems, vlen 256), 4096 slots, mvec 5.
    A run's time is a host clock around a launch and a device synchronise.  `equal` records that both arms'
    outputs (X and F of the loop; final iterates, steps, statuses and norms of the queue) were bit-identical.
(b) effect: a queue on the Family below (2^16 problems, vlen 256, 4096 slots, mvec 5, atol = 0,
    rtol = 1e-10, maxit = 100) at restart_growth 0, 1 and 2.  Per arm: the count per status, the mean steps
    of the converged problems, the total restarts, the slot-iterations (WHILE bodies times 4096, counted by
    the residual graph) and the median ms of R launches.  The family's loop histories at restart_growth = 0
    are summarised first (`growth_checks`: the share of checks k >= 1 of running problems with r_k > r_{k-1},
    over the first 4096 problems as one loop launch).
The card's name and power limit are read in the same run.  Without a GPU the tool fails, except with
--dry-run, which parses the arguments, builds a small Family on the CPU and evaluates its residual once.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import loop_time    # noqa: E402
import queue_time   # noqa: E402

K = 20
NEVER = 1e300
GAMMAS = (0.0, 1.0, 2.0)
EFFECT_PROBLEMS, EFFECT_VLEN, EFFECT_MAXIT, EFFECT_RTOL = 2**16, 256, 100, 1e-10


class Family:
    """A seeded family of problems on which accelerated steps sometimes raise the residual: per problem p,
    F = a_p (B_p - X) - e_p X^3 + h_p lap(X) (zero ends), a_p in [0.2, 0.9], e_p in [0, 1.5], h_p in
    [0, 0.2], B_p uniform in [-1, 1], X0 = 0.  At the larger e_p the plain step X += F is unstable at the
    solution (its slope there is below -1), so the accelerator has to carry the solve; where its model is
    poor a step can grow the residual.  Rows find their problem through slot_problem; `calls` counts
    residual evaluations."""

    def __init__(self, torch, nproblems, n, nslots, device="cuda", seed=23):
        self.torch = torch
        g = torch.Generator(device=device).manual_seed(seed)
        f64 = dict(dtype=torch.float64, device=device)
        self.a = 0.2 + 0.7 * torch.rand(nproblems, 1, generator=g, **f64)
        self.e = 1.5 * torch.rand(nproblems, 1, generator=g, **f64)
        self.h = 0.2 * torch.rand(nproblems, 1, generator=g, **f64)
        self.B = 2.0 * torch.rand(nproblems, n, generator=g, **f64) - 1.0
        self.X0 = torch.zeros(nproblems, n, **f64)
        self.X = torch.zeros(nslots, n, **f64)
        self.F = torch.zeros(nslots, n, **f64)
        self.slot = torch.full((nslots,), -1, dtype=torch.int32, device=device)
        self.calls = torch.zeros(1, dtype=torch.int64, device=device)

    def residual(self):
        idx = self.slot.clamp(min=0).long()
        X, F = self.X, self.F
        F.copy_(self.a.index_select(0, idx) * (self.B.index_select(0, idx) - X) - self.e.index_select(0, idx) * X * X * X)
        F[:, 1:-1] += self.h.index_select(0, idx) * (X[:, :-2] - 2.0 * X[:, 1:-1] + X[:, 2:])
        self.calls += 1


def _stats(t):
    return float(np.median(t)), float(min(t)), float(max(t))


def loop_cost(torch, nbatch, n, mvec, reps):
    g = torch.Generator(device="cuda").manual_seed(7)
    B = torch.rand(nbatch, n, dtype=torch.float64, device="cuda", generator=g) - 0.5
    arms = {}
    for gamma in (0.0, NEVER):
        a = loop_time.Arm(torch, nbatch, n, mvec, B)
        arms[gamma] = (a, a.acc.fixed_point_loop(a.residual, a.X, a.F, atol=0.0, rtol=0.0, maxit=K,
                                                 restart_growth=gamma))
    times = {gamma: [] for gamma in arms}
    for r in range(reps + 1):                 # rep 0 warms up
        for gamma, (a, loop) in arms.items():
            a.reset()
            t0 = time.perf_counter()
            loop.run()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r:
                times[gamma].append((t1 - t0) * 1e3)
    outs = {gamma: (a.X.cpu().numpy().view(np.uint64), a.F.cpu().numpy().view(np.uint64)) for gamma, (a, _) in arms.items()}
    res = {"case": "loop_cost", "nbatch": nbatch, "n": n, "mvec": mvec, "iters": K, "reps": reps,
           "equal": bool(all(np.array_equal(outs[0.0][i], outs[NEVER][i]) for i in (0, 1))),
           "all_took_K_steps": all(loop.results()[0].tolist() == [K] * nbatch for _, loop in arms.values()),
           "never_restarts": int(arms[NEVER][1].restarts().sum())}
    for gamma, tag in ((0.0, "gamma0"), (NEVER, "never")):
        res[tag + "_ms"], res[tag + "_ms_min"], res[tag + "_ms_max"] = _stats(times[gamma])
    res["never_over_gamma0"] = res["never_ms"] / res["gamma0_ms"]
    for a, loop in arms.values():
        loop.destroy()
        a.acc.delete()
    return res


def queue_cost(torch, reps, nproblems=2**18, n=256):
    from nka_b200 import BatchNKA
    arms = {}
    for gamma in (0.0, NEVER):
        w = queue_time.Work(torch, nproblems, n)
        acc = BatchNKA(queue_time.NSLOTS, n, queue_time.MVEC, 0.01)
        out = torch.zeros_like(w.X0)
        q = acc.fixed_point_queue(w.residual, w.X, w.F, w.slot, w.X0, out, atol=queue_time.ATOL, rtol=queue_time.RTOL,
                                  maxit=queue_time.MAXIT, restart_growth=gamma)
        arms[gamma] = (w, acc, out, q)
    times = {gamma: [] for gamma in arms}
    outs = {}
    for r in range(reps + 1):                 # run 0 warms up (and is the one compared)
        for gamma, (w, acc, out, q) in arms.items():
            w.reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            q.run()
            res = q.results()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r == 0:
                outs[gamma] = (out.cpu().numpy().view(np.uint64), *res)
            else:
                times[gamma].append((t1 - t0) * 1e3)
    equal = all(np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
                for a, b in zip(outs[0.0], outs[NEVER]))
    res = {"case": "queue_cost", "nslots": queue_time.NSLOTS, "nproblems": nproblems, "vlen": n, "mvec": queue_time.MVEC,
           "reps": reps, "equal": bool(equal), "never_restarts": int(arms[NEVER][3].restarts().sum())}
    for gamma, tag in ((0.0, "gamma0"), (NEVER, "never")):
        res[tag + "_ms"], res[tag + "_ms_min"], res[tag + "_ms_max"] = _stats(times[gamma])
    res["never_over_gamma0"] = res["never_ms"] / res["gamma0_ms"]
    for w, acc, out, q in arms.values():
        q.destroy()
        acc.delete()
    return res


def family_histories(torch):
    """The Family's first 4096 problems as one loop launch at restart_growth = 0: how often a check grows."""
    from nka_b200 import BatchNKA
    ns = queue_time.NSLOTS
    w = Family(torch, ns, EFFECT_VLEN, ns)
    w.slot.copy_(torch.arange(ns, dtype=torch.int32, device="cuda"))
    acc = BatchNKA(ns, EFFECT_VLEN, queue_time.MVEC, 0.01)
    loop = acc.fixed_point_loop(w.residual, w.X, w.F, atol=0.0, rtol=EFFECT_RTOL, maxit=EFFECT_MAXIT)
    w.X.zero_()
    loop.run()
    it, st, _ = loop.results()
    h = loop.history()
    grew = total = 0
    problems_with_growth = 0
    for b in range(ns):
        r = h[:it[b] + 1, b]
        d = r[1:] > r[:-1]
        grew += int(d.sum())
        total += d.size
        problems_with_growth += bool(d.any())
    res = {"case": "family_loop_histories", "problems": ns, "vlen": EFFECT_VLEN, "mvec": queue_time.MVEC,
           "maxit": EFFECT_MAXIT, "rtol": EFFECT_RTOL, "growth_checks": grew / max(total, 1),
           "problems_with_growth": problems_with_growth,
           "status_counts": {str(s): int((st == s).sum()) for s in np.unique(st)}}
    loop.destroy()
    acc.delete()
    return res


def effect(torch, reps):
    from nka_b200 import BatchNKA
    res = {"case": "effect", "nslots": queue_time.NSLOTS, "nproblems": EFFECT_PROBLEMS, "vlen": EFFECT_VLEN,
           "mvec": queue_time.MVEC, "maxit": EFFECT_MAXIT, "atol": 0.0, "rtol": EFFECT_RTOL, "reps": reps}
    for gamma in GAMMAS:
        w = Family(torch, EFFECT_PROBLEMS, EFFECT_VLEN, queue_time.NSLOTS)
        acc = BatchNKA(queue_time.NSLOTS, EFFECT_VLEN, queue_time.MVEC, 0.01)
        q = acc.fixed_point_queue(w.residual, w.X, w.F, w.slot, w.X0, torch.zeros_like(w.X0), atol=0.0,
                                  rtol=EFFECT_RTOL, maxit=EFFECT_MAXIT, restart_growth=gamma)
        times = []
        for r in range(reps + 1):             # run 0 warms up and is the one counted
            w.calls.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            q.run()
            it, st, _ = q.results()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r == 0:
                bodies = int(w.calls.item())
                rst = q.restarts()
                counts = {str(s): int((st == s).sum()) for s in np.unique(st)}
                conv = st == 1
                mean_conv = float(it[conv].mean()) if conv.any() else None
            else:
                times.append((t1 - t0) * 1e3)
        tag = "gamma%g" % gamma
        res[tag + "_status_counts"] = counts
        res[tag + "_mean_steps_converged"] = mean_conv
        res[tag + "_restarts"] = int(rst.sum())
        res[tag + "_slot_iterations"] = bodies * queue_time.NSLOTS
        res[tag + "_ms"] = float(np.median(times))
        q.destroy()
        acc.delete()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--effect-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--dry-run", action="store_true", help="CPU only: build a small Family and evaluate it once")
    args = ap.parse_args()
    import torch
    if args.dry_run:
        w = Family(torch, 64, 16, 8, device="cpu")
        w.slot.copy_(torch.arange(8, dtype=torch.int32))
        w.residual()
        print(json.dumps({"dry_run": True, "F_shape": list(w.F.shape), "F_finite": bool(torch.isfinite(w.F).all()),
                          "calls": int(w.calls.item()), "sizes": loop_time.SIZES, "gammas": GAMMAS}))
        return
    if not torch.cuda.is_available():
        raise SystemExit("restart_time.py needs a CUDA device")
    info = loop_time.card()
    rows = []

    def emit(r):
        r.update(info)
        rows.append(r)
        print(json.dumps(r), flush=True)

    for nbatch, n, mvec in loop_time.SIZES:
        emit(loop_cost(torch, nbatch, n, mvec, args.reps))
    emit(queue_cost(torch, args.reps))
    torch.cuda.empty_cache()
    emit(family_histories(torch))
    emit(effect(torch, args.effect_reps))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
