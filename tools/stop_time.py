#!/usr/bin/env python3
"""Time per-problem stopping tests on device-side loops and queues (B200; one JSON line per case).

    python tools/stop_time.py [--reps R] [--out FILE]

(a) loop: BatchNKA.fixed_point_loop solves of exactly K = 20 steps (atol = rtol = 0, maxit = 20) at
    tools/loop_time.py's four sizes and residual, three arms alternated in one process:
      - scalar: atol, rtol, maxit as numbers (the existing rule);
      - arrays: the same values as per-member tensors (atol_dev, rtol_dev, maxit_dev);
      - scale:  the arrays plus a scale of 1.0 ([nbatch, n], read after every residual).
    A solve's time is a host clock around a launch and a device synchronise, from X = 0 after a restart;
    given per arm are the median, min and max of R solves.  `equal` records that the three arms' final X and
    F were bit-identical (a scale of 1.0 leaves the norms' bits alone).
(b) queue: 2^16 problems of vlen 256 through 4096 slots, mvec 5, with tools/queue_time.py's seeded
    problems (5..60 steps, then F = 0, which stops them on atol = 1e-300), except that one problem in eight
    has no fixed point: its residual is F = 1.1^c B_p at its c-th evaluation, finite and growing.  maxit =
    100; dtol = 0 (those problems run to MAXIT) against dtol = 10 (they stop DIVERGED at c = 25).  Reported
    per arm: median ms of R launches, slot-iterations (WHILE bodies times 4096, counted by the residual
    graph) and statuses; `equal_nondivergent` records that every other problem's final iterate, steps,
    status and norm were bit-identical between the two arms.
The card's name and power limit are read in the same run.
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


def loop_case(torch, nbatch, n, mvec, reps):
    g = torch.Generator(device="cuda").manual_seed(7)
    B = torch.rand(nbatch, n, dtype=torch.float64, device="cuda", generator=g) - 0.5
    f64 = dict(dtype=torch.float64, device="cuda")
    arms = {}
    for name in ("scalar", "arrays", "scale"):
        a = loop_time.Arm(torch, nbatch, n, mvec, B)
        if name == "scalar":
            kw = dict(atol=0.0, rtol=0.0, maxit=K)
        else:
            kw = dict(atol=torch.zeros(nbatch, **f64), rtol=torch.zeros(nbatch, **f64),
                      maxit=torch.full((nbatch,), K, dtype=torch.int32, device="cuda"))
            if name == "scale":
                kw["scale"] = torch.ones(nbatch, n, **f64)
        arms[name] = (a, a.acc.fixed_point_loop(a.residual, a.X, a.F, **kw))
    times = {name: [] for name in arms}
    for r in range(reps + 1):                 # rep 0 warms up
        for name, (a, loop) in arms.items():
            a.reset()
            t0 = time.perf_counter()
            loop.run()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r:
                times[name].append((t1 - t0) * 1e3)
    outs = {name: (a.X.cpu().numpy().view(np.uint64), a.F.cpu().numpy().view(np.uint64)) for name, (a, _) in arms.items()}
    steps = {name: loop.results()[0].tolist() for name, (_, loop) in arms.items()}
    equal = all(np.array_equal(outs[name][i], outs["scalar"][i]) for name in outs for i in (0, 1))
    res = {"case": "loop", "nbatch": nbatch, "n": n, "mvec": mvec, "iters": K, "reps": reps, "equal": bool(equal),
           "all_took_K_steps": all(s == [K] * nbatch for s in steps.values())}
    for name, t in times.items():
        res[name + "_ms"] = float(np.median(t))
        res[name + "_ms_min"], res[name + "_ms_max"] = float(min(t)), float(max(t))
    for name, (a, loop) in arms.items():
        loop.destroy()
        a.acc.delete()
    return res


class DivergentWork(queue_time.Work):
    """queue_time.Work with every eighth problem divergent: F = 1.1^c B_p at its c-th evaluation."""

    def __init__(self, torch, nproblems, n):
        super().__init__(torch, nproblems, n)
        self.div_host = np.arange(nproblems) % 8 == 3
        self.div = torch.from_numpy(self.div_host).cuda().unsqueeze(1)

    def residual(self):
        torch = self.torch
        super().residual()
        idx = self.slot.clamp(min=0).long()
        grow = torch.pow(1.1, self.count.to(torch.float64)).unsqueeze(1) * self.B.index_select(0, idx)
        self.F.copy_(torch.where(self.div.index_select(0, idx), grow, self.F))


def queue_case(torch, reps, nproblems=2**16, n=256):
    from nka_b200 import BatchNKA
    arms = {}
    for dtol in (0.0, 10.0):
        w = DivergentWork(torch, nproblems, n)
        acc = BatchNKA(queue_time.NSLOTS, n, queue_time.MVEC, 0.01)
        out = torch.zeros_like(w.X0)
        q = acc.fixed_point_queue(w.residual, w.X, w.F, w.slot, w.X0, out, atol=queue_time.ATOL, rtol=queue_time.RTOL,
                                  maxit=100, dtol=dtol)
        arms[dtol] = (w, acc, out, q)
    times = {d: [] for d in arms}
    outs, bodies = {}, {}
    for r in range(reps + 1):                 # run 0 warms up (and is the one compared)
        for d, (w, acc, out, q) in arms.items():
            w.reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            q.run()
            res = q.results()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r == 0:
                outs[d] = (out.cpu().numpy().view(np.uint64), *res)
                bodies[d] = int(w.calls.item())
            else:
                times[d].append((t1 - t0) * 1e3)
    keep = ~arms[0.0][0].div_host
    equal = all(np.array_equal(np.asarray(a)[keep].view(np.uint8), np.asarray(b)[keep].view(np.uint8))
                for a, b in zip(outs[0.0], outs[10.0]))
    res = {"case": "queue", "nslots": queue_time.NSLOTS, "nproblems": nproblems, "vlen": n, "mvec": queue_time.MVEC,
           "maxit": 100, "divergent": int((~keep).sum()), "reps": reps, "equal_nondivergent": bool(equal)}
    for d in arms:
        tag = "dtol%g" % d
        st = outs[d][2]
        res[tag + "_ms"] = float(np.median(times[d]))
        res[tag + "_slot_iterations"] = bodies[d] * queue_time.NSLOTS
        res[tag + "_status_counts"] = {str(s): int((st == s).sum()) for s in np.unique(st)}
        res[tag + "_divergent_steps"] = sorted(set(outs[d][1][~keep].tolist()))[:5]
    res["speedup_dtol10_vs_dtol0"] = res["dtol0_ms"] / res["dtol10_ms"]
    for w, acc, out, q in arms.values():
        q.destroy()
        acc.delete()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--queue-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stop_time.py needs a CUDA device")
    info = loop_time.card()
    rows = []
    for nbatch, n, mvec in loop_time.SIZES:
        rows.append(loop_case(torch, nbatch, n, mvec, args.reps))
    rows.append(queue_case(torch, args.queue_reps))
    for r in rows:
        r.update(info)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
