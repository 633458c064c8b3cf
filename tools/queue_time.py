#!/usr/bin/env python3
"""Time many small fixed-point solves two ways (B200; one JSON line per size).

    python tools/queue_time.py [--reps R] [--out FILE]

Setup: mvec 5, 4096 slots (batch members), nproblems = 2^18 at vlen 256 and 2^16 at vlen 4096.  Problem p
takes a seeded number of steps s_p, uniform in 5..60: its residual is F = a_p (B_p - X) - 0.01 X^3 while
the slot has evaluated it fewer than s_p times since the problem arrived, then exactly 0, which stops it
on atol (atol = 1e-300, rtol = 0, maxit = 64).  The residual finds each row's problem through slot_problem.
  - queue: BatchNKA.fixed_point_queue, one graph launch for every problem (slots refilled on the device);
  - chunked: the existing BatchNKA.fixed_point_loop driven from the host chunk by chunk: slot_problem and
    the chunk's initial guesses in, restart, one loop launch, results and X out.  Each chunk lasts as long
    as its slowest problem.
A run's time is a host clock around it, ending in a device synchronise; the median of R runs is given, each
from the same initial guesses.  Reported: ms per full set of problems, problems/s, and slot-iterations
(bodies of the WHILE node times 4096, counted by the residual graph) against the useful sum of (s_p + 1)
residual checks.  `equal` records that both arms' final iterates, steps, statuses and norms were bit-identical.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NSLOTS, MVEC = 4096, 5
SIZES = [(2**18, 256), (2**16, 4096)]
ATOL, RTOL, MAXIT = 1e-300, 0.0, 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


class Work:
    """The problems, and the slots' X, F, slot_problem and residual state."""

    def __init__(self, torch, nproblems, n, seed=11):
        self.torch = torch
        g = torch.Generator(device="cuda").manual_seed(seed)
        cuda = dict(dtype=torch.float64, device="cuda")
        self.B = torch.rand(nproblems, n, generator=g, **cuda) - 0.5
        self.a = 0.3 + 0.6 * torch.rand(nproblems, 1, generator=g, **cuda)
        rng = np.random.default_rng(seed)
        self.steps_host = rng.integers(5, 61, nproblems).astype(np.int32)
        self.steps = torch.from_numpy(self.steps_host).cuda()
        self.X0 = 0.1 * (torch.rand(nproblems, n, generator=g, **cuda) - 0.5)
        self.X = torch.zeros(NSLOTS, n, **cuda)
        self.F = torch.zeros(NSLOTS, n, **cuda)
        self.slot = torch.full((NSLOTS,), -1, dtype=torch.int32, device="cuda")
        self.owner = torch.full((NSLOTS,), -2, dtype=torch.int32, device="cuda")
        self.count = torch.zeros(NSLOTS, dtype=torch.int32, device="cuda")
        self.calls = torch.zeros(1, dtype=torch.int64, device="cuda")

    def residual(self):
        torch = self.torch
        sp, X = self.slot, self.X
        idx = sp.clamp(min=0).long()
        self.count.copy_(torch.where(sp != self.owner, torch.zeros_like(self.count), self.count + 1))
        self.owner.copy_(sp)
        done = (self.count >= self.steps.index_select(0, idx)).unsqueeze(1)
        F = self.a.index_select(0, idx) * (self.B.index_select(0, idx) - X) - 0.01 * X * X * X
        self.F.copy_(torch.where(done, torch.zeros_like(F), F))
        self.calls += 1

    def reset(self):
        self.owner.fill_(-2)
        self.calls.zero_()


def measure(torch, nproblems, n, reps):
    from nka_b200 import BatchNKA
    nchunks = nproblems // NSLOTS

    wq = Work(torch, nproblems, n)
    accq = BatchNKA(NSLOTS, n, MVEC, 0.01)
    outq = torch.zeros_like(wq.X0)
    queue = accq.fixed_point_queue(wq.residual, wq.X, wq.F, wq.slot, wq.X0, outq, atol=ATOL, rtol=RTOL, maxit=MAXIT)

    def queue_run():
        queue.run()
        it, st, norm = queue.results()
        return it, st, norm

    wc = Work(torch, nproblems, n)
    accc = BatchNKA(NSLOTS, n, MVEC, 0.01)
    outc = torch.zeros_like(wc.X0)
    loop = accc.fixed_point_loop(wc.residual, wc.X, wc.F, atol=ATOL, rtol=RTOL, maxit=MAXIT)
    ids = torch.arange(nproblems, dtype=torch.int32, device="cuda")

    def chunked_run():
        it = np.zeros(nproblems, dtype=np.int32)
        st = np.zeros(nproblems, dtype=np.int32)
        norm = np.zeros(nproblems)
        for c in range(nchunks):
            rows = slice(c * NSLOTS, (c + 1) * NSLOTS)
            wc.slot.copy_(ids[rows])
            wc.X.copy_(wc.X0[rows])
            accc.restart()
            loop.run()
            it[rows], st[rows], norm[rows] = loop.results()
            outc[rows].copy_(wc.X)
        return it, st, norm

    arms = {"queue": (wq, outq, queue_run), "chunked": (wc, outc, chunked_run)}
    times = {name: [] for name in arms}
    outs, bodies = {}, {}
    for r in range(reps + 1):                 # run 0 warms up (and is the one compared)
        for name, (w, out, run) in arms.items():
            w.reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = run()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if r == 0:
                outs[name] = (out.cpu().numpy().view(np.uint64), *res)
                bodies[name] = int(w.calls.item())
            else:
                times[name].append((t1 - t0) * 1e3)
    equal = all(np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
                for a, b in zip(outs["queue"], outs["chunked"]))
    it, st = outs["queue"][1], outs["queue"][2]
    res = {"nslots": NSLOTS, "nproblems": nproblems, "vlen": n, "mvec": MVEC, "reps": reps, "equal": bool(equal),
           "steps_as_set": bool(np.array_equal(it, wq.steps_host) and np.all(st == 1)),
           "mean_steps": float(wq.steps_host.mean()),
           "useful_slot_iterations": int((wq.steps_host.astype(np.int64) + 1).sum())}
    for name in arms:
        ms = float(np.median(times[name]))
        res[name + "_ms"] = ms
        res[name + "_problems_per_s"] = nproblems / (ms * 1e-3)
        res[name + "_slot_iterations"] = bodies[name] * NSLOTS
    res["speedup_queue_vs_chunked"] = res["chunked_ms"] / res["queue_ms"]
    queue.destroy()
    loop.destroy()
    accq.delete()
    accc.delete()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("queue_time.py needs a CUDA device")
    info = card()
    rows = []
    for nproblems, n in SIZES:
        r = measure(torch, nproblems, n, args.reps)
        r.update(info)
        rows.append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
