#!/usr/bin/env python3
"""Time a batched fixed-point solve three ways (B200; one JSON line per size).

    python tools/loop_time.py [--iters K] [--reps R] [--out FILE]

Each solve takes exactly K accelerated steps of every member (atol = rtol = 0, maxit = K), so the three
arms do identical work: K + 1 residual evaluations, K batched updates, K steps X += F.
  - device: BatchNKA.fixed_point_loop, one graph launch per solve (a WHILE node; stop tests on the device);
  - replay: one CUDA-graph replay per iteration (update, step, residual, row norms), then the row norms are
    copied to the host and checked there, as a user without device-side loops does it;
  - eager: the same calls one by one, with the same host check.
The residual is a cheap elementwise G: F = 0.5 (B - X) - 0.01 X^3.  A solve's time is a host clock
around it, ending in a device synchronise (the device arm: launch, then synchronise); the median of R
solves is given, each from X = 0 after a restart of the accelerator.  `equal` records that the three arms'
final X and F were bit-identical.  The card's name and power limit are read in the same run.
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

SIZES = [(1, 2**12, 5), (1, 2**20, 5), (64, 2**14, 10), (4096, 4096, 5)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


class Arm:
    def __init__(self, torch, nbatch, n, mvec, B, stream=None):
        from nka_b200 import BatchNKA
        self.torch = torch
        self.B = B
        self.X = torch.zeros(nbatch, n, dtype=torch.float64, device="cuda")
        self.F = torch.zeros_like(self.X)
        self.acc = BatchNKA(nbatch, n, mvec, 0.01, stream=stream)

    def residual(self):
        X = self.X
        self.F.copy_(0.5 * (self.B - X) - 0.01 * X * X * X)

    def reset(self):
        self.acc.restart()
        self.X.zero_()
        self.torch.cuda.synchronize()


def measure(torch, nbatch, n, mvec, K, reps):
    g = torch.Generator(device="cuda").manual_seed(7)
    B = torch.rand(nbatch, n, dtype=torch.float64, device="cuda", generator=g) - 0.5
    s = torch.cuda.Stream()

    dev = Arm(torch, nbatch, n, mvec, B)
    loop = dev.acc.fixed_point_loop(dev.residual, dev.X, dev.F, atol=0.0, rtol=0.0, maxit=K)

    def device_solve():
        loop.run()
        torch.cuda.synchronize()

    eag = Arm(torch, nbatch, n, mvec, B)

    def eager_solve():
        eag.residual()
        norms = torch.linalg.vector_norm(eag.F, dim=1)
        for k in range(K + 1):
            if not (k < K and np.isfinite(norms.cpu().numpy()).all()):
                break
            eag.acc.accel_update(eag.F)
            eag.X += eag.F
            eag.residual()
            norms = torch.linalg.vector_norm(eag.F, dim=1)
        torch.cuda.synchronize()

    rep = Arm(torch, nbatch, n, mvec, B, stream=s.cuda_stream)
    with torch.cuda.stream(s):
        rep.residual()
        torch.linalg.vector_norm(rep.F, dim=1)
    torch.cuda.synchronize()
    first, step = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(first, stream=s):
        rep.residual()
        norms0 = torch.linalg.vector_norm(rep.F, dim=1)
    with torch.cuda.graph(step, stream=s):
        rep.acc.accel_update(rep.F)
        rep.X += rep.F
        rep.residual()
        norms1 = torch.linalg.vector_norm(rep.F, dim=1)

    def replay_solve():
        with torch.cuda.stream(s):
            first.replay()
            norms = norms0
            for k in range(K + 1):
                if not (k < K and np.isfinite(norms.cpu().numpy()).all()):
                    break
                step.replay()
                norms = norms1
        torch.cuda.synchronize()

    arms = {"device": (dev, device_solve), "replay": (rep, replay_solve), "eager": (eag, eager_solve)}
    times = {name: [] for name in arms}
    outs = {}
    for r in range(reps + 1):                 # solve 0 warms up (and is the one compared)
        for name, (arm, solve) in arms.items():
            arm.reset()
            t0 = time.perf_counter()
            solve()
            t1 = time.perf_counter()
            if r == 0:
                outs[name] = (arm.X.cpu().numpy().view(np.uint64), arm.F.cpu().numpy().view(np.uint64))
            else:
                times[name].append((t1 - t0) * 1e3)
    it, st, _ = loop.results()
    assert np.all(it[np.isfinite(loop.history()[0])] == K), it
    equal = all(np.array_equal(outs["device"][i], outs[a][i]) for a in ("replay", "eager") for i in (0, 1))
    res = {"nbatch": nbatch, "n": n, "mvec": mvec, "iters": K, "reps": reps, "equal": bool(equal)}
    for name in arms:
        ms = float(np.median(times[name]))
        res[name + "_solve_ms"] = ms
        res[name + "_ms_per_iter"] = ms / K
    res["speedup_device_vs_replay"] = res["replay_solve_ms"] / res["device_solve_ms"]
    res["speedup_device_vs_eager"] = res["eager_solve_ms"] / res["device_solve_ms"]
    for arm, _ in arms.values():
        arm.acc.delete()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("loop_time.py needs a CUDA device")
    info = card()
    rows = []
    for nbatch, n, mvec in SIZES:
        r = measure(torch, nbatch, n, mvec, args.iters, args.reps)
        r.update(info)
        rows.append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
