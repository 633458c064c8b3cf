#!/usr/bin/env python3
"""Time the batched accelerator against a loop over single handles (B200; one JSON line per size).

    python tools/batch_time.py [--steps K] [--warmup W] [--out FILE]

For each (nbatch, n, mvec): ms per batched update (all nbatch members), eager and replayed from a CUDA
graph, and the same nbatch updates as a loop over nbatch single NKA handles, eager and replayed (one graph
holding all of them).  Achieved bandwidth counts the algorithmic (2 mvec + 4) n 8 bytes per member update
and is also given as a fraction of a device-to-device copy rate measured in the same run.  Every update
takes fresh i.i.d. inputs, copied into f before its timed region (so part of f may sit in L2 when the
update starts), after at least mvec + 3 warm-up updates: every list is full.  Batch and loop are fed the
same inputs from the same start (the singles in the capacity shape, into which one capture switches
them), and `equal` records that their last outputs were bit-identical.  A last line gives the
per-kernel times of one size from torch.profiler.  The card's name and power limit are read in the same run.
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

SIZES = [(4096, 4096, 5), (1024, 16384, 10), (256, 65536, 10), (64, 2**20, 10)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def timed(torch, fn, reps):
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    beg.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return beg.elapsed_time(end) / reps


def copy_rate(torch):
    """Device-to-device copy of 2 GiB: bytes read + written per second."""
    a = torch.empty(2**28, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    ms = timed(torch, lambda: b.copy_(a), 20)
    del a, b
    return 2 * 2**28 * 8 / (ms * 1e-3)


def measure(torch, nbatch, n, mvec, steps, warmup):
    from nka_b200 import NKA, BatchNKA
    s = torch.cuda.Stream()
    gen = torch.Generator(device="cuda")
    warmup = max(warmup, mvec + 3)                   # every list full: the steady state is what is timed
    with torch.cuda.stream(s):
        batch = BatchNKA(nbatch, n, mvec, 0.01, stream=s.cuda_stream)
        singles = [NKA(n, mvec, 0.01, stream=s.cuda_stream) for _ in range(nbatch)]
        for acc in singles:                          # the capacity shape, as every batch member runs
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                acc.set_vec_tol(0.01)
        X = torch.empty(nbatch, n, dtype=torch.float64, device="cuda")
        Fb = torch.empty_like(X)
        Fs = torch.empty_like(X)
        rows = [Fs[b] for b in range(nbatch)]

        def batch_update():
            batch.accel_update(Fb)

        def loop_update():
            for acc, f in zip(singles, rows):
                acc.accel_update(f)

        gb, gl = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gb, stream=s):
            batch_update()
        with torch.cuda.graph(gl, stream=s):
            loop_update()
        beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def run(fn, dst, reps, seed):
            """reps updates, each on fresh i.i.d. inputs copied in before the timed region; ms per update"""
            gen.manual_seed(seed)
            total = 0.0
            for _ in range(reps):
                torch.rand(X.shape, generator=gen, dtype=torch.float64, device="cuda", out=X)
                dst.copy_(X)
                beg.record(s)
                fn()
                end.record(s)
                end.synchronize()
                total += beg.elapsed_time(end)
            return total / reps

        out = {"nbatch": nbatch, "n": n, "mvec": mvec, "steps": steps, "warmup": warmup}
        # batch and loop see the same input sequence: eager warm-up, eager timed, replayed warm-up, replayed timed
        for phase, (fb, fl) in enumerate(((batch_update, loop_update), (gb.replay, gl.replay))):
            mode = ("eager", "replay")[phase]
            for fn, dst, who in ((fb, Fb, "batch"), (fl, Fs, "loop")):
                run(fn, dst, warmup, 10 * phase + 1)
                out["%s_%s_ms" % (who, mode)] = run(fn, dst, steps, 10 * phase + 2)
        out["equal"] = bool(torch.equal(Fb.view(torch.int64), Fs.view(torch.int64)))
    nbytes = (2 * mvec + 4) * n * 8 * nbatch
    out["alg_bytes"] = nbytes
    for key in ("batch_eager_ms", "batch_replay_ms", "loop_eager_ms", "loop_replay_ms"):
        out[key.replace("_ms", "_GBps")] = nbytes / (out[key] * 1e-3) / 1e9
    out["speedup_batch_eager_vs_loop_eager"] = out["loop_eager_ms"] / out["batch_eager_ms"]
    batch.delete()
    for acc in singles:
        acc.delete()
    return out


def kernel_times(torch, nbatch, n, mvec, reps=20):
    from torch.profiler import ProfilerActivity, profile
    from nka_b200 import BatchNKA
    b = BatchNKA(nbatch, n, mvec, 0.01)
    F = torch.from_numpy(np.random.default_rng(1).uniform(-0.5, 0.5, (nbatch, n))).cuda()
    for _ in range(mvec + 3):
        b.accel_update(F)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            b.accel_update(F)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if "nka_batch" in ev.name:
            key = ev.name.split("<")[0].split("(")[0].replace("void ", "")
            per[key] = per.get(key, 0.0) + ev.device_time / 1e3 / reps
    b.delete()
    return {"kernel_ms_per_update": per, "nbatch": nbatch, "n": n, "mvec": mvec}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tools/batch_time.py needs a CUDA device")
    info = card()
    rate = copy_rate(torch)
    lines = []
    for nb, n, m in SIZES:
        r = measure(torch, nb, n, m, args.steps, args.warmup)
        r.update(info)
        r["d2d_copy_GBps"] = rate / 1e9
        for key in ("batch_eager", "batch_replay", "loop_eager", "loop_replay"):
            r[key + "_frac_copy"] = r[key + "_GBps"] * 1e9 / rate
        lines.append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    k = kernel_times(torch, *SIZES[0])
    k.update(info)
    lines.append(k)
    print(json.dumps(k), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            for r in lines:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
