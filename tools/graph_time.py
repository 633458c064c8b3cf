"""Per-update time of accel_update: eager calls against replays of a CUDA graph holding one update.

Usage: python tools/graph_time.py [--out FILE] [--log2n 12,16,20,24] [--mvec 5,10] [--reps 5]

Steady state (list full, one eviction per call), i.i.d. uniform(-0.5, 0.5) inputs from a pool of
mvec + 3 device vectors.  Each timed call copies the next pool vector into f and then updates it:
eagerly on handle E, or by replaying the graph captured on handle G.  The copy alone is timed too and
subtracted.  Both handles fill their lists eagerly before G captures its update, and they see the same
inputs in the same order, so their outputs must be equal bit for bit (the capacity shape of a captured
handle is the eager shape in steady state); `outputs_equal` records it.
Each window is timed twice: CUDA events on the stream, and a host clock that ends in a synchronise.
Arms alternate within every repetition; the median over repetitions is reported.
Prints a header line with the card, then one JSON line per (n, mvec)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nka_b200 import NKA  # noqa: E402


def card():
    line = {"gpu": torch.cuda.get_device_name(0), "torch": torch.__version__, "cuda": torch.version.cuda}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        line.update({"power_limit": power, "max_sm_clock": clock})
    except Exception as exc:                           # recorded, not hidden
        line["power_limit"] = "unknown (%s)" % type(exc).__name__
    return line


def measure(n, mvec, reps, vtol=0.01):
    s = torch.cuda.Stream()
    calls = int(min(5000, max(100, (1 << 28) // n)))
    gen = torch.Generator(device="cuda").manual_seed(n + mvec)
    pool = [torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) - 0.5 for _ in range(mvec + 3)]
    fe = torch.empty(n, dtype=torch.float64, device="cuda")
    fg = torch.empty_like(fe)
    fc = torch.empty_like(fe)
    e = NKA(n, mvec, vtol, stream=s.cuda_stream)
    g_acc = NKA(n, mvec, vtol, stream=s.cuda_stream)
    graph = None                                       # captured once both lists are full
    count = {"eager": 0, "graph": 0, "copy": 0}

    def run(arm, k):
        for _ in range(k):
            x = pool[count[arm] % len(pool)]
            count[arm] += 1
            if arm == "copy":
                fc.copy_(x)
            elif arm == "eager":
                fe.copy_(x)
                e.accel_update(fe)
            else:
                fg.copy_(x)
                if graph is None:
                    g_acc.accel_update(fg)
                else:
                    graph.replay()

    times = {arm: {"dev": [], "host": []} for arm in count}
    with torch.cuda.stream(s):
        for arm in count:                              # warm-up, eager on both handles: fills both lists
            run(arm, 2 * mvec + 4)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            g_acc.accel_update(fg)
        for arm in ("eager", "graph"):
            run(arm, 4)
        torch.cuda.synchronize()
        for _ in range(reps):
            for arm in ("eager", "graph", "copy"):
                b, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                b.record(s)
                run(arm, calls)
                en.record(s)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                times[arm]["dev"].append(b.elapsed_time(en) / calls)
                times[arm]["host"].append(1e3 * (t1 - t0) / calls)
    assert count["eager"] == count["graph"]
    equal = bool(torch.equal(fe, fg))
    med = {arm: {k: float(np.median(v)) for k, v in t.items()} for arm, t in times.items()}
    line = {"n": n, "log2n": n.bit_length() - 1, "mvec": mvec, "calls_per_window": calls, "reps": reps,
            "num_vec": [e.num_vec(), g_acc.num_vec()], "outputs_equal": equal,
            "ms_per_call": med,
            "ms_per_update_eager": {k: med["eager"][k] - med["copy"][k] for k in ("dev", "host")},
            "ms_per_update_graph": {k: med["graph"][k] - med["copy"][k] for k in ("dev", "host")},
            "spread_dev": {arm: [float(min(t["dev"])), float(max(t["dev"]))] for arm, t in times.items()}}
    e.delete()
    g_acc.delete()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--log2n", default="12,16,20,24")
    ap.add_argument("--mvec", default="5,10")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("graph_time.py needs a CUDA device")
    torch.cuda.set_device(0)
    lines = [dict(card(), what="accel_update per-update time, eager vs CUDA-graph replay (tools/graph_time.py)")]
    print(json.dumps(lines[0]), flush=True)
    for lg in (int(x) for x in args.log2n.split(",")):
        for m in (int(x) for x in args.mvec.split(",")):
            lines.append(measure(1 << lg, m, args.reps))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
