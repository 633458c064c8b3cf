#!/usr/bin/env python
"""bench.py -- accel_update throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is ONE accel_update in steady state (subspace full, one eviction per
call) on synthetic fp64 vectors, n = 2^28, mvec = 10, vtol = 0.01
(BASELINE.json configs[2], the configuration the metric is quoted on).  With
N > 1 (launched by torchrun, one process per GPU) every vector is split into N
contiguous slabs (strong scaling: n is fixed) and the only exchange is one
66-double NCCL all-reduce per update.

Prints one JSON line (rank 0).  `value` is device-resident throughput;
`e2e` is the same metric through the reference-facing C entry point
nka_accel_update(NKA, double*) with HOST (pinned) buffers, so each step pays
the host->device and device->host copy of f.  `cpu_baseline` / `--impl
reference` time the reference's own serial C implementation (oracle/_ref,
compiled from /root/reference; else the oracle port) on a bounded slice of the
same workload on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_FULL = 1 << 28
MVEC = 10
VTOL = 0.01


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_FULL, help="global vector length (default 2^28)")
    ap.add_argument("--mvec", type=int, default=MVEC)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pageable", action="store_true", help="skip the pageable-host-memory e2e figure")
    ap.add_argument("--no-probe", action="store_true", help="skip the cross-rank oracle parity probe")
    ap.add_argument("--no-sweep", action="store_true", help="skip the mvec 2/5/10/20 sweep (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the corrected f of the last timed step to DIR/f.npy (float64; "
                         "a fixed sample of %d elements when f is longer, see dump_index)" % DUMP_MAX)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1 (the number of timed accel_update calls)")
    return args


# --dump-outputs keeps at most this many doubles (32 MiB), so that two builds can be compared output for output
DUMP_MAX = 1 << 22


def dump_index(n: int):
    """The positions of a length-n output that --dump-outputs writes, in increasing order: all of them up to
    DUMP_MAX, else one position drawn with a fixed seed from each of DUMP_MAX equal blocks, so every run
    with the same n samples the same positions."""
    import numpy as np
    if n <= DUMP_MAX:
        return np.arange(n, dtype=np.int64)
    edges = np.arange(DUMP_MAX + 1, dtype=np.int64) * n // DUMP_MAX
    u = np.random.default_rng(12345).random(DUMP_MAX)
    return edges[:-1] + (u * np.diff(edges)).astype(np.int64)


def write_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def algorithmic_bytes(n: int, m: int) -> int:
    """SURVEY.md 8(d): reads M w + M v + f, writes f_out + new w + new v."""
    return (2 * m + 4) * n * 8


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float) -> dict:
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 9:
                continue
            try:
                clk, mx = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            smax.append(mx)
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                for nm, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------
# the reference arm / cpu baseline: the reference's own serial C accel_update
# --------------------------------------------------------------------------
def cpu_reference_run(n_full: int, mvec: int, steps: int, warmup: int, budget_s: float, n_cap: int = 1 << 26,
                      dump_dir: str | None = None):
    """Time the reference's C accel_update (1 thread: the reference is serial) on a bounded sample
    of the workload: the largest power-of-two length <= n_cap (2^26: BASELINE.md section 3; the
    unmodified source overflows int at (mvec+1)*n >= 2^31, src-C/...c:235,241) whose whole run fits
    in ~budget_s.  Returns updates/s scaled linearly to n_full, labelled as extrapolated, beside
    the real per-call time of the sample.  With dump_dir, the last timed call's corrected f (of the
    sample's length) is written there as f.npy."""
    import numpy as np
    from oracle import api
    calls = steps + warmup + mvec + 2
    # ~0.78 s per update at n = 2^24, mvec = 10 on this class of host (BENCH_r01), (8M+13) streams
    per_elem = 0.8 / (1 << 24) * (8 * mvec + 13) / 93.0
    n_s = 1 << 16
    while n_s * 2 <= min(n_full, n_cap) and (mvec + 1) * (n_s * 2) < 2 ** 31 \
            and (n_s * 2) * per_elem * calls <= budget_s:
        n_s *= 2
    kind = "reference" if api.ref_lib() is not None else "port"
    acc = api.RefNKA(n_s, mvec, VTOL) if kind == "reference" else api.OracleNKA(n_s, mvec, VTOL)
    rng = np.random.default_rng(1234)
    pool = [rng.random(n_s) - 0.5 for _ in range(mvec + 3)]
    k = 0
    for _ in range(mvec + 2 + warmup):
        acc.accel_update(pool[k % len(pool)])
        k += 1
    t0 = time.perf_counter()
    for _ in range(steps):
        acc.accel_update(pool[k % len(pool)])
        k += 1
    dt = time.perf_counter() - t0
    if dump_dir:
        write_outputs(dump_dir, {"f": pool[(k - 1) % len(pool)][dump_index(n_s)]})
    nvec = acc.num_vec()
    acc.close()
    ups_sample = steps / dt
    factor = n_full // n_s
    value = ups_sample / factor
    sample = ("%s C accel_update (gcc -O3 -DNDEBUG, serial, default dp) timed at n=2^%d, mvec=%d, %d steady-state "
              "calls (num_vec=%d), %.1f ms per call; updates/s EXTRAPOLATED x1/%d (linear in n) to n=2^%d"
              % ("reference src-C" if kind == "reference" else "oracle port of the reference",
                 n_s.bit_length() - 1, mvec, steps, nvec, 1e3 * dt / steps, factor, n_full.bit_length() - 1))
    return {"value": value, "unit": "updates/s", "cores": 1, "kind": kind, "sample": sample,
            "host_cores": os.cpu_count(), "ms_per_update_sample": 1e3 * dt / steps, "n_sample": n_s,
            "extrapolation_factor": factor, "updates_per_s_sample": ups_sample}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    res = cpu_reference_run(args.n, args.mvec, args.steps, args.warmup, budget_s=240.0, dump_dir=args.dump_outputs)
    line = {
        "impl": "reference",
        "metric": "accel_update/sec", "value": res["value"], "unit": "updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # what was really timed: one step = one reference call on the n_sample slice
        "ms_per_step": res["ms_per_update_sample"],
        "ms_per_step_extrapolated": 1e3 / res["value"],
        "extrapolated": {"from_n": res["n_sample"], "to_n": args.n, "factor": res["extrapolation_factor"],
                         "why": "the unmodified reference overflows int at (mvec+1)*n >= 2^31 "
                                "(src-C/nonlinear_krylov_accelerator.c:235,241)"},
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "hbm_gbs": res["value"] * algorithmic_bytes(args.n, args.mvec) / 1e9,
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args):
    """Identical for both arms (the driver compares them)."""
    return {
        "workload": "synthetic accel_update microbench (BASELINE.json configs[2]): n=2^%d fp64, mvec=%d, vtol=%g, "
                    "steady state (subspace full, one eviction per call), f_t i.i.d. uniform(-0.5,0.5)"
                    % (args.n.bit_length() - 1, args.mvec, VTOL),
        "n": args.n, "mvec": args.mvec, "vtol": VTOL,
        "l2": "inputs larger than L2: every column is %.0f MiB per GPU, no flush needed"
              % (args.n / max(args.gpus, 1) * 8 / 2 ** 20),
        "parallelism": ("row slabs over %d GPUs, one small sum per update" % args.gpus) if args.gpus > 1
                       else "single GPU",
    }


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------
def bind_near_gpu(local_rank: int) -> dict:
    """Run this process (and first-touch its host buffers) on the NUMA node the GPU hangs off:
    with 8 ranks staging host vectors at once, buffers on the far socket share one inter-socket
    link.  No-op when the platform does not expose the topology (VMs report node -1)."""
    info = {"node": None, "bound": False}
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        with open(path) as fh:
            node = int(fh.read().strip())
        info["node"] = node
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["bound"] = True
            info["cpus"] = len(allowed)
    except Exception as exc:                      # topology not visible: stay unbound
        info["error"] = type(exc).__name__
    return info


def parity_probe(world, rank, local_rank):
    """Before anything is timed: the N ranks together run two scenario sequences through the same
    library path the timed region uses (row slabs, in-kernel cross-rank sum) and rank 0 compares the
    joined corrections and every drop / eviction / relax decision with the CPU oracle
    (oracle/api.py, the checker: bit-identical to the compiled reference).
      A  picard_n500_m5_v2   vtol drops fire; odd slab sizes at N = 4, 8
      B  i.i.d. n = 2^20 + 38, mvec = 10, 14 calls: strict 1e-12 against the long-double arbiter
    Returns the dict for the JSON line on rank 0 (None elsewhere); ok=False fails the run."""
    import numpy as np
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scenarios as S
    from nka_b200 import NKA
    from nka_b200.distributed import distributed_nka, slab_bounds

    n_b = (1 << 20) + 38
    cases = [("picard_n500_m5_v2",) + S.SCENARIOS["picard_n500_m5_v2"],
             ("iid_n%d_m10" % n_b, n_b, 10, VTOL, lambda: S.iid(n_b, 14, 77))]
    report = {"scenarios": [], "max_rel_err": 0.0, "decisions_equal": True, "ok": True, "comm_mode": None,
              "ranks": world}
    for name, n, mvec, vtol, mk in cases:
        ops = mk()
        if world > 1:
            acc, lo, hi = distributed_nka(n, mvec, vtol, device=local_rank)
        else:
            acc, lo, hi = NKA(n, mvec, vtol, device=local_rank), 0, n
        maxlen = max(slab_bounds(n, world, r)[1] - slab_bounds(n, world, r)[0] for r in range(world))
        outs, decisions = [], []
        for op in ops:
            if op[0] == "update":
                d = torch.zeros(maxlen, dtype=torch.float64, device="cuda")
                d[: hi - lo].copy_(torch.from_numpy(np.ascontiguousarray(op[1][lo:hi])))
                acc.accel_update(d[: hi - lo])
                if world > 1:
                    allv = torch.empty(world * maxlen, dtype=torch.float64, device="cuda")
                    dist.all_gather_into_tensor(allv, d)
                else:
                    allv = d
                if rank == 0:
                    host = allv.cpu().numpy().reshape(world, maxlen)
                    outs.append(np.concatenate([host[r, : slab_bounds(n, world, r)[1] - slab_bounds(n, world, r)[0]]
                                                for r in range(world)]))
                st = acc.state()
                decisions.append((st["ndrop_last"], st["relaxed_last"], st["evicted_last"], st["error"], acc.num_vec()))
            elif op[0] == "relax":
                acc.relax()
            else:
                acc.restart()
        mode = acc.comm_mode()
        acc.delete()
        if world > 1:
            alld = [None] * world
            dist.all_gather_object(alld, decisions)
        else:
            alld = [decisions]
        if rank != 0:
            continue
        from oracle import api
        inputs = [op[1] for op in ops if op[0] == "update"]
        serial, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), ops)
        arbiter, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), ops)
        scales, tols = S.tolerances(serial, arbiter, inputs)
        if name.startswith("iid"):
            tols = [1e-12] * len(tols)
        orc = api.OracleNKA(n, mvec, vtol, dotmode=0)
        want_dec = []
        for op in ops:
            if op[0] == "update":
                orc.accel_update(op[1].copy())
                want_dec.append((orc.ndrop_last(), int(orc.relaxed_last()), int(orc.evicted_last()), 0, orc.num_vec()))
            elif op[0] == "relax":
                orc.relax()
            else:
                orc.restart()
        dec_ok = all(list(map(tuple, d)) == want_dec for d in alld)
        errs = [float(np.linalg.norm(o - a) / sc) for o, a, sc in zip(outs, arbiter, scales)]
        err_ok = all(e <= t for e, t in zip(errs, tols))
        report["scenarios"].append({"name": name, "n": n, "mvec": mvec, "vtol": vtol, "calls": len(inputs),
                                    "drops": int(sum(d[0] for d in want_dec)), "max_rel_err": max(errs),
                                    "tol": max(tols), "decisions_equal": dec_ok, "ok": bool(dec_ok and err_ok)})
        report["max_rel_err"] = max(report["max_rel_err"], max(errs))
        report["decisions_equal"] = report["decisions_equal"] and dec_ok
        report["ok"] = report["ok"] and dec_ok and err_ok
        report["comm_mode"] = mode
    return report if rank == 0 else None


def example_probe(world, rank, local_rank):
    """The example's physics on the N ranks' row slabs (BASELINE.json configs[3] in miniature, 200 x 131: odd slab
    sizes at every N) against the CPU oracle on rank 0: u <- u - z and the fused residual (halo rows from the
    neighbouring ranks, global norm), three SSOR sweeps that cross every slab boundary strip by strip through NVLink
    peer memory, and a second application -- all np.array_equal to the serial loops.  Returns the dict for the JSON
    line on rank 0 (None elsewhere); ok=False fails the run."""
    import numpy as np
    import torch.distributed as dist
    from nka_b200.example import System, distributed_system, FIELD_U, FIELD_R, FIELD_Z
    nx, ny, nsweep = 200, 131, 3
    rng = np.random.default_rng(42)
    u = rng.uniform(0.0, 0.3, (ny, nx))
    z = rng.uniform(-0.01, 0.01, (ny, nx))
    sy = distributed_system(0.02, nx, ny, scaling=1, device=local_rank) if world > 1 else System(0.02, nx, ny, scaling=1, device=local_rank)
    k0, k1 = (sy.k0, sy.k1) if world > 1 else (0, ny)
    sy.set(FIELD_U, u[k0:k1])
    sy.set(FIELD_Z, z[k0:k1])
    mine = {"rows": (k0, k1), "rnorm": sy.residual(subtract_z=True), "u": sy.get(FIELD_U), "r": sy.get(FIELD_R)}
    err = 0
    try:
        sy.pc_ssor(nsweep, 1.4)
        mine["z"] = sy.get(FIELD_Z)
        sy.pc_ssor(1, 1.4)
        mine["z2"] = sy.get(FIELD_Z)
        sy.residual(subtract_z=False)       # picks up the sweeps' device-side status ...
        sy.pc_ssor(1, 1.4)                  # ... which the next call reports (include/nka_example.h)
    except RuntimeError:
        err = 1
        mine.setdefault("z", np.zeros((k1 - k0, nx))); mine.setdefault("z2", np.zeros((k1 - k0, nx)))
    mine["error"] = err
    sy.delete()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    else:
        parts = [mine]
    if rank != 0:
        return None
    try:
        from oracle import api
        orc = api.OracleSystem(nx, ny, 0.02, 1)
        unew = u - z
        pad = np.zeros((ny + 2, nx + 2)); pad[1:-1, 1:-1] = unew
        r = orc.residual(pad).reshape(ny, nx)
        want = {"u": unew, "r": r, "z": orc.pc_ssor(nsweep, 1.4, r.ravel().copy()).reshape(ny, nx),
                "z2": orc.pc_ssor(1, 1.4, r.ravel().copy()).reshape(ny, nx)}
        norm_want = orc.norm2(r.ravel())
    except Exception as exc:            # the checker itself is unavailable: say so, do not call it a pass or a failure
        return {"grid": [nx, ny], "ranks": world, "ok": None, "checker_error": "%s: %s" % (type(exc).__name__, exc)}
    parts.sort(key=lambda d: d["rows"][0])
    equal = {k: bool(np.array_equal(np.concatenate([d[k] for d in parts], axis=0), w)) for k, w in want.items()}
    norms_same = all(d["rnorm"] == parts[0]["rnorm"] for d in parts)
    norm_err = abs(parts[0]["rnorm"] - norm_want) / parts[0]["rnorm"]
    ok = all(equal.values()) and norms_same and norm_err <= 1e-13 and all(d["error"] == 0 for d in parts)
    return {"grid": [nx, ny], "ranks": world, "slab_rows": [d["rows"][1] - d["rows"][0] for d in parts],
            "bit_identical": equal, "norm_same_on_every_rank": norms_same, "norm_rel_err": norm_err,
            "device_errors": [d["error"] for d in parts], "ok": bool(ok)}


def sample_of_slabs(f, lo, hi, n, world, torch):
    """The dump_index(n) elements of the global vector whose elements lo:hi this rank holds in f (device), on
    every rank.  Slabs are contiguous and in rank order, so the ranks' parts join in index order."""
    import numpy as np
    idx = dump_index(n)
    mine = idx[(idx >= lo) & (idx < hi)] - lo
    part = f.index_select(0, torch.from_numpy(mine).to(f.device)).cpu().numpy()
    if world == 1:
        return part
    import torch.distributed as dist
    parts = [None] * world
    dist.all_gather_object(parts, part)
    return np.concatenate(parts)


def time_updates(acc, pool, k, steps, stream, torch):
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(steps):
            acc.accel_update(pool[k % len(pool)]); k += 1
        ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1), k


def mvec_sweep(n, pool, gen, stream, peak, torch):
    """BASELINE.json configs[2]: mvec 2/5/10/20 at the same n, 3 x 10 steady-state steps each (median reported), outside the
    headline's timed region (device-resident inputs; mvec = 20 needs 84 GiB of subspace)."""
    from nka_b200 import NKA
    out = []
    for m in (2, 5, 10, 20):
        need = (2 * (m + 1) + max(0, m + 3 - len(pool))) * n * 8
        free, _ = torch.cuda.mem_get_info()
        if free < need + (2 << 30):
            out.append({"mvec": m, "skipped": "needs %.0f GiB, %.0f free" % (need / 2 ** 30, free / 2 ** 30)})
            continue
        while len(pool) < m + 3:
            pool.append(torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) - 0.5)
        acc = NKA(n, m, VTOL, stream=stream.cuda_stream)
        k = 0
        with torch.cuda.stream(stream):
            for _ in range(2 * m + 10):         # fill the subspace, then settle: the first ~20 updates on fresh allocations run up to 8 % slow
                acc.accel_update(pool[k % (m + 3)]); k += 1
        torch.cuda.synchronize()
        steps = 10
        runs = []
        for _ in range(3):                      # three back-to-back timings: short runs under a power cap scatter by several per cent
            ms, k = time_updates(acc, pool[: m + 3], k, steps, stream, torch)
            runs.append(ms / steps)
        ms_upd = sorted(runs)[1]                # the median one is reported
        ups = 1e3 / ms_upd
        gbs = ups * algorithmic_bytes(n, m) / 1e9
        out.append({"mvec": m, "updates_per_s": ups, "ms_per_update": ms_upd, "hbm_gbs": gbs, "frac": gbs / peak,
                    "num_vec": acc.num_vec(), "steps": steps, "ms_per_update_runs": runs})
        acc.delete()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun with %d processes (one per GPU)" % (args.gpus, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: nka_b200 has no CPU path")
    numa = bind_near_gpu(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from nka_b200 import NKA
    from nka_b200.distributed import distributed_nka

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- parity first: a fast kernel whose results differ from the reference's is not done ----
    probe = None
    if not args.no_probe:
        probe = parity_probe(world, rank, local_rank)
        flag = torch.tensor([1 if (probe is None or probe["ok"]) else 0], device="cuda")
        if world > 1:
            dist.broadcast(flag, src=0)
        if int(flag.item()) == 0:
            if rank == 0:
                print(json.dumps({"error": "parity probe failed", "parity_probe": probe}))
            raise SystemExit(3)

    ex_probe = None
    if not args.no_probe:
        ex_probe = example_probe(world, rank, local_rank)
        flag = torch.tensor([0 if (ex_probe is not None and ex_probe["ok"] is False) else 1], device="cuda")
        if world > 1:
            dist.broadcast(flag, src=0)
        if int(flag.item()) == 0:
            if rank == 0:
                print(json.dumps({"error": "example probe failed", "example_probe": ex_probe}))
            raise SystemExit(3)

    n, m = args.n, args.mvec
    stream = torch.cuda.Stream()
    if world > 1:
        acc, lo, hi = distributed_nka(n, m, VTOL, device=local_rank, stream=stream.cuda_stream)
    else:
        acc, lo, hi = NKA(n, m, VTOL, device=local_rank, stream=stream.cuda_stream), 0, n
    n_local = hi - lo

    # synthetic inputs, resident in HBM: a pool of mvec+3 independent vectors used round-robin.
    # accel_update overwrites f with f + (a tiny projection), so a revisited buffer is again an
    # i.i.d.-like vector unrelated to the subspace, which by then has evicted everything built from it.
    pool_n = m + 3
    gen = torch.Generator(device="cuda").manual_seed(1000 + rank)
    pool = [torch.rand(n_local, dtype=torch.float64, device="cuda", generator=gen) - 0.5 for _ in range(pool_n)]
    torch.cuda.synchronize()

    k = 0
    with torch.cuda.stream(stream):
        for _ in range(m + 2):                      # reach steady state (not counted as warm-up)
            acc.accel_update(pool[k % pool_n]); k += 1
        for _ in range(max(args.warmup, 0)):
            acc.accel_update(pool[k % pool_n]); k += 1
    barrier()
    assert acc.num_vec() == m, "not in steady state: num_vec=%d" % acc.num_vec()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    launches0 = acc.launch_count()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            acc.accel_update(pool[k % pool_n]); k += 1
        ev1.record(stream)
    barrier()
    t_wall1 = time.time()
    elapsed_ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = acc.launch_count() - launches0
    if args.dump_outputs:                         # before the steps below overwrite the pool buffers in place
        f_last = sample_of_slabs(pool[(k - 1) % pool_n], lo, hi, n, world, torch)
        if rank == 0:
            write_outputs(args.dump_outputs, {"f": f_last})

    # Per-kernel durations (roofline): the same steps again with a CUDA event pair around every
    # launch (the library's timing mode, events on the handle's stream).  Kept out of the headline
    # region because an event record between two kernels turns off their programmatic dependent
    # launch overlap; `span_ms_per_step` is this region's own time per step, for comparison.
    ksteps = max(1, min(args.steps, 50))
    acc.timing_enable(True)
    acc.timing_reset()
    barrier()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(ksteps):
            acc.accel_update(pool[k % pool_n]); k += 1
        ev1.record(stream)
    barrier()
    span_ms = max_over_ranks(ev0.elapsed_time(ev1))
    kt = acc.timing_read()
    acc.timing_enable(False)
    nvec_end = acc.num_vec()
    st = acc.state()
    geom = acc.launch_geometry()
    comm_mode = acc.comm_mode()

    # ---- e2e: the reference-facing entry point with HOST buffers (H2D + kernels + D2H per step) ----
    e2e = None
    if not args.no_e2e:
        import numpy as np
        from nka_b200 import _lib
        lib = _lib.load()
        h = acc._handle()

        def timed_host_calls(ptrs):
            j = 0
            for _ in range(2):
                lib.nka_accel_update(h, ptrs[j % len(ptrs)]); j += 1
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                lib.nka_accel_update(h, ptrs[j % len(ptrs)]); j += 1     # synchronous: returns with f updated
            torch.cuda.synchronize()
            return max_over_ranks(time.perf_counter() - t0)

        host = [torch.empty(n_local, dtype=torch.float64, pin_memory=True) for _ in range(3)]
        for hb, src in zip(host, pool):
            hb.copy_(src)
        torch.cuda.synchronize()
        dt = timed_host_calls([hb.data_ptr() for hb in host])

        # the floor of any implementation: the coefficients need every element of f before any output
        # element exists, so one H2D of the slab, then one D2H -- all ranks at once, bare copies
        scratch = pool[0]
        floor = 1e30
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            scratch.copy_(host[0], non_blocking=True)
            host[0].copy_(scratch, non_blocking=True)
            torch.cuda.synchronize()
            floor = min(floor, max_over_ranks(time.perf_counter() - t0))

        # the same with a barrier between the two copies: in an update no byte can return before the
        # LAST rank's last byte has arrived (the coefficients need the global dot products), so on a
        # box whose ranks share PCIe bandwidth the unsynchronised figure above is not attainable
        floor_sync = 1e30
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            scratch.copy_(host[0], non_blocking=True)
            barrier()
            host[0].copy_(scratch, non_blocking=True)
            torch.cuda.synchronize()
            floor_sync = min(floor_sync, max_over_ranks(time.perf_counter() - t0))

        # pageable host memory: what an unmodified reference caller passes (src-C/nka_example.c:139, malloc)
        pageable = None
        if not args.no_pageable:
            pg = [np.empty(n_local, dtype=np.float64) for _ in range(2)]
            for a, hb in zip(pg, host):
                a[:] = hb.numpy()
            dtp = timed_host_calls([a.ctypes.data for a in pg])
            pageable = {"value": args.e2e_steps / dtp, "unit": "updates/s", "ms_per_step": 1e3 * dtp / args.e2e_steps,
                        "host_memory": "pageable (malloc), as src-C/nka_example.c:139 passes it"}
            del pg
        e2e = {"value": args.e2e_steps / dt, "unit": "updates/s",
               "h2d_bytes_per_step": n_local * 8 * world, "d2h_bytes_per_step": n_local * 8 * world,
               "steps": args.e2e_steps, "ms_per_step": 1e3 * dt / args.e2e_steps,
               "host_memory": "pinned (cudaHostAlloc)",
               "pcie_floor_ms": 1e3 * floor, "frac_of_pcie_floor": floor / (dt / args.e2e_steps),
               "pcie_floor_synced_ms": 1e3 * floor_sync, "frac_of_pcie_floor_synced": floor_sync / (dt / args.e2e_steps),
               "pcie_floor": "bare cudaMemcpyAsync H2D then D2H of each rank's slab, all ranks at once, best of 3, "
                             "max over ranks; synced = with a barrier between the two copies, as the update's global "
                             "reduction imposes",
               "pageable": pageable, "numa": numa,
               "api": "nka_accel_update(NKA, double* host_f) -- include/nonlinear_krylov_accelerator.h"}
        del host

    if rank == 0:
        sampler.stop()

    peak, peak_kind = measured_peak()
    sweep = None
    if rank == 0 and world == 1 and not args.no_sweep and n == N_FULL:
        acc.delete()
        acc = None
        sweep = mvec_sweep(n, pool, gen, stream, peak, torch)

    if rank == 0:
        ups = args.steps / (elapsed_ms * 1e-3)
        algo = algorithmic_bytes(n, m)
        gbs = ups * algo / 1e9
        # dominant kernel = pass B (f + M Z-column reads, 3 column writes).  Its share of the
        # algorithmic bytes: the M "v" columns + the three writes (f_out, new w, new v) = (M+3) n 8;
        # pass A's share: the M "w" columns + f = (M+1) n 8 (it streams exactly that: lazy last column).
        kb = kt["pass_b"]
        ka = kt["pass_a"]
        algo_b = (m + 3) * n_local * 8
        algo_a = (m + 1) * n_local * 8
        ms_b = kb["ms"] / max(kb["count"], 1)
        ms_a = ka["ms"] / max(ka["count"], 1)
        traffic = None
        traffic_how = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                with open(tpath) as fh:
                    tj = json.load(fh)
                key = "n%d_m%d_g%d" % (n, m, world)
                traffic = tj.get(key, {}).get("pass_b")
                traffic_how = "ncu --set full capture of this configuration (profiles/traffic.json)"
                if traffic is None:
                    # no capture of this rank count (ncu is a one-GPU tool here): the same kernel streams the same
                    # columns over the rank's slab, so the one-GPU capture scales with the slab length
                    one = tj.get("n%d_m%d_g1" % (n, m), {}).get("pass_b")
                    if one is not None:
                        traffic = one * (n_local / n)
                        traffic_how = "one-GPU ncu capture scaled by n_local / n (no ncu capture at %d ranks)" % world
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "kernel": "nka_pass_b<%d,2>" % m,
                    "achieved": algo_b / (ms_b * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": algo_b / (ms_b * 1e-3) / 1e9 / peak, "traffic": traffic,
                    "traffic_source": traffic_how if traffic is not None else None,
                    "peak_kind": "of " + peak_kind, "algorithmic_bytes_per_launch": algo_b,
                    "avg_launch_ms": ms_b, "launches_timed": kb["count"]}
        line = {
            "metric": "accel_update/sec", "value": ups, "unit": "updates/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "n_local": n_local,
            "comm_mode": comm_mode,
            "parity_probe": probe, "example_probe": ex_probe,
            "hbm_gbs": gbs, "roofline_frac_update": gbs / (peak * world),
            "roofline_update": {"algorithmic_bytes": algo, "formula": "(2M+4)*n*8", "achieved_gbs": gbs,
                                "peak_gbs": peak * world, "frac": gbs / (peak * world),
                                "peak_kind": "of " + peak_kind},
            "clocks": sampler.summary(t_wall0, t_wall1),
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "kernels": {
                "pass_a": {"avg_ms": ms_a, "algorithmic_gbs": algo_a / (ms_a * 1e-3) / 1e9,
                           "frac": algo_a / (ms_a * 1e-3) / 1e9 / peak, "count": ka["count"]},
                "pass_b": {"avg_ms": ms_b, "algorithmic_gbs": algo_b / (ms_b * 1e-3) / 1e9,
                           "frac": algo_b / (ms_b * 1e-3) / 1e9 / peak, "count": kb["count"]},
                "state": {"avg_ms": kt["state"]["ms"] / max(kt["state"]["count"], 1)},
                "materialise": {"avg_ms": kt["materialise"]["ms"] / max(kt["materialise"]["count"], 1)},
                "allreduce": {"avg_ms": kt["allreduce"]["ms"] / max(kt["allreduce"]["count"], 1)},
                "geometry": geom,
                "how": "CUDA event pair around every launch over %d further steps right after the timed region "
                       "(events between kernels disable their dependent-launch overlap)" % ksteps,
                "span_ms_per_step": span_ms / ksteps,
            },
            "num_vec": nvec_end, "state_error": st["error"],
            "mvec_sweep": sweep,
        }
        if not args.no_cpu_baseline and world == 1:
            del pool
            torch.cuda.empty_cache()
            line["cpu_baseline"] = cpu_reference_run(n, m, steps=5, warmup=0, budget_s=20.0, n_cap=1 << 24)
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    if acc is not None:
        acc.delete()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
