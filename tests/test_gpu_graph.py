"""CUDA-graph capture of accel_update, relax and restart (-m gpu).

A replay runs on whatever the list holds by then, so a captured handle launches the capacity shape
(include/nka_b200.h, "CUDA graphs"): pass A at full width, the fix-up kernel always queued, pass B
at mvec pairs.  These tests drive the scenarios through graph replays and compare with the oracle
under the bars of test_gpu_parity.py: identical decisions on every call, corrections within
S.tolerances of the long-double arbiter.  In steady state a replay is bit-identical to an eager call.
"""
import os
import resource
import socket
import subprocess
import sys

import numpy as np
import pytest

import scenarios as S
from oracle import api

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch():
    import torch
    return torch


class Captured:
    """A fresh handle on a side stream with one graph each for update (captured at the empty list),
    relax and restart.  The update graph reads and writes `f`, a view `offset` doubles into a buffer
    that torch aligns to 512 bytes."""

    def __init__(self, n, mvec, vtol, offset=0):
        torch = _torch()
        from nka_b200 import NKA
        self.s = torch.cuda.Stream()
        self.acc = NKA(n, mvec, vtol, stream=self.s.cuda_stream)
        self.base = torch.zeros(n + 2, dtype=torch.float64, device="cuda")
        self.f = self.base[offset:offset + n]
        self.graphs = {}
        for op in ("update", "relax", "restart"):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.s):
                if op == "update":
                    self.acc.accel_update(self.f)
                else:
                    getattr(self.acc, op)()
            self.graphs[op] = g

    def replay(self, op):
        torch = _torch()
        with torch.cuda.stream(self.s):
            self.graphs[op].replay()

    def update(self, fin):
        torch = _torch()
        with torch.cuda.stream(self.s):
            self.f.copy_(torch.from_numpy(fin))
            self.graphs["update"].replay()
            return self.f.cpu().numpy()

    def eager_update(self, fin):
        torch = _torch()
        with torch.cuda.stream(self.s):
            self.f.copy_(torch.from_numpy(fin))
            self.acc.accel_update(self.f)
            return self.f.cpu().numpy()


def drive_against_oracle(acc, n, mvec, vtol, ops, update, relax, restart, tag):
    """Run `ops` through the callables; after every op the decisions equal the serial oracle's and
    every correction lies within S.tolerances of the long-double arbiter."""
    inputs = [op[1] for op in ops if op[0] == "update"]
    serial, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), ops)
    arbiter, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), ops)
    scales, tols = S.tolerances(serial, arbiter, inputs)
    orc = api.OracleNKA(n, mvec, vtol, dotmode=0)
    it = 0
    for k, op in enumerate(ops):
        if op[0] == "update":
            want = op[1].copy()
            orc.accel_update(want)
            got = update(it, op[1])
            if hasattr(acc, "state"):
                st = acc.state()
                assert st["error"] == 0, (tag, it)
                assert (st["ndrop_last"], bool(st["relaxed_last"]), bool(st["evicted_last"])) == \
                       (orc.ndrop_last(), orc.relaxed_last(), orc.evicted_last()), (tag, it)
            err = np.linalg.norm(got - arbiter[it]) / scales[it]
            assert err <= tols[it], (tag, it, err, tols[it])
            it += 1
        elif op[0] == "relax":
            orc.relax()
            relax()
        else:
            orc.restart()
            restart()
        assert acc.num_vec() == orc.num_vec(), (tag, k)
    assert acc.defined()


# ---------------------------------------------------------------------------------------------
# 1. every scenario through graphs captured on a fresh handle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(S.SCENARIOS))
def test_scenarios_replayed_from_graphs_match_oracle(name):
    """The update graph is captured at the empty list, so it must serve the first call, the growth
    of the list, the steady state, vtol drops that need the fix-up, relax and restart."""
    n, mvec, vtol, mk = S.SCENARIOS[name]
    c = Captured(n, mvec, vtol)
    drive_against_oracle(c.acc, n, mvec, vtol, mk(), lambda it, fin: c.update(fin),
                         lambda: c.replay("relax"), lambda: c.replay("restart"), name)
    c.acc.delete()


# ---------------------------------------------------------------------------------------------
# 2. steady state: a replay is an eager call, bit for bit
# ---------------------------------------------------------------------------------------------
def steady_state_bits(mvec, offset, n=3001):
    """Handles A and B take the same inputs eagerly until the list is full; then B captures one
    update and replays it for 2 mvec calls while A keeps calling eagerly."""
    torch = _torch()
    from nka_b200 import NKA
    rng = np.random.default_rng(1000 + mvec)
    fill = [rng.uniform(-0.5, 0.5, n) for _ in range(mvec + 3)]
    more = [rng.uniform(-0.5, 0.5, n) for _ in range(2 * mvec)]
    s = torch.cuda.Stream()
    a = NKA(n, mvec, 0.01, stream=s.cuda_stream)
    b = NKA(n, mvec, 0.01, stream=s.cuda_stream)
    ba = torch.zeros(n + 1, dtype=torch.float64, device="cuda")
    bb = torch.zeros(n + 1, dtype=torch.float64, device="cuda")
    fa, fb = ba[offset:offset + n], bb[offset:offset + n]
    assert (fa.data_ptr() % 16 == 0) == (offset == 0)

    def states_equal():
        sa, sb = a.state(), b.state()
        for key in ("ndrop_last", "evicted_last", "relaxed_last", "error", "first", "next", "pending", "chained"):
            assert sa[key] == sb[key], (mvec, offset, key)
        for key in ("c", "s", "h"):
            assert np.array_equal(sa[key], sb[key]), (mvec, offset, key)

    with torch.cuda.stream(s):
        for x in fill:
            for acc, f in ((a, fa), (b, fb)):
                f.copy_(torch.from_numpy(x))
                acc.accel_update(f)
            assert torch.equal(fa, fb)
        assert a.num_vec() == b.num_vec() == mvec
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            b.accel_update(fb)
        assert b.launch_geometry() == a.launch_geometry()
        for t, x in enumerate(more):
            fa.copy_(torch.from_numpy(x))
            a.accel_update(fa)
            fb.copy_(torch.from_numpy(x))
            g.replay()
            assert torch.equal(fa, fb), (mvec, offset, t)
            states_equal()
    a.delete()
    b.delete()


@pytest.mark.parametrize("offset", [0, 1], ids=["f16B", "f8Boff"])
@pytest.mark.parametrize("mvec", [1, 2, 5, 10, 32])
def test_steady_state_replay_bit_identical_to_eager(mvec, offset):
    steady_state_bits(mvec, offset)


def test_steady_state_replay_bit_identical_to_eager_without_lazy_column():
    """The same with NKA_LAZY_LAST=0: pass A streams all mvec + 1 columns in both."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r + '/tests'); import test_gpu_graph as T\n"
            "for m in (1, 2, 5, 10, 32):\n"
            "    for o in (0, 1): T.steady_state_bits(m, o)\n"
            "print('ok')" % (ROOT, ROOT))
    env = dict(os.environ, NKA_LAZY_LAST="0")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------
# 3. eager calls after replays: the host must not trust what it knew before the capture
# ---------------------------------------------------------------------------------------------
def _fill_drop_relax():
    ops = S.fill_then_collinear(300, 8, 10, 25)
    return ops[:12] + [("relax",)] + ops[12:15] + [("relax",), ("relax",)] + ops[15:]


@pytest.mark.parametrize("case", ["fill_drop_relax", "mixed_n257_m5"])
@pytest.mark.parametrize("k", [0, 3])
def test_eager_calls_after_replays_match_oracle(case, k):
    """Capture, replay k updates (k = 0: capture only), then go on eagerly on the same handle through
    vtol drops at a full list (the fix-up), relax and restart."""
    if case == "fill_drop_relax":
        n, mvec, vtol, ops = 300, 4, 0.1, _fill_drop_relax()
    else:
        n, mvec, vtol, mk = S.SCENARIOS[case]
        ops = mk()
    c = Captured(n, mvec, vtol)
    state = {"replays": 0}

    def update(it, fin):
        if it < k:
            state["replays"] += 1
            return c.update(fin)
        return c.eager_update(fin)

    def other(op):
        with _torch().cuda.stream(c.s):
            if state["replays"] < k:
                c.replay(op)
            else:
                getattr(c.acc, op)()

    drive_against_oracle(c.acc, n, mvec, vtol, ops, update, lambda: other("relax"), lambda: other("restart"),
                         "%s/k=%d" % (case, k))
    c.acc.delete()


# ---------------------------------------------------------------------------------------------
# 4. torch.cuda.graph around a whole iteration
# ---------------------------------------------------------------------------------------------
def test_torch_graph_of_a_fixed_point_iteration_matches_eager():
    """x <- x + f with f = NKA(g(x) - x): the torch op that forms f, accel_update and the update of x
    in one graph.  Replays follow the same iteration run eagerly, and each call's correction lies
    within the oracle tolerance of the reference on that call's input."""
    torch = _torch()
    from nka_b200 import NKA
    n, mvec, vtol, steps = 1000, 5, 0.01, 16
    rng = np.random.default_rng(31)
    b = torch.from_numpy(rng.uniform(0.5, 1.5, n)).cuda()
    x0 = torch.from_numpy(rng.uniform(0.1, 1.0, n)).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())

    def step(acc, x, f, fin):
        torch.sub(b / (1.0 + 0.5 * torch.roll(x, 1) + 0.3 * x * x), x, out=f)
        fin.copy_(f)
        acc.accel_update(f)
        x.add_(f)

    runs = {}
    with torch.cuda.stream(s):
        for kind in ("eager", "graph"):
            acc = NKA(n, mvec, vtol, stream=s.cuda_stream)
            x, f, fin = x0.clone(), torch.empty_like(x0), torch.empty_like(x0)
            if kind == "graph":
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=s):
                    step(acc, x, f, fin)
            rec = {"in": [], "out": [], "x": [], "nvec": []}
            for _ in range(steps):
                if kind == "graph":
                    g.replay()
                else:
                    step(acc, x, f, fin)
                rec["in"].append(fin.cpu().numpy())
                rec["out"].append(f.cpu().numpy())
                rec["x"].append(x.cpu().numpy())
                rec["nvec"].append(acc.num_vec())
            acc.delete()
            runs[kind] = rec
    for kind, rec in runs.items():
        ops = [("update", fi) for fi in rec["in"]]
        serial, nv = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), ops)
        arbiter, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), ops)
        scales, tols = S.tolerances(serial, arbiter, rec["in"])
        assert rec["nvec"] == nv, kind
        for t in range(steps):
            assert np.linalg.norm(rec["out"][t] - arbiter[t]) / scales[t] <= tols[t], (kind, t)
    assert runs["graph"]["nvec"] == runs["eager"]["nvec"]
    for t in range(steps):
        xe, xg = runs["eager"]["x"][t], runs["graph"]["x"][t]
        assert np.linalg.norm(xg - xe) <= 1e-9 * np.linalg.norm(xe), t


# ---------------------------------------------------------------------------------------------
# 5. the gpu_vector flavour
# ---------------------------------------------------------------------------------------------
def test_vector_flavour_accel_update_captures():
    torch = _torch()
    from nka_b200.vector import GpuVector, VectorNKA
    name = "picard_n500_m5_v2"
    n, mvec, vtol, mk = S.SCENARIOS[name]
    s = torch.cuda.Stream()
    f = GpuVector(n, stream=s.cuda_stream)
    acc = VectorNKA().init(f, mvec, vtol)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        acc.accel_update(f)

    def update(it, fin):
        f.set(fin)
        with torch.cuda.stream(s):
            g.replay()
        return f.get()

    drive_against_oracle(acc, n, mvec, vtol, mk(), update, acc.relax, acc.restart, name)
    acc.delete()


# ---------------------------------------------------------------------------------------------
# 6. refusals, and what a capture leaves untouched
# ---------------------------------------------------------------------------------------------
_REFUSED_C = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r)
import torch
from nka_b200 import NKA, _lib
from nka_b200.nka import DP_FUNC
lib = _lib.load()
s = torch.cuda.Stream()
acc = NKA(64, 3, 0.01, stream=s.cuda_stream)
h = acc._h
d = torch.zeros(64, dtype=torch.float64, device="cuda")
host = (C.c_double * 64)()
view = _lib.StateView()
ms, cnt = (C.c_double * 5)(), (C.c_ulonglong * 5)()
cb = DP_FUNC(lambda m, x, y: x[0] * y[0])
which = %(which)r
if which == "dp":
    lib.nka_set_dot_prod(h, C.cast(cb, C.c_void_p))
calls = {
    "nka_accel_update_host": lambda: lib.nka_accel_update_host(h, C.addressof(host)),
    "nka_accel_update with a host pointer": lambda: lib.nka_accel_update(h, C.addressof(host)),
    "dp": lambda: lib.nka_accel_update_dev(h, d.data_ptr()),
    "nka_num_vec": lambda: lib.nka_num_vec(h),
    "nka_defined": lambda: lib.nka_defined(h),
    "nka_get_state": lambda: lib.nka_get_state(h, C.byref(view)),
    "nka_timing_read": lambda: lib.nka_timing_read(h, ms, cnt),
    "nka_timing_reset": lambda: lib.nka_timing_reset(h),
    "nka_timing_enable": lambda: lib.nka_timing_enable(h, 1),
    "nka_set_stream": lambda: lib.nka_set_stream(h, None),
    "nka_synchronize": lambda: lib.nka_synchronize(h),
    "nka_set_dot_prod": lambda: lib.nka_set_dot_prod(h, None),
    "nka_comm_init": lambda: lib.nka_comm_init(h, 2, 0, C.create_string_buffer(128)),
    "nka_comm_adopt": lambda: lib.nka_comm_adopt(h, None, 2, 0),
}
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g, stream=s):
    assert lib.nka_stream_capturing(h) == 1
    calls[which]()
print("returned")
"""

_REFUSED = ["nka_accel_update_host", "nka_accel_update with a host pointer", "dp", "nka_num_vec", "nka_defined",
            "nka_get_state", "nka_timing_read", "nka_timing_reset", "nka_timing_enable", "nka_set_stream",
            "nka_synchronize", "nka_set_dot_prod", "nka_comm_init", "nka_comm_adopt"]


def _no_core():
    resource.setrlimit(resource.RLIMIT_CORE, (0, 0))


def test_refused_calls_abort_with_their_message(tmp_path):
    """Through the C-ABI each refused call stops the process before it reaches the stream, with a
    message that names it (one process per call, run side by side)."""
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "which": w}], cwd=str(tmp_path),
                                 stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, preexec_fn=_no_core)
             for w in _REFUSED}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        name = "nka_accel_update" if w == "dp" else w
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert "nka_b200: " in err and (name + " cannot be captured in a CUDA graph") in err, (w, err)
        if w == "dp":
            assert "host callback" in err, err


def test_refused_calls_raise_in_python_and_a_capture_runs_nothing():
    torch = _torch()
    from nka_b200 import NKA, NKAError
    from nka_b200.nka import DP_FUNC
    n, mvec = 512, 3
    rng = np.random.default_rng(5)
    s = torch.cuda.Stream()
    acc = NKA(n, mvec, 0.01, stream=s.cuda_stream)
    hooked = NKA(n, mvec, 0.01, stream=s.cuda_stream)
    cb = DP_FUNC(lambda m, x, y: x[0] * y[0])
    hooked.set_dot_prod(cb)
    d = torch.zeros(n, dtype=torch.float64, device="cuda")
    d2 = torch.zeros(n, dtype=torch.float64, device="cuda")
    acc.timing_enable(True)
    with torch.cuda.stream(s):
        for _ in range(3):
            d.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, n)))
            acc.accel_update(d)
    timing0 = acc.timing_read()
    launches0 = acc.launch_count()
    assert acc.stream_capturing() == 0
    refused = {
        "accel_update(numpy)": lambda: acc.accel_update(np.zeros(n)),
        "accel_update(cpu tensor)": lambda: acc.accel_update(torch.zeros(n, dtype=torch.float64)),
        "accel_update with dp": lambda: hooked.accel_update(d2),
        "num_vec": acc.num_vec, "defined": acc.defined, "state": acc.state,
        "timing_read": acc.timing_read, "timing_reset": acc.timing_reset,
        "timing_enable": lambda: acc.timing_enable(False),
        "set_stream": lambda: acc.set_stream(None), "synchronize": acc.synchronize,
        "set_dot_prod": lambda: acc.set_dot_prod(None),
        "comm_init": lambda: acc.comm_init(2, 0, b"\0" * 128),
    }
    errors = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        capturing = acc.stream_capturing()
        acc.accel_update(d)
        for name, call in refused.items():
            try:
                call()
                errors[name] = None
            except NKAError as exc:
                errors[name] = str(exc)
    assert capturing == 1
    assert acc.stream_capturing() == 0
    for name in refused:
        assert errors[name] and "cannot be captured in a CUDA graph" in errors[name], (name, errors[name])
    assert acc.launch_count() == launches0
    with torch.cuda.stream(s):
        for _ in range(4):
            d.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, n)))
            g.replay()
    assert acc.launch_count() == launches0
    assert acc.timing_read() == timing0
    assert acc.num_vec() == mvec
    with torch.cuda.stream(s):
        acc.accel_update(d)
    assert acc.launch_count() > launches0
    t1 = acc.timing_read()
    assert t1["pass_a"]["count"] == timing0["pass_a"]["count"] + 1
    assert t1["pass_b"]["count"] == timing0["pass_b"]["count"] + 1
    acc.delete()
    hooked.delete()


# ---------------------------------------------------------------------------------------------
# 7. two GPUs: peer and NCCL reductions inside the graph
# ---------------------------------------------------------------------------------------------
def _free_port():
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    return port


def _multi_worker(rank, world, port, name, mode, q):
    os.environ["NKA_PEER_REDUCE"] = "1" if mode == "peer" else "0"
    os.environ["NKA_PEER_TIMEOUT_S"] = "30"
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scenarios as S_
    from nka_b200.distributed import distributed_nka
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        n, mvec, vtol, mk = S_.SCENARIOS[name]
        s = torch.cuda.Stream()
        acc, lo, hi = distributed_nka(n, mvec, vtol, device=rank, stream=s.cuda_stream)
        f = torch.zeros(hi - lo, dtype=torch.float64, device="cuda")
        graphs = {}
        for op in ("update", "relax", "restart"):          # every rank: the same graphs, in the same order
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                if op == "update":
                    acc.accel_update(f)
                else:
                    getattr(acc, op)()
            graphs[op] = g
        outs, nvec, decisions = [], [], []
        with torch.cuda.stream(s):
            for op in mk():
                if op[0] == "update":
                    f.copy_(torch.from_numpy(np.ascontiguousarray(op[1][lo:hi])))
                graphs[op[0]].replay()
                if op[0] == "update":
                    outs.append(f.cpu().numpy())
                    st = acc.state()
                    decisions.append((st["ndrop_last"], st["relaxed_last"], st["evicted_last"], st["error"]))
                nvec.append(acc.num_vec())
        q.put((rank, {"outs": outs, "nvec": nvec, "decisions": decisions, "comm_mode": acc.comm_mode()}))
        acc.delete()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name", ["picard_n500_m5_v2", "relax_restart_n96_m4", "fullthendrop_n300_m4"])
@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_two_gpu_captured_slabs_match_serial_oracle(name, mode):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_multi_worker, args=(r, world, port, name, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=180) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n, mvec, vtol, mk = S.SCENARIOS[name]
    ops = mk()
    inputs = [op[1] for op in ops if op[0] == "update"]
    serial, nv_ref = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), ops)
    arbiter, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), ops)
    scales, tols = S.tolerances(serial, arbiter, inputs)
    orc = api.OracleNKA(n, mvec, vtol, dotmode=0)
    want_decisions = []
    for op in ops:
        if op[0] == "update":
            orc.accel_update(op[1].copy())
            want_decisions.append((orc.ndrop_last(), int(orc.relaxed_last()), int(orc.evicted_last()), 0))
        elif op[0] == "relax":
            orc.relax()
        else:
            orc.restart()
    assert got[0]["comm_mode"] == got[1]["comm_mode"] == mode
    assert got[0]["nvec"] == got[1]["nvec"] == nv_ref
    assert got[0]["decisions"] == got[1]["decisions"] == want_decisions
    for t in range(len(inputs)):
        joined = np.concatenate([got[0]["outs"][t], got[1]["outs"][t]])
        assert np.linalg.norm(joined - arbiter[t]) / scales[t] <= tols[t], (name, t)
