"""The batched accelerator on the GPU (-m gpu).

Every member of a BatchNKA must be bit-identical to a single NKA handle in the capacity shape that is fed
that member's calls: outputs and every field of state() after every call, whatever nbatch, the member's
index, the other members' data (NaN included) and the masks.  A single handle enters the capacity shape
for good with its first capture; here that is one captured set_vec_tol on a fresh handle.
"""
import hashlib
import json
import os
import resource
import subprocess
import sys

import numpy as np
import pytest

import scenarios as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))


def _torch():
    import torch
    return torch


def capacity_single(n, mvec, vtol, stream):
    """A single handle on `stream`, switched to the capacity shape by one captured set_vec_tol."""
    torch = _torch()
    from nka_b200 import NKA
    acc = NKA(n, mvec, vtol, stream=stream.cuda_stream)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        acc.set_vec_tol(vtol)
    return acc


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def assert_state_equal(sa, sb, ctx):
    assert sa.keys() == sb.keys()
    for k in sa:
        if isinstance(sa[k], np.ndarray) or isinstance(sa[k], float):
            assert np.array_equal(_bits(sa[k]), _bits(sb[k])), (ctx, k, sa[k], sb[k])
        else:
            assert sa[k] == sb[k], (ctx, k, sa[k], sb[k])


class Singles:
    """One capacity-shape single handle per member, each with f at the alignment the batch row has."""

    def __init__(self, nb, n, mvec, vtol, stream, aligned):
        torch = _torch()
        self.accs = [capacity_single(n, mvec, vtol, stream) for _ in range(nb)]
        self.off = 0 if aligned else 1
        self.buf = [torch.zeros(n + 2, dtype=torch.float64, device="cuda") for _ in range(nb)]
        self.f = [b[self.off:self.off + n] for b in self.buf]
        self.s = stream

    def update(self, b, x):
        torch = _torch()
        with torch.cuda.stream(self.s):
            self.f[b].copy_(torch.from_numpy(x))
            self.accs[b].accel_update(self.f[b])
            return self.f[b].cpu().numpy()

    def delete(self):
        for a in self.accs:
            a.delete()


def member_schedule(ops, nb, skip=True):
    """Member 0 runs the ops as listed; member b >= 1 starts b steps late and (skip) leaves out one
    mid-sequence update.  Returns, per global step, per member, the op or None."""
    sched = []
    per = []
    for b in range(nb):
        mine = list(ops)
        if b > 0 and skip:
            k = len(mine) // 2 + b - 2
            while mine[k][0] != "update":
                k += 1
            mine = mine[:k] + [None] + mine[k + 1:]      # None: the member sits this step out
        per.append([None] * b + mine)
    T = max(len(p) for p in per)
    for t in range(T):
        sched.append([p[t] if t < len(p) else None for p in per])
    return sched


def run_scenario(name, nb=4):
    """Drive a batch and nb capacity-shape singles through the scenario; returns a digest of every output
    and state (for comparing runs under different environment switches)."""
    torch = _torch()
    from nka_b200 import BatchNKA
    n, mvec, vtol, build = S.SCENARIOS[name]
    ops = build()
    rng = np.random.default_rng(4242)
    perms = [np.arange(n)] + [rng.permutation(n) for _ in range(nb - 1)]
    s = torch.cuda.Stream()
    batch = BatchNKA(nb, n, mvec, vtol, stream=s.cuda_stream)
    F = torch.zeros(nb, n, dtype=torch.float64, device="cuda")          # ldf = n: V = 2 iff n is even
    singles = Singles(nb, n, mvec, vtol, s, aligned=(n % 2 == 0))
    digest = hashlib.sha256()
    nan_row = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    for t, step in enumerate(member_schedule(ops, nb)):
        for kind in ("relax", "restart"):
            sel = [b for b in range(nb) if step[b] is not None and step[b][0] == kind]
            if sel:
                mask = torch.zeros(nb, dtype=torch.bool, device="cuda")
                mask[sel] = True
                with torch.cuda.stream(s):
                    getattr(batch, kind)(mask)
                for b in sel:
                    getattr(singles.accs[b], kind)()
        upd = [b for b in range(nb) if step[b] is not None and step[b][0] == "update"]
        if upd:
            active = torch.zeros(nb, dtype=torch.uint8, device="cuda")
            active[upd] = 1
            with torch.cuda.stream(s):
                for b in range(nb):
                    if b in upd:
                        F[b].copy_(torch.from_numpy(step[b][1][perms[b]]))
                    else:
                        F[b].copy_(nan_row)                 # an inactive row: never read, never written
                batch.accel_update(F, active)
                out = F.cpu().numpy()
            for b in range(nb):
                if b in upd:
                    want = singles.update(b, step[b][1][perms[b]])
                    assert np.array_equal(_bits(out[b]), _bits(want)), (name, t, b)
                    digest.update(_bits(out[b]).tobytes())
                else:
                    assert np.all(np.isnan(out[b])), (name, t, b)
        for b in range(nb):
            sb = batch.state(b)
            assert_state_equal(sb, singles.accs[b].state(), (name, t, b))
            digest.update(repr(sorted((k, _bits(v).tobytes() if isinstance(v, (np.ndarray, float)) else v)
                                      for k, v in sb.items())).encode())
    assert list(batch.num_vec()) == [a.num_vec() for a in singles.accs]
    assert batch.defined()
    batch.delete()
    singles.delete()
    return digest.hexdigest()


# ---------------------------------------------------------------------------------------------
# 1. bit identity to single handles, every scenario
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(S.SCENARIOS))
def test_every_member_is_bit_identical_to_a_capacity_shape_single(name):
    run_scenario(name)


_SUB = """
import sys, json
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_batch as T
out = {name: T.run_scenario(name) for name in %(names)r}
out["launches"] = T.launches_per_update()
print("RESULT " + json.dumps(out))
"""

LAZY_OFF = ["fullthendrop_n700_m32", "fullthendrop_n300_m4", "iid_n513_m32", "relax_restart_n96_m4", "mixed_n257_m5"]


def _no_core():
    resource.setrlimit(resource.RLIMIT_CORE, (0, 0))


def _run_sub(env_extra, names):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, "-c", _SUB % {"root": ROOT, "here": HERE, "names": names}], env=env,
                       capture_output=True, text=True, timeout=1800, preexec_fn=_no_core)
    assert r.returncode == 0, (env_extra, r.stdout[-3000:], r.stderr[-3000:])
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def launches_per_update():
    """Launches one batched update adds, at nbatch 1 and 4096."""
    torch = _torch()
    from nka_b200 import BatchNKA
    out = []
    for nb in (1, 4096):
        b = BatchNKA(nb, 64, 3, 0.01)
        F = torch.ones(nb, 64, dtype=torch.float64, device="cuda")
        c0 = b.launch_count()
        b.accel_update(F)
        out.append(b.launch_count() - c0)
        b.synchronize()
        b.delete()
    return out


def test_without_the_lazy_column():
    """NKA_LAZY_LAST=0: pass A at mvec + 1 columns (33 at mvec = 32), no fix-up launch."""
    res = _run_sub({"NKA_LAZY_LAST": "0"}, LAZY_OFF)
    assert res.pop("launches") == [3, 3]


def test_launch_count_is_four_whatever_nbatch():
    assert launches_per_update() == [4, 4]


def test_poisoned_allocations_give_the_same_bits():
    names = ["fullthendrop_n300_m4", "relax_restart_n96_m4", "zeros_n33_m3", "picard_n500_m5", "iid_n513_m32",
             "n3_m5_rankdef", "mixed_n257_m5"]
    clean = {name: run_scenario(name) for name in names}
    poisoned = _run_sub({"NKA_POISON_ALLOC": "1"}, names)
    poisoned.pop("launches")
    assert poisoned == clean


# ---------------------------------------------------------------------------------------------
# 2. independence of the member's index, the batch size and the neighbours
# ---------------------------------------------------------------------------------------------
def _member_run(nb, idx, neighbours, n=1000, mvec=10, ncall=16):
    torch = _torch()
    from nka_b200 import BatchNKA
    rng = np.random.default_rng(77)
    seq = [rng.uniform(-0.5, 0.5, n) for _ in range(ncall)]
    nrng = np.random.default_rng(1000 + nb + idx)
    s = torch.cuda.Stream()
    batch = BatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    F = torch.zeros(nb, n, dtype=torch.float64, device="cuda")
    active = torch.ones(nb, dtype=torch.bool, device="cuda")
    if neighbours == "inactive":
        active[:] = False
        active[idx] = True
    outs = []
    with torch.cuda.stream(s):
        for x in seq:
            if neighbours == "nan":
                F.fill_(float("nan"))
            elif neighbours == "random":
                F.copy_(torch.from_numpy(nrng.uniform(-1, 1, (nb, n))))
            F[idx].copy_(torch.from_numpy(x))
            batch.accel_update(F, active)
            outs.append(F[idx].cpu().numpy())
    st = batch.state(idx)
    batch.delete()
    return outs, st


def test_member_bits_do_not_depend_on_index_batch_size_or_neighbours():
    ref_out, ref_st = _member_run(1, 0, "none")
    for nb in (7, 300):
        for idx in (0, nb // 2, nb - 1):
            for nbr in ("random", "nan", "inactive"):
                outs, st = _member_run(nb, idx, nbr)
                for t, (a, b) in enumerate(zip(outs, ref_out)):
                    assert np.array_equal(_bits(a), _bits(b)), (nb, idx, nbr, t)
                assert_state_equal(st, ref_st, (nb, idx, nbr))


# ---------------------------------------------------------------------------------------------
# 3. large members: the SM-capped partition, the V = 2 tail, padded rows, V = 1 by misalignment
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("misalign", [False, True], ids=["f16B", "f8Boff"])
def test_large_members_match_singles(misalign):
    torch = _torch()
    from nka_b200 import BatchNKA
    n, mvec, nb, ncall = 2**20 + 3, 10, 3, 15
    ldf = n + 1                                           # padded and even: the 8-byte offset alone decides V
    rng = np.random.default_rng(2024)
    s = torch.cuda.Stream()
    batch = BatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    singles = Singles(nb, n, mvec, 0.01, s, aligned=not misalign)
    off = 1 if misalign else 0
    store = torch.full((nb * ldf + 2,), -7.25, dtype=torch.float64, device="cuda")
    F = store[off:off + nb * ldf].view(nb, ldf)[:, :n]
    assert F.stride(0) == ldf and (F.data_ptr() % 16 == 0) == (not misalign)
    for t in range(ncall):
        xs = [rng.uniform(-0.5, 0.5, n) * 0.9 ** t for _ in range(nb)]
        with torch.cuda.stream(s):
            for b in range(nb):
                F[b].copy_(torch.from_numpy(xs[b]))
            batch.accel_update(F)
            out = F.cpu().numpy()
            pad = store[off:off + nb * ldf].view(nb, ldf)[:, n:].cpu().numpy()
        assert np.all(pad == -7.25), t                    # the padding columns keep their bits
        for b in range(nb):
            want = singles.update(b, xs[b])
            assert np.array_equal(_bits(out[b]), _bits(want)), (t, b)
            assert_state_equal(batch.state(b), singles.accs[b].state(), (t, b))
    assert list(batch.num_vec()) == [mvec] * nb
    batch.delete()
    singles.delete()


# ---------------------------------------------------------------------------------------------
# 4. masks
# ---------------------------------------------------------------------------------------------
def test_masked_members_are_untouched():
    torch = _torch()
    from nka_b200 import BatchNKA
    nb, n, mvec = 5, 300, 4
    rng = np.random.default_rng(3)
    s = torch.cuda.Stream()
    batch = BatchNKA(nb, n, mvec, 0.1, stream=s.cuda_stream)
    F = torch.zeros(nb, n, dtype=torch.float64, device="cuda")
    with torch.cuda.stream(s):
        for _ in range(mvec + 2):
            F.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, (nb, n))))
            batch.accel_update(F)
    before = [batch.state(b) for b in range(nb)]
    chosen = [1, 0, 1, 0, 0]
    sel = torch.tensor(chosen, dtype=torch.uint8, device="cuda")
    row = np.full(n, np.nan)
    row[::3] = 1.5
    with torch.cuda.stream(s):
        F.copy_(torch.from_numpy(np.tile(row, (nb, 1))))
        batch.accel_update(F, torch.zeros(nb, dtype=torch.bool, device="cuda"))
        out = F.cpu().numpy()
    assert np.array_equal(_bits(out), _bits(np.tile(row, (nb, 1))))
    for b in range(nb):
        assert_state_equal(batch.state(b), before[b], ("no-op update", b))
    for op in ("relax", "restart"):
        prev = [batch.state(b) for b in range(nb)]
        with torch.cuda.stream(s):
            getattr(batch, op)(sel)
        for b in range(nb):
            now = batch.state(b)
            if chosen[b]:
                assert now["pending"] == 0, (op, b)
                if op == "restart":
                    assert now["first"] == -1, b
            else:
                assert_state_equal(now, prev[b], (op, b))
    nv = batch.num_vec()
    assert list(nv) == [0, mvec, 0, mvec, mvec]
    batch.delete()


# ---------------------------------------------------------------------------------------------
# 5. graphs
# ---------------------------------------------------------------------------------------------
def _picard_setup(nb, n, seed=15):
    torch = _torch()
    rng = np.random.default_rng(seed)
    X = torch.from_numpy(rng.uniform(0.1, 1.0, (nb, n))).cuda()
    Bv = torch.from_numpy(rng.uniform(0.5, 1.5, (nb, n))).cuda()
    return X, Bv


def _picard_iteration(batch, X, Bv, F, active, tol):
    """One batched fixed-point iteration: each member applies picard_like's map with its own b, the
    members whose residual norm is above tol are accelerated and step; the others sit still."""
    torch = _torch()
    G = Bv / (1.0 + 0.5 * torch.roll(X, 1, dims=1) + 0.3 * X * X)
    torch.sub(X, G, out=F)
    torch.gt(torch.linalg.vector_norm(F, dim=1), tol, out=active)
    batch.accel_update(F, active)
    X.sub_(F * active.unsqueeze(1))


def test_torch_graph_of_a_batched_fixed_point_iteration_matches_eager():
    torch = _torch()
    from nka_b200 import BatchNKA, NKAError
    nb, n, mvec, iters, tol = 33, 500, 5, 20, 1e-9
    s = torch.cuda.Stream()
    eager = BatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    capt = BatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    Xe, Bv = _picard_setup(nb, n)
    Xg = Xe.clone()
    Fe = torch.zeros(nb, n, dtype=torch.float64, device="cuda")
    Fg = torch.zeros_like(Fe)
    ae = torch.zeros(nb, dtype=torch.bool, device="cuda")
    ag = torch.zeros_like(ae)
    torch.cuda.synchronize()
    launches0 = capt.launch_count()
    g = torch.cuda.CUDAGraph()
    refused = {"num_vec": capt.num_vec, "defined": capt.defined, "state": lambda: capt.state(0),
               "set_stream": lambda: capt.set_stream(None), "synchronize": capt.synchronize}
    errors = {}
    with torch.cuda.graph(g, stream=s):
        capturing = capt.stream_capturing()
        _picard_iteration(capt, Xg, Bv, Fg, ag, tol)
        for name, call in refused.items():
            try:
                call()
                errors[name] = None
            except NKAError as exc:
                errors[name] = str(exc)
    assert capturing == 1 and capt.stream_capturing() == 0
    for name in refused:
        assert errors[name] and "cannot be captured in a CUDA graph" in errors[name], (name, errors[name])
    assert capt.launch_count() == launches0
    nactive = []
    with torch.cuda.stream(s):
        for it in range(iters):
            _picard_iteration(eager, Xe, Bv, Fe, ae, tol)
            g.replay()
            assert np.array_equal(_bits(Xe.cpu().numpy()), _bits(Xg.cpu().numpy())), it
            assert torch.equal(ae, ag), it
            nactive.append(int(ae.sum()))
    assert capt.launch_count() == launches0
    for b in range(nb):
        assert_state_equal(eager.state(b), capt.state(b), b)
    assert nactive[0] == nb
    eager.delete()
    capt.delete()


_REFUSED_C = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r)
import torch
from nka_b200 import _lib
lib = _lib.load()
s = torch.cuda.Stream()
h = lib.nka_batch_init(4, 100, 3, 0.01, -1, s.cuda_stream)
F = torch.zeros(4, 100, dtype=torch.float64, device="cuda")
out = (C.c_int * 4)()
view = _lib.StateView()
calls = {"nka_batch_num_vec": lambda: lib.nka_batch_num_vec(h, out),
         "nka_batch_defined": lambda: lib.nka_batch_defined(h),
         "nka_batch_get_state": lambda: lib.nka_batch_get_state(h, 0, C.byref(view)),
         "nka_batch_set_stream": lambda: lib.nka_batch_set_stream(h, None),
         "nka_batch_synchronize": lambda: lib.nka_batch_synchronize(h)}
torch.cuda.synchronize()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g, stream=s):
    lib.nka_batch_accel_update(h, F.data_ptr(), 100, None)
    calls[%(which)r]()
print("returned")
"""


def test_refused_calls_abort_with_their_message(tmp_path):
    names = ["nka_batch_num_vec", "nka_batch_defined", "nka_batch_get_state", "nka_batch_set_stream",
             "nka_batch_synchronize"]
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "which": w}], cwd=str(tmp_path),
                                 stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, preexec_fn=_no_core)
             for w in names}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert "nka_b200: " in err and (w + " cannot be captured in a CUDA graph") in err, (w, err)
