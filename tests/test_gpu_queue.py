"""Device-side work queues (BatchNKA.fixed_point_queue) on the GPU.  Every problem's final iterate, steps,
status and norm must be bit for bit what the existing device loop (BatchNKA.fixed_point_loop) gives it on
a member just restarted with its X row set to the problem's initial guess, through the same slot_problem
and residual -- whatever slot it lands in, whatever nbatch and whatever ran in the slot before."""
import hashlib
import os
import resource
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
RUNNING, CONVERGED, MAXIT, NONFINITE = 0, 1, 2, 3


def _torch():
    import torch
    return torch


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


# problem kinds: coefficients (a, h, e, nan, x0_is_b) of F = a (B - X) - e X^3 + h lap(X) [+ sqrt(1 - X^2)]
FAST = (1.0, 0.0, 0.0, False, False)    # X1 = B up to rounding: converges at check 1
SLOW = (0.05, 0.2, 0.0, False, False)   # far from converged in maxit steps: MAXIT
NAN = (1.0, 0.0, 0.0, True, False)      # X1 = B + 1 leaves [-1, 1]: NONFINITE at check 1
ZERO = (1.0, 0.0, 0.0, False, True)     # X0 = B: F = 0 at check 0, CONVERGED on atol with 0 steps


def _kind(rng):
    """Contraction factors spread widely: a few steps to maxit."""
    return (rng.uniform(0.03, 0.95), rng.uniform(0.0, 0.2), rng.uniform(0.0, 0.05), False, False)


def kinds_for(nproblems, seed):
    rng = np.random.default_rng(seed)
    k = [_kind(rng) for _ in range(nproblems)]
    for p in range(nproblems):            # the special kinds early, so clean problems follow them in their slots
        if p % 7 == 1:
            k[p] = NAN
        elif p % 7 == 3:
            k[p] = ZERO
        elif p % 7 == 4:
            k[p] = SLOW
        elif p % 11 == 5:
            k[p] = FAST
    return k


class Problems:
    """nproblems problems of length n solved on nb slots.  X, X0 and every Xout from rows() have row stride
    n + 1.  With n odd that stride is even, every row is 16-byte aligned and the queue moves rows 16 bytes at
    a time plus a one-element tail; with n even it moves them 8 bytes at a time.  F has row stride n + 3,
    16-byte aligned or 8 bytes off."""

    def __init__(self, kinds, n, nb, seed, aligned=True):
        torch = _torch()
        P = len(kinds)
        rng = np.random.default_rng(seed)
        cuda = dict(dtype=torch.float64, device="cuda")
        self.n, self.nb, self.P = n, nb, P
        self.a = torch.tensor([[k[0]] for k in kinds], **cuda)
        self.h = torch.tensor([[k[1]] for k in kinds], **cuda)
        self.e = torch.tensor([[k[2]] for k in kinds], **cuda)
        self.nan = torch.tensor([[k[3]] for k in kinds], dtype=torch.bool, device="cuda")
        B = rng.uniform(-0.5, 0.5, (P, n))
        x0 = rng.uniform(-0.1, 0.1, (P, n))
        for p, k in enumerate(kinds):
            if k[4]:
                x0[p] = B[p]
        self.B = torch.from_numpy(B).cuda()
        self.X0 = self.rows()
        self.X0.copy_(torch.from_numpy(x0))
        self.X = torch.zeros(nb, n + 1, **cuda)[:, :n]
        ldf = n + 3
        off = 0 if aligned else 1
        self.fbuf = torch.zeros(nb * ldf + 2, **cuda)
        self.F = self.fbuf[off:off + nb * ldf].view(nb, ldf)[:, :n]
        self.slot = torch.full((nb,), -1, dtype=torch.int32, device="cuda")

    def rows(self):
        """Zeros [nproblems, n] at X0's row stride n + 1: an Xout laid out as X0 and X are."""
        torch = _torch()
        return torch.zeros(self.P, self.n + 1, dtype=torch.float64, device="cuda")[:, :self.n]

    def wide_rows(self):
        """Whether the queue moves this layout's rows 16 bytes at a time (X, X0, rows() 16-byte aligned)."""
        return all(T.data_ptr() % 16 == 0 and T.stride(0) % 2 == 0 for T in (self.X, self.X0, self.rows()))

    def residual(self):
        torch = _torch()
        X, F = self.X, self.F
        idx = self.slot.clamp(min=0).long()
        a, h, e = self.a.index_select(0, idx), self.h.index_select(0, idx), self.e.index_select(0, idx)
        F.copy_(a * (self.B.index_select(0, idx) - X) - e * X * X * X)
        F[:, 1:-1] += h * (X[:, :-2] - 2.0 * X[:, 1:-1] + X[:, 2:])
        F.copy_(torch.where(self.nan.index_select(0, idx), F + torch.sqrt(1.0 - X * X), F))


def reference(acc, pr, atol, rtol, maxit):
    """The existing device loop on the same batch, problems loaded nb at a time into restarted members
    through the same slot_problem and residual.  Returns (X rows, steps, status, norm) per problem."""
    torch = _torch()
    nb, P = pr.nb, pr.P
    loop = acc.fixed_point_loop(pr.residual, pr.X, pr.F, atol=atol, rtol=rtol, maxit=maxit)
    X = np.zeros((P, pr.n))
    it = np.zeros(P, dtype=np.int32)
    st = np.zeros(P, dtype=np.int32)
    norm = np.zeros(P)
    for g0 in range(0, P, nb):
        ids = np.arange(g0, min(g0 + nb, P))
        sp = np.full(nb, -1, dtype=np.int32)
        sp[:len(ids)] = ids
        pr.slot.copy_(torch.from_numpy(sp))
        pr.X.zero_()
        pr.X[:len(ids)] = pr.X0[torch.from_numpy(ids).cuda()]
        acc.restart()
        loop.run()
        i, s, r = loop.results()
        X[ids] = pr.X[:len(ids)].cpu().numpy()
        it[ids], st[ids], norm[ids] = i[:len(ids)], s[:len(ids)], r[:len(ids)]
    loop.destroy()
    return X, it, st, norm


def run_queue(acc, pr, atol, rtol, maxit, Xout=None, launches=1):
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, Xout, atol=atol, rtol=rtol, maxit=maxit)
    c0 = acc.launch_count()
    out = []
    for _ in range(launches):
        q.run()
        it, st, norm = q.results()
        assert acc.launch_count() == c0
        assert pr.slot.cpu().tolist() == [-1] * pr.nb
        out.append((q.Xout.cpu().numpy(), it, st, norm))
    q.destroy()
    return out


def assert_same(a, b, ctx):
    (Xa, ia, sa, na), (Xb, ib, sb, nb_) = a, b
    assert np.array_equal(ia, ib), (ctx, "steps", np.nonzero(ia != ib)[0][:10])
    assert np.array_equal(sa, sb), (ctx, "status", np.nonzero(sa != sb)[0][:10])
    assert np.array_equal(_bits(na), _bits(nb_)), (ctx, "norm")
    bad = np.nonzero(np.any(_bits(Xa) != _bits(Xb), axis=1))[0]
    assert bad.size == 0, (ctx, "X", bad[:10])


def compare(kinds, n, nb, mvec, aligned=True, atol=1e-8, rtol=1e-10, maxit=12, seed=3):
    from nka_b200 import BatchNKA
    pr = Problems(kinds, n, nb, seed, aligned)
    acc = BatchNKA(nb, n, mvec, 0.01)
    X0 = pr.X0.clone()
    Xout = pr.rows()
    assert Xout.stride(0) == pr.X0.stride(0) == pr.X.stride(0) == n + 1
    (got,) = run_queue(acc, pr, atol, rtol, maxit, Xout=Xout)
    assert _torch().equal(pr.X0, X0)               # a separate Xout leaves X0 alone, bit for bit
    assert np.array_equal(_bits(pr.X0.cpu().numpy()), _bits(X0.cpu().numpy()))
    want = reference(acc, pr, atol, rtol, maxit)
    assert_same(got, want, (n, nb, mvec, aligned))
    acc.delete()
    return got


# ---------------------------------------------------------------------------------------------
# bit identity with the device loop; every status; slots reused after NaN, MAXIT and check-0 problems
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mvec", [1, 5, 32])
@pytest.mark.parametrize("aligned", [True, False])
def test_queue_is_bit_identical_to_the_device_loop(mvec, aligned):
    assert Problems([FAST], 1001, 8, 0).wide_rows()        # n odd: 16-byte row moves with a one-element tail
    X, it, st, norm = compare(kinds_for(29, mvec), 1001, 8, mvec, aligned)     # 29 problems, 8 slots
    assert st[1] == NONFINITE and it[1] == 1
    assert st[3] == CONVERGED and it[3] == 0
    assert st[4] == MAXIT and it[4] == 12
    assert set(st.tolist()) == {CONVERGED, MAXIT, NONFINITE}
    assert len(set(it.tolist())) >= 4, it


def test_fewer_problems_than_slots_and_maxit_zero():
    assert not Problems([FAST], 300, 8, 0).wide_rows()     # n even: 8-byte row moves
    X, it, st, norm = compare(kinds_for(5, 1), 300, 8, 5)
    assert np.all(st != RUNNING)
    X, it, st, norm = compare(kinds_for(13, 2), 300, 4, 5, maxit=0)
    assert np.all(it == 0)
    assert set(st.tolist()) <= {CONVERGED, MAXIT, NONFINITE}


def test_problem_bits_do_not_depend_on_nbatch():
    from nka_b200 import BatchNKA
    kinds = kinds_for(40, 7)
    ref = None
    for nb in (1, 7, 300):
        pr = Problems(kinds, 257, nb, 5)
        acc = BatchNKA(nb, 257, 5, 0.01)
        assert pr.wide_rows()
        (got,) = run_queue(acc, pr, 1e-8, 1e-10, 15, Xout=pr.rows())   # X0 kept for the reference
        if nb == 7:
            assert_same(got, reference(acc, pr, 1e-8, 1e-10, 15), nb)
        acc.delete()
        if ref is None:
            ref = got
        else:
            assert_same(got, ref, nb)


def test_more_problems_than_the_member_cap():
    from nka_b200 import BatchNKA
    P = 200000
    rng = np.random.default_rng(1)
    kinds = [(rng.uniform(0.2, 0.95), rng.uniform(0.0, 0.2), rng.uniform(0.0, 0.05), False, False) for _ in range(P)]
    for p in range(0, P, 997):
        kinds[p] = NAN
    pr = Problems(kinds, 16, 4096, 2)
    acc = BatchNKA(4096, 16, 5, 0.01)
    (got,) = run_queue(acc, pr, 1e-10, 1e-12, 30, Xout=pr.rows())   # X0 kept for the reference
    assert np.all(got[2] != RUNNING)
    assert_same(got, reference(acc, pr, 1e-10, 1e-12, 30), "200000")
    acc.delete()


# ---------------------------------------------------------------------------------------------
# in place, relaunch, eager calls after a launch
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [500, 257])                # 8-byte row moves; 16-byte ones with a tail
def test_in_place_relaunch_and_eager_calls(n):
    from nka_b200 import BatchNKA
    kinds = kinds_for(23, 4)
    pr = Problems(kinds, n, 6, 8)
    assert pr.wide_rows() == (n % 2 == 1)
    acc = BatchNKA(6, n, 5, 0.01)
    X0 = pr.X0.clone()
    sep = pr.rows()
    (a, b) = run_queue(acc, pr, 1e-8, 1e-10, 12, Xout=sep, launches=2)
    assert_same(a, b, "relaunch, separate Xout")
    # in place: the same bits as a separate Xout
    (c, d) = run_queue(acc, pr, 1e-8, 1e-10, 12, launches=2)
    assert_same(a, c, "in place")
    conv = c[2] == CONVERGED
    assert conv.any()
    # the second launch continues from the solutions: converged problems stop at check 0 and keep their rows
    assert np.all(d[1][conv] == 0) and np.all(d[2][conv] == CONVERGED)
    assert np.array_equal(_bits(d[0][conv]), _bits(c[0][conv]))
    assert np.all(d[2][c[2] == NONFINITE] == NONFINITE)
    # eager batch calls after a launch, then a launch from the original guesses again
    pr.X0.copy_(X0)
    acc.accel_update(pr.F)
    acc.restart()
    acc.synchronize()
    (e,) = run_queue(acc, pr, 1e-8, 1e-10, 12, Xout=sep)
    assert_same(a, e, "after eager calls")
    assert_same(a, reference(acc, pr, 1e-8, 1e-10, 12), "against the device loop")
    acc.delete()


# ---------------------------------------------------------------------------------------------
# NKA_LAZY_LAST=0 and NKA_POISON_ALLOC=1
# ---------------------------------------------------------------------------------------------
def run_digest():
    X, it, st, norm = compare(kinds_for(17, 9), 1001, 5, 5, aligned=False)
    return hashlib.sha256(_bits(X).tobytes() + it.tobytes() + st.tobytes() + _bits(norm).tobytes()).hexdigest()


_SUB = """
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_queue as T
print("RESULT " + T.run_digest())
"""


def _no_core():
    resource.setrlimit(resource.RLIMIT_CORE, (0, 0))


def _run_sub(env_extra):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, "-c", _SUB % {"root": ROOT, "here": HERE}], env=env, capture_output=True,
                       text=True, timeout=1800, preexec_fn=_no_core)
    assert r.returncode == 0, (env_extra, r.stdout[-3000:], r.stderr[-3000:])
    return [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):]


def test_lazy_column_off_and_poisoned_allocations():
    clean = run_digest()
    assert _run_sub({"NKA_POISON_ALLOC": "1"}) == clean
    _run_sub({"NKA_LAZY_LAST": "0"})            # matches its own device loop inside


# ---------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------
def test_python_refuses_inside_a_capture():
    from nka_b200 import BatchNKA, NKAError
    torch = _torch()
    s = torch.cuda.Stream()
    pr = Problems(kinds_for(10, 1), 256, 4, 0)
    acc = BatchNKA(4, 256, 3, 0.01, stream=s.cuda_stream)
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, maxit=5)
    s.wait_stream(torch.cuda.current_stream())
    q.run()
    q.results()
    errors = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        pr.residual()
        for name, call in (("run", q.run), ("results", q.results)):
            try:
                call()
                errors[name] = None
            except NKAError as exc:
                errors[name] = str(exc)
    for name, msg in errors.items():
        assert msg and "cannot be captured" in msg, (name, msg)
    acc.delete()
    assert q._h is None


_REFUSED_C = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import torch
import test_gpu_queue as T
from nka_b200 import _lib
lib = _lib.load()
s = torch.cuda.Stream()
pr = T.Problems([T.FAST] * 6, 100, 4, 0)
g = torch.cuda.CUDAGraph(keep_graph=True)
with torch.cuda.graph(g):
    pr.residual()
h = lib.nka_batch_init(4, 100, 3, 0.01, -1, s.cuda_stream)
Q = lib.nka_batch_queue_create(h, g.raw_cuda_graph(), pr.X.data_ptr(), 101, pr.F.data_ptr(), 103, pr.slot.data_ptr(),
                               pr.X0.data_ptr(), 101, pr.X0.data_ptr(), 101, 6, 0.0, 1e-8, 5)
assert Q
it, st, nrm = (C.c_int * 6)(), (C.c_int * 6)(), (C.c_double * 6)()
calls = {"nka_batch_queue_launch": lambda: lib.nka_batch_queue_launch(Q),
         "nka_batch_queue_results": lambda: lib.nka_batch_queue_results(Q, it, st, nrm)}
torch.cuda.synchronize()
g2 = torch.cuda.CUDAGraph()
with torch.cuda.graph(g2, stream=s):
    lib.nka_batch_accel_update(h, pr.F.data_ptr(), 103, None)
    calls[%(which)r]()
print("returned")
"""


def test_c_entry_points_abort_inside_a_capture(tmp_path):
    names = ["nka_batch_queue_launch", "nka_batch_queue_results"]
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "here": HERE, "which": w}],
                                 cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                 preexec_fn=_no_core)
             for w in names}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert "nka_b200: " in err and (w + " cannot be captured in a CUDA graph") in err, (w, err)


# A residual graph with a host node: CUDA refuses it in a conditional body; create returns NULL (NKAError
# in Python), no error is left behind, and the batch keeps working.
_HOST_NODE = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r)
import torch
from nka_b200 import BatchNKA, NKAError, _lib
torch.zeros(1, device="cuda")
try:
    rt = C.CDLL("libcudart.so.12")
except OSError:
    rt = C.CDLL("/usr/local/cuda/lib64/libcudart.so")
HOSTFN = C.CFUNCTYPE(None, C.c_void_p)
noop = HOSTFN(lambda p: None)
class HostParams(C.Structure):
    _fields_ = [("fn", C.c_void_p), ("userData", C.c_void_p)]
graph, node = C.c_void_p(), C.c_void_p()
assert rt.cudaGraphCreate(C.byref(graph), 0) == 0
hp = HostParams(C.cast(noop, C.c_void_p), None)
assert rt.cudaGraphAddHostNode(C.byref(node), graph, None, C.c_size_t(0), C.byref(hp)) == 0
acc = BatchNKA(4, 64, 3, 0.01)
X = torch.zeros(4, 64, dtype=torch.float64, device="cuda")
F = torch.ones(4, 64, dtype=torch.float64, device="cuda")
X0 = torch.zeros(9, 64, dtype=torch.float64, device="cuda")
slot = torch.zeros(4, dtype=torch.int32, device="cuda")
lib = _lib.load()
Q = lib.nka_batch_queue_create(acc._h, graph, X.data_ptr(), 64, F.data_ptr(), 64, slot.data_ptr(), X0.data_ptr(), 64,
                               X0.data_ptr(), 64, 9, 0.0, 1e-8, 5)
print("C:", "NULL" if not Q else "QUEUE")
def residual():
    F.copy_(0.5 * X)
    rt.cudaLaunchHostFunc(C.c_void_p(torch.cuda.current_stream().cuda_stream), noop, None)
try:
    acc.fixed_point_queue(residual, X, F, slot, X0, maxit=5)
    print("PY: QUEUE")
except NKAError as exc:
    print("PY: NKAError", exc)
acc.accel_update(F)
acc.synchronize()
print("CLEAN", acc.defined())
"""


def test_a_residual_graph_cuda_refuses_gives_null_and_nkaerror(tmp_path):
    r = subprocess.run([sys.executable, "-c", _HOST_NODE % {"root": ROOT}], cwd=str(tmp_path), capture_output=True,
                       text=True, timeout=600, preexec_fn=_no_core)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert "C: NULL" in r.stdout and "PY: NKAError" in r.stdout, (r.stdout, r.stderr)
    assert "CLEAN True" in r.stdout, (r.stdout, r.stderr)
    assert "nka_b200: nka_batch_queue_create" in r.stderr, r.stderr
