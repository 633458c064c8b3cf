"""Device-side fixed-point loops (BatchNKA.fixed_point_loop) on the GPU: one graph launch per solve must
give each member the bits of a host-driven loop (eager residual, BatchNKA.accel_update with the same
masks, X[b] += F[b]) whose stop decisions are read from the loop's own recorded norms."""
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


def assert_state_equal(sa, sb, ctx):
    assert sa.keys() == sb.keys()
    for k in sa:
        if isinstance(sa[k], np.ndarray) or isinstance(sa[k], float):
            assert np.array_equal(_bits(sa[k]), _bits(sb[k])), (ctx, k, sa[k], sb[k])
        else:
            assert sa[k] == sb[k], (ctx, k, sa[k], sb[k])


# member kinds: coefficients (a, h, e, nan) of F = a (B - X) - e X^3 + h lap(X) [+ sqrt(1 - X^2)]
FAST = (1.0, 0.0, 0.0, False)       # X1 = B up to rounding: converges at check 1
SLOW = (0.05, 0.2, 0.0, False)      # spectrum of the step map in [0.15, 0.95]: far from converged in 12 steps
NAN = (1.0, 0.0, 0.0, True)         # X1 = B + 1 leaves [-1, 1]: F is NaN at check 1


def _kind(rng):
    return (rng.uniform(0.3, 0.9), rng.uniform(0.0, 0.1), rng.uniform(0.0, 0.05), False)


class Problem:
    """nb members of length n; F at row stride ldf = n + 2, 16-byte aligned or 8 bytes off."""

    def __init__(self, kinds, n, seed, aligned=True):
        torch = _torch()
        nb = len(kinds)
        rng = np.random.default_rng(seed)
        self.n, self.nb = n, nb
        cuda = dict(dtype=torch.float64, device="cuda")
        self.a = torch.tensor([[k[0]] for k in kinds], **cuda)
        self.h = torch.tensor([[k[1]] for k in kinds], **cuda)
        self.e = torch.tensor([[k[2]] for k in kinds], **cuda)
        self.nan = torch.tensor([[k[3]] for k in kinds], dtype=torch.bool, device="cuda")
        self.B = torch.from_numpy(rng.uniform(-0.5, 0.5, (nb, n))).cuda()
        self.X = torch.zeros(nb, n, **cuda)
        ldf = n + 2
        off = 0 if aligned else 1
        self.fbuf = torch.zeros(nb * ldf + 2, **cuda)
        self.F = self.fbuf[off:off + nb * ldf].view(nb, ldf)[:, :n]

    def residual(self):
        X, F = self.X, self.F
        F.copy_(self.a * (self.B - X) - self.e * X * X * X)
        F[:, 1:-1] += self.h * (X[:, :-2] - 2.0 * X[:, 1:-1] + X[:, 2:])
        F.copy_(_torch().where(self.nan, F + _torch().sqrt(1.0 - X * X), F))


def host_loop(acc, p, hist, atol, rtol, maxit, check_norms=True):
    """The host-driven loop: decisions from the device loop's recorded norms, which are checked against
    numpy's norm of this loop's F and against the rule.  Returns (steps, status)."""
    torch = _torch()
    nb = p.nb
    k = np.zeros(nb, dtype=np.int32)
    st = np.full(nb, RUNNING, dtype=np.int32)
    r0 = np.zeros(nb)
    for _ in range(maxit + 1):
        p.residual()
        Fh = p.F.cpu().numpy()
        for b in np.nonzero(st == RUNNING)[0]:
            r = hist[k[b], b]
            if check_norms:
                want = np.linalg.norm(Fh[b])
                if np.isfinite(want):
                    assert abs(r - want) <= 1e-14 * max(want, 1e-300), (b, k[b], r, want)
                else:
                    assert not np.isfinite(r), (b, k[b], r)
            if k[b] == 0:
                r0[b] = r
            if not np.isfinite(r):
                st[b] = NONFINITE
            elif r < max(atol, rtol * r0[b]):
                st[b] = CONVERGED
            elif k[b] >= maxit:
                st[b] = MAXIT
        on = st == RUNNING
        assert np.all(np.isfinite(Fh[on])), "a non-finite row would reach the accelerator"
        mask = torch.from_numpy(on.astype(np.uint8)).cuda()
        acc.accel_update(p.F, mask)
        for b in np.nonzero(on)[0]:
            p.X[b] += p.F[b]
        k[on] += 1
        if not on.any():
            break
    torch.cuda.synchronize()
    return k, st


def _same(pa, pb, acca, accb, members, ctx):
    Xa, Xb = pa.X.cpu().numpy(), pb.X.cpu().numpy()
    Fa, Fb = pa.F.cpu().numpy(), pb.F.cpu().numpy()
    for b in members:
        assert np.array_equal(_bits(Xa[b]), _bits(Xb[b])), (ctx, "X", b)
        assert np.array_equal(_bits(Fa[b]), _bits(Fb[b])), (ctx, "F", b)
        assert_state_equal(acca.state(b), accb.state(b), (ctx, b))


def compare_with_host(kinds, n, mvec, aligned, atol=1e-8, rtol=1e-10, maxit=12, seed=3, relaunch=False):
    """Device loop against the host-driven loop; returns the device loop's results for further checks."""
    from nka_b200 import BatchNKA
    nb = len(kinds)
    pd, ph = Problem(kinds, n, seed, aligned), Problem(kinds, n, seed, aligned)
    dev, host = BatchNKA(nb, n, mvec, 0.01), BatchNKA(nb, n, mvec, 0.01)
    loop = dev.fixed_point_loop(pd.residual, pd.X, pd.F, atol=atol, rtol=rtol, maxit=maxit)
    out = []
    for launch in range(2 if relaunch else 1):
        if launch == 1:
            dev.restart()
            host.restart()
        c0 = dev.launch_count()
        loop.run()
        it, st, norm = loop.results()
        hist = loop.history()
        assert dev.launch_count() == c0
        kh, sh = host_loop(host, ph, hist, atol, rtol, maxit)
        ctx = (n, mvec, aligned, launch)
        assert np.array_equal(it, kh), (ctx, it, kh)
        assert np.array_equal(st, sh), (ctx, st, sh)
        for b in range(nb):
            assert np.array_equal(_bits(norm[b]), _bits(hist[it[b], b])), (ctx, b)
            assert np.all(np.isnan(hist[it[b] + 1:, b])), (ctx, b)
            assert np.all(~np.isnan(hist[:it[b] + 1, b]) | (st[b] == NONFINITE)), (ctx, b)
        _same(pd, ph, dev, host, range(nb), ctx)
        out.append((it, st, norm, hist))
    loop.destroy()
    dev.delete()
    host.delete()
    return out


# ---------------------------------------------------------------------------------------------
# 1./2. bit identity with the host-driven loop, every status
# ---------------------------------------------------------------------------------------------
def _kinds(nb, seed):
    rng = np.random.default_rng(seed)
    k = [_kind(rng) for _ in range(nb)]
    k[1], k[3], k[5] = FAST, NAN, SLOW
    return k


@pytest.mark.parametrize("mvec", [1, 5, 32])
@pytest.mark.parametrize("aligned", [True, False])
def test_device_loop_is_bit_identical_to_a_host_driven_loop(mvec, aligned):
    (it, st, norm, hist), = compare_with_host(_kinds(8, mvec), 1001, mvec, aligned)
    assert st[1] == CONVERGED and st[3] == NONFINITE and st[5] == MAXIT, st
    assert it[3] == 1 and it[5] == 12


def test_every_status_and_maxit_zero():
    from nka_b200 import BatchNKA
    torch = _torch()
    (it, st, norm, hist), = compare_with_host(_kinds(8, 2), 512, 5, True)
    assert set(st.tolist()) == {CONVERGED, MAXIT, NONFINITE}
    assert np.all(it[st == MAXIT] == 12)
    # maxit = 0: one residual evaluation, no step, X untouched
    p = Problem(_kinds(8, 2), 512, 3)
    acc = BatchNKA(8, 512, 5, 0.01)
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, atol=0.0, rtol=0.5, maxit=0)
    loop.run()
    it, st, norm = loop.results()
    assert np.all(it == 0) and np.all(st == MAXIT)
    assert torch.count_nonzero(p.X).item() == 0
    assert np.array_equal(loop.history().shape, (1, 8))
    assert acc.num_vec().tolist() == [0] * 8
    # atol = rtol = 0: every finite member takes exactly maxit steps
    loop2 = acc.fixed_point_loop(p.residual, p.X, p.F, atol=0.0, rtol=0.0, maxit=4)
    loop2.run()
    it, st, _ = loop2.results()
    assert it.tolist() == [4 if b != 3 else 1 for b in range(8)], it
    acc.delete()
    assert loop._h is None and loop2._h is None


# ---------------------------------------------------------------------------------------------
# 3. independence of nbatch, index and neighbours
# ---------------------------------------------------------------------------------------------
def _member(nb, idx, neighbours, n=1000, mvec=5):
    from nka_b200 import BatchNKA
    rng = np.random.default_rng(11)
    me = _kind(rng)
    kinds = []
    for b in range(nb):
        if b == idx:
            kinds.append(me)
        elif neighbours == "nan":
            kinds.append(NAN)
        elif neighbours == "converged":
            kinds.append(FAST)
        else:
            kinds.append(_kind(rng))
    p = Problem(kinds, n, 0)
    p.B[idx] = Problem([me], n, 5).B[0]
    acc = BatchNKA(nb, n, mvec, 0.01)
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, atol=1e-8, rtol=1e-10, maxit=15)
    loop.run()
    it, st, norm = loop.results()
    hist = loop.history()
    s = acc.state(idx)
    out = (int(it[idx]), int(st[idx]), _bits(hist[:, idx]).tobytes(), _bits(p.X[idx].cpu().numpy()).tobytes(),
           _bits(p.F[idx].cpu().numpy()).tobytes(), repr({k: (_bits(v).tobytes() if isinstance(v, (np.ndarray, float))
                                                               else v) for k, v in s.items()}))
    acc.delete()
    return out


def test_member_bits_do_not_depend_on_batch_size_index_or_neighbours():
    ref = _member(1, 0, "random")
    for nb, idx, nbrs in [(7, 3, "random"), (7, 6, "nan"), (7, 0, "converged"), (300, 217, "random"),
                          (300, 5, "nan")]:
        assert _member(nb, idx, nbrs) == ref, (nb, idx, nbrs)


# ---------------------------------------------------------------------------------------------
# 4. relaunch
# ---------------------------------------------------------------------------------------------
def test_second_launch_continues_and_eager_restart_matches_the_batch():
    from nka_b200 import BatchNKA
    kinds = _kinds(8, 9)
    p = Problem(kinds, 700, 4)
    acc = BatchNKA(8, 700, 5, 0.01)
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, atol=1e-8, rtol=1e-10, maxit=12)
    loop.run()
    it1, st1, norm1 = loop.results()
    loop.run()
    it2, st2, norm2 = loop.results()
    hist2 = loop.history()
    conv = st1 == CONVERGED
    assert conv.any()
    assert np.all(it2[conv] == 0) and np.all(st2[conv] == CONVERGED)
    assert np.array_equal(_bits(hist2[0, conv]), _bits(norm1[conv]))
    assert st2[3] == NONFINITE and it2[3] == 0
    acc.delete()
    # an eager restart between launches: the second launch still matches the host-driven loop
    compare_with_host(kinds, 700, 5, True, seed=4, relaunch=True)


# ---------------------------------------------------------------------------------------------
# 5. NKA_LAZY_LAST=0 and NKA_POISON_ALLOC=1
# ---------------------------------------------------------------------------------------------
def run_digest():
    (it, st, norm, hist), = compare_with_host(_kinds(8, 5), 1001, 5, False)
    return hashlib.sha256(it.tobytes() + st.tobytes() + _bits(hist).tobytes()).hexdigest()


_SUB = """
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_loop as T
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
    _run_sub({"NKA_LAZY_LAST": "0"})            # matches its own host-driven loop inside


# ---------------------------------------------------------------------------------------------
# 6./7. refusals, launch count
# ---------------------------------------------------------------------------------------------
def test_python_refuses_inside_a_capture():
    from nka_b200 import BatchNKA, NKAError
    torch = _torch()
    s = torch.cuda.Stream()
    p = Problem(_kinds(8, 1), 256, 0)
    acc = BatchNKA(8, 256, 3, 0.01, stream=s.cuda_stream)
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, maxit=5)
    c0 = acc.launch_count()
    s.wait_stream(torch.cuda.current_stream())
    loop.run()
    loop.results()
    assert acc.launch_count() == c0
    errors = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        p.residual()
        for name, call in (("run", loop.run), ("results", loop.results), ("history", loop.history)):
            try:
                call()
                errors[name] = None
            except NKAError as exc:
                errors[name] = str(exc)
    for name, msg in errors.items():
        assert msg and "cannot be captured" in msg, (name, msg)
    acc.delete()


_REFUSED_C = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import torch
import test_gpu_loop as T
from nka_b200 import _lib
lib = _lib.load()
s = torch.cuda.Stream()
p = T.Problem([T.FAST] * 4, 100, 0)
g = torch.cuda.CUDAGraph(keep_graph=True)
with torch.cuda.graph(g):
    p.residual()
h = lib.nka_batch_init(4, 100, 3, 0.01, -1, s.cuda_stream)
L = lib.nka_batch_loop_create(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102, 0.0, 1e-8, 5)
assert L
it, st, nrm = (C.c_int * 4)(), (C.c_int * 4)(), (C.c_double * 4)()
hist = (C.c_double * 24)()
calls = {"nka_batch_loop_launch": lambda: lib.nka_batch_loop_launch(L),
         "nka_batch_loop_results": lambda: lib.nka_batch_loop_results(L, it, st, nrm),
         "nka_batch_loop_history": lambda: lib.nka_batch_loop_history(L, hist)}
torch.cuda.synchronize()
g2 = torch.cuda.CUDAGraph()
with torch.cuda.graph(g2, stream=s):
    lib.nka_batch_accel_update(h, p.F.data_ptr(), 102, None)
    calls[%(which)r]()
print("returned")
"""


def test_c_entry_points_abort_inside_a_capture(tmp_path):
    names = ["nka_batch_loop_launch", "nka_batch_loop_results", "nka_batch_loop_history"]
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "here": HERE, "which": w}],
                                 cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                 preexec_fn=_no_core)
             for w in names}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert "nka_b200: " in err and (w + " cannot be captured in a CUDA graph") in err, (w, err)


# A residual graph with a host node, built with libcudart through ctypes (and, for the Python binding, a
# residual that queues a host function): CUDA refuses it in a conditional body; create returns NULL, no
# error is left behind, and the batch keeps working.
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
lib = _lib.load()
L = lib.nka_batch_loop_create(acc._h, graph, X.data_ptr(), 64, F.data_ptr(), 64, 0.0, 1e-8, 5)
print("C:", "NULL" if not L else "LOOP")
def residual():
    F.copy_(0.5 * X)
    rt.cudaLaunchHostFunc(C.c_void_p(torch.cuda.current_stream().cuda_stream), noop, None)
try:
    acc.fixed_point_loop(residual, X, F, maxit=5)
    print("PY: LOOP")
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
    assert "nka_b200: nka_batch_loop_create" in r.stderr, r.stderr
