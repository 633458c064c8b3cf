"""Per-problem stopping tests (the _stop creates; fixed_point_loop / fixed_point_queue with tensor atol, rtol,
maxit, a scale and dtol) on the GPU.  Uniform arrays must give the scalar API's bits; a scale of 1.0 the
unscaled bits; a scale's bits must not depend on where its rows sit; per-member rules must match a
host-driven loop replaying the rule; a queue's problems must match the loop on a just-restarted member
carrying the problem's entries, at any nbatch."""
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
sys.path.insert(0, HERE)
RUNNING, CONVERGED, MAXIT, NONFINITE, DIVERGED = 0, 1, 2, 3, 4

import test_gpu_loop as TL        # noqa: E402
import test_gpu_queue as TQ       # noqa: E402
from test_gpu_loop import _bits   # noqa: E402


def _torch():
    import torch
    return torch


def _cuda(a, dtype=None):
    torch = _torch()
    return torch.tensor(np.asarray(a), dtype=dtype or torch.float64, device="cuda")


# ---------------------------------------------------------------------------------------------
# fixtures: a member family with a divergent kind, and scale rows placed aligned or 8 bytes off
# ---------------------------------------------------------------------------------------------
EXP = "exp"      # F = 2 exp(X) from X = 0: r1 = e^2 r0 (scaled by 1/(1+|X|): r1 = e^2/3 r0), DIVERGED at dtol 2


def _even_ld(n):
    """An even row stride >= n + 2: with a 16-byte aligned base every row is 16-byte aligned."""
    return n + 2 + n % 2


def access_width(T):
    """The access width the check takes for rows T: 2 (16 bytes) when every row is 16-byte aligned."""
    return 2 if T.data_ptr() % 16 == 0 and T.stride(0) % 2 == 0 else 1


class Problem(TL.Problem):
    """test_gpu_loop's members plus EXP members.  F (unlike test_gpu_loop's, whose stride n + 2 is odd for odd
    n) and S have even row strides, so `aligned` / `scale_aligned` pick the 16-byte paths (V = 2, a 16-byte
    scale) and 8 bytes off the 8-byte ones, at odd n too.  rewrite: the residual writes S = 1 / (1 + |X|)
    from X in every evaluation."""

    def __init__(self, kinds, n, seed, aligned=True, scale_aligned=True, rewrite=False, scale=None):
        torch = _torch()
        exp = [k == EXP for k in kinds]
        super().__init__([TL.FAST if k == EXP else k for k in kinds], n, seed, aligned)
        self.exp = torch.tensor([[e] for e in exp], dtype=torch.bool, device="cuda")
        ld = _even_ld(n)
        off = 0 if aligned else 1
        self.fbuf = torch.zeros(self.nb * ld + 2, dtype=torch.float64, device="cuda")
        self.F = self.fbuf[off:off + self.nb * ld].view(self.nb, ld)[:, :n]
        off = 0 if scale_aligned else 1
        self.sbuf = torch.zeros(self.nb * ld + 2, dtype=torch.float64, device="cuda")
        self.S = self.sbuf[off:off + self.nb * ld].view(self.nb, ld)[:, :n]
        self.S.copy_(scale if scale is not None else torch.ones(self.nb, n, dtype=torch.float64))
        self.rewrite = rewrite
        assert access_width(self.F) == (2 if aligned else 1)
        assert access_width(self.S) == (2 if scale_aligned else 1)

    def residual(self):
        torch = _torch()
        super().residual()
        self.F.copy_(torch.where(self.exp, 2.0 * torch.exp(self.X), self.F))
        if self.rewrite:
            self.S.copy_(1.0 / (1.0 + self.X.abs()))


def _kinds(nb, seed):
    k = TL._kinds(nb, seed)
    k[6] = EXP
    return k


def loop_stop_c(acc, p, atol, rtol, maxit, dtol, bound, scale=None):
    """A FixedPointLoop built through the C entry point nka_batch_loop_create_stop (entries the Python binding
    refuses, such as maxit entries above the bound or below 0, included)."""
    from nka_b200 import _lib
    from nka_b200.batch import FixedPointLoop, _capture
    st = _lib.StopTest()
    st.atol, st.rtol, st.dtol, st.maxit = 0.0, 0.0, dtol, bound
    st.atol_dev, st.rtol_dev, st.maxit_dev = atol.data_ptr(), rtol.data_ptr(), maxit.data_ptr()
    if scale is not None:
        st.scale_dev, st.ldscale = scale.data_ptr(), scale.stride(0)
    graph = _capture(p.residual, p.F.device)
    loop = FixedPointLoop(acc, graph, p.X, p.F, bound)
    loop._stop = (atol, rtol, maxit, scale)
    loop._h = acc._lib.nka_batch_loop_create_stop(acc._h, graph.raw_cuda_graph(), p.X.data_ptr(), p.X.stride(0),
                                                  p.F.data_ptr(), p.F.stride(0), st)
    assert loop._h
    acc._loops.add(loop)
    return loop


def host_loop(acc, p, hist, atol, rtol, maxit, dtol, bound, scaled):
    """test_gpu_loop.host_loop with per-member atol, rtol and (clamped) maxit, a scale and dtol: decisions
    from the device loop's recorded norms, which are checked against numpy's ||s_b * F_b||."""
    torch = _torch()
    nb = p.nb
    k = np.zeros(nb, dtype=np.int32)
    st = np.full(nb, RUNNING, dtype=np.int32)
    r0 = np.zeros(nb)
    for _ in range(bound + 1):
        p.residual()
        Fh = p.F.cpu().numpy()
        Sh = p.S.cpu().numpy() if scaled else np.ones_like(Fh)
        for b in np.nonzero(st == RUNNING)[0]:
            r = hist[k[b], b]
            want = np.linalg.norm(Sh[b] * Fh[b])
            if np.isfinite(want):
                assert abs(r - want) <= 1e-14 * max(want, 1e-300), (b, k[b], r, want)
            else:
                assert not np.isfinite(r), (b, k[b], r)
            if k[b] == 0:
                r0[b] = r
            if not np.isfinite(r):
                st[b] = NONFINITE
            elif r < max(atol[b], rtol[b] * r0[b]):
                st[b] = CONVERGED
            elif dtol > 0 and r > dtol * r0[b]:
                st[b] = DIVERGED
            elif k[b] >= maxit[b]:
                st[b] = MAXIT
        on = st == RUNNING
        acc.accel_update(p.F, torch.from_numpy(on.astype(np.uint8)).cuda())
        for b in np.nonzero(on)[0]:
            p.X[b] += p.F[b]
        k[on] += 1
        if not on.any():
            break
    torch.cuda.synchronize()
    return k, st


def _outcome(acc, p, loop, nb):
    it, st, norm = loop.results()
    X, F = p.X.cpu().numpy(), p.F.cpu().numpy()
    states = [acc.state(b) for b in range(nb)]
    return it, st, norm, loop.history(), X, F, states


def assert_outcomes_equal(a, b, ctx):
    for name, x, y in zip(("steps", "status"), a[:2], b[:2]):
        assert np.array_equal(x, y), (ctx, name, x, y)
    for name, x, y in zip(("norm", "history", "X", "F"), a[2:6], b[2:6]):
        assert x.shape == y.shape and np.array_equal(_bits(x), _bits(y)), (ctx, name)
    for m, (sa, sb) in enumerate(zip(a[6], b[6])):
        TL.assert_state_equal(sa, sb, (ctx, m))


# ---------------------------------------------------------------------------------------------
# 1. uniform arrays give the scalar API's bits (loop and queue)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mvec", [1, 5, 32])
@pytest.mark.parametrize("aligned", [True, False])
def test_uniform_arrays_are_the_scalar_apis_bits(mvec, aligned):
    from nka_b200 import BatchNKA
    torch = _torch()
    kinds, n, nb = TL._kinds(8, mvec), 1001, 8
    atol, rtol, maxit = 1e-8, 1e-10, 12
    outs = []
    for arrays in (False, True):
        p = Problem(kinds, n, 3, aligned)             # F at V = 2 when aligned, V = 1 when 8 bytes off
        acc = BatchNKA(nb, n, mvec, 0.01)
        if arrays:
            kw = dict(atol=torch.full((nb,), atol, dtype=torch.float64, device="cuda"),
                      rtol=torch.full((nb,), rtol, dtype=torch.float64, device="cuda"),
                      maxit=torch.full((nb,), maxit, dtype=torch.int32, device="cuda"))
        else:
            kw = dict(atol=atol, rtol=rtol, maxit=maxit)
        loop = acc.fixed_point_loop(p.residual, p.X, p.F, **kw)
        loop.run()
        outs.append(_outcome(acc, p, loop, nb))
        acc.delete()
    assert set(outs[0][1].tolist()) == {CONVERGED, MAXIT, NONFINITE}
    assert_outcomes_equal(outs[0], outs[1], (mvec, aligned))
    # the queue: every problem's Xout row, steps, status and norm
    qk = TQ.kinds_for(40, mvec)
    got = []
    for arrays in (False, True):
        pr = TQ.Problems(qk, 257, 7, 5, aligned)
        assert access_width(pr.F) == (2 if aligned else 1)
        acc = BatchNKA(7, 257, mvec, 0.01)
        if arrays:
            kw = dict(atol=torch.full((40,), atol, dtype=torch.float64, device="cuda"),
                      rtol=torch.full((40,), rtol, dtype=torch.float64, device="cuda"),
                      maxit=torch.full((40,), maxit, dtype=torch.int32, device="cuda"))
        else:
            kw = dict(atol=atol, rtol=rtol, maxit=maxit)
        q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, pr.rows(), **kw)
        q.run()
        it, st, norm = q.results()
        got.append((q.Xout.cpu().numpy(), it, st, norm))
        acc.delete()
    TQ.assert_same(got[0], got[1], ("queue", mvec, aligned))


# ---------------------------------------------------------------------------------------------
# 2. scale: 1.0 is the unscaled norm; the bits do not depend on where the scale rows sit.  With F aligned
#    (V = 2) the aligned and 8-bytes-off scale rows take the 16-byte and the 8-byte scale loads; n = 1001
#    is odd, so the tail element is scaled too.
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("aligned", [True, False])
def test_unit_scale_is_unscaled_and_scale_placement_does_not_matter(aligned):
    from nka_b200 import BatchNKA
    torch = _torch()
    kinds, n, nb, mvec = TL._kinds(8, 4), 1001, 8, 5

    def run(scale_kind, scale_aligned=True):
        w = torch.from_numpy(np.random.default_rng(2).uniform(0.5, 20.0, (nb, n)))
        p = Problem(kinds, n, 3, aligned, scale_aligned, scale=w if scale_kind == "w" else None)
        acc = BatchNKA(nb, n, mvec, 0.01)
        scale = None if scale_kind == "none" else p.S
        loop = acc.fixed_point_loop(p.residual, p.X, p.F, atol=1e-8, rtol=1e-10, maxit=12, scale=scale)
        loop.run()
        out = _outcome(acc, p, loop, nb)
        acc.delete()
        return out

    plain = run("none")
    assert_outcomes_equal(plain, run("ones", True), ("ones aligned", aligned))
    assert_outcomes_equal(plain, run("ones", False), ("ones off", aligned))
    wa = run("w", True)
    assert_outcomes_equal(wa, run("w", False), ("weights", aligned))
    assert not np.array_equal(_bits(wa[3][0]), _bits(plain[3][0]))       # the weights did change the norms


# ---------------------------------------------------------------------------------------------
# 3. per-member rules against a host-driven loop: every status, clamped maxit entries, a rewritten scale
# ---------------------------------------------------------------------------------------------
def compare_with_host(n=1001, mvec=5, aligned=True, rewrite=True, scale_aligned=True, seed=3):
    from nka_b200 import BatchNKA
    torch = _torch()
    nb = 9
    kinds = _kinds(nb, 7)
    kinds[8] = TL.SLOW
    bound, dtol = 12, 2.0
    atol = np.array([1e-8, 1e-8, 1e-6, 1e-8, 1e-4, 0.0, 1e-8, 1e-3, 0.0])
    rtol = np.array([1e-10, 0.0, 1e-3, 1e-10, 1e-10, 0.0, 1e-10, 1e-2, 0.0])
    # member 5 (SLOW, atol = rtol = 0) runs to the bound: its entry 40 must be clamped to 12; also below 0, 0
    maxit_dev = np.array([12, 40, 7, 12, -3, 40, 12, 3, 0], dtype=np.int32)
    maxit = np.minimum(np.maximum(maxit_dev, 0), bound)
    res = []
    for side in ("device", "host"):
        p = Problem(kinds, n, seed, aligned, scale_aligned, rewrite=rewrite)
        acc = BatchNKA(nb, n, mvec, 0.01)
        res.append((p, acc))
    (pd, dev), (ph, host) = res
    a, r, m = _cuda(atol), _cuda(rtol), _cuda(maxit_dev, torch.int32)
    loop = loop_stop_c(dev, pd, a, r, m, dtol, bound, scale=pd.S if rewrite else None)
    loop.run()
    it, st, norm = loop.results()
    hist = loop.history()
    kh, sh = host_loop(host, ph, hist, atol, rtol, maxit, dtol, bound, scaled=rewrite)
    assert hist.shape == (bound + 1, nb)
    ctx = (n, mvec, aligned, rewrite, scale_aligned)
    assert np.array_equal(it, kh), (ctx, it, kh)
    assert np.array_equal(st, sh), (ctx, st, sh)
    for b in range(nb):
        assert np.array_equal(_bits(norm[b]), _bits(hist[it[b], b])), (ctx, b)
        assert np.all(np.isnan(hist[it[b] + 1:, b])), (ctx, b)
    TL._same(pd, ph, dev, host, range(nb), ctx)
    out = (it, st, norm, hist)
    dev.delete()
    host.delete()
    return out


# (F aligned, scale aligned, scale rewritten): V = 2 with the 16-byte and the 8-byte scale loads, V = 1,
# and no scale at V = 2 and V = 1; n = 1001 is odd, so the scaled tail is replayed too
@pytest.mark.parametrize("aligned,scale_aligned,rewrite", [(True, True, True), (True, False, True), (False, True, True),
                                                           (True, True, False), (False, True, False)])
def test_per_member_rules_match_a_host_driven_loop(aligned, scale_aligned, rewrite):
    it, st, norm, hist = compare_with_host(aligned=aligned, rewrite=rewrite, scale_aligned=scale_aligned)
    assert set(st.tolist()) == {CONVERGED, MAXIT, NONFINITE, DIVERGED}, st
    assert st[6] == DIVERGED and it[6] == 1
    assert st[3] == NONFINITE
    assert st[4] == MAXIT and it[4] == 0          # maxit entry -3: clamped to 0
    assert st[8] == MAXIT and it[8] == 0
    assert st[5] == MAXIT and it[5] == 12         # entry 40: clamped to the bound 12
    assert np.all(np.isfinite(hist[:, 5]))        # every row of the (bound + 1)-row history holds a check
    assert it[1] <= 12
    assert np.all(np.isfinite(hist[:it[6] + 1, 6]))


def test_python_checks_entries_and_lengths_at_create():
    from nka_b200 import BatchNKA
    torch = _torch()
    p = TL.Problem(TL._kinds(8, 1), 64, 0)
    acc = BatchNKA(8, 64, 3, 0.01)
    f = dict(dtype=torch.float64, device="cuda")
    bad = [(dict(atol=torch.zeros(7, **f)), "atol"), (dict(rtol=torch.zeros(9, **f)), "rtol"),
           (dict(maxit=torch.zeros(3, dtype=torch.int32, device="cuda")), "maxit"),
           (dict(atol=torch.tensor([0.0] * 7 + [-1.0], **f)), "atol"),
           (dict(rtol=torch.tensor([0.0] * 7 + [float("nan")], **f)), "rtol"),
           (dict(maxit=torch.tensor([3] * 7 + [-1], dtype=torch.int32, device="cuda")), "maxit"),
           (dict(atol=torch.zeros(16, **f)[::2]), "atol"),
           (dict(scale=torch.zeros(8, 65, **f)), "scale")]
    for kw, what in bad:
        with pytest.raises(ValueError, match=what):
            acc.fixed_point_loop(p.residual, p.X, p.F, **kw)
    # a maxit tensor: the history has max(maxit) + 1 rows
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, maxit=torch.tensor([1, 2, 3, 4, 5, 6, 7, 2], dtype=torch.int32,
                                                                         device="cuda"), rtol=0.0)
    loop.run()
    it, st, _ = loop.results()
    assert loop.history().shape == (8, 8)
    assert it.tolist() == [1, 2, 3, 1, 5, 6, 7, 2], it          # member 3 is NONFINITE at check 1
    acc.delete()


# ---------------------------------------------------------------------------------------------
# 4. queues with per-problem values
# ---------------------------------------------------------------------------------------------
class Problems(TQ.Problems):
    """test_gpu_queue's problems plus EXP problems (F = 2 exp(X), found through slot_problem); the residual
    writes the slots' scale rows S = 1 / (1 + |X|).  With `aligned` F and S rows are 16-byte aligned (V = 2,
    16-byte scale loads), otherwise both are 8 bytes off (V = 1)."""

    def __init__(self, kinds, n, nb, seed, aligned=True):
        torch = _torch()
        super().__init__([TQ.FAST if k == EXP else k for k in kinds], n, nb, seed, aligned)
        self.exp = torch.tensor([[k == EXP] for k in kinds], dtype=torch.bool, device="cuda")
        ld, off = _even_ld(n), 0 if aligned else 1
        self.S = torch.ones(nb * ld + 2, dtype=torch.float64, device="cuda")[off:off + nb * ld].view(nb, ld)[:, :n]
        assert access_width(self.F) == access_width(self.S) == (2 if aligned else 1)

    def residual(self):
        torch = _torch()
        super().residual()
        idx = self.slot.clamp(min=0).long()
        self.F.copy_(torch.where(self.exp.index_select(0, idx), 2.0 * torch.exp(self.X), self.F))
        self.S.copy_(1.0 / (1.0 + self.X.abs()))


def queue_kinds(P, seed):
    k = TQ.kinds_for(P, seed)
    for p in range(P):
        if p % 9 == 2:
            k[p] = EXP
    return k


def queue_entries(P, seed):
    rng = np.random.default_rng(seed)
    atol = rng.choice([1e-8, 1e-6, 1e-10], P)      # > 0: a ZERO problem converges at check 0
    rtol = rng.choice([1e-10, 1e-4, 0.0], P)
    maxit = rng.integers(2, 16, P).astype(np.int32)
    for p in range(P):
        if p % 7 == 4:
            maxit[p] = 3                 # SLOW problems: a per-problem MAXIT
    return atol, rtol, maxit


def run_queue_stop(pr, acc, atol, rtol, maxit, dtol):
    torch = _torch()
    Xout = pr.rows()
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, Xout, atol=_cuda(atol), rtol=_cuda(rtol),
                              maxit=_cuda(maxit, torch.int32), dtol=dtol, scale=pr.S)
    q.run()
    it, st, norm = q.results()
    assert pr.slot.cpu().tolist() == [-1] * pr.nb
    out = (q.Xout.cpu().numpy(), it, st, norm)
    q.destroy()
    return out


def queue_reference(pr, acc, atol, rtol, maxit, dtol):
    """fixed_point_loop with the _stop rule, problems loaded nb at a time into restarted members, the members'
    entries rewritten to their problems' entries before each launch (the loop reads them at every launch)."""
    torch = _torch()
    nb, P = pr.nb, pr.P
    am = torch.zeros(nb, dtype=torch.float64, device="cuda")
    rm = torch.zeros_like(am)
    mm = torch.full((nb,), int(maxit.max()), dtype=torch.int32, device="cuda")
    loop = acc.fixed_point_loop(pr.residual, pr.X, pr.F, atol=am, rtol=rm, maxit=mm, dtol=dtol, scale=pr.S)
    X = np.zeros((P, pr.n))
    it = np.zeros(P, dtype=np.int32)
    st = np.zeros(P, dtype=np.int32)
    norm = np.zeros(P)
    for g0 in range(0, P, nb):
        ids = np.arange(g0, min(g0 + nb, P))
        sp = np.full(nb, -1, dtype=np.int32)
        sp[:len(ids)] = ids
        full = np.where(sp >= 0, sp, 0)
        am.copy_(_cuda(atol[full]))
        rm.copy_(_cuda(rtol[full]))
        mm.copy_(_cuda(maxit[full], torch.int32))
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


def queue_case(nb, P=60, n=129, mvec=5, dtol=2.0, aligned=True, reference=False, seed=5):
    from nka_b200 import BatchNKA
    kinds = queue_kinds(P, seed)
    atol, rtol, maxit = queue_entries(P, seed)
    pr = Problems(kinds, n, nb, seed, aligned)
    acc = BatchNKA(nb, n, mvec, 0.01)
    got = run_queue_stop(pr, acc, atol, rtol, maxit, dtol)
    if reference:
        TQ.assert_same(got, queue_reference(pr, acc, atol, rtol, maxit, dtol), (nb, P, n, mvec, aligned))
    acc.delete()
    return got


@pytest.mark.parametrize("aligned", [True, False])
def test_queue_per_problem_rules_match_the_loop_on_restarted_members(aligned):
    got = queue_case(7, aligned=aligned, reference=True)
    st, it = got[2], got[1]
    kinds = queue_kinds(60, 5)
    _, _, maxit = queue_entries(60, 5)
    assert set(st.tolist()) == {CONVERGED, MAXIT, NONFINITE, DIVERGED}, st
    assert all(st[p] == DIVERGED and it[p] == 1 for p in range(60) if kinds[p] == EXP)
    assert all(it[p] == maxit[p] for p in range(60) if st[p] == MAXIT)
    # problems after a DIVERGED or a per-problem MAXIT in their slot still finish
    assert all(s != RUNNING for s in st)


def test_queue_bits_do_not_depend_on_nbatch():
    ref = queue_case(7)
    for nb in (1, 300):
        TQ.assert_same(queue_case(nb), ref, ("nbatch", nb))


# ---------------------------------------------------------------------------------------------
# 5. NKA_POISON_ALLOC=1 and NKA_LAZY_LAST=0; C preconditions
# ---------------------------------------------------------------------------------------------
def run_digest():
    it, st, norm, hist = compare_with_host(aligned=True, rewrite=True)
    X, qi, qs, qn = queue_case(7, reference=True)
    return hashlib.sha256(it.tobytes() + st.tobytes() + _bits(hist).tobytes() + _bits(X).tobytes() + qi.tobytes()
                          + qs.tobytes() + _bits(qn).tobytes()).hexdigest()


_SUB = """
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_stop as T
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
    _run_sub({"NKA_LAZY_LAST": "0"})            # matches its own host-driven loop and reference inside


_REFUSED_C = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import torch
import test_gpu_loop as T
from nka_b200 import _lib
lib = _lib.load()
p = T.Problem([T.FAST] * 4, 100, 0)
g = torch.cuda.CUDAGraph(keep_graph=True)
with torch.cuda.graph(g):
    p.residual()
h = lib.nka_batch_init(4, 100, 3, 0.01, -1, None)
S = torch.ones(4, 100, dtype=torch.float64, device="cuda")
slot = torch.full((4,), -1, dtype=torch.int32, device="cuda")
st = _lib.StopTest(0.0, 1e-8, 0.0, 5)
which = %(which)r
if which == "atol": st.atol = -1.0
if which == "rtol": st.rtol = float("nan")
if which == "maxit": st.maxit = -1
if which == "dtol": st.dtol = 0.5
if which == "ldscale": st.scale_dev, st.ldscale = S.data_ptr(), 99
arg = None if which == "null" else st
if which == "queue dtol":
    st.dtol = float("nan")
    Q = lib.nka_batch_queue_create_stop(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102, slot.data_ptr(),
                                        p.X.data_ptr(), 100, p.X.data_ptr(), 100, 4, st)
else:
    L = lib.nka_batch_loop_create_stop(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102, arg)
print("returned")
"""

_REFUSALS = {"null": "nka_batch_loop_create: null stop test",
             "atol": "nka_batch_loop_create: atol and rtol must be >= 0",
             "rtol": "nka_batch_loop_create: atol and rtol must be >= 0",
             "maxit": "nka_batch_loop_create: maxit must be >= 0",
             "dtol": "nka_batch_loop_create: dtol must be 0 (off) or >= 1",
             "ldscale": "nka_batch_loop_create: ldscale must be >= vlen",
             "queue dtol": "nka_batch_queue_create: dtol must be 0 (off) or >= 1"}


def test_c_preconditions_abort(tmp_path):
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "here": HERE, "which": w}],
                                 cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                 preexec_fn=_no_core)
             for w in _REFUSALS}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert _REFUSALS[w] in err and "nka_batch_loop.cu:" in err, (w, err)
