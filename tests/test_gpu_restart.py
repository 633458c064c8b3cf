"""Residual-growth restarts (restart_growth) of device-side loops and queues on the GPU.  A rule that never
fires must give the bits of restart_growth = 0; a rule that fires must give each member the bits of a
host-driven loop that restarts the members the rule picks (from the device loop's recorded norms) before its
masked update; each queue problem must get the bits of the loop with the same rule on a just-restarted
member, whatever slot it lands in and whatever nbatch.  The residual multiplies F by BUMP at seeded
evaluations of seeded problems, so growth happens at known points."""
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

CMAX = 64          # evaluations covered by the bump table
BUMP = 100.0       # F is multiplied by this at a bumped evaluation
NEVER = 1e300      # a restart_growth that never fires on these problems
EXP = "exp"        # F = 2 exp(8 X): r1 > 1e5 r0, DIVERGED at check 1 with dtol = 1e4


def _torch():
    import torch
    return torch


def _kinds(P, seed):
    """test_gpu_queue's kinds (NAN, ZERO, SLOW, FAST and random contractions)."""
    return TQ.kinds_for(P, seed)


def _targets(kinds, seed):
    """The problems whose residual is bumped: every third one of the plain random kinds."""
    plain = [p for p, k in enumerate(kinds) if k not in (TQ.NAN, TQ.ZERO, TQ.SLOW, TQ.FAST, EXP)]
    return plain[::3]


class Problems(TQ.Problems):
    """test_gpu_queue's problems with a per-row evaluation counter, reset whenever slot_problem changes for the
    row (so one residual serves loops, where slot_problem is fixed, and queues), and F multiplied by BUMP at
    the seeded evaluations of the target problems.  EXP problems have F = 2 exp(8 X).  `scale`: fixed weights
    for the stop test's norm, per slot."""

    def __init__(self, kinds, n, nb, seed, aligned=True, targets=None):
        torch = _torch()
        P = len(kinds)
        super().__init__([TQ.FAST if k == EXP else k for k in kinds], n, nb, seed, aligned)
        self.exp = torch.tensor([[k == EXP] for k in kinds], dtype=torch.bool, device="cuda")
        self.targets = _targets(kinds, seed) if targets is None else list(targets)
        rng = np.random.default_rng(seed + 1000)
        bump = np.zeros((P, CMAX), dtype=bool)
        for p in self.targets:
            c = int(rng.integers(2, 5))
            while c < CMAX - 1:
                bump[p, c] = True
                c += int(rng.integers(3, 8))
        self.bump_host = bump
        self.bump = torch.from_numpy(bump.reshape(-1)).cuda()
        self.owner = torch.full((nb,), -2, dtype=torch.int32, device="cuda")
        self.count = torch.zeros(nb, dtype=torch.int64, device="cuda")
        self.S = torch.from_numpy(np.random.default_rng(seed + 7).uniform(0.5, 4.0, (nb, n))).cuda()

    def reset(self):
        """The next evaluation of every row is its problem's evaluation 0."""
        self.owner.fill_(-2)

    def residual(self):
        torch = _torch()
        super().residual()
        sp = self.slot
        self.count.copy_(torch.where(sp != self.owner, torch.zeros_like(self.count), self.count + 1))
        self.owner.copy_(sp)
        idx = sp.clamp(min=0).long()
        hit = self.bump.index_select(0, idx * CMAX + self.count.clamp(max=CMAX - 1)).unsqueeze(1)
        F = torch.where(self.exp.index_select(0, idx), 2.0 * torch.exp(8.0 * self.X), self.F)
        self.F.copy_(torch.where(hit, BUMP * F, F))


def loop_problems(kinds, n, seed, aligned=True):
    """nb = P members, member b solving problem b from its X0 row."""
    torch = _torch()
    p = Problems(kinds, n, len(kinds), seed, aligned)
    p.slot.copy_(torch.arange(len(kinds), dtype=torch.int32, device="cuda"))
    p.X.copy_(p.X0)
    return p


def host_replay(acc, p, hist, gamma, atol, rtol, maxit, dtol=0.0):
    """The host-driven loop: stop decisions and the rule's picks from the device loop's recorded norms;
    residual, restart(picked), accel_update(F, running), X[b] += F[b].  Returns (steps, status, restarts, the
    num_vec of each restarted member just before its restart)."""
    torch = _torch()
    nb = p.nb
    k = np.zeros(nb, dtype=np.int32)
    st = np.full(nb, RUNNING, dtype=np.int32)
    r0 = np.zeros(nb)
    nrst = np.zeros(nb, dtype=np.int32)
    before = []
    p.reset()
    for _ in range(maxit + 1):
        p.residual()
        pick = np.zeros(nb, dtype=bool)
        for b in np.nonzero(st == RUNNING)[0]:
            r = hist[k[b], b]
            if k[b] == 0:
                r0[b] = r
            if not np.isfinite(r):
                st[b] = NONFINITE
            elif r < max(atol, rtol * r0[b]):
                st[b] = CONVERGED
            elif dtol > 0 and r > dtol * r0[b]:
                st[b] = DIVERGED
            elif k[b] >= maxit:
                st[b] = MAXIT
            elif gamma > 0 and k[b] >= 1 and r > gamma * hist[k[b] - 1, b]:
                pick[b] = True
        on = st == RUNNING
        if pick.any():
            nv = acc.num_vec()
            before += [(int(b), int(nv[b])) for b in np.nonzero(pick)[0]]
            acc.restart(torch.from_numpy(pick.astype(np.uint8)).cuda())
            nrst[pick] += 1
        acc.accel_update(p.F, torch.from_numpy(on.astype(np.uint8)).cuda())
        for b in np.nonzero(on)[0]:
            p.X[b] += p.F[b]
        k[on] += 1
        if not on.any():
            break
    torch.cuda.synchronize()
    return k, st, nrst, before


def run_loop(acc, p, gamma, atol=1e-10, rtol=1e-12, maxit=24, dtol=0.0, scale=False):
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, atol=atol, rtol=rtol, maxit=maxit, dtol=dtol,
                                scale=p.S if scale else None, restart_growth=gamma)
    p.reset()
    loop.run()
    it, st, norm = loop.results()
    out = dict(it=it, st=st, norm=norm, hist=loop.history(), nrst=loop.restarts(), X=p.X.cpu().numpy(),
               F=p.F.cpu().numpy(), states=[acc.state(b) for b in range(p.nb)])
    loop.destroy()
    return out


def replay_case(gamma, mvec=5, aligned=True, n=1001, seed=3, P=10, scale=False, dtol=0.0, kinds=None):
    """The device loop at `gamma` against host_replay; returns the device outcome and the replay's picks."""
    from nka_b200 import BatchNKA
    kinds = kinds or _kinds(P, seed)
    pd, ph = loop_problems(kinds, n, seed, aligned), loop_problems(kinds, n, seed, aligned)
    dev, host = BatchNKA(len(kinds), n, mvec, 0.01), BatchNKA(len(kinds), n, mvec, 0.01)
    d = run_loop(dev, pd, gamma, maxit=24, dtol=dtol, scale=scale)
    kh, sh, rh, before = host_replay(host, ph, d["hist"], gamma, 1e-10, 1e-12, 24, dtol)
    ctx = (gamma, mvec, aligned, n, scale, dtol)
    assert np.array_equal(d["it"], kh), (ctx, d["it"], kh)
    assert np.array_equal(d["st"], sh), (ctx, d["st"], sh)
    assert np.array_equal(d["nrst"], rh), (ctx, d["nrst"], rh)
    TL._same(pd, ph, dev, host, range(len(kinds)), ctx)
    dev.delete()
    host.delete()
    return d, before, pd


def _access_width(T):
    return 2 if T.data_ptr() % 16 == 0 and T.stride(0) % 2 == 0 else 1


# ---------------------------------------------------------------------------------------------
# 1. forced growth: the targets restart with a non-empty subspace, nothing else restarts
# ---------------------------------------------------------------------------------------------
def test_forced_growth_restarts_the_targets_only():
    d, before, p = replay_case(2.0, P=12)
    targets = set(p.targets)
    assert targets
    for t in targets:
        assert any(b == t and nv > 0 for b, nv in before), (t, before)
    for b in range(p.nb):
        if b not in targets:
            assert d["nrst"][b] == 0, (b, d["nrst"])
    # the queue: the same problems, per-problem counts
    from nka_b200 import BatchNKA
    kinds = _kinds(12, 3)
    pr = Problems(kinds, 1001, 4, 3)
    acc = BatchNKA(4, 1001, 5, 0.01)
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, pr.rows(), atol=1e-10, rtol=1e-12, maxit=24,
                              restart_growth=2.0)
    pr.reset()
    q.run()
    rq = q.restarts()
    assert rq.dtype == np.int32 and rq.shape == (12,)
    assert np.array_equal(rq, d["nrst"]), (rq, d["nrst"])       # a problem's counts are its loop member's
    assert all(rq[t] >= 1 for t in targets), rq
    assert all(rq[p_] == 0 for p_ in range(12) if p_ not in targets), rq
    acc.delete()


# ---------------------------------------------------------------------------------------------
# 2. a rule that never fires gives restart_growth = 0's bits (loop and queue)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mvec", [1, 5, 32])
@pytest.mark.parametrize("aligned", [True, False])
def test_never_firing_rule_is_restart_growth_zero(mvec, aligned):
    from nka_b200 import BatchNKA
    kinds = _kinds(10, mvec)
    outs = []
    for gamma in (0.0, NEVER):
        p = loop_problems(kinds, 1001, 3, aligned)
        assert _access_width(p.F) == (2 if aligned else 1)
        acc = BatchNKA(10, 1001, mvec, 0.01)
        outs.append(run_loop(acc, p, gamma))
        acc.delete()
    a, b = outs
    for key in ("it", "st"):
        assert np.array_equal(a[key], b[key]), (key, a[key], b[key])
    for key in ("norm", "hist", "X", "F"):
        assert np.array_equal(_bits(a[key]), _bits(b[key])), key
    for m, (sa, sb) in enumerate(zip(a["states"], b["states"])):
        TL.assert_state_equal(sa, sb, m)
    assert not a["nrst"].any() and not b["nrst"].any()
    assert set(a["st"].tolist()) >= {CONVERGED, NONFINITE}, a["st"]
    got = []
    for gamma in (0.0, NEVER):
        pr = Problems(_kinds(29, mvec), 1001, 8, 5, aligned)
        acc = BatchNKA(8, 1001, mvec, 0.01)
        q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, pr.rows(), atol=1e-10, rtol=1e-12,
                                  maxit=24, restart_growth=gamma)
        pr.reset()
        q.run()
        it, st, norm = q.results()
        assert not q.restarts().any()
        got.append((q.Xout.cpu().numpy(), it, st, norm))
        acc.delete()
    TQ.assert_same(got[0], got[1], ("queue", mvec, aligned))


# ---------------------------------------------------------------------------------------------
# 3. a rule that fires: the loop against the host replay
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gamma", [1.0, 0.5])
@pytest.mark.parametrize("mvec", [1, 5, 32])
@pytest.mark.parametrize("aligned", [True, False])
def test_loop_matches_the_host_replay(gamma, mvec, aligned):
    d, before, p = replay_case(gamma, mvec, aligned, seed=mvec)
    assert _access_width(p.F) == (2 if aligned else 1)
    assert d["nrst"].sum() > 0
    assert any(nv > 0 for _, nv in before)


def test_loop_matches_the_host_replay_with_a_scale_and_dtol():
    kinds = _kinds(10, 3)
    kinds[2] = EXP
    d, before, p = replay_case(1.0, scale=True, dtol=1e4, kinds=kinds)      # above any bump (BUMP = 100)
    assert d["st"][2] == DIVERGED and d["it"][2] == 1 and d["nrst"][2] == 0      # DIVERGED wins over a restart
    assert d["hist"][1, 2] > d["hist"][0, 2]
    assert d["nrst"].sum() > 0


# ---------------------------------------------------------------------------------------------
# 4. queues against the loop on restarted members; nbatch; in place; relaunch
# ---------------------------------------------------------------------------------------------
def queue_reference(acc, pr, gamma, atol, rtol, maxit):
    """fixed_point_loop with the same rule, problems loaded nb at a time into restarted members."""
    torch = _torch()
    nb, P = pr.nb, pr.P
    loop = acc.fixed_point_loop(pr.residual, pr.X, pr.F, atol=atol, rtol=rtol, maxit=maxit, restart_growth=gamma)
    X = np.zeros((P, pr.n))
    it = np.zeros(P, dtype=np.int32)
    st = np.zeros(P, dtype=np.int32)
    norm = np.zeros(P)
    nrst = np.zeros(P, dtype=np.int32)
    for g0 in range(0, P, nb):
        ids = np.arange(g0, min(g0 + nb, P))
        sp = np.full(nb, -1, dtype=np.int32)
        sp[:len(ids)] = ids
        pr.slot.copy_(torch.from_numpy(sp))
        pr.X.zero_()
        pr.X[:len(ids)] = pr.X0[torch.from_numpy(ids).cuda()]
        acc.restart()
        pr.reset()
        loop.run()
        i, s, r = loop.results()
        X[ids] = pr.X[:len(ids)].cpu().numpy()
        it[ids], st[ids], norm[ids] = i[:len(ids)], s[:len(ids)], r[:len(ids)]
        nrst[ids] = loop.restarts()[:len(ids)]
    loop.destroy()
    return (X, it, st, norm), nrst


def run_queue(acc, pr, gamma, Xout, launches=1, atol=1e-10, rtol=1e-12, maxit=24):
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, Xout, atol=atol, rtol=rtol, maxit=maxit,
                              restart_growth=gamma)
    out = []
    for _ in range(launches):
        pr.reset()
        q.run()
        it, st, norm = q.results()
        assert pr.slot.cpu().tolist() == [-1] * pr.nb
        out.append(((q.Xout.cpu().numpy(), it, st, norm), q.restarts()))
    q.destroy()
    return out


@pytest.mark.parametrize("n", [1001, 1000])             # 16-byte row moves with a tail; 8-byte ones
def test_queue_matches_the_loop_on_restarted_members(n):
    from nka_b200 import BatchNKA
    pr = Problems(_kinds(29, 4), n, 8, 5)
    assert pr.wide_rows() == (n % 2 == 1)
    acc = BatchNKA(8, n, 5, 0.01)
    (got, rq), (again, rq2) = run_queue(acc, pr, 1.0, pr.rows(), launches=2)
    want, rl = queue_reference(acc, pr, 1.0, 1e-10, 1e-12, 24)
    TQ.assert_same(got, want, ("queue", n))
    assert np.array_equal(rq, rl), (rq, rl)
    assert rq.sum() > 0
    TQ.assert_same(got, again, ("relaunch", n))
    assert np.array_equal(rq, rq2)
    # in place (Xout is X0): the same bits
    ((inplace, rqi),) = run_queue(acc, pr, 1.0, None)
    TQ.assert_same(got, inplace, ("in place", n))
    assert np.array_equal(rq, rqi)
    acc.delete()


def queue_case(nb, P=40, n=257, gamma=1.0):
    from nka_b200 import BatchNKA
    pr = Problems(_kinds(P, 7), n, nb, 5)
    acc = BatchNKA(nb, n, 5, 0.01)
    ((got, rq),) = run_queue(acc, pr, gamma, pr.rows())
    acc.delete()
    return got, rq


def test_queue_bits_do_not_depend_on_nbatch():
    ref, rref = queue_case(7)
    assert rref.sum() > 0
    for nb in (1, 300):
        got, rq = queue_case(nb)
        TQ.assert_same(got, ref, ("nbatch", nb))
        assert np.array_equal(rq, rref), nb


# ---------------------------------------------------------------------------------------------
# 5. NKA_POISON_ALLOC=1 (rprev is 0xFF bytes until check 0 writes it) and NKA_LAZY_LAST=0
# ---------------------------------------------------------------------------------------------
def run_digest():
    d, _, _ = replay_case(1.0, aligned=False)
    (X, it, st, norm), rq = queue_case(7)
    return hashlib.sha256(d["it"].tobytes() + d["st"].tobytes() + d["nrst"].tobytes() + _bits(d["hist"]).tobytes()
                          + _bits(X).tobytes() + it.tobytes() + st.tobytes() + _bits(norm).tobytes()
                          + rq.tobytes()).hexdigest()


_SUB = """
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_restart as T
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
    _run_sub({"NKA_LAZY_LAST": "0"})            # matches its own host replay and loop inside


# ---------------------------------------------------------------------------------------------
# 6. refusals
# ---------------------------------------------------------------------------------------------
def test_restarts_refused_inside_a_capture():
    from nka_b200 import BatchNKA, NKAError
    torch = _torch()
    s = torch.cuda.Stream()
    p = loop_problems(_kinds(4, 1), 256, 0)
    acc = BatchNKA(4, 256, 3, 0.01, stream=s.cuda_stream)
    loop = acc.fixed_point_loop(p.residual, p.X, p.F, maxit=5, restart_growth=1.0)
    pr = Problems(_kinds(10, 1), 256, 4, 0)
    q = acc.fixed_point_queue(pr.residual, pr.X, pr.F, pr.slot, pr.X0, maxit=5, restart_growth=1.0)
    s.wait_stream(torch.cuda.current_stream())
    loop.run()
    assert loop.restarts().shape == (4,)
    q.run()
    assert q.restarts().shape == (10,)
    errors = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        p.residual()
        for name, call in (("loop", loop.restarts), ("queue", q.restarts)):
            try:
                call()
                errors[name] = None
            except NKAError as exc:
                errors[name] = str(exc)
    for name, msg in errors.items():
        assert msg and "restarts cannot be captured" in msg, (name, msg)
    acc.delete()


_REFUSED_C = r"""
import sys
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
slot = torch.full((4,), -1, dtype=torch.int32, device="cuda")
st = _lib.StopTest(0.0, 1e-8, 0.0, 5)
which = %(which)r
if which == "loop negative":
    L = lib.nka_batch_loop_create_restart(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102, st, -1.0)
elif which == "loop nan":
    L = lib.nka_batch_loop_create_restart(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102, st,
                                          float("nan"))
else:
    Q = lib.nka_batch_queue_create_restart(h, g.raw_cuda_graph(), p.X.data_ptr(), 100, p.F.data_ptr(), 102,
                                           slot.data_ptr(), p.X.data_ptr(), 100, p.X.data_ptr(), 100, 4, st,
                                           float("inf") if which == "queue inf" else -0.5)
print("returned")
"""

_REFUSALS = {"loop negative": "nka_batch_loop_create: restart_growth must be",
             "loop nan": "nka_batch_loop_create: restart_growth must be",
             "queue negative": "nka_batch_queue_create: restart_growth must be",
             "queue inf": "nka_batch_queue_create: restart_growth must be"}


def test_c_preconditions_abort(tmp_path):
    procs = {w: subprocess.Popen([sys.executable, "-c", _REFUSED_C % {"root": ROOT, "here": HERE, "which": w}],
                                 cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                 preexec_fn=_no_core)
             for w in _REFUSALS}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert _REFUSALS[w] in err and ".cu:" in err, (w, err)
