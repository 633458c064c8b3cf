"""The interleaved batched accelerator on the GPU (-m gpu).

Every member of an InterleavedBatchNKA must give, bit for bit, what the reference's C accelerator
(OracleNKA(dotmode=0, flavour=0), pinned to the compiled reference by test_oracle.py) gives when fed that
member's calls: every correction vector, num_vec, the lists, the Gram factor among list slots, the
coefficients, min_margin and the last update's drop / eviction / relax flags, after every call, whatever
nbatch, the member's index, the other members' data (NaN, zeros) and masks, ldf and f's alignment.
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
GOLD = os.path.join(HERE, "golden", "accel_golden.json")
SENTINEL = -7.25


def _torch():
    import torch
    return torch


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


# ---------------------------------------------------------------------------------------------
# member sequences: families of scenarios.py with other seeds, late starts, a sat-out step, NaN members
# ---------------------------------------------------------------------------------------------
FAMILIES = [
    S.iid, S.contraction, S.collinear, S.with_repeats, S.picard_like, S.relax_restart, S.zeros_then_iid,
    S.mixed_stress, lambda n, k, seed: S.fill_then_collinear(n, k // 2, k - k // 2, seed), None,
]


def member_ops(b, n, ncall):
    """Member b >= 1: a family of scenarios.py (or, for every tenth kind, all-NaN inputs), started b % 3
    steps late, sitting one mid-sequence step out (None)."""
    fam = FAMILIES[b % len(FAMILIES)]
    ncall = max(ncall, 8)
    if fam is None:
        ops = [("update", np.full(n, np.nan)) for _ in range(ncall)]
        ops.insert(3, ("relax",))
    else:
        ops = fam(n, ncall, 7919 * b + 11)
    k = len(ops) // 2
    return [None] * (b % 3) + ops[:k] + [None] + ops[k:]


def is_nan_member(b):
    return FAMILIES[b % len(FAMILIES)] is None


class Oracle:
    """OracleNKA plus the comparison of its state with a member's."""

    def __init__(self, n, mvec, vtol):
        from oracle import api
        self.o = api.OracleNKA(n, mvec, vtol, dotmode=0, flavour=0)

    def apply(self, op):
        if op[0] == "update":
            f = op[1].copy()
            self.o.accel_update(f)
            return f
        getattr(self.o, op[0])()
        return None

    def check(self, st, nv, ctx):
        o = self.o
        assert nv == o.num_vec(), (ctx, nv, o.num_vec())
        lists = o.lists()
        for k in ("subspace", "pending", "first", "last", "free", "next", "prev"):
            assert st[k] == lists[k], (ctx, k, st[k], lists[k])
        slots = []
        k = lists["first"]
        if lists["pending"] and k != -1:
            k = lists["next"][k]
        while k != -1:
            slots.append(k)
            k = lists["next"][k]
        if slots:
            ix = np.ix_(slots, slots)
            assert np.array_equal(_bits(st["h"][ix]), _bits(o.h()[ix])), (ctx, "h")
            if lists["subspace"]:
                assert np.array_equal(_bits(st["c"][slots]), _bits(o.coeffs())), (ctx, "c")
        assert _bits(st["min_margin"]) == _bits(o.min_margin()), (ctx, "min_margin", st["min_margin"], o.min_margin())
        assert (st["ndrop_last"], bool(st["evicted_last"]), bool(st["relaxed_last"])) == \
            (o.ndrop_last(), o.evicted_last(), o.relaxed_last()), ctx


class Run:
    """An InterleavedBatchNKA whose F is a [nbatch, vlen] view with member stride 1 and component stride ldf,
    `offset` doubles into a store filled with SENTINEL."""

    def __init__(self, nb, n, mvec, vtol, ldf=None, offset=0):
        torch = _torch()
        from nka_b200 import InterleavedBatchNKA
        self.nb, self.n = nb, n
        self.ldf = ldf or nb
        self.s = torch.cuda.Stream()
        self.acc = InterleavedBatchNKA(nb, n, mvec, vtol, stream=self.s.cuda_stream)
        self.offset = offset
        self.store = torch.full((offset + n * self.ldf + 1,), SENTINEL, dtype=torch.float64, device="cuda")
        self.F = self.store[offset:offset + n * self.ldf].view(n, self.ldf)[:, :nb].t()
        assert self.F.stride() == (1, self.ldf)

    def step(self, kinds, rows):
        """kinds: per member None / 'update' / 'relax' / 'restart'; rows: [nb, n] host array, NaN except the
        updating members' f.  Returns F after the step (host) or None if nothing updated."""
        torch = _torch()
        out = None
        with torch.cuda.stream(self.s):
            for kind in ("relax", "restart"):
                sel = kinds == kind
                if sel.any():
                    getattr(self.acc, kind)(torch.from_numpy(sel).cuda())
            upd = kinds == "update"
            if upd.any():
                self.F.copy_(torch.from_numpy(rows))
                self.acc.accel_update(self.F, torch.from_numpy(upd).cuda())
                out = self.F.cpu().numpy()
                full = self.store.cpu().numpy()
        if out is not None:
            assert np.array_equal(_bits(out[~upd]), _bits(rows[~upd])), "an inactive member's f was touched"
            pad = full[self.offset:self.offset + self.n * self.ldf].reshape(self.n, self.ldf)[:, self.nb:]
            assert np.all(pad == SENTINEL) and full[:self.offset].tolist() == [SENTINEL] * self.offset \
                and full[-1] == SENTINEL, "the padding around F was touched"
        return out


def _kinds_rows(step, nb, n):
    kinds = np.array([op[0] if op is not None else None for op in step], dtype=object)
    rows = np.full((nb, n), np.nan)
    for b, op in enumerate(step):
        if op is not None and op[0] == "update":
            rows[b] = op[1]
    return kinds, rows


def drive(nb, n, mvec, vtol, ops, compare, ldf=None, offset=0):
    """Run the members' op lists; compare the members in `compare` with their oracles after every step.
    Returns (member 0's outputs, member 0's num_vec after each of its ops, a digest of every output)."""
    run = Run(nb, n, mvec, vtol, ldf, offset)
    oracles = {b: Oracle(n, mvec, vtol) for b in compare}
    T = max(len(o) for o in ops)
    outs0, nv0 = [], []
    digest = hashlib.sha256()
    for t in range(T):
        step = [o[t] if t < len(o) else None for o in ops]
        kinds, rows = _kinds_rows(step, nb, n)
        out = run.step(kinds, rows)
        if out is not None:
            digest.update(_bits(out).tobytes())
        nv = run.acc.num_vec()
        digest.update(nv.tobytes())
        if step[0] is not None:
            if step[0][0] == "update":
                outs0.append(out[0].copy())
            nv0.append(int(nv[0]))
        for b, orc in oracles.items():
            if step[b] is None:
                continue
            want = orc.apply(step[b])
            if want is not None:
                assert np.array_equal(_bits(out[b]), _bits(want)), (t, b)
            orc.check(run.acc.state(b), int(nv[b]), (t, b))
    assert run.acc.defined()
    run.acc.delete()
    return outs0, nv0, digest.hexdigest()


def scenario_members(name, nb):
    n, mvec, vtol, build = S.SCENARIOS[name]
    ops0 = build()
    nupd = sum(1 for op in ops0 if op[0] == "update")
    return (n, mvec, vtol), [ops0] + [member_ops(b, n, nupd) for b in range(1, nb)]


# ---------------------------------------------------------------------------------------------
# 1 + 2. goldens for member 0, the oracle's bits for every member
# ---------------------------------------------------------------------------------------------
with open(GOLD) as _fh:
    _GOLD = json.load(_fh)


@pytest.mark.parametrize("name", sorted(S.SCENARIOS))
def test_member_zero_gives_the_golden_bits_and_every_member_its_oracles(name):
    nb = 37
    (n, mvec, vtol), ops = scenario_members(name, nb)
    compare = [b for b in range(nb) if not is_nan_member(b)]
    outs0, nv0, _ = drive(nb, n, mvec, vtol, ops, compare)
    g = _GOLD[name]
    assert nv0 == g["num_vec"]
    assert [hashlib.sha256(o.tobytes()).hexdigest() for o in outs0] == g["sha256"]


@pytest.mark.parametrize("nb", [1, 7, 300])
def test_every_member_matches_its_oracle_at_any_batch_size(nb):
    name = "mixed_n257_m5"
    (n, mvec, vtol), ops = scenario_members(name, nb)
    outs0, nv0, _ = drive(nb, n, mvec, vtol, ops, [b for b in range(nb) if not is_nan_member(b)])
    assert [hashlib.sha256(o.tobytes()).hexdigest() for o in outs0] == _GOLD[name]["sha256"]


def test_beyond_65535_members_sampled_oracles_and_digests_of_a_small_batch():
    """70 001 members, member b running kind b % K: sampled members against their oracles, every member
    bit-identical to member b % K of a batch of K."""
    torch = _torch()
    nb, n, mvec, vtol, K = 70001, 16, 5, 0.05, 20
    kinds_ops = [S.iid(n, 24, 5)] + [member_ops(k, n, 24) for k in range(1, K)]
    T = max(len(o) for o in kinds_ops)
    small = Run(K, n, mvec, vtol)
    big = Run(nb, n, mvec, vtol)
    which = np.arange(nb) % K
    sample = [0, 1, 2, 31, 32, 33, 65534, 65535, 65536, 69999, 70000]
    sample = [b for b in sample if not is_nan_member(which[b])]
    oracles = {b: Oracle(n, mvec, vtol) for b in sample}
    for t in range(T):
        step = [o[t] if t < len(o) else None for o in kinds_ops]
        kinds, rows = _kinds_rows(step, K, n)
        out_s = small.step(kinds, rows)
        out_b = big.step(kinds[which], rows[which])
        if out_s is not None:
            assert np.array_equal(_bits(out_b), _bits(out_s)[which]), t
        nv_s, nv_b = small.acc.num_vec(), big.acc.num_vec()
        assert np.array_equal(nv_b, nv_s[which]), t
        for b, orc in oracles.items():
            op = step[which[b]]
            if op is None:
                continue
            want = orc.apply(op)
            if want is not None:
                assert np.array_equal(_bits(out_b[b]), _bits(want)), (t, b)
            orc.check(big.acc.state(b), int(nv_b[b]), (t, b))
    assert big.acc.defined() and small.acc.defined()
    big.acc.delete()
    small.acc.delete()
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------
# 3. layout: padded ldf and an 8-byte offset give the same bits
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["fullthendrop_n300_m4", "iid_n513_m32"])
def test_padding_and_misalignment_give_the_same_bits(name):
    nb = 37
    (n, mvec, vtol), ops = scenario_members(name, nb)
    _, _, plain = drive(nb, n, mvec, vtol, ops, [])
    _, _, padded = drive(nb, n, mvec, vtol, ops, [], ldf=nb + 13)
    _, _, shifted = drive(nb, n, mvec, vtol, ops, [], ldf=nb + 3, offset=1)
    assert plain == padded == shifted


# ---------------------------------------------------------------------------------------------
# 4. graphs
# ---------------------------------------------------------------------------------------------
def _interleaved(rows):
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(rows.T)).cuda()
    return t.t()


def _iteration(acc, X, Bv, F, active, relax, tol):
    """One fixed-point iteration of picard_like's map per member, with device-computed masks: members above
    tol are accelerated and step; members that just dropped below 100*tol relax their pending pair."""
    torch = _torch()
    G = Bv / (1.0 + 0.5 * torch.roll(X, 1, dims=1) + 0.3 * X * X)
    torch.sub(X, G, out=F)
    norm = torch.linalg.vector_norm(F, dim=1)
    torch.lt(norm, 100 * tol, out=relax)
    acc.relax(relax)
    torch.gt(norm, tol, out=active)
    acc.accel_update(F, active)
    X.sub_(F * active.unsqueeze(1))


def test_captured_iteration_gives_the_eager_bits():
    torch = _torch()
    from nka_b200 import InterleavedBatchNKA, NKAError
    nb, n, mvec, iters, tol = 45, 200, 5, 25, 1e-10
    rng = np.random.default_rng(15)
    x0 = rng.uniform(0.1, 1.0, (nb, n))
    s = torch.cuda.Stream()
    eager = InterleavedBatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    capt = InterleavedBatchNKA(nb, n, mvec, 0.01, stream=s.cuda_stream)
    Bv = _interleaved(rng.uniform(0.5, 1.5, (nb, n)))
    Xe, Xg = _interleaved(x0), _interleaved(x0)
    Fe, Fg = _interleaved(np.zeros((nb, n))), _interleaved(np.zeros((nb, n)))
    ae, ag, re_, rg = (torch.zeros(nb, dtype=torch.bool, device="cuda") for _ in range(4))
    with torch.cuda.stream(s):
        eager.set_vec_tol(0.02)
    torch.cuda.synchronize()
    launches0 = capt.launch_count()
    g = torch.cuda.CUDAGraph()
    refused = {"num_vec": capt.num_vec, "defined": capt.defined, "state": lambda: capt.state(0),
               "set_stream": lambda: capt.set_stream(None), "synchronize": capt.synchronize}
    errors = {}
    with torch.cuda.graph(g, stream=s):
        capturing = capt.stream_capturing()
        capt.set_vec_tol(0.02)
        _iteration(capt, Xg, Bv, Fg, ag, rg, tol)
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
            _iteration(eager, Xe, Bv, Fe, ae, re_, tol)
            g.replay()
            assert np.array_equal(_bits(Xe.cpu().numpy()), _bits(Xg.cpu().numpy())), it
            assert torch.equal(ae, ag) and torch.equal(re_, rg), it
            nactive.append(int(ae.sum()))
    assert capt.launch_count() == launches0
    assert list(eager.num_vec()) == list(capt.num_vec())
    for b in range(nb):
        se, sg = eager.state(b), capt.state(b)
        for k in se:
            if isinstance(se[k], np.ndarray) or isinstance(se[k], float):
                assert np.array_equal(_bits(se[k]), _bits(sg[k])), (b, k)
            else:
                assert se[k] == sg[k], (b, k)
    assert nactive[0] == nb and capt.state(0)["vtol"] == 0.02
    eager.delete()
    capt.delete()


def test_one_launch_per_update_whatever_nbatch():
    torch = _torch()
    from nka_b200 import InterleavedBatchNKA
    for nb in (1, 100000):
        acc = InterleavedBatchNKA(nb, 8, 3, 0.01)
        F = _interleaved(np.ones((nb, 8)))
        c0 = acc.launch_count()
        acc.accel_update(F)
        acc.relax()
        acc.restart()
        assert acc.launch_count() - c0 == 3
        acc.synchronize()
        acc.delete()
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------
# 5. environment and aborts
# ---------------------------------------------------------------------------------------------
POISON_NAMES = ["fullthendrop_n300_m4", "relax_restart_n96_m4", "zeros_n33_m3", "iid_n513_m32", "n3_m5_rankdef"]


def digests(names):
    out = {}
    for name in names:
        (n, mvec, vtol), ops = scenario_members(name, 37)
        out[name] = drive(37, n, mvec, vtol, ops, [])[2]
    return out


def _no_core():
    resource.setrlimit(resource.RLIMIT_CORE, (0, 0))


_SUB = """
import sys, json
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_ibatch as T
print("RESULT " + json.dumps(T.digests(%(names)r)))
"""


def test_poisoned_allocations_give_the_same_bits():
    clean = digests(POISON_NAMES)
    env = dict(os.environ, NKA_POISON_ALLOC="1")
    r = subprocess.run([sys.executable, "-c", _SUB % {"root": ROOT, "here": HERE, "names": POISON_NAMES}], env=env,
                       capture_output=True, text=True, timeout=1800, preexec_fn=_no_core)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    assert json.loads(line[len("RESULT "):]) == clean


_ABORT = r"""
import ctypes as C, sys
sys.path.insert(0, %(root)r)
from nka_b200 import _lib
lib = _lib.load()
view = _lib.StateView()
def handle():
    return lib.nka_ibatch_init(4, 8, 2, 0.01, -1, None)
calls = {
    "nbatch": lambda: lib.nka_ibatch_init(0, 8, 2, 0.01, -1, None),
    "vlen": lambda: lib.nka_ibatch_init(4, 0, 2, 0.01, -1, None),
    "mvec": lambda: lib.nka_ibatch_init(4, 8, 33, 0.01, -1, None),
    "vtol": lambda: lib.nka_ibatch_init(4, 8, 2, 0.0, -1, None),
    "null f": lambda: lib.nka_ibatch_accel_update(handle(), None, 4, None),
    "ldf": lambda: lib.nka_ibatch_accel_update(handle(), 4096, 3, None),
    "member": lambda: lib.nka_ibatch_get_state(handle(), 4, C.byref(view)),
    "set_vec_tol": lambda: lib.nka_ibatch_set_vec_tol(handle(), 0.0),
}
calls[%(which)r]()
print("returned")
"""

_ABORT_MSG = {"nbatch": "nbatch must be in 1..2^31-1", "vlen": "vlen must be >= 1", "mvec": "mvec > 32",
              "vtol": "vtol must be > 0", "null f": "null f", "ldf": "ldf must be >= nbatch",
              "member": "member out of range", "set_vec_tol": "nka_ibatch_set_vec_tol: vtol must be > 0"}


def test_c_preconditions_abort_with_file_and_line(tmp_path):
    procs = {w: subprocess.Popen([sys.executable, "-c", _ABORT % {"root": ROOT, "which": w}], cwd=str(tmp_path),
                                 stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, preexec_fn=_no_core)
             for w in _ABORT_MSG}
    for w, p in procs.items():
        out, err = p.communicate(timeout=600)
        assert p.returncode != 0 and "returned" not in out, (w, out, err)
        assert "nka_b200: " in err and "nka_ibatch.cu:" in err and _ABORT_MSG[w] in err, (w, err)
