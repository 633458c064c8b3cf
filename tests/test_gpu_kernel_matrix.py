"""Every pass A / pass B instantiation at both access widths, against the reference (-m gpu, one GPU).

accel_update runs one of 132 compiled kernels: nka_pass_a<NC, V> (NC = 1..33) and nka_pass_b<NZ, V>
(NZ = 0..32), V = 2 doubles per access when f is 16-byte aligned and 1 otherwise (nka_capi.cu:
update_shape).  Each kernel has a predicate-free FULL body and a general one (drops, chain breaks,
nz != NZ).  The sweep below drives every width mvec = 1..32 with f aligned and at an 8-byte offset,
in three modes (lazy oldest column, NKA_LAZY_LAST=0, a one-process dp hook), and on every call checks
the decisions against the serial reference and the output, the projection coefficients c, the factor
h and min_margin against the long-double arbiter.  A host model run alongside (tests/model/) tells
which kernel and which body the device ran; the ledger at the end requires all 132 kernels and both
bodies of every NC >= 2 and NZ >= 1.

The second half reads nothing it has not written: with NKA_POISON_ALLOC=1 the library's data buffers
start as NaN bytes instead of cudaMalloc's usual zeros, so a stale column multiplied by a zero
coefficient turns into NaN, and NaN guard words around f catch reads and writes past its ends.  Runs
are deterministic, so poisoned and guarded runs must equal plain ones bit for bit.
"""
import numpy as np
import pytest

import scenarios as S
from model import ModelNKA
from oracle import api
from parity_log import record_parity

pytestmark = pytest.mark.gpu

VTOL = 0.1
N_ODD = 1001        # odd: the V = 2 kernels also run their scalar tail element
N_SMALL = 201       # below one CTA's thread count: the fold has a single partial row
SMALL_N_WIDTHS = (1, 13, 24, 32)
POISON_WIDTHS = (1, 12, 13, 23, 24, 32)
MODES = ("lazy", "eager", "dp")
PLACEMENTS = ("aligned", "offset")
NCOLLINEAR = 12
MAXSLOT = 33
THREADS_A = 256

# Kernel / body combinations the sweep does not reach, each with the reason.  (None at present: the
# ledger requires the FULL and the general body of every NC >= 2 and NZ >= 1, and all 132 kernels.)
UNREACHED = {}


def _torch():
    import torch
    return torch


def sweep_ops(n, mvec, seed=None):
    """mvec + 4 i.i.d. calls (the list grows to capacity and evicts: FULL bodies), then near-collinear
    calls (vtol drops at a full list: general bodies) with one relax() in their middle.  The relax comes
    after the i.i.d. calls because it breaks the chain of every pair then on the list, and a full,
    fully chained list is what the FULL bodies of the widest kernels need."""
    nfill = mvec + 4
    ops = S.fill_then_collinear(n, nfill, NCOLLINEAR, 1000 + mvec if seed is None else seed)
    ops.insert(nfill + NCOLLINEAR // 2, ("relax",))
    return ops, nfill


class Placed:
    """f on the device: buf[0:n] of a fresh tensor (16-byte aligned: V = 2) or buf[1:n+1] (8 bytes
    off: V = 1).  guard=True fills the words around f with NaN sentinels of a recognisable payload:
    buf[n] (same 16-byte word as the last element of an aligned f with odd n), or buf[0] and buf[n+1]."""
    SENTINEL = 0x7FF4DEADBEEF0001    # a NaN whose payload no computation produces

    def __init__(self, n, placement, guard=False):
        torch = _torch()
        self.n, self.off = n, (0 if placement == "aligned" else 1)
        self.buf = torch.zeros(n + 2, dtype=torch.float64, device="cuda")
        self.f = self.buf[self.off:self.off + n]
        assert self.f.data_ptr() % 16 == (0 if placement == "aligned" else 8)
        self.guards = []
        if guard:
            self.guards = [n] if self.off == 0 else [0, n + 1]
            bits = self.buf.view(torch.int64)
            for g in self.guards:
                bits[g] = self.SENTINEL
        self.V = 2 if self.off == 0 else 1

    def load(self, x):
        self.f.copy_(_torch().from_numpy(x))

    def read(self):
        return self.f.cpu().numpy()

    def guards_intact(self):
        bits = self.buf.view(_torch().int64).cpu().numpy()
        return all(int(bits[g]) == self.SENTINEL for g in self.guards)


def _list_slots(first, nxt, skip_head):
    out, k = [], first
    while k != -1:
        out.append(k)
        k = nxt[k]
    return out[1:] if skip_head and out else out


def _rel_inf(a, b):
    return float(np.max(np.abs(a - b))) / max(float(np.max(np.abs(b))), 1e-300) if b.size else 0.0


class Spread:
    """The S.tolerances policy for one quantity: 1e-12, or 4x the reference's own serial-vs-long-double
    spread of it so far (a running maximum), whichever is larger."""

    def __init__(self):
        self.worst = 0.0

    def tol(self, serial_vs_arbiter):
        self.worst = max(self.worst, serial_vs_arbiter)
        return max(1e-12, 4.0 * self.worst)


def _make_device(n, mvec, mode):
    from nka_b200 import NKA
    from nka_b200.nka import DP_FUNC
    acc = NKA(n, mvec, VTOL)
    if mode == "dp":
        cb = DP_FUNC(lambda m, x, y: x[0] * y[0])    # one process: the partial sum is the global sum
        acc.set_dot_prod(cb)
    return acc


def run_checked(n, mvec, placement, mode, ledger_a, ledger_b, worst):
    """One sweep sequence on the device beside the serial reference, the long-double arbiter and the
    host model; asserts on every call, adds (NC, V, full) / (NZ, V, full) to the ledgers."""
    ops, nfill = sweep_ops(n, mvec)
    lazy = mode == "lazy"
    fused = mode != "dp"
    ser = api.OracleNKA(n, mvec, VTOL, dotmode=0)
    arb = api.OracleNKA(n, mvec, VTOL, dotmode=1)
    mod = ModelNKA(n, mvec, VTOL, lazy=lazy)
    acc = _make_device(n, mvec, mode)
    dev = Placed(n, placement)
    sp_out, sp_c, sp_h, sp_m = Spread(), Spread(), Spread(), Spread()
    it = 0
    for op in ops:
        if op[0] == "relax":
            ser.relax(); arb.relax(); mod.relax(); acc.relax()
            assert acc.num_vec() == ser.num_vec() == mod.num_vec()
            continue
        fin = op[1]
        where = (mode, placement, n, mvec, it)
        # the kernels this call runs, worked out as nka_capi.cu does (update_shape, nz_expected)
        L, pending = mod.ub_len(), bool(mod.host_pending())
        ncol, skip, submask = mod.plan_a()
        NZ = min(max(L - 1 if pending else L, 0), mvec)
        assert acc.launch_geometry()["threads"] == THREADS_A * 10000 + (256 if NZ >= 24 else 512), where
        if L > 0:
            NC = mvec if (fused and lazy and pending and L == mvec + 1) else L
            allbits = (1 << NC) - 1
            ledger_a.add((NC, dev.V, ncol - skip == NC and (submask & allbits) == allbits))
        a, b = fin.copy(), fin.copy()
        ser.accel_update(a)
        arb.accel_update(b)
        mod.accel_update(fin.copy())
        dev.load(fin)
        acc.accel_update(dev.f)
        got = dev.read()
        nz, has_pair, write_f, nmat = mod.plan_b()
        ledger_b.add((NZ, dev.V, nz == NZ and bool(has_pair) and bool(write_f) and nmat == 0))

        st = acc.state()
        assert st["error"] == 0, where
        decisions = (st["ndrop_last"], bool(st["relaxed_last"]), bool(st["evicted_last"]))
        assert decisions == (ser.ndrop_last(), ser.relaxed_last(), ser.evicted_last()), where
        assert decisions == (mod.ndrop_last(), bool(mod.relaxed_last()), bool(mod.evicted_last())), where
        assert acc.num_vec() == ser.num_vec() == mod.num_vec(), where

        # the output: the S.tolerances bar against the arbiter
        scale = max(np.linalg.norm(b), np.linalg.norm(fin), 1e-300)
        err = np.linalg.norm(got - b) / scale
        assert np.all(np.isfinite(got)) and err <= sp_out.tol(np.linalg.norm(a - b) / scale), (where, err)
        worst["out"] = max(worst["out"], err)

        # the list: the reference's slots, newest first (DESIGN.md section 3)
        lst_arb = arb.lists()
        assert (st["first"], st["pending"]) == (lst_arb["first"], lst_arb["pending"]), where
        slots = _list_slots(st["first"], st["next"], skip_head=bool(st["pending"]))
        assert slots == _list_slots(lst_arb["first"], lst_arb["next"], skip_head=bool(lst_arb["pending"])), where

        iid = it < nfill
        # projection coefficients, in list order without the new pending head
        c_arb, c_ser = arb.coeffs(), ser.coeffs()
        c_dev = st["c"][slots] if st["subspace"] else np.zeros(0)
        assert c_dev.size == c_arb.size == c_ser.size, where
        e_c = _rel_inf(c_dev, c_arb)
        tol_c = sp_c.tol(_rel_inf(c_ser, c_arb))
        assert e_c <= (1e-12 if iid else tol_c), (where, "c", e_c, tol_c)
        worst["c_iid" if iid else "c_collinear"] = max(worst["c_iid" if iid else "c_collinear"], e_c)

        # the Gram entries (newer, older), the factor (older, newer) and its diagonal among those pairs
        if slots:
            ix = np.ix_(slots, slots)
            h_dev, h_arb, h_ser = st["h"][ix], arb.h()[ix], ser.h()[ix]
            e_h = _rel_inf(h_dev, h_arb)
            tol_h = sp_h.tol(_rel_inf(h_ser, h_arb))
            assert e_h <= (1e-12 if iid else tol_h), (where, "h", e_h, tol_h)
            worst["h_iid" if iid else "h_collinear"] = max(worst["h_iid" if iid else "h_collinear"], e_h)

        # min over the Cholesky rows of hkk - vtol^2 (no row: the arbiter says inf, the device 1e300)
        m_arb, m_ser, m_dev = arb.min_margin(), ser.min_margin(), st["min_margin"]
        if np.isinf(m_arb):
            assert m_dev >= 1e299 and np.isinf(m_ser), where
        else:
            e_m = abs(m_dev - m_arb)
            tol_m = sp_m.tol(abs(m_ser - m_arb))
            assert e_m <= (1e-12 if iid else tol_m), (where, "min_margin", e_m, tol_m)
            worst["margin"] = max(worst["margin"], e_m)
        it += 1
    assert acc.defined()
    acc.delete()


def _sweep_shapes():
    for mvec in range(1, 33):
        for placement in PLACEMENTS:
            yield N_ODD, mvec, placement
            if mvec in SMALL_N_WIDTHS:
                yield N_SMALL, mvec, placement


_MODE_LEDGERS = {}


def _run_mode(mode):
    """The whole sweep in one mode (memoised: the ledger test reuses what the per-mode tests ran)."""
    if mode not in _MODE_LEDGERS:
        ledger_a, ledger_b = set(), set()
        with pytest.MonkeyPatch.context() as mp:
            if mode == "eager":
                mp.setenv("NKA_LAZY_LAST", "0")     # read when the handle is created
            else:
                mp.delenv("NKA_LAZY_LAST", raising=False)
            worst = {}
            for n, mvec, placement in _sweep_shapes():
                w = worst.setdefault(mvec, dict.fromkeys(("out", "c_iid", "c_collinear", "h_iid", "h_collinear",
                                                          "margin"), 0.0))
                run_checked(n, mvec, placement, mode, ledger_a, ledger_b, w)
            for mvec, w in worst.items():
                record_parity("kernel_matrix_%s_m%02d" % (mode, mvec), mvec=mvec, vtol=VTOL,
                              **{"worst_" + k: v for k, v in w.items()})
        _MODE_LEDGERS[mode] = (ledger_a, ledger_b)
    return _MODE_LEDGERS[mode]


@pytest.mark.parametrize("mode", MODES)
def test_kernel_matrix_matches_reference(mode):
    """Every width 1..32, f aligned and 8 bytes off, odd n = 1001 (and n = 201 at a few widths).  Per call:
    decisions equal to the serial reference; output within the S.tolerances bar of the long-double arbiter;
    c, h (the pairs on the list, the reference's slots) and min_margin within 1e-12 of it during the i.i.d.
    calls and within 4x the reference's own serial-vs-long-double spread during the collinear ones.
    eager: NKA_LAZY_LAST=0, pass A streams NC = 33 at mvec = 32.  dp: the reference's dot-product hook,
    so pass A is not fused with the state step, which runs as a kernel of its own with up to 33 columns."""
    _run_mode(mode)


def test_every_kernel_and_body_ran():
    """The ledger of the three sweeps: all 66 pass A and all 66 pass B kernels ran, and both the FULL and
    the general body of every NC >= 2 and NZ >= 1, at V = 1 and V = 2."""
    ran = set()
    for mode in MODES:
        la, lb = _run_mode(mode)
        ran |= {("A",) + k for k in la} | {("A",) + k[:2] for k in la}
        ran |= {("B",) + k for k in lb} | {("B",) + k[:2] for k in lb}
    want = [("A", nc, v) for nc in range(1, MAXSLOT + 1) for v in (1, 2)]
    want += [("B", nz, v) for nz in range(0, MAXSLOT) for v in (1, 2)]
    want += [("A", nc, v, full) for nc in range(2, MAXSLOT + 1) for v in (1, 2) for full in (True, False)]
    want += [("B", nz, v, full) for nz in range(1, MAXSLOT) for v in (1, 2) for full in (True, False)]
    kernels = [k for k in want if len(k) == 3 and k in ran]
    print("kernel ledger: %d pass A and %d pass B kernels ran; %d (kernel, V, FULL) bodies"
          % (sum(k[0] == "A" for k in kernels), sum(k[0] == "B" for k in kernels), sum(len(k) == 4 for k in ran)))
    assert not [k for k in want if k not in ran and k not in UNREACHED]
    assert not [k for k in UNREACHED if k in ran], "listed as unreached but ran"
    assert len(kernels) == 132


# ---------------------------------------------------------------------------------------------------
# Poisoned allocations and guard words
# ---------------------------------------------------------------------------------------------------
def _run_device(n, mvec, vtol, ops, placement="aligned", guard=False):
    """Outputs and (c, h, s) after every update of a device run; guards checked after every update."""
    from nka_b200 import NKA
    acc = NKA(n, mvec, vtol)
    dev = Placed(n, placement, guard=guard)
    outs, states = [], []
    for op in ops:
        if op[0] == "update":
            dev.load(op[1])
            acc.accel_update(dev.f)
            outs.append(dev.read())
            st = acc.state()
            assert st["error"] == 0
            states.append(np.concatenate([st["c"], st["h"].ravel(), st["s"]]))
            assert dev.guards_intact(), ("write past the ends of f", n, mvec, placement, len(outs))
        elif op[0] == "relax":
            acc.relax()
        else:
            acc.restart()
    acc.delete()
    return outs, states


def _poisoned_equals_plain(n, mvec, vtol, ops, placement="aligned"):
    with pytest.MonkeyPatch.context() as mp:
        mp.delenv("NKA_POISON_ALLOC", raising=False)
        plain = _run_device(n, mvec, vtol, ops, placement)
        mp.setenv("NKA_POISON_ALLOC", "1")          # read when the handle is created
        poisoned = _run_device(n, mvec, vtol, ops, placement)
    for k, (a, b) in enumerate(zip(plain[0] + plain[1], poisoned[0] + poisoned[1])):
        assert np.all(np.isfinite(b)), ("non-finite result with poisoned buffers", n, mvec, placement, k)
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), ("poison changed a result", n, mvec, placement, k)


@pytest.mark.parametrize("name", sorted(S.SCENARIOS))
def test_poisoned_buffers_change_nothing_scenarios(name):
    """NKA_POISON_ALLOC=1 fills W and Z (whole pools, padding included), the partial rows and dots with NaN
    bytes: outputs and c, h, s after every call are bit-identical to a run on cudaMalloc's memory, and finite.
    A stale value read under a zero coefficient is invisible on zeroed memory and NaN here."""
    n, mvec, vtol, mk = S.SCENARIOS[name]
    _poisoned_equals_plain(n, mvec, vtol, mk())


@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("mvec", POISON_WIDTHS)
def test_poisoned_buffers_change_nothing_sweep(mvec, placement):
    """The kernel-matrix sequence at the widths where pass B changes shape (12 | 13: coefficients move to
    shared memory; 23 | 24: 256 threads) and at both ends, f aligned and 8 bytes off."""
    ops, _ = sweep_ops(N_ODD, mvec)
    _poisoned_equals_plain(N_ODD, mvec, VTOL, ops, placement)


def test_poisoned_buffers_change_nothing_chunked_host_path():
    """Host f through the chunked pipeline (NKA_HOST_CHUNK_BYTES=256: up to 16 chunks, several launches per
    sweep folding one set of partial rows), with the staging buffer poisoned too: bit-identical."""
    from nka_b200 import _lib
    lib = _lib.load()

    def run():
        outs = []
        for name in ("odd_n1023_m7", "picard_n500_m5_v2", "mixed_n257_m5", "iid_n1000_m10"):
            n, mvec, vtol, mk = S.SCENARIOS[name]
            h = lib.nka_init(n, mvec, vtol, None)
            for op in mk():
                if op[0] == "update":
                    got = op[1].copy()
                    lib.nka_accel_update(h, got.ctypes.data)
                    outs.append(got)
                elif op[0] == "relax":
                    lib.nka_relax(h)
                else:
                    lib.nka_restart(h)
            assert lib.nka_defined(h)
            lib.nka_delete(h)
        return outs

    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("NKA_HOST_CHUNK_BYTES", "256")
        mp.delenv("NKA_POISON_ALLOC", raising=False)
        plain = run()
        mp.setenv("NKA_POISON_ALLOC", "1")
        poisoned = run()
    assert len(plain) == len(poisoned)
    for a, b in zip(plain, poisoned):
        assert np.all(np.isfinite(b)) and np.array_equal(a.view(np.int64), b.view(np.int64))


@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("mvec", (1, 13, 24, 32))
def test_guard_words_around_f(mvec, placement):
    """NaN sentinels next to f (aligned f with odd n: buf[n], in the last element's 16-byte word; f 8 bytes
    off: buf[0] and buf[n+1]) keep their bits through every update (nothing is written out of range), and
    the results equal those of a run with zeros there (nothing out of range is read)."""
    for n in (N_ODD, N_SMALL):
        ops, _ = sweep_ops(n, mvec)
        plain = _run_device(n, mvec, VTOL, ops, placement)
        guarded = _run_device(n, mvec, VTOL, ops, placement, guard=True)
        for a, b in zip(plain[0] + plain[1], guarded[0] + guarded[1]):
            assert np.array_equal(a.view(np.int64), b.view(np.int64)), (n, mvec, placement)
