"""Pin the oracle: the C restatement against the reference's own golden
tables and against outputs of the compiled reference (SURVEY.md 8c).

CPU only.  The goldens under tests/golden/ were produced by tests/golden/make_golden.py
from the reference's sources and compiled library (accel_dp_golden.json names its own
source); nothing here reads the reference's sources.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import scenarios as S
from oracle import api

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _table_blocks():
    with open(os.path.join(GOLD, "example_c_f95.txt")) as fh:
        text = fh.read()
    acc, unacc = text.split("UNACCELERATED SOLVE")
    pick = lambda blk: [ln for ln in blk.splitlines() if ln[:4].strip().rstrip(":").isdigit() and ":" in ln[:4]]
    return pick(acc), pick(unacc)


def test_example_table_f95_c_accelerated():
    """src-F95/reference_output:5-31 == src-C/reference_output: 26 iterations, every line."""
    want, _ = _table_blocks()
    got = api.format_table(api.example_solve(mvec=5, scaling=0, flavour=0)["rnorm"])
    assert len(want) == 27
    assert got == want


def test_example_table_f95_c_unaccelerated():
    """src-F95/reference_output:36-403: 367 iterations, every line."""
    _, want = _table_blocks()
    got = api.format_table(api.example_solve(mvec=0, scaling=0)["rnorm"])
    assert len(want) == 368
    assert got == want


def test_example_f08_last_lines():
    """src-F08/reference_output:7,16,25 (== src-F08-vector/reference_output)."""
    with open(os.path.join(GOLD, "example_f08.json")) as fh:
        runs = json.load(fh)["runs"]
    assert len(runs) == 3
    for run in runs:
        args = run["args"]
        mvec = int(args[args.index("--nka-vec") + 1]) if "--nka-vec" in args else 0
        nsweep = int(args[args.index("--sweeps") + 1]) if "--sweeps" in args else 2
        res = api.example_solve(mvec=mvec, nsweep=nsweep, scaling=1, flavour=1)
        assert api.format_table(res["rnorm"])[-1] == run["last_line"]


def test_example_num_vec_sequence():
    """SURVEY.md 3.3: num_vec after each call is 0,1,2,3,4,5,5,... and no vtol drop fires."""
    res = api.example_solve(mvec=5, record=True)
    assert list(res["nvec"]) == [0, 1, 2, 3, 4] + [5] * 21


with open(os.path.join(GOLD, "accel_golden.json")) as _fh:
    _GOLD = json.load(_fh)


@pytest.mark.parametrize("name", sorted(S.SCENARIOS))
def test_oracle_bit_identical_to_compiled_reference(name):
    """Every correction vector of the port has the sha256 the compiled
    reference library produced; num_vec (i.e. every drop decision) matches."""
    n, mvec, vtol, mk = S.SCENARIOS[name]
    g = _GOLD[name]
    assert (g["n"], g["mvec"], g["vtol"]) == (n, mvec, vtol)
    ops = mk()
    assert [op[0] for op in ops] == g["ops"]
    assert [hashlib.sha256(op[1].tobytes()).hexdigest() for op in ops if op[0] == "update"] == g["in_sha256"]
    acc = api.OracleNKA(n, mvec, vtol, dotmode=0, flavour=0)
    outs, nvecs = S.run_ops(acc, ops)
    assert acc.defined()
    assert nvecs == g["num_vec"]
    assert [hashlib.sha256(o.tobytes()).hexdigest() for o in outs] == g["sha256"]


def test_small_goldens_match_npz():
    small = np.load(os.path.join(GOLD, "accel_small.npz"))
    for name in small.files:
        n, mvec, vtol, mk = S.SCENARIOS[name]
        outs, _ = S.run_ops(api.OracleNKA(n, mvec, vtol), mk())
        assert np.array_equal(np.stack(outs), small[name])


@pytest.mark.parametrize("name", ["iid_n1000_m10", "picard_n500_m5", "contraction_n200_m5"])
def test_long_double_arbiter_close_to_serial(name):
    """The long-double-dot arbiter (used above n = 2^18) agrees with the serial
    reference to rounding on small problems, with identical drop decisions."""
    n, mvec, vtol, mk = S.SCENARIOS[name]
    a, nva = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), mk())
    b, nvb = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), mk())
    assert nva == nvb
    for x, y in zip(a, b):
        assert np.linalg.norm(x - y) <= 1e-9 * np.linalg.norm(x)


def test_flavours_differ_only_by_rounding():
    n, mvec, vtol, mk = S.SCENARIOS["iid_n1000_m10"]
    a, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, flavour=0), mk())
    b, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, flavour=1), mk())
    for x, y in zip(a, b):
        assert np.linalg.norm(x - y) <= 1e-14 * np.linalg.norm(x)


with open(os.path.join(GOLD, "accel_dp_golden.json")) as _fh:
    _GOLD_DP = json.load(_fh)


def test_compiled_reference_matches_port_when_present():
    """The long-double arbiter (the port with dotmode = 1, and the port with the same dot product
    handed to its dp hook) reproduces the stored digests of every call and num_vec; the file's
    "source" says what produced them.  If oracle/_ref/libnka_ref.so travelled with the tree, the
    reference itself is cross-checked live as well, in serial mode and through its dp hook."""
    n, mvec, vtol, mk = S.SCENARIOS["picard_n500_m5_v2"]
    g = _GOLD_DP["picard_n500_m5_v2"]
    assert (g["n"], g["mvec"], g["vtol"]) == (n, mvec, vtol)
    hook = C.cast(api.oracle_lib().orc_dp_long_double, C.c_void_p)
    for acc in (api.OracleNKA(n, mvec, vtol, dotmode=1), api.OracleNKA(n, mvec, vtol, dp=hook)):
        outs, nvecs = S.run_ops(acc, mk())
        assert nvecs == g["num_vec"]
        assert [hashlib.sha256(o.tobytes()).hexdigest() for o in outs] == g["sha256"]
    if api.ref_lib() is None:
        return
    a, nva = S.run_ops(api.RefNKA(n, mvec, vtol), mk())
    b, nvb = S.run_ops(api.OracleNKA(n, mvec, vtol), mk())
    assert nva == nvb
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    # and the arbiter through the reference's own dp hook
    c, _ = S.run_ops(api.RefNKA(n, mvec, vtol, long_double_dp=True), mk())
    d, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), mk())
    assert all(np.array_equal(x, y) for x, y in zip(c, d))


def test_queries_and_preconditions():
    acc = api.OracleNKA(10, 3, 0.02)
    assert (acc.vec_len(), acc.max_vec(), acc.vec_tol(), acc.num_vec()) == (10, 3, 0.02, 0)
    acc.set_vec_tol(0.5)
    assert acc.vec_tol() == 0.5
    assert acc.defined()
    with pytest.raises(ValueError):
        api.OracleNKA(10, 0, 0.01)
    with pytest.raises(ValueError):
        api.OracleNKA(10, 3, 0.0)
