"""CPU check of the device algorithm's scalar half.

tests/model/ compiles nka_b200/csrc/nka_state.h -- the exact code the state
kernel runs on the device -- for the host, with plain-loop stand-ins for the
streaming kernels.  Run against the oracle this pins the raw-chain storage
scheme, the materialisation rule, the drop/evict/relax decisions and the host
bookkeeping (pending flag, list-length bound) without a GPU.  The product
never uses this model; the -m gpu tests check the real kernels.
"""
import os
import subprocess

import numpy as np
import pytest

import scenarios as S
from model import ModelNKA
from oracle import api

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("lazy", [True, False])
@pytest.mark.parametrize("name", sorted(S.SCENARIOS))
def test_model_matches_oracle(name, lazy):
    n, mvec, vtol, mk = S.SCENARIOS[name]
    ops = mk()
    inputs = [op[1] for op in ops if op[0] == "update"]
    serial, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=0), ops)
    arbiter, _ = S.run_ops(api.OracleNKA(n, mvec, vtol, dotmode=1), ops)
    scales, tols = S.tolerances(serial, arbiter, inputs)
    orc = api.OracleNKA(n, mvec, vtol, dotmode=1)
    mod = ModelNKA(n, mvec, vtol, lazy=lazy)
    it = 0
    for op in ops:
        if op[0] == "update":
            fin = op[1]
            a, b = fin.copy(), fin.copy()
            orc.accel_update(a)
            mod.accel_update(b)
            assert (orc.ndrop_last(), orc.relaxed_last(), orc.evicted_last()) == \
                   (mod.ndrop_last(), bool(mod.relaxed_last()), bool(mod.evicted_last()))
            assert np.linalg.norm(a - b) / scales[it] <= tols[it], (name, it)
            it += 1
        elif op[0] == "relax":
            orc.relax(); mod.relax()
        else:
            orc.restart(); mod.restart()
        assert orc.num_vec() == mod.num_vec()
        assert mod.defined() and mod.error() == 0
        assert mod.host_pending() == mod.dev_pending()
        assert mod.list_len() <= mod.ub_len()
    assert mod.bound_violations() == 0


def test_model_materialises_only_on_breaks():
    """No vtol drop, no relax, no s == 0: the chain is never materialised."""
    n, mvec, vtol, mk = S.SCENARIOS["iid_n1000_m10"]
    mod = ModelNKA(n, mvec, vtol)
    S.run_ops(mod, mk())
    assert mod.mat_entries() == 0
    n, mvec, vtol, mk = S.SCENARIOS["relax_restart_n96_m4"]
    mod = ModelNKA(n, mvec, vtol)
    S.run_ops(mod, mk())
    assert mod.mat_entries() > 0


def test_lazy_last_column_fixup_is_exercised_and_bit_identical():
    """Skipping the doomed oldest column must not change a single bit: when a vtol drop (or the
    s == 0 guard) keeps that column after all, the fix-up supplies its two dot products."""
    for name in ("picard_n500_m5_v2", "repeats_n128_m4", "mixed_n257_m5"):
        n, mvec, vtol, mk = S.SCENARIOS[name]
        lazy, eager = ModelNKA(n, mvec, vtol, lazy=True), ModelNKA(n, mvec, vtol, lazy=False)
        a, nva = S.run_ops(lazy, mk())
        b, nvb = S.run_ops(eager, mk())
        assert lazy.fixups() > 0 and eager.fixups() == 0
        assert nva == nvb
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _write_sequence(path, n, mvec, vtol, ops):
    """The op-sequence file tests/model/lanes_test.cpp reads."""
    with open(path, "wb") as fh:
        fh.write(np.array([n, mvec, len(ops)], dtype=np.int32).tobytes())
        fh.write(np.array([vtol], dtype=np.float64).tobytes())
        for op in ops:
            fh.write(np.array([("update", "relax", "restart").index(op[0])], dtype=np.int32).tobytes())
            if op[0] == "update":
                fh.write(np.ascontiguousarray(op[1], dtype=np.float64).tobytes())


def _lanes_inputs(tmp_path):
    files = []
    for name in sorted(S.SCENARIOS):
        n, mvec, vtol, mk = S.SCENARIOS[name]
        files.append(str(tmp_path / (name + ".seq")))
        _write_sequence(files[-1], n, mvec, vtol, mk())
    return files


def _build_lanes(tmp_path, *flags):
    exe = tmp_path / "lanes_test"
    r = subprocess.run(["g++", "-std=c++17", "-ffp-contract=off", "-pthread", "-Wall", *flags,
                        os.path.join(HERE, "model", "lanes_test.cpp"), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


def test_state_step_is_bit_identical_on_any_number_of_lanes(tmp_path):
    """The device runs the state step on the 32 lanes of a warp, synchronised by __syncwarp() (nka_state.h:
    par.sync()); the host model runs it on one.  Here every scenario, lazy column on and off, runs on 2, 3, 32
    and 33 host threads whose par.sync() is a barrier (tests/model/lanes_test.cpp): outputs and h, c, s after
    every op equal the one-lane run bit for bit.  The same driver also starts the one-lane model from a state
    filled with 0xFF bytes (NaN doubles) before nka_state_init, and requires the same bits: init sets
    everything the step reads, as it must on the device, where the state lives in uninitialised memory."""
    exe = _build_lanes(tmp_path, "-O2")
    r = subprocess.run([exe, *_lanes_inputs(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "lanes ok" in r.stdout, r.stdout + r.stderr


def test_state_step_lanes_have_no_data_race(tmp_path):
    """The same driver under ThreadSanitizer: a par.sync() missing between a write and a read of another
    lane is reported as a data race even in a run whose bits happen to come out right."""
    exe = _build_lanes(tmp_path, "-O1", "-g", "-fsanitize=thread")
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=1 exitcode=66")
    r = subprocess.run([exe, *_lanes_inputs(tmp_path)], capture_output=True, text=True, timeout=1200, env=env)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[-4000:]
    assert r.returncode == 0 and "lanes ok" in r.stdout, r.stdout + r.stderr[-4000:]
