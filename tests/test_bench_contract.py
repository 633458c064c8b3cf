"""bench.py's contract on the CPU: the reference arm prints one JSON line with the keys the driver reads (timed
on a small slice here), ranks other than 0 stay silent, and our own arm refuses to run without a CUDA device
instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run(["--impl", "reference", "--n", str(1 << 18), "--mvec", "4", "--steps", "3", "--warmup", "1"])
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "accel_update/sec" and d["unit"] == "updates/s"
    assert d["higher_is_better"] is True and d["steps"] == 3 and d["warmup"] == 1 and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 1 and cb["value"] == d["value"]
    assert cb["n_sample"] * cb["extrapolation_factor"] == 1 << 18
    assert d["e2e"] == {"value": d["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["n"] == 1 << 18


def test_reference_arm_other_ranks_exit_silently():
    r = _run(["--impl", "reference", "--gpus", "2", "--n", str(1 << 16), "--steps", "1", "--warmup", "1"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dumps_the_output_of_its_last_timed_step(tmp_path):
    """--dump-outputs writes the f the last of the --steps timed calls returned: the same calls on the port
    (bit-identical to the reference in serial mode) give it bit for bit."""
    import numpy as np
    from oracle import api
    n, mvec, steps, warmup = 1 << 16, 4, 3, 1
    r = _run(["--impl", "reference", "--n", str(n), "--mvec", str(mvec), "--steps", str(steps), "--warmup", str(warmup),
              "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.splitlines()[-1])["cpu_baseline"]["n_sample"] == n
    got = np.load(tmp_path / "f.npy")
    rng = np.random.default_rng(1234)
    pool = [rng.random(n) - 0.5 for _ in range(mvec + 3)]
    acc = api.OracleNKA(n, mvec, 0.01)
    calls = mvec + 2 + warmup + steps
    for k in range(calls):
        acc.accel_update(pool[k % len(pool)])
    assert got.dtype == np.float64 and np.array_equal(got, pool[(calls - 1) % len(pool)])


@pytest.mark.gpu
def test_our_arm_dumps_a_fixed_sample_of_its_last_timed_step(tmp_path):
    """Above bench.DUMP_MAX elements --dump-outputs writes a fixed sample of the last timed step's f; the same
    inputs and number of calls through the library directly give the same values bit for bit (fixed-order
    reductions).  This checks what is dumped and where it is sampled; the values themselves are checked
    against the oracle by the parity tests."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from nka_b200 import NKA
    n, mvec, steps, warmup = (1 << 22) + 6, 4, 3, 1
    r = _run(["--n", str(n), "--mvec", str(mvec), "--steps", str(steps), "--warmup", str(warmup), "--no-e2e",
              "--no-cpu-baseline", "--no-probe", "--no-sweep", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.splitlines()[-1])["steps"] == steps
    got = np.load(tmp_path / "f.npy")
    idx = bench.dump_index(n)
    assert got.dtype == np.float64 and got.shape == idx.shape == (bench.DUMP_MAX,)
    assert np.all(np.diff(idx) > 0) and idx[-1] < n
    gen = torch.Generator(device="cuda").manual_seed(1000)
    pool = [torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) - 0.5 for _ in range(mvec + 3)]
    acc = NKA(n, mvec, 0.01)
    calls = mvec + 2 + warmup + steps
    for k in range(calls):
        acc.accel_update(pool[k % len(pool)])
    torch.cuda.synchronize()
    want = pool[(calls - 1) % len(pool)].cpu().numpy()[idx]
    acc.delete()
    assert np.array_equal(got, want)


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "CUDA device" in (r.stderr + r.stdout)
