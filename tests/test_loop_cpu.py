"""Device-side fixed-point loops without a GPU: the argument checks of BatchNKA.fixed_point_loop that raise
before any CUDA call, and the code generation of the loop's kernels (cuobjdump on nka_batch_loop.o)."""
import os
import re
import subprocess

import pytest

from test_batch_cpu import _unbuilt


def test_fixed_point_loop_validates_before_any_cuda_call():
    import numpy as np
    import torch
    b = _unbuilt(4, 10)
    good = torch.zeros(4, 10, dtype=torch.float64)          # a CPU tensor: fails the last check, on "CUDA"
    bad = {
        "numpy": (np.zeros((4, 10)), "CUDA float64"),
        "float32": (torch.zeros(4, 10, dtype=torch.float32), "float64"),
        "rows": (torch.zeros(5, 10, dtype=torch.float64), "shape"),
        "column stride": (torch.zeros(10, 4, dtype=torch.float64).t(), "stride"),
        "row stride": (torch.zeros(40, dtype=torch.float64).as_strided((4, 10), (5, 1)), "row stride"),
        "cpu tensor": (good, "CUDA"),
    }
    for name, (T, what) in bad.items():
        with pytest.raises(ValueError, match=what):
            b.fixed_point_loop(lambda: None, T, good)
        with pytest.raises(ValueError):
            b.fixed_point_loop(lambda: None, good, T)
    # tolerances and maxit are checked first
    for kw, what in [(dict(atol=-1.0), "atol"), (dict(atol=float("nan")), "atol"), (dict(rtol=-1e-8), "rtol"),
                     (dict(rtol="1e-8"), "rtol"), (dict(maxit=-1), "maxit"), (dict(maxit=2.5), "maxit"),
                     (dict(maxit=True), "maxit")]:
        with pytest.raises(ValueError, match=what):
            b.fixed_point_loop(lambda: None, good, good, **kw)


@pytest.fixture(scope="module")
def obj():
    from nka_b200 import build
    build.build_library()
    return os.path.join(build.LIB_DIR, "nka_batch_loop.o")


def _res_usage(path):
    out = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True, check=True).stdout
    return {m.group(1): int(m.group(2))
            for m in re.finditer(r"Function (\S+):\s*\n\s*REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:(\d+)", out)}


def _sass(path, fun):
    return subprocess.run(["cuobjdump", "-sass", "-fun", fun, path], capture_output=True, text=True, check=True).stdout


def test_loop_kernels_have_no_local_memory(obj):
    res = _res_usage(obj)
    assert len(res) == 6, sorted(res)                 # reset, decide, check<1|2>, step<1|2>
    assert all(local == 0 for local in res.values()), res


def test_loop_check_and_step_use_16_byte_accesses(obj):
    res = _res_usage(obj)
    check = [n for n in res if n.startswith("_Z14nka_loop_checkILi2E")]
    step = [n for n in res if n.startswith("_Z13nka_loop_stepILi2E")]
    assert len(check) == 1 and len(step) == 1
    assert "LDG.E.128" in _sass(obj, check[0])
    sass = _sass(obj, step[0])
    assert "LDG.E.128" in sass and "STG.E.128" in sass
