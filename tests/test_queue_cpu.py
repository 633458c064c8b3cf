"""Device-side work queues without a GPU: the argument checks of BatchNKA.fixed_point_queue that raise before
any CUDA call, and the code generation of the queue's kernels (cuobjdump on nka_batch_queue.o)."""
import os

import pytest

from test_batch_cpu import _unbuilt
from test_loop_cpu import _res_usage, _sass


def test_fixed_point_queue_validates_before_any_cuda_call():
    import numpy as np
    import torch
    b = _unbuilt(4, 10)
    f64 = dict(dtype=torch.float64)
    rows = torch.zeros(4, 10, **f64)                      # CPU tensors: each case fails before the device checks
    slot = torch.zeros(4, dtype=torch.int32)
    X0 = torch.zeros(9, 10, **f64)
    for kw, what in [(dict(atol=-1.0), "atol"), (dict(rtol=float("nan")), "rtol"), (dict(maxit=-1), "maxit"),
                     (dict(maxit=1.5), "maxit")]:
        with pytest.raises(ValueError, match=what):
            b.fixed_point_queue(lambda: None, rows, rows, slot, X0, **kw)
    bad_slot = [np.zeros(4, dtype=np.int32), torch.zeros(4, dtype=torch.int64), torch.zeros(5, dtype=torch.int32),
                torch.zeros(4, 1, dtype=torch.int32), torch.zeros(8, dtype=torch.int32)[::2]]
    for sp in bad_slot:
        with pytest.raises(ValueError, match="slot_problem"):
            b.fixed_point_queue(lambda: None, rows, rows, sp, X0)
    bad_rows = {
        "numpy": (np.zeros((9, 10)), "CUDA float64"),
        "float32": (torch.zeros(9, 10, dtype=torch.float32), "float64"),
        "1-D": (torch.zeros(90, **f64), "shape"),
        "vlen": (torch.zeros(9, 11, **f64), "shape"),
        "no problems": (torch.zeros(0, 10, **f64), "problems"),
        "column stride": (torch.zeros(10, 9, **f64).t(), "stride"),
        "row stride": (torch.zeros(90, **f64).as_strided((9, 10), (5, 1)), "row stride"),
    }
    for name, (T, what) in bad_rows.items():
        with pytest.raises(ValueError, match=what):
            b.fixed_point_queue(lambda: None, rows, rows, slot, T)
        if name != "no problems":
            with pytest.raises(ValueError, match="Xout" if what != "CUDA float64" else what):
                b.fixed_point_queue(lambda: None, rows, rows, slot, X0, T)
    with pytest.raises(ValueError, match="Xout"):
        b.fixed_point_queue(lambda: None, rows, rows, slot, X0, torch.zeros(8, 10, **f64))
    # structurally good arguments: the first device check refuses the CPU tensors
    with pytest.raises(ValueError, match="slot_problem must be a CUDA tensor"):
        b.fixed_point_queue(lambda: None, rows, rows, slot, X0)


@pytest.fixture(scope="module")
def obj():
    from nka_b200 import build
    build.build_library()
    return os.path.join(build.LIB_DIR, "nka_batch_queue.o")


def test_queue_kernels_have_no_local_memory(obj):
    res = _res_usage(obj)
    assert len(res) == 4, sorted(res)                 # reset, claim, rows<1|2>
    assert all(local == 0 for local in res.values()), res


def test_queue_rows_use_16_byte_accesses(obj):
    res = _res_usage(obj)
    rows = [n for n in res if n.startswith("_Z14nka_queue_rowsILi2E")]
    assert len(rows) == 1
    sass = _sass(obj, rows[0])
    assert "LDG.E.128" in sass and "STG.E.128" in sass


def test_claim_stays_in_static_shared_memory(obj):
    """One CTA of 1024 threads whatever nbatch is: its scan keeps one int per warp in a static shared array
    of its own, a few hundred bytes, so it fits any SM without asking for dynamic shared memory."""
    import re
    import subprocess
    out = subprocess.run(["cuobjdump", "-elf", obj], capture_output=True, text=True, check=True).stdout
    usage = subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True, check=True).stdout
    claim = [n for n in _res_usage(obj) if n.startswith("_Z15nka_queue_claim")]
    assert len(claim) == 1
    assert ".nv.shared." + claim[0] in out                  # a static shared section of its own
    shared = int(re.search(r"Function %s:\s*\n\s*REG:\d+ STACK:\d+ SHARED:(\d+)" % re.escape(claim[0]), usage).group(1))
    assert 32 * 4 <= shared <= 2048, shared                 # the warp totals (plus what the toolchain reserves)
