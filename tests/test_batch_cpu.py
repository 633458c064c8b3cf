"""The batched accelerator without a GPU: argument checks of BatchNKA that raise before any CUDA call,
and the code-generation properties of the batched kernels (cuobjdump on the objects nvcc wrote)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batch_init_validates_before_any_cuda_call():
    from nka_b200 import BatchNKA
    b = BatchNKA()
    for bad in [dict(nbatch=0, vlen=10, mvec=3), dict(nbatch=65536, vlen=10, mvec=3), dict(nbatch=-1, vlen=10, mvec=3),
                dict(nbatch=4, vlen=10, mvec=33), dict(nbatch=4, vlen=10, mvec=0), dict(nbatch=4, vlen=0, mvec=3),
                dict(nbatch=4, vlen=10, mvec=3, vtol=0.0)]:
        with pytest.raises(ValueError):
            b.init(**bad)
    assert not b.defined()


def _unbuilt(nbatch, vlen):
    """A BatchNKA that knows its shape but holds no handle: any call reaching the library would fail."""
    from nka_b200 import BatchNKA
    b = BatchNKA()
    b.nbatch, b.vlen, b.mvec = nbatch, vlen, 3
    return b


def test_batch_update_validates_f_and_masks_before_any_cuda_call():
    import numpy as np
    import torch
    b = _unbuilt(4, 10)
    cases = {
        "numpy": (np.zeros((4, 10)), "CUDA float64"),
        "float32": (torch.zeros(4, 10, dtype=torch.float32), "float64"),
        "1-D": (torch.zeros(40, dtype=torch.float64), "shape"),
        "rows": (torch.zeros(5, 10, dtype=torch.float64), "shape"),
        "cols": (torch.zeros(4, 11, dtype=torch.float64), "shape"),
        "column stride": (torch.zeros(10, 4, dtype=torch.float64).t(), "stride"),
        "row stride": (torch.zeros(40, dtype=torch.float64).as_strided((4, 10), (5, 1)), "row stride"),
        "cpu tensor": (torch.zeros(4, 10, dtype=torch.float64), "CUDA"),
    }
    for name, (F, what) in cases.items():
        with pytest.raises(ValueError, match=what):
            b.accel_update(F)
    for mask in (np.ones(4, dtype=bool), torch.ones(4, dtype=torch.bool), torch.ones(4, dtype=torch.int32),
                 torch.ones(5, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            b.relax(mask)
        with pytest.raises(ValueError):
            b.restart(mask)
    with pytest.raises(ValueError):
        b.set_vec_tol(0.0)
    with pytest.raises(ValueError):
        b.state(4)


# ---------------------------------------------------------------------------------------------
# code generation of the batched kernels
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def objdir():
    from nka_b200 import build
    build.build_library()
    return build.LIB_DIR


def _res_usage(obj):
    out = subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True, check=True).stdout
    res = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out):
        res[m.group(1)] = {"reg": int(m.group(2)), "stack": int(m.group(3)), "shared": int(m.group(4)),
                           "local": int(m.group(5))}
    return res


def _sass(obj, fun):
    return subprocess.run(["cuobjdump", "-sass", "-fun", fun, obj], capture_output=True, text=True, check=True).stdout


def test_batched_kernels_do_not_spill(objdir):
    seen = 0
    for obj in ("nka_batch.o", "nka_batch_pass_a.o", "nka_batch_pass_b.o"):
        for name, r in _res_usage(os.path.join(objdir, obj)).items():
            assert r["local"] == 0, (obj, name, r)
            seen += 1
    assert seen == 2 * 33 + 2 * 33 + 8


def test_batched_sweeps_fit_their_ctas_and_are_vectorised(objdir):
    a = _res_usage(os.path.join(objdir, "nka_batch_pass_a.o"))
    b = _res_usage(os.path.join(objdir, "nka_batch_pass_b.o"))
    names_b = [n for n in b if n.startswith("_Z16nka_batch_pass_bILi")]
    assert len(names_b) == 66
    for name in names_b:
        nz = int(re.match(r"_Z16nka_batch_pass_bILi(\d+)E", name).group(1))
        # 512-thread CTAs below 24 columns (coefficients in registers below 13): 65536 registers per SM / 512
        assert b[name]["reg"] <= (128 if nz < 24 else 255), (name, b[name])
    assert len([n for n in a if n.startswith("_Z16nka_batch_pass_aILi")]) == 66
    fa = [n for n in a if n.startswith("_Z16nka_batch_pass_aILi10ELi2E")][0]
    assert "LDG.E.128" in _sass(os.path.join(objdir, "nka_batch_pass_a.o"), fa)
    fb = [n for n in b if n.startswith("_Z16nka_batch_pass_bILi10ELi2E")][0]
    sass = _sass(os.path.join(objdir, "nka_batch_pass_b.o"), fb)
    assert "LDG.E.128" in sass and "STG.E.128" in sass


def test_batched_state_kernel_staging_fits_without_opt_in(objdir):
    res = _res_usage(os.path.join(objdir, "nka_batch.o"))
    st = [n for n in res if "nka_batch_state_kernel" in n]
    assert len(st) == 1
    assert 3 * 12 * 1024 <= res[st[0]]["shared"] <= 48 * 1024, res[st[0]]
