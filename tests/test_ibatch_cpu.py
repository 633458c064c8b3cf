"""The interleaved batched accelerator without a GPU: argument checks of InterleavedBatchNKA that raise before
any CUDA call, its ctypes signatures against the header, and the code generation of its kernels (cuobjdump on
the object nvcc wrote, and on the same translation unit rebuilt with -fmad=false)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_init_validates_before_any_cuda_call():
    from nka_b200 import InterleavedBatchNKA
    acc = InterleavedBatchNKA()
    for bad in [dict(nbatch=0, vlen=10, mvec=3), dict(nbatch=2**31, vlen=10, mvec=3), dict(nbatch=-1, vlen=10, mvec=3),
                dict(nbatch=4, vlen=10, mvec=33), dict(nbatch=4, vlen=10, mvec=0), dict(nbatch=4, vlen=0, mvec=3),
                dict(nbatch=4, vlen=10, mvec=3, vtol=0.0), dict(nbatch=4, vlen=10, mvec=3, vtol=float("nan"))]:
        with pytest.raises(ValueError):
            acc.init(**bad)
    assert not acc.defined()


def _unbuilt(nbatch, vlen):
    """An InterleavedBatchNKA that knows its shape but holds no handle: any call reaching the library fails."""
    from nka_b200 import InterleavedBatchNKA
    acc = InterleavedBatchNKA()
    acc.nbatch, acc.vlen, acc.mvec = nbatch, vlen, 3
    return acc


def test_update_validates_f_and_masks_before_any_cuda_call():
    import numpy as np
    import torch
    acc = _unbuilt(4, 10)
    cases = {
        "numpy": (np.zeros((10, 4)).T, "CUDA float64"),
        "float32": (torch.zeros(10, 4, dtype=torch.float32).t(), "float64"),
        "1-D": (torch.zeros(40, dtype=torch.float64), "shape"),
        "rows": (torch.zeros(10, 5, dtype=torch.float64).t(), "shape"),
        "cols": (torch.zeros(11, 4, dtype=torch.float64).t(), "shape"),
        "row-major": (torch.zeros(4, 10, dtype=torch.float64), "interleaved"),
        "component stride": (torch.zeros(40, dtype=torch.float64).as_strided((4, 10), (1, 3)), "component stride"),
        "cpu tensor": (torch.zeros(10, 4, dtype=torch.float64).t(), "CUDA"),
    }
    for name, (F, what) in cases.items():
        with pytest.raises(ValueError, match=what):
            acc.accel_update(F)
    for mask in (np.ones(4, dtype=bool), torch.ones(4, dtype=torch.bool), torch.ones(4, dtype=torch.int32),
                 torch.ones(5, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            acc.relax(mask)
        with pytest.raises(ValueError):
            acc.restart(mask)
    with pytest.raises(ValueError):
        acc.set_vec_tol(0.0)
    with pytest.raises(ValueError):
        acc.state(4)
    with pytest.raises(ValueError):
        acc.state(-1)


def test_one_member_or_one_component_takes_any_unused_stride():
    """With nbatch == 1 the member stride addresses nothing, with vlen == 1 the component stride: any is
    accepted there (and fails only at the CPU check here)."""
    import torch
    for nb, vlen, F in [(1, 10, torch.zeros(1, 10, dtype=torch.float64)),
                        (4, 1, torch.zeros(4, 1, dtype=torch.float64))]:
        with pytest.raises(ValueError, match="must be a CUDA tensor"):
            _unbuilt(nb, vlen).accel_update(F)


# ---------------------------------------------------------------------------------------------
# the ctypes table against the header
# ---------------------------------------------------------------------------------------------
def _ibatch_prototypes():
    text = open(os.path.join(ROOT, "include", "nka_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = {}
    for m in re.finditer(r"\n([\w ]+?[\s\*]+)(nka_ibatch_\w+)\s*\((.*?)\)\s*;", text, re.S):
        out[m.group(2)] = (m.group(1).strip(), [p.strip() for p in m.group(3).split(",")])
    return out


def _ctype_of(decl):
    import ctypes as C
    from nka_b200 import _lib
    if "nka_state_view" in decl:
        return C.POINTER(_lib.StateView)
    if "int *" in decl:
        return C.POINTER(C.c_int)
    if "*" in decl:
        return C.c_void_p
    words = decl.split()
    base = " ".join(words[:-1]) if len(words) > 1 and words[-1] not in ("int", "double", "size_t", "long") else decl
    return {"int": C.c_int, "size_t": C.c_size_t, "double": C.c_double, "void": None,
            "unsigned long long": C.c_ulonglong}[base]


def test_ctypes_signatures_match_the_header():
    from nka_b200 import _lib
    protos = _ibatch_prototypes()
    assert len(protos) == 13
    for name, (ret, params) in protos.items():
        restype, argtypes = _lib.SYMBOLS[name]
        assert restype == _ctype_of(ret + " x"), (name, ret, restype)
        assert argtypes == [_ctype_of(p) for p in params], (name, params, argtypes)


# ---------------------------------------------------------------------------------------------
# code generation
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def obj():
    from nka_b200 import build
    build.build_library()
    return os.path.join(build.LIB_DIR, "nka_ibatch.o")


def _res_usage(path):
    out = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True, check=True).stdout
    res = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out):
        res[m.group(1)] = {"reg": int(m.group(2)), "stack": int(m.group(3)), "local": int(m.group(5))}
    return res


def _sass(path):
    text = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    return [ln.strip() for ln in text.splitlines() if re.match(r"\s*(Function :|/\*[0-9a-f]{4,}\*/)", ln)]


def test_kernels_use_no_local_memory(obj):
    res = _res_usage(obj)
    updates = [n for n in res if n.startswith("_Z17nka_ibatch_updateILi")]
    assert sorted(int(re.match(r"_Z17nka_ibatch_updateILi(\d+)E", n).group(1)) for n in updates) == list(range(2, 34))
    assert len(res) == 32 + 6
    for name, r in res.items():
        assert r["local"] == 0 and r["stack"] == 0, (name, r)


def test_sass_is_identical_without_contraction(obj, tmp_path):
    """Every multiply, add and subtract of the update is an explicit round-to-nearest intrinsic, so forbidding
    FMA contraction changes no instruction (division and sqrt keep their own internal FMAs either way)."""
    from nka_b200 import build
    nofma = str(tmp_path / "nka_ibatch_nofma.o")
    src = os.path.join(build.CSRC, "nka_ibatch.cu")
    subprocess.run([os.environ.get("NVCC", "nvcc"), *build.NVCC_FLAGS, "-fmad=false", "-c", src, "-o", nofma],
                   check=True, capture_output=True)
    a, b = _sass(obj), _sass(nofma)
    assert len(a) > 10000
    assert a == b
