"""Per-problem stopping tests without a GPU: the argument checks of fixed_point_loop / fixed_point_queue that
raise before any CUDA call, the layout of nka_stop_test in C, ctypes and Fortran, and the scaled sweep of
the 16-byte check kernel in the generated code."""
import os
import re
import subprocess

import pytest

from test_batch_cpu import _unbuilt
from test_loop_cpu import _res_usage, _sass

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_stop_arguments_are_validated_before_any_cuda_call():
    import numpy as np
    import torch
    b = _unbuilt(4, 10)
    f64 = dict(dtype=torch.float64)
    rows = torch.zeros(4, 10, **f64)                      # CPU tensors: each case fails before the device checks
    bad = [
        (dict(atol=torch.zeros(4, dtype=torch.float32)), "atol"),
        (dict(atol=torch.zeros(4, **f64)), "atol"),                       # not CUDA
        (dict(atol=torch.zeros(4, 1, **f64)), "atol"),
        (dict(rtol=torch.zeros(4, dtype=torch.int32)), "rtol"),
        (dict(rtol=np.zeros(4)), "rtol"),
        (dict(maxit=torch.zeros(4, dtype=torch.int64)), "maxit"),
        (dict(maxit=torch.zeros(4, dtype=torch.int32)), "maxit"),         # not CUDA
        (dict(maxit=np.zeros(4, dtype=np.int32)), "maxit"),
        (dict(dtol=0.5), "dtol"), (dict(dtol=-1.0), "dtol"), (dict(dtol=float("nan")), "dtol"),
        (dict(dtol=True), "dtol"), (dict(dtol="10"), "dtol"), (dict(dtol=1e-300), "dtol"),
    ]
    for kw, what in bad:
        with pytest.raises(ValueError, match=what):
            b.fixed_point_loop(lambda: None, rows, rows, **kw)
        with pytest.raises(ValueError, match=what):
            b.fixed_point_queue(lambda: None, rows, rows, torch.zeros(4, dtype=torch.int32), torch.zeros(9, 10, **f64),
                                **kw)
    bad_scale = {
        "numpy": (np.zeros((4, 10)), "CUDA float64"),
        "float32": (torch.zeros(4, 10, dtype=torch.float32), "float64"),
        "rows": (torch.zeros(5, 10, **f64), "shape"),
        "column stride": (torch.zeros(10, 4, **f64).t(), "stride"),
        "row stride": (torch.zeros(40, **f64).as_strided((4, 10), (5, 1)), "row stride"),
        "cpu tensor": (rows, "scale must be a CUDA tensor"),
    }
    for name, (T, what) in bad_scale.items():
        with pytest.raises(ValueError, match=what):
            b.fixed_point_loop(lambda: None, rows, rows, scale=T)
    # dtol = 0 and dtol >= 1 are accepted: the next check refuses the CPU X
    for dtol in (0, 0.0, 1.0, 10, 1e300, float("inf")):
        with pytest.raises(ValueError, match="X must be a CUDA tensor"):
            b.fixed_point_loop(lambda: None, rows, rows, dtol=dtol)


_LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "nka_b200.h"
#define F(m) printf(#m " %zu %zu\n", offsetof(nka_stop_test, m), sizeof(((nka_stop_test *)0)->m));
int main(void)
{
  printf("sizeof %zu\n", sizeof(nka_stop_test));
  F(atol) F(rtol) F(dtol) F(maxit) F(atol_dev) F(rtol_dev) F(maxit_dev) F(scale_dev) F(ldscale)
  printf("DIVERGED %d\n", NKA_LOOP_DIVERGED);
  return 0;
}
"""


def test_stop_test_layout_matches_in_c_ctypes_and_fortran(tmp_path):
    import ctypes as C
    from nka_b200 import _lib, batch
    src = tmp_path / "layout.c"
    src.write_text(_LAYOUT_C)
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    c_size = int(out[0].split()[1])
    c_fields = [(ln.split()[0], int(ln.split()[1]), int(ln.split()[2])) for ln in out[1:] if ln and ln.split()[0] != "DIVERGED"]
    assert "DIVERGED 4" in out and batch.DIVERGED == 4
    S = _lib.StopTest
    assert C.sizeof(S) == c_size
    py_fields = [(name, getattr(S, name).offset, getattr(S, name).size) for name, _ in S._fields_]
    assert py_fields == c_fields
    # the Fortran bind(C) type: the same components in the same order, with interoperable kinds
    text = open(os.path.join(ROOT, "nka_b200", "fortran", "nka_b200_c.F90")).read()
    body = re.search(r"type,\s*bind\(C\)\s*::\s*nka_stop_test\s*\n(.*?)\n\s*end type", text, re.S | re.I).group(1)
    comps = []
    for line in body.splitlines():
        line = line.split("!")[0]
        if "::" in line:
            kind, names = line.split("::")
            comps += [(n.strip(), kind.strip().replace(" ", "").lower()) for n in names.split(",")]
    kinds = {"real(c_double)": 8, "integer(c_int)": 4, "type(c_ptr)": C.sizeof(C.c_void_p), "integer(c_size_t)": C.sizeof(C.c_size_t)}
    assert [n for n, _ in comps] == [n for n, _, _ in c_fields]
    assert [kinds[k] for _, k in comps] == [size for _, _, size in c_fields]


def _loops(sass):
    """Instruction lists of the loop bodies: from a backward branch's target to the branch."""
    ins = [(int(m.group(1), 16), m.group(2)) for m in re.finditer(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", sass)]
    out = []
    for addr, text in ins:
        m = re.search(r"\bBRA\s+(?:\S+,\s*)?0x([0-9a-f]+)", text)
        if m and int(m.group(1), 16) < addr:
            out.append([t for a, t in ins if int(m.group(1), 16) <= a <= addr])
    return out


def test_scaled_check_sweep_loads_f_and_scale_16_bytes_at_a_time():
    """At V = 2 with 16-byte scale rows, the scaled sweep is as wide as the plain one: a loop whose body
    loads F and the scale with LDG.E.128 (and no 8-byte load) before multiplying them."""
    from nka_b200 import build
    build.build_library()
    obj = os.path.join(build.LIB_DIR, "nka_batch_loop.o")
    check = [n for n in _res_usage(obj) if n.startswith("_Z14nka_loop_checkILi2E")]
    assert len(check) == 1
    loops = _loops(_sass(obj, check[0]))
    assert loops
    wide = [body for body in loops
            if sum("LDG.E.128" in t for t in body) >= 2 and any(t.split()[0].startswith("DMUL") or " DMUL" in t for t in body)
            and not any("LDG.E.64" in t for t in body)]
    assert wide, "no scaled sweep with two 16-byte load sites"
    # the 8-byte-scale sweep exists too (F 16 bytes, the scale 8 bytes at a time)
    assert any(any("LDG.E.128" in t for t in body) and any("LDG.E.64" in t for t in body) for body in loops)
