"""Generate the golden fixtures from the reference itself.

Run in the build container (needs /root/reference and gcc):

    python tests/golden/make_golden.py

Writes, next to this file:

* ``example_c_f95.txt``      -- stdout of the reference's own C example
  (oracle/_ref/nka_example_ref, compiled from /root/reference/src-C); checked
  here to be byte-identical to src-C/reference_output and to
  src-F95/reference_output before it is written.
* ``example_f08.json``       -- the three final table lines the F08 / F08-vector
  fixtures pin (src-F08/reference_output:7,16,25), parsed from that file.
* ``accel_golden.json``      -- for every scenario in tests/scenarios.py, what
  the compiled reference library (oracle/_ref/libnka_ref.so) returned:
  num_vec after every op and the sha256 of every correction vector's bytes
  (the oracle port is bit-identical to the reference, so a digest pins it).
* ``accel_small.npz``        -- full correction vectors for the scenarios with
  n <= 128, for eyeballing and for tolerance tests without the oracle.
* ``accel_dp_golden.json``   -- the same digests for DP_SCENARIOS with a long-double
  dot product handed to the reference through its ``dp`` hook: the arbiter the GPU
  tests compare with.  ``--dp-from-port`` writes this file alone from the port
  (dotmode = 1) where the reference is not at hand; its "source" field says which.
"""
from __future__ import annotations

import hashlib
import json
import os
import re
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import api, build  # noqa: E402
import scenarios as S  # noqa: E402

REF = "/root/reference"
DP_SCENARIOS = ["picard_n500_m5_v2"]


def _digests(acc, ops) -> dict:
    outs, nvecs = S.run_ops(acc, ops)
    acc.close()
    return {"num_vec": nvecs, "sha256": [hashlib.sha256(o.tobytes()).hexdigest() for o in outs]}


def write_dp_golden(from_port: bool) -> None:
    gold = {"source": "oracle port, dotmode=1 (long-double dots)" if from_port
            else "compiled reference src-C, long-double dp through nka_init's dp hook"}
    for name in DP_SCENARIOS:
        n, mvec, vtol, mk = S.SCENARIOS[name]
        acc = api.OracleNKA(n, mvec, vtol, dotmode=1) if from_port else api.RefNKA(n, mvec, vtol, long_double_dp=True)
        gold[name] = {"n": n, "mvec": mvec, "vtol": vtol, **_digests(acc, mk())}
    with open(os.path.join(HERE, "accel_dp_golden.json"), "w") as fh:
        json.dump(gold, fh, indent=0)


def main() -> None:
    if "--dp-from-port" in sys.argv:
        write_dp_golden(from_port=True)
        return
    if not build.reference_available():
        raise SystemExit("needs /root/reference (build container only)")
    built = build.build_all()

    # 1. the example's full table
    out = subprocess.run([built["ref_example"]], capture_output=True, check=True).stdout
    for flavour in ("src-C", "src-F95"):
        with open(os.path.join(REF, flavour, "reference_output"), "rb") as fh:
            if fh.read() != out:
                raise SystemExit("compiled reference example differs from %s/reference_output" % flavour)
    with open(os.path.join(HERE, "example_c_f95.txt"), "wb") as fh:
        fh.write(out)

    # 2. the F08 fixture's pinned lines
    with open(os.path.join(REF, "src-F08", "reference_output")) as fh:
        text = fh.read()
    with open(os.path.join(REF, "src-F08-vector", "reference_output")) as fh:
        if fh.read() != text:
            raise SystemExit("F08 and F08-vector fixtures differ")
    runs = []
    for block in text.split("% nka_example")[1:]:
        args = block.split("\n", 1)[0].split()
        last = [ln for ln in block.splitlines() if re.match(r"^\s*\d+:", ln)][-1]
        runs.append({"args": args, "last_line": last})
    with open(os.path.join(HERE, "example_f08.json"), "w") as fh:
        json.dump({"source": "src-F08/reference_output == src-F08-vector/reference_output", "runs": runs},
                  fh, indent=1)

    # 3./4. per-call goldens from the compiled reference library
    gold = {}
    small = {}
    for name, (n, mvec, vtol, mk) in S.SCENARIOS.items():
        ops = mk()
        ref = api.RefNKA(n, mvec, vtol)
        outs, nvecs = S.run_ops(ref, ops)
        ref.close()
        gold[name] = {
            "n": n, "mvec": mvec, "vtol": vtol,
            "ops": [op[0] for op in ops],
            "num_vec": nvecs,
            "sha256": [hashlib.sha256(o.tobytes()).hexdigest() for o in outs],
            "in_sha256": [hashlib.sha256(op[1].tobytes()).hexdigest() for op in ops if op[0] == "update"],
        }
        if n <= 128:
            small[name] = np.stack(outs)
    with open(os.path.join(HERE, "accel_golden.json"), "w") as fh:
        json.dump(gold, fh, indent=0)
    np.savez_compressed(os.path.join(HERE, "accel_small.npz"), **small)
    write_dp_golden(from_port=False)
    print("wrote goldens for %d scenarios" % len(gold))


if __name__ == "__main__":
    main()
