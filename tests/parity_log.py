"""Achieved-error table of the GPU parity tests.

Per scenario: how far the CUDA path is from the long-double arbiter and from the unmodified
(serial-sum) reference, beside the tolerance that was applied.  Written at session end to
build/parity_errors.json (a run's output, kept out of git); tools/merge_parity.py merges it into
profiles/parity_errors.json (the copy that is committed)."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "build", "parity_errors.json")
_PARITY = {}
WHAT = ("max over the calls of a scenario of ||got - ref|| / max(||ref||, ||f_in||); arbiter = the reference "
        "algorithm with long-double dot products (its dp hook), serial = the unmodified reference (serial sums)")


def record_parity(name: str, **fields) -> None:
    _PARITY[name] = {k: (float(v) if isinstance(v, float) or hasattr(v, "dtype") else v) for k, v in fields.items()}


def flush() -> None:
    if not _PARITY:
        return
    try:
        os.makedirs(os.path.dirname(PATH), exist_ok=True)
        old = {}
        if os.path.exists(PATH):
            try:
                with open(PATH) as fh:
                    old = json.load(fh).get("scenarios", {})
            except Exception:
                old = {}
        old.update(_PARITY)
        with open(PATH, "w") as fh:
            json.dump({"what": WHAT, "scenarios": dict(sorted(old.items()))}, fh, indent=1)
    except OSError:
        pass
