"""Merge the achieved-error table of a GPU test run (build/parity_errors.json) into the committed copy
(profiles/parity_errors.json): entries of the new run replace older ones of the same name."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
new = json.load(open(os.path.join(ROOT, "build", "parity_errors.json")))
path = os.path.join(ROOT, "profiles", "parity_errors.json")
old = json.load(open(path)) if os.path.exists(path) else {"what": new["what"], "scenarios": {}}
old["what"] = new["what"]
old["scenarios"].update(new["scenarios"])
old["scenarios"] = dict(sorted(old["scenarios"].items()))
json.dump(old, open(path, "w"), indent=1)
print(len(new["scenarios"]), "entries merged,", len(old["scenarios"]), "in", path)
