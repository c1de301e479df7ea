"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/api_behaviour.json: what the REAL reference does in each scenario
of oracle/api_scenarios.py.  Needs the reference staged in oracle/_ref/site (oracle/stage_reference.sh):

    python oracle/gen_api_golden.py
"""
from __future__ import annotations

import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "_ref", "site"))
sys.path.insert(1, os.path.join(HERE, ".."))
import datasketch  # noqa: E402  (the reference)

from oracle.api_scenarios import SCENARIOS  # noqa: E402

assert os.path.dirname(datasketch.__file__).startswith(os.path.join(HERE, "_ref")), datasketch.__file__
out = {name: fn(datasketch) for name, fn in SCENARIOS.items()}
with open(os.path.join(HERE, "..", "tests", "golden", "api_behaviour.json"), "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
    f.write("\n")
print({k: len(v) for k, v in out.items()})
