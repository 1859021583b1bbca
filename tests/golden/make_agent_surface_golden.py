#!/usr/bin/env python
"""Record the reference side of the agent-surface harnesses (tests/agent_surface/) that tests/test_agent_surface.py compares against,
under tests/golden/agent_surface/ (apart from the trajectory goldens that helpers.golden_names() collects).

    python tests/golden/make_agent_surface_golden.py        (needs the reference checkout at tests/agent_surface/harness.py:REF)

kwargs_matrix_reference.npz (kwargs_matrix_harness.py --impl reference): per case, as JSON under `cases`, the verdict, the summary, the
solver, the number of state rows, the terminated flags and — for constant references — the rewards.  The state trajectories are stored
as float64 arrays `states/<case>` holding the rows `rows/<case>`: the reset and the five fixed steps (rows 0..6) and every 8th row
after them, which keeps the file under 1 MB.

integration_stub_reference.json (integration_stub_harness.py --impl reference): every value the INTEGRATION.md stub reads from the
reference's SCMLSystem."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT_DIR = os.path.join(HERE, "agent_surface")
HARNESS_DIR = os.path.normpath(os.path.join(HERE, "..", "agent_surface"))
sys.path.insert(0, HARNESS_DIR)
from harness import REF  # noqa: E402


def sampled_rows(n):
    return [i for i in range(n) if i < 7 or i % 8 == 0]


def run_reference(harness):
    with tempfile.TemporaryDirectory() as cwd:  # example code may create files under the cwd
        out = subprocess.run([sys.executable, os.path.join(HARNESS_DIR, harness), "--impl", "reference"], capture_output=True, text=True, check=True,
                             cwd=cwd)
    return json.loads(out.stdout.strip().splitlines()[-1])


def main():
    if not os.path.isdir(os.path.join(REF, "src", "gym_electric_motor")):
        raise SystemExit(f"no gym-electric-motor checkout at {REF}")
    cases, arrays = {}, {}
    for name, rec in run_reference("kwargs_matrix_harness.py").items():
        tr = rec["trajectory"]
        if tr is not None:
            rows = sampled_rows(len(tr["states"]))
            arrays[f"rows/{name}"] = np.asarray(rows, dtype=np.int32)
            arrays[f"states/{name}"] = np.asarray([tr["states"][i] for i in rows], dtype=np.float64)
            tr = dict(n_states=len(tr["states"]), terminated=tr["terminated"], rewards=tr["rewards"], solver=tr["solver"])
        cases[name] = dict(verdict=rec["verdict"], summary=rec["summary"], trajectory=tr)
    np.savez_compressed(os.path.join(OUT_DIR, "kwargs_matrix_reference.npz"), cases=json.dumps(cases), **arrays)
    with open(os.path.join(OUT_DIR, "integration_stub_reference.json"), "w") as f:
        json.dump(run_reference("integration_stub_harness.py")["reads"], f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
