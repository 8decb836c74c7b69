"""The oracle against the unmodified upstream gym-pybullet-drones Python, live (not through fixtures): random configurations
replayed in both.  The upstream sources are not part of this repository: point GPD_REFERENCE at a checkout of them (the
directory holding gym_pybullet_drones/), or stage a copy into oracle/_ref (oracle/stage_reference.py).  Without either, the
test cannot run and says so; the oracle is then checked only against the recorded upstream trajectories in tests/golden."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = next((r for r in (os.environ.get("GPD_REFERENCE"), os.path.join(ROOT, "oracle", "_ref"))
            if r and os.path.isdir(os.path.join(r, "gym_pybullet_drones"))), None)


@pytest.mark.skipif(REF is None, reason="needs the upstream gym-pybullet-drones sources, which this repository does not "
                                        "contain: set GPD_REFERENCE to a checkout of them (or stage them into oracle/_ref)")
def test_oracle_matches_live_reference_on_random_configs():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "fuzz_vs_reference.py"), "--ref", REF, "--seeds", "60"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert out.returncode == 0 and lines, out.stderr[-2000:] + out.stdout[-2000:]
    d = json.loads(lines[-1])
    assert d["cases"] == 60 and d["failures"] == []
    assert d["open_loop_worst"] <= 1e-10 and d["closed_loop_worst"] <= 1e-6
