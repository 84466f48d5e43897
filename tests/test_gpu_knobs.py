"""The remaining A/B knob sets the hash tables' capacity (DESIGN.md section 6): with it set, the pipeline must
still produce the oracle's bits.  The knob is read once per process, so each case runs
``__graft_entry__.smoke()`` - front end, voxel grid, radius outliers, RANSAC ground removal on a 32 768-point
scan, compared bit for bit with the CPU oracle - in a fresh interpreter with the knob set."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KNOBS = [
    {"APC_HASH_SLOTS_PER_POINT": "2"},      # 2 slots per point instead of 4 in the hash tables
]


@pytest.mark.parametrize("knobs", KNOBS, ids=lambda k: "+".join(f"{a}={b}" for a, b in k.items()))
def test_knob_variants_match_the_oracle(knobs):
    env = dict(os.environ, **knobs)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "__graft_entry__.py"), "smoke"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "smoke ok" in r.stdout
