"""Lock-step fuzz against the UNMODIFIED reference -- only where the original CarlaBEV package can be imported
(CARLABEV_REFERENCE_ROOT, or the copy oracle/make_ref.py stages under oracle/_ref/); it is not part of this repository,
so these tests skip elsewhere.  Its recorded snapshots and trajectories are compared everywhere by test_host_logic.py and
test_oracle_golden.py.  They run a small slice of oracle/fuzz_scenes.py and oracle/fuzz_steps.py (the full runs are
recorded in DESIGN.md section 2)."""
import os
import subprocess
import sys

import pytest

from golden_util import ROOT
from oracle.ref_loader import reference_available

pytestmark = pytest.mark.skipif(not reference_available(), reason="the original CarlaBEV package is not available")


def _run(script, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", script), *map(str, args)], capture_output=True,
                       text=True, timeout=600)
    tail = (r.stdout + r.stderr)[-2000:]
    assert r.returncode == 0, tail
    return r.stdout.strip().splitlines()[-1]


def test_scene_generators_equal_the_reference_on_random_options():
    last = _run("fuzz_scenes.py", 24, 77)
    assert last.endswith("0 mismatches"), last


def test_oracle_step_equals_the_reference_on_random_episodes():
    last = _run("fuzz_steps.py", 5, 78, 60)
    assert last.endswith("0 mismatching episodes"), last
