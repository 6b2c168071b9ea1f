"""Seeded slices of the CPU fuzzers (tools/fuzz_cpu.py, tools/fuzz_lod_cpu.py,
tools/fuzz_misc_cpu.py):
compiled reference == oracle == kernel bodies (host build) over random points
of the parameter space, the reference's outputs replayed from
tests/golden/reference_tape.npz.  The full sweeps are developer tools; these
keep a few dozen configurations in the regular suite."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("tool,cases,seed", [("fuzz_cpu.py", 40, 101), ("fuzz_lod_cpu.py", 30, 102),
                                             ("fuzz_misc_cpu.py", 30, 103)])
def test_fuzz_slice(tool, cases, seed):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool), str(cases), str(seed)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert f"{cases} cases, 0 mismatches" in r.stdout
