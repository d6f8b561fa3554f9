"""The reference-compatible C++ front end (tinympc_b200/shim): every function the reference's headers define for the solve
path is exported with C linkage (tiny_api.hpp:10-62, admm.hpp:9-34), and tiny_initialize_sensitivity_matrices leaves in the
cache exactly what the reference's does (tiny_api.cpp:479-540, stored in tests/golden/).  No GPU needed (nothing is solved)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tinympc_b200", "lib", "libtinympc_shim.so")

TINY_API = ["tiny_setup", "tiny_set_bound_constraints", "tiny_set_cone_constraints", "tiny_set_linear_constraints",
            "tiny_set_tv_linear_constraints", "tiny_precompute_and_set_cache", "tiny_solve", "tiny_update_settings",
            "tiny_set_default_settings", "tiny_set_x0", "tiny_set_x_ref", "tiny_set_u_ref", "tiny_initialize_sensitivity_matrices"]
ADMM = ["solve", "update_linear_cost", "backward_pass_grad", "forward_pass", "update_slack", "update_dual", "termination_condition"]

pytestmark = pytest.mark.skipif(not os.path.exists(SHIM), reason="shim library not built (needs Eigen headers at build time)")


def test_shim_exports_the_reference_interface():
    out = subprocess.run(["nm", "-D", "--defined-only", SHIM], capture_output=True, text=True, check=True).stdout
    have = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    missing = [n for n in TINY_API + ADMM if n not in have]
    assert not missing, missing
    assert len(TINY_API) == 13


def test_sensitivity_tables_equal_the_reference():
    """Against the tables the reference's tiny_initialize_sensitivity_matrices leaves (tests/golden/make_golden.py)."""
    gold = H.load_reference("sensitivity_tables")
    shapes = [(4, 12), (12, 12), (4, 4), (12, 12)]
    ref = [np.asfortranarray(gold[n]) for n in ("dKinf_drho", "dPinf_drho", "dC1_drho", "dC2_drho")]
    assert [a.shape for a in ref] == shapes
    lib = C.CDLL(SHIM)
    mine = [np.zeros(s, np.float64, order="F") for s in shapes]
    assert lib.tinympc_shim_sensitivity_tables(*[C.c_void_p(a.ctypes.data) for a in mine]) == 0
    for a, b in zip(mine, ref):
        assert a.tobytes(order="F") == b.tobytes(order="F")
    assert np.abs(ref[1]).max() > 1.0  # the dPinf_drho table is not all zeros
