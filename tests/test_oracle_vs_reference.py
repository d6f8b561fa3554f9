"""The C restatement (oracle/tinympc_oracle.c) must be BIT-IDENTICAL to the unmodified reference compiled
with the pinned flags on every parity case, through warm-started closed loops.  The reference's outputs (and the cache
its tiny_setup computed) are stored in tests/golden/ by tests/golden/make_golden.py; here the port runs the cases
from their definitions (tests/helpers.py), simulating the plant itself, and must reproduce them."""
import os

import numpy as np
import pytest

import helpers as H
from oracle import oracle

CASES = H.make_cases()


def _solve(impl):
    def fn(prob, settings, x0, Xref, Uref, state, cold, want):
        return oracle.solve_batch(prob, settings, x0, Xref, Uref, state=state, cold_start=cold, want_state=want, impl=impl)
    return fn


@pytest.mark.parametrize("name", sorted(CASES))
def test_port_bit_identical_to_reference(name):
    c = CASES[name]
    gold = np.load(os.path.join(H.GOLDEN_DIR, name + ".npz"))
    prob = H.problem_from_spec(c["spec"], c["dtype"], H.stored_setup(gold, "prob"))
    st = c["spec"].settings
    port, x0s = H.closed_loop(prob, st, c["inst"], c["steps"], c["reset_duals"], c["state"], _solve("port"))
    assert H.bits_equal(np.stack(x0s), gold["x0_seq"])
    moved = 0
    for k, p in enumerate(port):
        for key in H.OUT_KEYS + c["state"]:
            assert H.bits_equal(gold[f"step{k}_{key}"], p[key]), f"{name} step {k}: {key} differs"
        moved += int(p["iter"].sum())
    assert moved > 0


def test_precompute_port_close_to_reference():
    for name in ("cartpole_f64", "quad_hover_N10_f64", "rocket_soc_N10_f64", "lti_8_2_f64"):
        c = CASES[name]
        gold = np.load(os.path.join(H.GOLDEN_DIR, name + ".npz"))
        pp = H.problem_from_spec(c["spec"], np.float64, oracle.port_setup)
        for f in H.CACHE_FIELDS:
            a, b = gold["prob_" + f], getattr(pp, f)
            assert np.allclose(a, b, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(a).max())), (name, f)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_port_bit_identical_to_reference_random_lti_sweep(dt):
    """Randomised sweep over the compiled (nx, nu) pairs and short horizons (BASELINE config 5's generator): warm-started
    three-step loops with active box bounds, restatement vs the unmodified reference, bit for bit."""
    gold = H.load_reference(f"lti_sweep_{np.dtype(dt).name}")
    want = dict(zip(gold["names"], gold["digests"]))
    for key, sp, inst in H.lti_sweep(dt):
        prob = H.problem_from_spec(sp, dt, H.stored_setup(gold, key))
        port, x0s = H.closed_loop(prob, sp.settings, inst, 3, False, H.BOX_STATE, _solve("port"))
        assert H.digest(np.stack(x0s)) == want[f"{key}_x0_seq"], key
        for k, p in enumerate(port):
            for name in H.OUT_KEYS + H.BOX_STATE:
                assert H.digest(p[name]) == want[f"{key}_step{k}_{name}"], f"{key} step {k}: {name} differs"


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_port_bit_identical_to_reference_constraint_families(dt):
    """Cones and hyperplanes, alone and combined with active box bounds, on every shape of tests/helpers.py:family_cases:
    warm-started three-step loops carrying all 20 state arrays, restatement vs the unmodified reference, bit for bit.  Every
    enabled constraint family must change the answer, and the cases together must hold instances that converge before
    max_iter and instances that run to it."""
    from tinympc_b200.problem import copy_settings

    gold = H.load_reference(f"families_{np.dtype(dt).name}")
    want = dict(zip(gold["names"], gold["digests"]))
    iters, max_iters = [], []
    for key, sp, inst in H.family_cases(dt):
        prob = H.problem_from_spec(sp, dt, H.stored_setup(gold, key))
        port, x0s = H.closed_loop(prob, sp.settings, inst, 3, False, H.ALL_STATE, _solve("port"))
        assert H.bits_equal(np.stack(x0s), gold[f"{key}_x0_seq"]), key
        for k, p in enumerate(port):
            for name in H.OUT_KEYS + H.ALL_STATE:
                assert H.digest(p[name]) == want[f"{key}_step{k}_{name}"], f"{key} step {k}: {name} differs"
            iters.append(p["iter"])
            max_iters.append(np.full_like(p["iter"], sp.settings.max_iter))
        for flag in H.FAMILY_FLAGS:
            if getattr(sp.settings, flag):
                off = copy_settings(sp.settings)
                setattr(off, flag, 0)
                o = _solve("port")(prob, off, inst["x0"], inst["Xref"], None, None, True, ())
                assert not (H.bits_equal(o["sol_x"], port[0]["sol_x"]) and H.bits_equal(o["sol_u"], port[0]["sol_u"])), \
                    f"{key}: {flag} does not change the solution"
    iters, max_iters = np.concatenate(iters), np.concatenate(max_iters)
    assert (iters < max_iters).any() and (iters == max_iters).any()
