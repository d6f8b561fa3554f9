"""Cones and hyperplanes on every lane mapping of the streamed lane-group kernel (GPS, csrc/gps_kernel.cuh) and on the
thread-per-instance kernel (TPI, csrc/tpi_kernel.cuh), alone and combined with active box bounds.

The cases (tests/helpers.py:family_cases) cover each (lanes per instance, instances per lane group) variant GPS compiles for
fp32 and fp64 with four constraint mixes: cones (family mask 1), static + time-varying hyperplanes (mask 6), cones + static
hyperplanes and cones + both hyperplane kinds (mask 7, where the cost terms of several families add up in one q / r / p).
STRICT mode is compared bit for bit with the unmodified reference's stored outputs (tests/golden/reference/families_*.npz)
or with the C restatement given the same inputs; FAST mode is held to the bar of test_gpu_parity.py's scatter test.
"""
import functools

import numpy as np
import pytest

import helpers as H
from oracle import oracle
from tinympc_b200 import abi
from tinympc_b200.problem import copy_settings

pytestmark = pytest.mark.gpu

KERNELS = {"gps": abi.KERNEL_GPS, "tpi": abi.KERNEL_TPI, "auto": abi.KERNEL_AUTO}
DTYPES = {"f32": np.float32, "f64": np.float64}
CASES = {(tag, key): (sp, inst) for tag, dt in DTYPES.items() for key, sp, inst in H.family_cases(dt)}
# the state arrays the answer of a warm-started solve depends on: rollout, box slacks (first linear cost) and duals.  The
# family slacks are re-initialised from the rollout at the start of a solve; v / z only enter the dual residual of the first
# iteration, which decides nothing unless an instance terminates there.
WARM_INPUTS = ["x", "u", "vnew", "znew", "g", "y", "gc", "yc", "gl", "yl", "gl_tv", "yl_tv"]
FAMILY_SLACKS = {"cones": ["vcnew", "zcnew"], "planes": ["vlnew", "zlnew"], "tv_planes": ["vlnew_tv", "zlnew_tv"]}
FAMILY_DUALS = ["gc", "yc", "gl", "yl", "gl_tv", "yl_tv"]


@functools.lru_cache(maxsize=None)
def _gold(tag):
    g = H.load_reference(f"families_{np.dtype(DTYPES[tag]).name}")
    return g, dict(zip(g["names"], g["digests"]))


def _solver(prob, st, kernel, mode=abi.MODE_STRICT):
    from tinympc_b200.solver import BatchedTinySolver

    return BatchedTinySolver(prob, st, device=0, mode=mode, kernel=KERNELS[kernel])


def _setup(spec, dt):
    from tinympc_b200.solver import setup_problem

    return setup_problem(spec, dt)


def _cuda_fn(solver):
    def fn(prob, settings, x0, Xref, Uref, state, cold, want):
        return solver.solve(x0, Xref, Uref, state=state, cold_start=cold, want_state=want)
    return fn


def _port(prob, st, x0, Xref, Uref, state, cold, want, nthreads=8):
    return oracle.solve_batch(prob, st, x0, Xref, Uref, state=state, cold_start=cold, want_state=want, impl="port",
                              nthreads=nthreads)


def _check_plan(stats, kernel, dt, nx, nu):
    """The solve ran on the intended kernel family and, for the lane groups, on the variant of FAMILY_VARIANTS."""
    if kernel == "tpi":
        assert stats["kernel_family"] == abi.KERNEL_TPI
        return
    assert stats["kernel_family"] == abi.KERNEL_GPS, (kernel, stats["kernel_family"])  # AUTO resolves to GPS as well
    L, per_warp = H.FAMILY_VARIANTS[dt][(nx, nu)]
    assert stats["lanes_per_instance"] == L, (nx, nu, stats["lanes_per_instance"], L)
    assert stats["instances_per_cta"] == per_warp * (stats["threads_per_cta"] // 32), (nx, nu, stats)


def _warm_state(prob, B, seed):
    """Every one of the 20 state arrays with its own seeded values, at the scale of a converged solve."""
    out = {}
    for i, name in enumerate(H.ALL_STATE):
        shape = (B, prob.N, prob.nx) if abi.STATE_IS_X[name] else (B, prob.N - 1, prob.nu)
        scale = 1.0 if name in ("x", "vnew", "v") else (0.5 if name in ("u", "znew", "z") else 0.2)
        out[name] = (scale * np.random.default_rng(seed + 17 * i).standard_normal(shape)).astype(prob.dtype)
    return out


def _copy(state, names=None):
    return {n: state[n].copy() for n in (names if names is not None else state)}


# ---------------------------------------------------------------------------------------------------------------------
# 1. closed loops against the reference's stored outputs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,key", sorted(CASES))
def test_closed_loop_bit_identical_to_reference(tag, key):
    """Warm-started three-step loops carrying all 20 state arrays, on GPS, TPI and AUTO: every output and state array of
    every step equals the reference's (stored as digests), and the solve ran on the intended variant."""
    sp, inst = CASES[(tag, key)]
    dt = DTYPES[tag]
    gold, want = _gold(tag)
    prob = H.problem_from_spec(sp, dt, H.stored_setup(gold, key))
    x0_seq = gold[f"{key}_x0_seq"]
    for kernel in ("gps", "tpi", "auto"):
        solver = _solver(prob, sp.settings, kernel)
        got, _ = H.closed_loop(prob, sp.settings, inst, 3, False, H.ALL_STATE, _cuda_fn(solver), x0_seq=x0_seq)
        _check_plan(solver.stats(), kernel, dt, sp.nx, sp.nu)
        for k, r in enumerate(got):
            for name in H.OUT_KEYS + H.ALL_STATE:
                assert H.digest(r[name]) == want[f"{key}_step{k}_{name}"], f"{key}/{kernel} step {k}: {name} differs"
        solver.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. arbitrary warm state, and which state arrays the caller asks for
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims", list(H.FAMILY_VARIANTS[np.float32]))
@pytest.mark.parametrize("tag", sorted(DTYPES))
def test_arbitrary_warm_state_and_state_requests(tag, dims):
    """A ragged batch warm-started from 20 unrelated random state arrays (so that a swapped field or a wrong slot offset in
    the GPS record shows), cones + both hyperplane kinds: every output and returned state array equals the restatement's.
    Then the same solve with fewer state arrays passed, which switches the record's region B (previous and family slacks) on
    and off per family: without family slacks and v / z, with one family's slacks, with only v / z.  The solution, iter, solved and
    residuals stay bit-identical, and every array passed comes back as in the full solve."""
    dt = DTYPES[tag]
    nx, nu = dims
    sp = H.family_spec(nx, nu, "ALL", seed=7)
    prob = _setup(sp, dt)
    B = 333
    x0 = H.family_x0(sp, np.random.default_rng(3), B).astype(dt)
    Xref = np.zeros((sp.N, nx), dt)
    warm = _warm_state(prob, B, seed=100 * nx + nu)
    o = _port(prob, sp.settings, x0, Xref, None, _copy(warm), False, ())
    requests = {"no slacks": WARM_INPUTS, "v / z": WARM_INPUTS + ["v", "z"]}
    requests.update({f"{f} slacks": WARM_INPUTS + s for f, s in FAMILY_SLACKS.items()})
    for kernel in ("gps", "tpi"):
        solver = _solver(prob, sp.settings, kernel)
        g = solver.solve(x0, Xref, None, state=_copy(warm), cold_start=False)
        _check_plan(solver.stats(), kernel, dt, nx, nu)
        for name in H.OUT_KEYS + H.ALL_STATE:
            assert H.bits_equal(g[name], o[name]), (kernel, name)
        for what, names in requests.items():
            r = solver.solve(x0, Xref, None, state=_copy(warm, names), cold_start=False)
            for name in H.OUT_KEYS + names:
                assert H.bits_equal(r[name], o[name]), (kernel, what, name)
        solver.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. slots refilled with family state over several waves
# ---------------------------------------------------------------------------------------------------------------------
def test_refill_over_several_waves():
    """(6,3) fp64 with cones and both hyperplane kinds on GPS, more instances than resident slots: finished instances hand
    their slot (and its family slacks / duals) to queued ones.  Iteration counts spread, so slots change hands at many
    different times; a strided sample and the last instances meet the restatement."""
    import torch

    dt = np.float64
    sp = H.family_spec(6, 3, "ALL", seed=60)
    prob = _setup(sp, dt)
    B = 20000
    rng = np.random.default_rng(11)
    x0 = (H.family_x0(sp, rng, B) * rng.uniform(0.02, 1.0, B)[:, None]).astype(dt)
    Xref = np.zeros((sp.N, 6), dt)
    solver = _solver(prob, sp.settings, "gps")
    # device pointers: one launch over the whole batch (the host-pointer path cuts big batches into pipelined chunks)
    batch, out = solver.make_device_batch(x0, Xref, None, cold_start=True)
    solver.solve_device(batch)
    torch.cuda.synchronize()
    g = {k: v.cpu().numpy() for k, v in out.items() if v is not None}
    stt = solver.stats()
    assert stt["kernel_launches"] == 1 and stt["instances"] == B
    _check_plan(stt, "gps", dt, 6, 3)
    print(f"\n(6,3) fp64 cones + hyperplanes on GPS: instances_per_cta={stt['instances_per_cta']} "
          f"threads_per_cta={stt['threads_per_cta']} ctas={stt['ctas']}")
    assert B > stt["ctas"] * stt["instances_per_cta"], stt  # more than one wave
    assert len(np.unique(g["iter"])) >= 5 and 0 < g["solved"].mean() < 1
    idx = np.unique(np.concatenate([np.arange(0, B, B // 256), np.arange(B - 8, B)]))
    o = _port(prob, sp.settings, x0[idx], Xref, None, None, True, ())
    for key in H.OUT_KEYS:
        assert H.bits_equal(g[key][idx], o[key]), key


# ---------------------------------------------------------------------------------------------------------------------
# 4. flag edges
# ---------------------------------------------------------------------------------------------------------------------
def _edge_spec(edge, nx, nu):
    if edge == "state_linear_without_rows":  # the reference still keeps (and updates) a slack and a dual for it
        sp = H.family_spec(nx, nu, "C", seed=5)
        sp.settings.en_state_linear = 1
    elif edge == "soc_without_cones":  # the reference skips the cone family
        sp = H.family_spec(nx, nu, "H", seed=5)
        sp.settings.en_state_soc = sp.settings.en_input_soc = 1
    else:
        sp = H.family_spec(nx, nu, "ALL", seed=5)
    s = sp.settings
    if edge == "input_side_only":
        s.en_state_soc = s.en_state_linear = s.en_tv_state_linear = 0
    elif edge == "state_side_only":
        s.en_input_soc = s.en_input_linear = s.en_tv_input_linear = 0
    elif edge == "time_varying_box":
        rng = np.random.default_rng(8)
        N = sp.N
        sp.constraints = dict(sp.constraints, x_min=-3.0 - rng.uniform(0, 1, (nx, N)), x_max=3.0 + rng.uniform(0, 1, (nx, N)),
                              u_min=-0.8 + 0.3 * rng.uniform(0, 1, (nu, N - 1)), u_max=0.8 - 0.3 * rng.uniform(0, 1, (nu, N - 1)))
    elif edge == "check_termination_3":
        s.check_termination = 3
    elif edge == "max_iter_0":
        s.max_iter = 0
    return sp


EDGES = ["state_linear_without_rows", "soc_without_cones", "input_side_only", "state_side_only", "time_varying_box",
         "check_termination_3", "max_iter_0"]


@pytest.mark.parametrize("edge", EDGES)
@pytest.mark.parametrize("tag,dims", [("f32", (12, 4)), ("f64", (8, 8))])
def test_flag_edges_vs_oracle(tag, dims, edge):
    """Flag combinations at the edges of the family dispatch, warm-started from random state, on GPS and TPI: every output
    and state array equals the restatement's."""
    dt = DTYPES[tag]
    nx, nu = dims
    sp = _edge_spec(edge, nx, nu)
    prob = _setup(sp, dt)
    B = 77
    x0 = H.family_x0(sp, np.random.default_rng(21), B).astype(dt)
    Xref = np.zeros((sp.N, nx), dt)
    warm = _warm_state(prob, B, seed=7)
    o = _port(prob, sp.settings, x0, Xref, None, _copy(warm), False, ())
    for kernel in ("gps", "tpi"):
        solver = _solver(prob, sp.settings, kernel)
        g = solver.solve(x0, Xref, None, state=_copy(warm), cold_start=False)
        _check_plan(solver.stats(), kernel, dt, nx, nu)
        for name in H.OUT_KEYS + H.ALL_STATE:
            assert H.bits_equal(g[name], o[name]), (edge, kernel, name)
        solver.close()
    if edge == "max_iter_0":  # no iteration: the duals come back unchanged, the enabled families' slacks are the rollout
        assert (o["iter"] == 0).all()
        for name in FAMILY_DUALS + ["g", "y"]:
            assert H.bits_equal(o[name], warm[name]), name
        for name in ("vcnew", "vlnew", "vlnew_tv"):
            assert H.bits_equal(o[name], o["x"]), name
        for name in ("zcnew", "zlnew", "zlnew_tv"):
            assert H.bits_equal(o[name], o["u"]), name
    if edge == "state_linear_without_rows":
        assert not H.bits_equal(o["gl"], warm["gl"])  # the slack / dual pair without rows was really carried
    if edge == "soc_without_cones":
        assert H.bits_equal(o["vcnew"], warm["vcnew"]) and H.bits_equal(o["gc"], warm["gc"])


# ---------------------------------------------------------------------------------------------------------------------
# 5. FAST mode with families
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", sorted(DTYPES))
def test_fast_mode_with_families_within_reference_scatter(tag):
    """FAST mode (FMA contraction) with cones and both hyperplane kinds on GPS and TPI, held to the bar of
    test_gpu_parity.py:test_fast_mode_within_reference_scatter: (a) at fixed work (tolerances 0, 20 iterations) x and u
    within 2e-4 relative (fp32) / 1e-10 (fp64) of the STRICT restatement; (b) run to convergence, at least as close to the
    fp64 restatement as the pinned fp32 restatement is (x2 slack)."""
    dt = DTYPES[tag]
    nx, nu = 12, 4
    sp = H.family_spec(nx, nu, "ALL", seed=9)
    prob = _setup(sp, dt)
    B = 512
    rng = np.random.default_rng(4)
    x0 = (H.family_x0(sp, rng, B) * rng.uniform(0.02, 1.0, B)[:, None]).astype(dt)
    Xref = np.zeros((sp.N, nx), dt)
    st = copy_settings(sp.settings)
    st.abs_pri_tol = st.abs_dua_tol = 0.0
    st.max_iter = 20
    o = _port(prob, st, x0, Xref, None, None, True, ("x", "u"))
    st2 = sp.settings
    o2 = _port(prob, st2, x0, Xref, None, None, True, ())
    o64 = _port(_setup(sp, np.float64), st2, x0.astype(np.float64), Xref.astype(np.float64), None, None, True, ())
    err_pinned = np.abs(o2["sol_u"].astype(np.float64) - o64["sol_u"]).max()
    tol = 2e-4 if dt == np.float32 else 1e-10
    for kernel in ("gps", "tpi"):
        solver = _solver(prob, st, kernel, mode=abi.MODE_FAST)
        g = solver.solve(x0, Xref, None, cold_start=True, want_state=("x", "u"))
        _check_plan(solver.stats(), kernel, dt, nx, nu)
        assert (g["iter"] == 20).all() and not g["solved"].any()
        for key in ("sol_x", "sol_u", "x", "u"):
            a, b = g[key].astype(np.float64), o[key].astype(np.float64)
            assert np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max()), (kernel, key, np.abs(a - b).max())
        assert not H.bits_equal(g["sol_x"], o["sol_x"]) or dt == np.float64  # FMA really changes fp32 bits
        solver2 = _solver(prob, st2, kernel, mode=abi.MODE_FAST)
        g2 = solver2.solve(x0, Xref, None, cold_start=True)
        err_fast = np.abs(g2["sol_u"].astype(np.float64) - o64["sol_u"]).max()
        assert err_fast <= max(2.0 * err_pinned, 1e-9), (kernel, err_fast, err_pinned)
        assert g2["iter"].mean() <= 1.1 * o2["iter"].mean() + 0.5, (kernel, g2["iter"].mean(), o2["iter"].mean())
        solver.close()
        solver2.close()
