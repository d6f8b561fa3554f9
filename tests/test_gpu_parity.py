"""Parity tests proper: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Bar (BASELINE.json north_star): STRICT mode is bit-identical to the pinned reference build in fp64 AND fp32 —
every solution/state scalar, all four residuals, iter and solved.  FAST mode (FMA contraction) is held to the
reference's own build-to-build scatter (SURVEY B.7): <= 2e-4 relative on x,u in fp32 (1e-9 in fp64), with
iteration counts allowed to move by one termination check on a small fraction of instances.
"""
import os

import numpy as np
import pytest

import helpers as H
from oracle import oracle
from tinympc_b200 import abi, workloads as wl
from tinympc_b200.solver import BatchedTinySolver, setup_problem

pytestmark = pytest.mark.gpu

# "gpi" = the lane-group kernels, planner's choice: state on chip (dual variables + d in tensor memory when that holds
# more instances per SM) for box-constrained problems that fit, else the streamed variant;
# "gpi_smem" forces the all-shared-memory on-chip variant (TINYMPC_GPI_TMEM=0); "gps" forces the streamed variant
KERNELS = {"tpi": abi.KERNEL_TPI, "gpi": abi.KERNEL_GPI, "gpi_smem": abi.KERNEL_GPI, "gps": abi.KERNEL_GPS, "auto": abi.KERNEL_AUTO}
ALLK = ["tpi", "gpi", "gpi_smem", "gps"]


@pytest.fixture(autouse=True)
def _default_gpi_variant():
    os.environ.pop("TINYMPC_GPI_TMEM", None)
    yield
    os.environ.pop("TINYMPC_GPI_TMEM", None)


def _mk_solver(prob, st, kernel, mode=abi.MODE_STRICT):
    from tinympc_b200._lib import TinyMPCError
    if kernel == "gpi_smem":
        os.environ["TINYMPC_GPI_TMEM"] = "0"
    else:
        os.environ.pop("TINYMPC_GPI_TMEM", None)
    try:
        s = BatchedTinySolver(prob, st, device=0, mode=mode, kernel=KERNELS[kernel])
    except TinyMPCError as e:  # pragma: no cover
        pytest.fail(str(e))
    return s


def _cuda_fn(solver):
    def fn(prob, settings, x0, Xref, Uref, state, cold, want):
        return solver.solve(x0, Xref, Uref, state=state, cold_start=cold, want_state=want)
    return fn


def _port(prob, settings, x0, Xref, Uref, state, cold, want, nthreads=8):
    return oracle.solve_batch(prob, settings, x0, Xref, Uref, state=state, cold_start=cold, want_state=want,
                              impl="port", nthreads=nthreads)


def _gpi_applicable(prob, st):
    ext = (st.en_state_soc and len(prob.Acx)) or (st.en_input_soc and len(prob.Acu)) or st.en_state_linear or \
        st.en_input_linear or st.en_tv_state_linear or st.en_tv_input_linear
    return not ext


@pytest.mark.parametrize("kernel", ALLK)
@pytest.mark.parametrize("name", H.golden_names())
def test_strict_bit_identical_to_reference_golden(name, kernel):
    prob, st, inst, meta, gold = H.load_golden(name)
    boxonly = _gpi_applicable(prob, st)
    if kernel == "gpi_smem" and not boxonly:
        pytest.skip("cones / hyperplanes always stream their state: covered by the 'gpi' and 'gps' cases")
    solver = _mk_solver(prob, st, kernel)
    got, _ = H.closed_loop(prob, st, inst, meta["steps"], meta["reset_duals"], meta["state"], _cuda_fn(solver),
                           x0_seq=meta["x0_seq"])
    for k, (g, r) in enumerate(zip(gold, got)):
        for key in H.OUT_KEYS + meta["state"]:
            assert H.bits_equal(g[key], r[key]), f"{name}/{kernel} step {k}: {key} differs from the reference"
    fam = solver.stats()["kernel_family"]
    if kernel == "gpi":  # on chip when the problem is box-constrained (every golden horizon fits), else streamed lane groups
        assert fam == (abi.KERNEL_GPI if boxonly else abi.KERNEL_GPS)
    else:
        assert fam == KERNELS[kernel]


@pytest.mark.parametrize("kernel", ALLK)
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_strict_batch_vs_oracle_ragged(dt, kernel):
    """A ragged batch (B not a multiple of the warp / group size) of randomised tracking instances, cold start,
    then one warm-started step; compared with the oracle on every scalar."""
    spec = wl.quadrotor(N=50)
    prob = setup_problem(spec, dt)
    st = spec.settings
    B = 333
    inst = wl.tracking_instances(B, N=50, seed=21, dtype=dt)
    solver = _mk_solver(prob, st, kernel)
    want = tuple(H.BOX_STATE)
    g1 = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
    o1 = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want)
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g1[key], o1[key]), key
    assert 1 < o1["iter"].min() and o1["iter"].max() < 100 and o1["solved"].all()
    # warm start from the returned state with perturbed measurements
    x0b = (inst["x0"] + dt(0.01)).astype(dt)
    state_g = {n: g1[n].copy() for n in H.BOX_STATE}
    state_o = {n: o1[n].copy() for n in H.BOX_STATE}
    g2 = solver.solve(x0b, inst["Xref"], None, state=state_g, cold_start=False)
    o2 = _port(prob, st, x0b, inst["Xref"], None, state_o, False, ())
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g2[key], o2[key]), "warm " + key


@pytest.mark.parametrize("kernel", ALLK)
def test_edge_cases(kernel):
    """B=1, B=33; max_iter=1; check_termination=3 (stale residual fields); per-instance Uref; shared refs."""
    spec = wl.quadrotor(N=10)
    dt = np.float32
    prob = setup_problem(spec, dt)
    rng = np.random.default_rng(0)
    for B, max_iter, check in ((1, 100, 1), (33, 1, 1), (33, 25, 3), (5, 7, 10)):
        st = abi.Settings.from_buffer_copy(spec.settings)
        st.max_iter, st.check_termination = max_iter, check
        inst = wl.tracking_instances(B, N=10, seed=B, dtype=dt)
        Uref = (0.05 * rng.standard_normal((B, 9, 4))).astype(dt)
        solver = _mk_solver(prob, st, kernel)
        want = tuple(H.BOX_STATE)
        g = solver.solve(inst["x0"], inst["Xref"], Uref, cold_start=True, want_state=want)
        o = _port(prob, st, inst["x0"], inst["Xref"], Uref, None, True, want, nthreads=1)
        for key in H.OUT_KEYS + H.BOX_STATE:
            assert H.bits_equal(g[key], o[key]), (B, max_iter, check, key)


@pytest.mark.parametrize("kernel", ALLK)
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_fast_mode_within_reference_scatter(dt, kernel):
    """FAST mode = same operation order with FMA contraction.  It cannot be bit-identical to any Eigen build
    (SURVEY B.7), so it is held to the reference's own build-to-build scatter:
      (a) fixed work (tolerances 0, 20 iterations): |x,u difference| vs the pinned oracle <= 2e-4 relative in fp32
          (1e-10 in fp64) — pure arithmetic difference, no termination effects;
      (b) run to convergence: every instance solves, and the solution is at least as close to the fp64 oracle as
          the pinned fp32 oracle is (x2 slack) — in fp32 the iteration count itself is rounding-sensitive
          (the same instance takes 8..18 iterations depending on rounding), so iter is compared on the mean."""
    spec = wl.quadrotor(N=50)
    prob = setup_problem(spec, dt)
    B = 512
    inst = wl.tracking_instances(B, N=50, seed=5, dtype=dt)
    st = abi.Settings.from_buffer_copy(spec.settings)
    st.abs_pri_tol = st.abs_dua_tol = 0.0
    st.max_iter = 20
    solver = _mk_solver(prob, st, kernel, mode=abi.MODE_FAST)
    g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=("x", "u"))
    o = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, ("x", "u"))
    tol = 2e-4 if dt == np.float32 else 1e-10
    assert (g["iter"] == 20).all() and not g["solved"].any()
    for key in ("sol_x", "sol_u", "x", "u"):
        a, b = g[key].astype(np.float64), o[key].astype(np.float64)
        assert np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max()), (key, np.abs(a - b).max())
    assert not H.bits_equal(g["sol_x"], o["sol_x"]) or dt == np.float64  # FMA really changes fp32 bits
    # (b) to convergence, against the fp64 oracle
    st2 = spec.settings
    solver2 = _mk_solver(prob, st2, kernel, mode=abi.MODE_FAST)
    g2 = solver2.solve(inst["x0"], inst["Xref"], None, cold_start=True)
    o2 = _port(prob, st2, inst["x0"], inst["Xref"], None, None, True, ())
    prob64 = setup_problem(spec, np.float64)
    inst64 = {k: (None if v is None else v.astype(np.float64)) for k, v in inst.items()}
    o64 = _port(prob64, st2, inst64["x0"], inst64["Xref"], None, None, True, ())
    assert g2["solved"].all()
    err_fast = np.abs(g2["sol_u"].astype(np.float64) - o64["sol_u"]).max()
    err_pinned = np.abs(o2["sol_u"].astype(np.float64) - o64["sol_u"]).max()
    assert err_fast <= max(2.0 * err_pinned, 1e-9), (err_fast, err_pinned)
    assert g2["iter"].mean() <= 1.1 * o2["iter"].mean() + 0.5


@pytest.mark.parametrize("kernel", ALLK)
def test_device_pointer_path_equals_host_path(kernel):
    import torch

    spec = wl.quadrotor(N=50)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = spec.settings
    inst = wl.tracking_instances(700, N=50, seed=8, dtype=dt)
    solver = _mk_solver(prob, st, kernel)
    h = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=("u",))
    batch, out = solver.make_device_batch(inst["x0"], inst["Xref"], None, cold_start=True, want_state=("u",))
    solver.solve_device(batch)
    torch.cuda.synchronize()
    for key in ("sol_x", "sol_u", "iter", "solved", "residuals", "u"):
        assert H.bits_equal(h[key], out[key].cpu().numpy()), key
    s = solver.stats()
    assert s["kernel_launches"] == 1 and s["kernel_ms"] > 0


def test_full_size_identical_instances_and_shard_invariance():
    """BASELINE config 2 at full size (B=65536 identical hovering instances, N=50, fp32): every instance must equal
    the oracle's single solve (size-independent property), and solving two halves separately gives the same bits."""
    spec = wl.quadrotor(N=50)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = spec.settings
    B = 65536
    inst = wl.hovering_instances(B, N=50, dtype=dt)
    o = _port(prob, st, inst["x0"][:1], inst["Xref"], None, None, True, ("u",), nthreads=1)
    for kernel in ("gpi", "gpi_smem", "tpi", "gps"):
        solver = _mk_solver(prob, st, kernel)
        g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=("u",))
        if kernel in ("gpi", "gpi_smem"):
            # (12,4,50) fp32: g, y and d (5 columns per knot point and thread) fit in tensor memory for 8 warps per SM,
            # twice what shared memory alone holds
            stt = solver.stats()
            assert stt["tmem_cols_per_cta"] == (512 if kernel == "gpi" else 0)
            assert stt["instances_per_cta"] == (64 if kernel == "gpi" else 32)
        for key in ("sol_x", "sol_u", "iter", "solved", "residuals", "u"):
            assert H.bits_equal(g[key][:1], o[key]), (kernel, key)
            assert (g[key] == g[key][:1]).all(), (kernel, key)
        half = solver.solve(inst["x0"][: B // 2], inst["Xref"], None, cold_start=True)
        assert H.bits_equal(half["sol_u"], g["sol_u"][: B // 2])
        assert int(g["iter"].sum()) == 100 * B and not g["solved"].any()  # SURVEY B.4: runs to max_iter


@pytest.mark.parametrize("kernel", ["auto", "gps"])
def test_full_size_tracking_sample_vs_oracle(kernel):
    """BASELINE config 3 at full size (B=65536 randomised tracking instances, per-instance references) on the path the
    bench numbers come from (AUTO = on-chip lane groups with tensor memory) and on the streamed lane groups: the oracle is
    run on a strided sample of 512 instances; iteration histogram sanity on the whole batch."""
    import torch

    spec = wl.quadrotor(N=50)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = spec.settings
    B = 65536
    inst = wl.tracking_instances(B, N=50, seed=0, dtype=dt)
    solver = _mk_solver(prob, st, kernel)
    batch, out = solver.make_device_batch(inst["x0"], inst["Xref"], None, cold_start=True)
    solver.solve_device(batch)
    torch.cuda.synchronize()
    stt = solver.stats()
    if kernel == "auto":
        assert stt["kernel_family"] == abi.KERNEL_GPI and stt["tmem_cols_per_cta"] == 512 and stt["instances_per_cta"] == 64
    else:
        assert stt["kernel_family"] == abi.KERNEL_GPS and stt["workspace_bytes"] > 0
    assert stt["kernel_launches"] == 1
    g = {k: v.cpu().numpy() for k, v in out.items() if v is not None}
    idx = np.unique(np.concatenate([np.arange(0, B, B // 512), np.arange(B - 8, B)]))
    o = _port(prob, st, inst["x0"][idx], inst["Xref"][idx], None, None, True, ())
    for key in H.OUT_KEYS:
        assert H.bits_equal(g[key][idx], o[key]), key
    assert g["solved"].all() and g["iter"].max() < 100


def test_errors_are_loud():
    from tinympc_b200._lib import TinyMPCError

    spec = wl.quadrotor(N=10)
    prob = setup_problem(spec, np.float32)
    prob.x_min = prob.x_max = None  # bounds never set but en_state_bound = 1 (UB in the reference, SURVEY A.3-7)
    solver = BatchedTinySolver(prob, spec.settings)
    inst = wl.hovering_instances(4, N=10)
    with pytest.raises(TinyMPCError) as e:
        solver.solve(inst["x0"], inst["Xref"])
    assert e.value.code == abi.ERR_NO_BOUNDS
    # overlapping cones: the reference applies them one after the other (admm.cpp:115-121), so the second sees the
    # first one's result; every kernel family reproduces that
    rs = wl.rocket(N=10)
    rs.constraints = dict(rs.constraints, Acx=[0, 2], qcx=[3, 3], cx=[0.25, 0.5])
    rp = setup_problem(rs, np.float64)
    ri = wl.rocket_instances(5, N=10, spread=0.5)
    o = _port(rp, rs.settings, ri["x0"], ri["Xref"], ri["Uref"], None, True, ())
    for k in (abi.KERNEL_GPS, abi.KERNEL_GPI, abi.KERNEL_TPI, abi.KERNEL_AUTO):
        s2 = BatchedTinySolver(rp, rs.settings, kernel=k)
        g = s2.solve(ri["x0"], ri["Xref"], ri["Uref"])
        for key in H.OUT_KEYS:
            assert H.bits_equal(g[key], o[key]), (k, key)
    # hyperplane count without its matrices is an argument error at create(), not a device fault later
    bad = setup_problem(wl.quadrotor(N=10), np.float32)
    cp = bad.to_c()
    cp.num_state_linear = 2
    import ctypes as C
    from tinympc_b200._lib import load
    h = C.c_void_p()
    assert load().tinympc_b200_create(C.byref(cp), 0, C.byref(h)) == abi.ERR_ARG


@pytest.mark.parametrize("kernel", ALLK)
def test_device_resident_closed_loop_matches_oracle(kernel):
    """SURVEY §8f-1: the reference's closed loop (set x0 -> solve warm-started -> x0 = A x0 + B u0) for 300 plants kept
    entirely on the GPU (DeviceMPCLoop + tinympc_b200_advance) equals the oracle stepping the same loop on the host."""
    from tinympc_b200.closed_loop import DeviceMPCLoop

    spec = wl.quadrotor(N=10)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = spec.settings
    B, steps = 300, 6
    inst = wl.tracking_instances(B, N=10, seed=12, dtype=dt)
    traj = inst["Xref"]
    loop = DeviceMPCLoop(_mk_solver(prob, st, kernel), inst["x0"], reset_duals=True)
    x0 = inst["x0"].copy()
    state = None
    A, Bm, f = prob.A, prob.B, prob.f
    for k in range(steps):
        Xref = np.ascontiguousarray(np.roll(traj, -k, axis=1))  # a different window every step
        out = loop.step(Xref)
        if state is not None:
            state["g"] = np.zeros_like(state["g"])
            state["y"] = np.zeros_like(state["y"])
        o = _port(prob, st, x0, Xref, None, state, state is None, tuple(H.BOX_STATE))
        for key in H.OUT_KEYS + list(loop.fields):
            assert H.bits_equal(out[key].cpu().numpy(), o[key]), (k, key)
        assert H.bits_equal(out["u0"].cpu().numpy(), np.ascontiguousarray(o["u"][:, 0, :])), (k, "u0")
        state = {n: o[n] for n in H.BOX_STATE}
        u0 = o["u"][:, 0, :]
        nxt = np.zeros_like(x0)
        for i in range(prob.nx):  # same ascending-k, no-FMA arithmetic as tinympc_b200_advance
            ax = A[i, 0] * x0[:, 0]
            for m in range(1, prob.nx):
                ax = ax + A[i, m] * x0[:, m]
            bu = Bm[i, 0] * u0[:, 0]
            for j in range(1, prob.nu):
                bu = bu + Bm[i, j] * u0[:, j]
            nxt[:, i] = (ax + bu) + f[i]
        x0 = nxt
        assert H.bits_equal(loop.x0.cpu().numpy(), x0), ("advance", k)


@pytest.mark.parametrize("kernel", ALLK)
@pytest.mark.parametrize("dims", [(4, 2), (4, 8), (6, 3), (8, 8), (12, 2), (12, 8), (16, 2), (16, 4), (16, 8)])
def test_every_compiled_dimension_vs_oracle(dims, kernel):
    """Random LTI problems for the other compiled (nx, nu) pairs (lane mappings L=4 and L=8, padding rows),
    fixed work and to-convergence, fp32, against the oracle on every scalar."""
    nx, nu = dims
    dt = np.float32
    for N, B in ((10, 70), (33, 41)):
        spec = wl.random_lti(nx, nu, N, seed=nx * 10 + nu)
        prob = setup_problem(spec, dt)
        st = abi.Settings.from_buffer_copy(spec.settings)
        st.max_iter = 30
        inst = wl.random_instances(B, nx, N, seed=N, dtype=dt)
        inst["x0"] = (3.0 * inst["x0"]).astype(dt)  # large enough for the input bounds to bite
        solver = _mk_solver(prob, st, kernel)
        want = tuple(H.BOX_STATE)
        g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
        o = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want)
        for key in H.OUT_KEYS + H.BOX_STATE:
            assert H.bits_equal(g[key], o[key]), (dims, N, key)
        assert (np.abs(o["znew"]) >= 1.0 - 1e-6).any()  # the box was active somewhere


@pytest.mark.parametrize("kernel", ALLK)
def test_time_varying_bounds(kernel):
    """Bounds are full nx x N / nu x (N-1) matrices in the reference API (types.hpp:117-120); every example passes
    constants, here they really vary along the horizon."""
    spec = wl.quadrotor(N=20)
    dt = np.float32
    rng = np.random.default_rng(3)
    N = spec.N
    cons = dict(spec.constraints)
    cons["x_min"] = (-5.0 - rng.uniform(0, 1, (12, N))).astype(dt)
    cons["x_max"] = (5.0 + rng.uniform(0, 1, (12, N))).astype(dt)
    cons["u_min"] = (-0.5 + 0.3 * rng.uniform(0, 1, (4, N - 1))).astype(dt)
    cons["u_max"] = (0.5 - 0.3 * rng.uniform(0, 1, (4, N - 1))).astype(dt)
    spec.constraints = cons
    prob = setup_problem(spec, dt)
    st = spec.settings
    inst = wl.tracking_instances(90, N=N, seed=4, dtype=dt)
    solver = _mk_solver(prob, st, kernel)
    want = tuple(H.BOX_STATE)
    g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
    o = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want)
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g[key], o[key]), key


@pytest.mark.parametrize("kernel", ALLK)
def test_max_iter_zero_returns_the_warm_state(kernel):
    """max_iter = 0: solve() skips its loop (admm.cpp:378) and reports solution = vnew/znew as they stand, iter = 0."""
    spec = wl.quadrotor(N=10)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = abi.Settings.from_buffer_copy(spec.settings)
    inst = wl.tracking_instances(40, N=10, seed=2, dtype=dt)
    solver = _mk_solver(prob, spec.settings, kernel)
    first = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=tuple(H.BOX_STATE))
    st.max_iter = 0
    solver0 = _mk_solver(prob, st, kernel)
    state_g = {n: first[n].copy() for n in H.BOX_STATE}
    state_o = {n: first[n].copy() for n in H.BOX_STATE}
    g = solver0.solve(inst["x0"], inst["Xref"], None, state=state_g, cold_start=False)
    o = _port(prob, st, inst["x0"], inst["Xref"], None, state_o, False, ())
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g[key], o[key]), key
    assert (g["iter"] == 0).all() and H.bits_equal(g["sol_x"], first["vnew"])


@pytest.mark.parametrize("kernel", ALLK)
@pytest.mark.parametrize("N", [2, 3, 5])
def test_tiny_horizons(N, kernel):
    """N = 2 is the smallest horizon the reference can represent (one input column)."""
    spec = wl.quadrotor(N=N)
    dt = np.float64
    prob = setup_problem(spec, dt)
    st = spec.settings
    inst = wl.tracking_instances(37, N=N, seed=N, dtype=dt)
    solver = _mk_solver(prob, st, kernel)
    want = tuple(H.BOX_STATE)
    g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
    o = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want, nthreads=1)
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g[key], o[key]), (N, key)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_heterogeneous_models_per_instance(dt):
    """SURVEY §8f-2: every instance has its own (A, B, Q, R, rho) and cache (tinympc_batch_t.models); the on-chip kernel keeps
    each instance's matrix rows in its lane group's registers.  Checked against the oracle solving each model separately."""
    from tinympc_b200.problem import MPCProblem
    from tinympc_b200.solver import setup_models, unpack_model

    nx, nu, N, Bn = 12, 4, 20, 45
    specs = [wl.random_lti(nx, nu, N, seed=300 + i) for i in range(Bn)]
    rhos = np.array([0.5 + 0.1 * (i % 9) for i in range(Bn)])
    blobs = setup_models(nx, nu, np.stack([s.A for s in specs]), np.stack([s.B for s in specs]), np.stack([s.f for s in specs]),
                         np.stack([s.Qdiag for s in specs]), np.stack([s.Rdiag for s in specs]), rhos, dtype=dt)
    cons = specs[0].constraints
    st = abi.Settings.from_buffer_copy(specs[0].settings)
    st.max_iter = 40
    probs = []
    for i in range(Bn):
        m = unpack_model(blobs[i], nx, nu)
        rho = m.pop("rho")
        probs.append(MPCProblem(nx=nx, nu=nu, N=N, dtype=dt, rho=rho, **m, **cons))
    inst = wl.random_instances(Bn, nx, N, seed=9, dtype=dt)
    inst["x0"] = (2.0 * inst["x0"]).astype(dt)
    solver = _mk_solver(probs[0], st, "auto")
    want = tuple(H.BOX_STATE)
    g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want, models=blobs)
    assert solver.stats()["kernel_family"] == abi.KERNEL_GPI
    for i in range(Bn):
        o = _port(probs[i], st, inst["x0"][i:i + 1], inst["Xref"], None, None, True, want, nthreads=1)
        for key in H.OUT_KEYS + H.BOX_STATE:
            assert H.bits_equal(g[key][i:i + 1], o[key]), (i, key)
    assert len(set(g["iter"].tolist())) > 3  # the models really behave differently
    # the streaming kernel cannot hold per-instance matrices: explicit request is refused loudly
    from tinympc_b200._lib import TinyMPCError
    s2 = _mk_solver(probs[0], st, "tpi")
    with pytest.raises(TinyMPCError) as e:
        s2.solve(inst["x0"], inst["Xref"], None, cold_start=True, models=blobs)
    assert e.value.code == abi.ERR_UNSUPPORTED


@pytest.mark.parametrize("dims", [(4, 1), (12, 4), (16, 8)])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_device_precompute_bit_identical_to_host_precompute(dt, dims):
    """SURVEY §8f-2: the batched cache precompute on the device (one warp per model) produces exactly the blobs of the
    host routine (which restates tiny_api.cpp:117-118,307-381), including the number of Riccati sweeps' effect."""
    import torch
    from tinympc_b200.solver import setup_models

    nx, nu = dims
    Bn = 67
    specs = [wl.random_lti(nx, nu, 10, seed=100 + i) for i in range(Bn)]
    rhos = np.array([0.5 + 0.25 * (i % 7) for i in range(Bn)])
    args = (np.stack([s.A for s in specs]), np.stack([s.B for s in specs]), np.stack([s.f for s in specs]),
            np.stack([s.Qdiag for s in specs]), np.stack([s.Rdiag for s in specs]), rhos)
    host = setup_models(nx, nu, *args, dtype=dt)
    prob = setup_problem(specs[0], dt)
    solver = _mk_solver(prob, specs[0].settings, "auto")
    dev, sweeps = solver.setup_models_device(*args, want_sweeps=True)
    torch.cuda.synchronize()
    assert H.bits_equal(dev.cpu().numpy(), host)
    sw = sweeps.cpu().numpy()
    assert (sw > 1).all() and (sw <= 1000).all() and len(set(sw.tolist())) > 1


# ---------------------------------------------------------------------------------------------------------------------
# launch plans of the on-chip kernel: every compiled (nx, nu) at the horizons of the BASELINE sweep (N = 50, 100), so that
# each distinct (lanes per instance, instances per SM, tensor memory) plan of profiles/*_sweep_1gpu.md meets the oracle
# ---------------------------------------------------------------------------------------------------------------------
ALL_DIMS = [(4, 1), (6, 3), (12, 4), (4, 2), (4, 4), (4, 8), (8, 2), (8, 4), (8, 8), (12, 2), (12, 8), (16, 2), (16, 4), (16, 8)]
# fp32 plans as measured in the round-1 sweep table: (lanes per instance, instances per SM, tensor-memory columns > 0)
_P50 = {(4, 2): (4, 64, True), (4, 4): (4, 64, True), (8, 2): (4, 64, True), (8, 4): (4, 64, True), (12, 2): (4, 64, True),
        (12, 4): (4, 64, True), (4, 8): (4, 32, True), (8, 8): (4, 32, True), (12, 8): (8, 32, True), (16, 2): (8, 32, True),
        (16, 4): (8, 32, True), (16, 8): (8, 32, True)}
_P100 = {(4, 2): (4, 32, True), (4, 4): (4, 32, True), (8, 2): (4, 32, True), (8, 4): (4, 32, True), (12, 2): (4, 32, True),
         (12, 4): (4, 32, True), (4, 8): (8, 16, True), (8, 8): (8, 16, True), (12, 8): (8, 16, True), (16, 2): (8, 16, True),
         (16, 4): (8, 16, True), (16, 8): (8, 16, True)}
EXPECTED_F32_PLANS = {50: _P50, 100: _P100}
# fp64: matrix rows re-read per sweep (narrower lane groups) + dual variables in tensor memory, two columns per value
EXPECTED_F64_PLANS = {50: {(12, 4): (8, 16, True), (4, 2): (4, 32, True), (8, 4): (4, 32, True), (16, 8): (16, 8, True)}}


@pytest.mark.parametrize("N", [50, 100])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("dims", ALL_DIMS)
def test_launch_plans_long_horizons_vs_oracle(dims, dt, N):
    """kernel = GPI (planner's choice), AUTO and GPS on a ragged batch: cold solve + one warm-started solve, every scalar vs
    the oracle.  fp32: the plan the bench tables quote is asserted through stats()."""
    nx, nu = dims
    spec = wl.random_lti(nx, nu, N, seed=7 * nx + nu)
    prob = setup_problem(spec, dt)
    st = abi.Settings.from_buffer_copy(spec.settings)
    st.max_iter = 12
    B = 37
    inst = wl.random_instances(B, nx, N, seed=N + nx, dtype=dt)
    inst["x0"] = (3.0 * inst["x0"]).astype(dt)
    want = tuple(H.BOX_STATE)
    o1 = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want)
    x0b = (inst["x0"] * dt(0.9)).astype(dt)
    o2 = _port(prob, st, x0b, inst["Xref"], None, {n: o1[n].copy() for n in H.BOX_STATE}, False, want)
    for kernel in ("gpi", "auto", "gps"):  # "gps": the streamed lane groups (TMA record ring) at the long horizons too
        solver = _mk_solver(prob, st, kernel)
        g1 = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
        stt = solver.stats()
        if kernel == "gps":
            assert stt["kernel_family"] == abi.KERNEL_GPS and stt["workspace_bytes"] > 0
        for key in H.OUT_KEYS + H.BOX_STATE:
            assert H.bits_equal(g1[key], o1[key]), (dims, N, kernel, key)
        g2 = solver.solve(x0b, inst["Xref"], None, state={n: g1[n].copy() for n in H.BOX_STATE}, cold_start=False, want_state=want)
        for key in H.OUT_KEYS + H.BOX_STATE:
            assert H.bits_equal(g2[key], o2[key]), (dims, N, kernel, "warm", key)
        if kernel == "gpi":
            assert stt["kernel_family"] in (abi.KERNEL_GPI, abi.KERNEL_GPS)
            exp64 = EXPECTED_F64_PLANS.get(N, {}).get(dims)
            if dt == np.float64 and exp64 is not None:
                assert stt["kernel_family"] == abi.KERNEL_GPI
                got = (stt["lanes_per_instance"], stt["instances_per_cta"], stt["tmem_cols_per_cta"] > 0)
                assert got == exp64, (dims, N, got, exp64)
            exp = EXPECTED_F32_PLANS[N].get(dims)
            if dt == np.float32 and exp is not None:
                assert stt["kernel_family"] == abi.KERNEL_GPI
                got = (stt["lanes_per_instance"], stt["instances_per_cta"], stt["tmem_cols_per_cta"] > 0)
                assert got == exp, (dims, N, got, exp)


def test_full_size_rocket_sample_vs_oracle():
    """BASELINE config 4 at full size (16384 rocket-landing instances, N = 100, fp64, cones, per-instance references as in
    bench.py) on the path AUTO picks (streamed lane groups): a strided 256-instance sample against the oracle, all scalars."""
    import torch

    spec = wl.rocket(N=100)
    dt = np.float64
    prob = setup_problem(spec, dt)
    st = spec.settings
    B = 16384
    inst = wl.rocket_instances(B, N=100, seed=0, dtype=dt, per_instance_refs=True)
    solver = _mk_solver(prob, st, "auto")
    batch, out = solver.make_device_batch(inst["x0"], inst["Xref"], inst["Uref"], cold_start=True)
    solver.solve_device(batch)
    torch.cuda.synchronize()
    stt = solver.stats()
    assert stt["kernel_family"] == abi.KERNEL_GPS and stt["kernel_launches"] == 1
    g = {k: v.cpu().numpy() for k, v in out.items() if v is not None}
    idx = np.unique(np.concatenate([np.arange(0, B, B // 248), np.arange(B - 8, B)]))
    o = _port(prob, st, inst["x0"][idx], inst["Xref"][idx], inst["Uref"][idx], None, True, ())
    for key in H.OUT_KEYS:
        assert H.bits_equal(g[key][idx], o[key]), key
    assert int(g["iter"].sum()) == 100 * B  # never converges in the reference either: fixed work


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_device_precompute_vs_reference_tiny_setup(dt):
    """SURVEY §8f-2 against the REFERENCE: the device precompute's blobs vs the cache the compiled reference's tiny_setup
    computed (tiny_api.cpp:21-147,307-381; stored in tests/golden/ by tests/golden/make_golden.py), per model.  fp64: <= 1e-9 of the matrix's largest entry (measured
    5e-14); fp32: <= 2e-5 where the Riccati fixed point converges in float (measured worst 1.1e-5: ~150 sweeps of fp32
    rounding under a 1e-5 stopping rule), <= 1e-4 where it never does (quadrotor 20 Hz: 1000 sweeps of a rounding-level limit
    cycle, measured 4.6e-5 — Eigen's inverse and the product's Gauss-Jordan differ in the last bits of every sweep)."""
    import torch
    from tinympc_b200.solver import unpack_model

    gold = H.load_reference(f"tiny_setup_{np.dtype(dt).name}")
    for nx, nu, specs in H.precompute_models():
        prob = setup_problem(specs[0], dt)
        solver = _mk_solver(prob, specs[0].settings, "auto")
        args = (np.stack([s.A for s in specs]), np.stack([np.asarray(s.B).reshape(nx, nu) for s in specs]), np.stack([s.f for s in specs]),
                np.stack([s.Qdiag for s in specs]), np.stack([s.Rdiag for s in specs]), np.array([s.rho for s in specs]))
        dev, sweeps = solver.setup_models_device(*args, want_sweeps=True)
        torch.cuda.synchronize()
        dev, sweeps = dev.cpu().numpy(), sweeps.cpu().numpy()
        for i, sp in enumerate(specs):
            ref = H.problem_from_spec(sp, dt, H.stored_setup(gold, f"{nx}_{nu}", i))
            m = unpack_model(dev[i], nx, nu)
            tol = 1e-9 if dt == np.float64 else (2e-5 if sweeps[i] < 1000 else 1e-4)
            for f in ("Q", "R", "Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf"):
                a, b = np.asarray(m[f], np.float64), np.asarray(getattr(ref, f), np.float64).reshape(np.shape(m[f]))
                scale = max(float(np.abs(b).max()), 1e-30)
                assert float(np.abs(a - b).max()) <= tol * scale, (sp.name, i, f, float(np.abs(a - b).max()) / scale, int(sweeps[i]))


def test_closed_loop_without_previous_slacks_equals_reference_with_v_z_zeroed():
    """DeviceMPCLoop(exact_first_residual=False) drops work->v / work->z between steps.  Parity statement: that mode is the
    reference's loop with work->v and work->z zeroed before every tiny_solve — bit for bit (v, z only enter the dual
    residual of a solve's first iteration, admm.cpp:315,317)."""
    from tinympc_b200.closed_loop import DeviceMPCLoop

    spec = wl.quadrotor(N=10)
    dt = np.float32
    prob = setup_problem(spec, dt)
    st = spec.settings
    B, steps = 200, 5
    inst = wl.tracking_instances(B, N=10, seed=5, dtype=dt)
    loop = DeviceMPCLoop(_mk_solver(prob, st, "auto"), inst["x0"], reset_duals=True, exact_first_residual=False)
    x0, state = inst["x0"].copy(), None
    for k in range(steps):
        Xref = np.ascontiguousarray(np.roll(inst["Xref"], -k, axis=1))
        out = loop.step(Xref)
        if state is not None:
            for n in ("g", "y", "v", "z"):
                state[n] = np.zeros_like(state[n])
        o = _port(prob, st, x0, Xref, None, state, state is None, tuple(H.BOX_STATE))
        for key in H.OUT_KEYS + list(loop.fields):
            assert H.bits_equal(out[key].cpu().numpy(), o[key]), (k, key)
        state = {n: o[n] for n in H.BOX_STATE}
        x0 = loop.x0.cpu().numpy().copy()  # the plant update itself is covered by test_device_resident_closed_loop_matches_oracle


@pytest.mark.parametrize("kernel", ALLK)
def test_bounds_with_signed_zeros(kernel):
    """Bounds that contain +0 / -0: Eigen's compare-select clamp and min / max instructions differ in the SIGN of a zero
    result there, so the on-chip kernel must fall back to the compare-select form (it uses min / max only when no bound is
    a zero).  Inputs are chosen so that slacks land exactly on the zero bounds."""
    spec = wl.quadrotor(N=10)
    dt = np.float32
    spec.constraints = dict(x_min=np.array([-5, -5, 0.0, -5, -5, -5, -0.0, -5, -5, -5, -5, -5]), x_max=np.array([5, 5, 5, 5, -0.0, 5, 5, 5, 5, 5, 0.0, 5]),
                            u_min=np.array([-0.0, -0.5, 0.0, -0.5]), u_max=np.array([0.5, 0.0, 0.5, -0.0]))
    prob = setup_problem(spec, dt)
    st = abi.Settings.from_buffer_copy(spec.settings)
    st.max_iter = 25
    B = 77
    inst = wl.tracking_instances(B, N=10, seed=9, dtype=dt)
    inst["x0"][: B // 2] = -inst["x0"][: B // 2]
    solver = _mk_solver(prob, st, kernel)
    want = tuple(H.BOX_STATE)
    g = solver.solve(inst["x0"], inst["Xref"], None, cold_start=True, want_state=want)
    o = _port(prob, st, inst["x0"], inst["Xref"], None, None, True, want)
    for key in H.OUT_KEYS + H.BOX_STATE:
        assert H.bits_equal(g[key], o[key]), (kernel, key)
    z = o["znew"]
    assert (z == 0).any() and np.signbit(z[z == 0]).any() and (~np.signbit(z[z == 0])).any()  # both zero signs occur


def test_device_resident_closed_loop_with_cones_matches_oracle():
    """The device-resident MPC loop on the conic path (rocket landing, fp64, streamed lane groups): slacks and duals of the box
    AND cone constraints stay in HBM between steps (examples/rocket_landing_mpc.cpp:118-136 pattern: warm start, x0 advanced
    with the rollout input); every step equals the oracle stepping the same loop on the host."""
    from tinympc_b200.closed_loop import DeviceMPCLoop

    spec = wl.rocket(N=20)
    dt = np.float64
    prob = setup_problem(spec, dt)
    st = abi.Settings.from_buffer_copy(spec.settings)
    st.max_iter = 40
    B, steps = 90, 4
    inst = wl.rocket_instances(B, N=20, seed=4, dtype=dt)
    # cone slacks are re-initialised from the previous rollout at the start of solve() (admm.cpp:352-376): work->x / work->u
    # belong to the warm-start state of the conic path, next to the cone slack / dual pairs
    soc = ("x", "u", "vcnew", "zcnew", "gc", "yc")
    solver = _mk_solver(prob, st, "auto")
    loop = DeviceMPCLoop(solver, inst["x0"], reset_duals=False, extra_state=soc)
    x0, state = inst["x0"].copy(), None
    for k in range(steps):
        out = loop.step(inst["Xref"], inst["Uref"])
        assert solver.stats()["kernel_family"] == abi.KERNEL_GPS
        o = _port(prob, st, x0, inst["Xref"], inst["Uref"], state, state is None, tuple(H.SOC_STATE))
        for key in H.OUT_KEYS + list(loop.fields):
            assert H.bits_equal(out[key].cpu().numpy(), o[key]), (k, key)
        assert H.bits_equal(out["u0"].cpu().numpy(), np.ascontiguousarray(o["u"][:, 0, :])), (k, "u0")
        state = {n: o[n] for n in H.SOC_STATE}
        x0 = loop.x0.cpu().numpy().copy()


def test_auto_rule_choices():
    """TINYMPC_KERNEL_AUTO follows the measured rules of DESIGN.md §5 (csrc/capi.cu: resolve_family): which family serves
    which (constraints, dtype, shape, batch size).  Two iterations per instance are enough to see the choice in stats()."""
    import torch

    big = 148 * 384 + 64  # "big batch": one thread per instance fills the GPU
    cases = [
        ("box fp32, fits 64/SM on chip", wl.random_lti(12, 4, 50, seed=1), np.float32, 64, abi.KERNEL_GPI),
        ("box fp32, 16/SM on chip, big batch -> thread per instance", wl.random_lti(4, 8, 100, seed=1), np.float32, big, abi.KERNEL_TPI),
        ("box fp32, 16/SM on chip, small batch -> on chip", wl.random_lti(4, 8, 100, seed=1), np.float32, 4096, abi.KERNEL_GPI),
        ("box fp32 (16,8,100): on chip even at 16/SM", wl.random_lti(16, 8, 100, seed=1), np.float32, big, abi.KERNEL_GPI),
        ("box fp64, four warps per SM on chip", wl.random_lti(12, 4, 50, seed=1), np.float64, big, abi.KERNEL_GPI),
        ("box fp64, one warp per SM on chip, small shape -> streamed lane groups", wl.random_lti(6, 3, 100, seed=1), np.float64, big, abi.KERNEL_GPS),
        ("cones -> streamed lane groups", wl.rocket(N=20), np.float64, 256, abi.KERNEL_GPS),
    ]
    for what, spec, dt, B, expect in cases:
        st = abi.Settings.from_buffer_copy(spec.settings)
        st.max_iter = 2
        prob = setup_problem(spec, dt)
        solver = _mk_solver(prob, st, "auto")
        x0 = np.zeros((B, spec.nx), dt)
        x0[:, 0] = np.linspace(-1, 1, B)
        Xref = np.zeros((spec.N, spec.nx), dt)
        batch, out = solver.make_device_batch(x0, Xref, None, cold_start=True)
        solver.solve_device(batch)
        torch.cuda.synchronize()
        assert solver.stats()["kernel_family"] == expect, (what, solver.stats()["kernel_family"])
        assert int(out["iter"].min().item()) >= 1
        solver.close()
        del batch, out
        torch.cuda.empty_cache()
