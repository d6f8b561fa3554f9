"""Shared test helpers: the parity cases (small versions of the BASELINE configs + the reference's example
workloads) and a closed-loop runner that feeds warm-start state back the way the reference's examples do."""
from __future__ import annotations

import hashlib
import os

import numpy as np

from tinympc_b200 import abi, workloads as wl
from tinympc_b200.problem import MPCProblem, copy_settings

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# further outputs of the unmodified reference (tests/golden/make_golden.py), kept apart from the closed-loop fixtures above
REF_DIR = os.path.join(GOLDEN_DIR, "reference")
CACHE_FIELDS = ("Q", "R", "Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf")
BOX_STATE = ["x", "u", "v", "z", "vnew", "znew", "g", "y"]
SOC_STATE = BOX_STATE + ["vcnew", "zcnew", "gc", "yc"]
LIN_STATE = BOX_STATE + ["vlnew", "zlnew", "gl", "yl"]
TVLIN_STATE = BOX_STATE + ["vlnew_tv", "zlnew_tv", "gl_tv", "yl_tv"]
ALL_STATE = list(abi.STATE_FIELDS)
OUT_KEYS = ["sol_x", "sol_u", "iter", "solved", "residuals"]


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def problem_from_spec(spec: wl.ModelSpec, dtype, setup) -> MPCProblem:
    """setup(nx,nu,N,rho,A,B,f,Qdiag,Rdiag,dtype=..., **constraints) -> MPCProblem (oracle.ref_setup / port_setup)."""
    return setup(spec.nx, spec.nu, spec.N, spec.rho, spec.A, spec.B, spec.f, spec.Qdiag, spec.Rdiag, dtype=dtype,
                 **spec.constraints)


def digest(a):
    """First 128 bits of the SHA-256 of an array's dtype, shape and bytes: comparing digests is a bit-for-bit comparison
    (bits_equal) against an array that need not be stored."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


def stored_setup(store, prefix, index=None):
    """A setup like oracle.ref_setup whose Q, R and cache are the ones the reference's tiny_setup computed, read from `store`
    (a golden .npz) as <prefix>_<field>, or as row `index` of it."""
    def setup(nx, nu, N, rho, A, B, f, Qdiag, Rdiag, dtype=np.float64, **constraints) -> MPCProblem:
        dt = np.dtype(dtype).type
        cache = {k: store[f"{prefix}_{k}"] if index is None else store[f"{prefix}_{k}"][index] for k in CACHE_FIELDS}
        return MPCProblem(nx=nx, nu=nu, N=N, dtype=dt, rho=float(dt(rho)), A=np.asfortranarray(A, dtype=dt),
                          B=np.asfortranarray(np.asarray(B, dtype=dt).reshape(nx, nu)), f=np.ascontiguousarray(f, dtype=dt),
                          **cache, **constraints)
    return setup


def load_reference(name):
    return np.load(os.path.join(REF_DIR, name + ".npz"))


def lti_sweep(dt):
    """Randomised sweep over the compiled (nx, nu) pairs and short horizons (BASELINE config 5's generator) ->
    [(key, spec, inst)]: warm-started three-step loops whose first x0 pushes the rollout into the box bounds."""
    dims = [(4, 1), (4, 2), (4, 8), (6, 3), (8, 4), (12, 2), (12, 8), (16, 4), (16, 8)]
    out = []
    for n, (nx, nu) in enumerate(dims):
        N = (3, 7, 12)[n % 3]
        sp = wl.random_lti(nx, nu, N, seed=40 + n)
        sp.settings.max_iter = 25
        sp.settings.check_termination = 1 + n % 3
        inst = wl.random_instances(5, nx, N, seed=70 + n, dtype=dt)
        inst["x0"] = (3.0 * inst["x0"]).astype(dt)
        out.append((f"{nx}_{nu}_{N}", sp, inst))
    return out


def precompute_models():
    """[(nx, nu, [spec])]: the models whose tiny_setup cache the device precompute is checked against."""
    return [(12, 4, [wl.quadrotor(N=10), wl.quadrotor(N=10, hz=50)] + [wl.random_lti(12, 4, 10, seed=i) for i in range(6)]),
            (6, 3, [wl.rocket(N=10)] + [wl.random_lti(6, 3, 10, seed=i) for i in range(5)]),
            (16, 8, [wl.random_lti(16, 8, 10, seed=i) for i in range(6)])]


EXAMPLES = ["cartpole_example", "quadrotor_hovering", "quadrotor_tracking", "rocket_landing_mpc", "quadrotor_linear_constraints",
            "quadrotor_tv_linear_constraints"]


def quad_linear_spec(tv=False, N=10):
    """examples/quadrotor_linear_constraints.cpp / quadrotor_tv_linear_constraints.cpp in spirit: the 50 Hz
    quadrotor with hyperplanes on the state and on the input; bounds disabled as the examples do (:70-71)."""
    spec = wl.quadrotor(N=N, hz=50)
    s = copy_settings(spec.settings)
    s.en_state_bound = 0
    s.en_input_bound = 0
    s.max_iter = 60
    rng = np.random.default_rng(5)
    cons = {}
    if not tv:
        Ax = np.zeros((2, 12)); Ax[0, 0] = 1.0; Ax[0, 1] = 0.5; Ax[1, 2] = -1.0; Ax[1, 0] = 0.25
        bx = np.array([0.3, -0.2])
        Au = np.array([[1.0, 1.0, 1.0, 1.0]]); bu = np.array([0.4])
        cons.update(Alin_x=Ax, blin_x=bx, Alin_u=Au, blin_u=bu)
        s.en_state_linear = 1
        s.en_input_linear = 1
    else:
        nsx, nsu = 2, 1
        Ax = np.zeros((nsx * N, 12))
        for k in range(N):
            Ax[nsx * k + 0, 0] = 1.0; Ax[nsx * k + 0, 1] = 0.1 * k
            Ax[nsx * k + 1, 2] = -1.0; Ax[nsx * k + 1, 1] = 0.3
        bx = 0.2 + 0.05 * rng.standard_normal((nsx, N))
        Au = np.tile(np.array([[1.0, -1.0, 1.0, 0.5]]), (nsu * (N - 1), 1)) * (1.0 + 0.1 * np.arange(N - 1))[:, None]
        bu = 0.3 + 0.02 * rng.standard_normal((nsu, N - 1))
        cons.update(tv_Alin_x=Ax, tv_blin_x=bx, tv_Alin_u=Au, tv_blin_u=bu)
        s.en_tv_state_linear = 1
        s.en_tv_input_linear = 1
    spec.constraints = cons
    spec.settings = s
    return spec


def make_cases():
    """name -> dict(spec, dtype, inst (x0,Xref,Uref), steps, reset_duals, state_names)"""
    cases = {}
    for dt, tag in ((np.float64, "f64"), (np.float32, "f32")):
        sp = wl.cartpole()
        cases[f"cartpole_{tag}"] = dict(spec=sp, dtype=dt, steps=40, reset_duals=False, state=BOX_STATE,
                                        inst=dict(x0=np.array([[0.5, 0, 0, 0]]), Xref=np.tile([1.0, 0, 0, 0], (sp.N, 1)), Uref=None))
        sp = wl.quadrotor(N=10)
        cases[f"quad_hover_N10_{tag}"] = dict(spec=sp, dtype=dt, steps=6, reset_duals=False, state=BOX_STATE,
                                              inst=wl.hovering_instances(3, N=10, dtype=dt))
        sp = wl.quadrotor(N=50)
        cases[f"quad_hover_N50_{tag}"] = dict(spec=sp, dtype=dt, steps=2, reset_duals=False, state=BOX_STATE,
                                              inst=wl.hovering_instances(2, N=50, dtype=dt))
        cases[f"quad_track_N50_{tag}"] = dict(spec=sp, dtype=dt, steps=3, reset_duals=True, state=BOX_STATE,
                                              inst=wl.tracking_instances(9, N=50, seed=3, dtype=dt))
        sp = wl.rocket(N=10)
        cases[f"rocket_soc_N10_{tag}"] = dict(spec=sp, dtype=dt, steps=5, reset_duals=False, state=SOC_STATE,
                                              inst=wl.rocket_instances(5, N=10, seed=1, dtype=dt))
        sp = wl.rocket(N=100)
        cases[f"rocket_soc_N100_{tag}"] = dict(spec=sp, dtype=dt, steps=1, reset_duals=False, state=SOC_STATE,
                                               inst=wl.rocket_instances(3, N=100, seed=2, dtype=dt))
        sp = wl.rocket(N=10)
        sp.constraints = dict(sp.constraints, cx=[0.1], cu=[0.02], Acx=[1], Acu=[0])  # both cone branches active
        cases[f"rocket_soc_tight_{tag}"] = dict(spec=sp, dtype=dt, steps=3, reset_duals=False, state=SOC_STATE,
                                                inst=wl.rocket_instances(4, N=10, seed=7, dtype=dt, spread=0.5))
        sp = quad_linear_spec(tv=False)
        rng = np.random.default_rng(11)
        x0 = 0.3 * rng.standard_normal((4, 12))
        cases[f"quad_lin_{tag}"] = dict(spec=sp, dtype=dt, steps=3, reset_duals=False, state=LIN_STATE,
                                        inst=dict(x0=x0, Xref=np.zeros((sp.N, 12)), Uref=None))
        sp = quad_linear_spec(tv=True)
        cases[f"quad_tvlin_{tag}"] = dict(spec=sp, dtype=dt, steps=3, reset_duals=False, state=TVLIN_STATE,
                                          inst=dict(x0=x0, Xref=np.zeros((sp.N, 12)), Uref=None))
        sp = wl.random_lti(8, 2, 10, seed=1)
        cases[f"lti_8_2_{tag}"] = dict(spec=sp, dtype=dt, steps=2, reset_duals=False, state=BOX_STATE,
                                       inst=wl.random_instances(6, 8, 10, seed=4, dtype=dt))
    return cases


def closed_loop(prob: MPCProblem, settings, inst, steps, reset_duals, state_names, solve_fn, x0_seq=None):
    """Run `steps` warm-started MPC steps (examples/quadrotor_tracking.cpp:77-106 pattern).

    solve_fn(prob, settings, x0, Xref, Uref, state, cold_start, want_state) -> result dict.
    If x0_seq is given (replay of a golden file) the measured states come from it; otherwise they are
    simulated as x0 <- A x0 + B u0 + f with the rollout input work->u[:,0].
    Returns (list of result dicts, list of x0 arrays used).
    """
    dt = prob.dtype
    x0 = np.ascontiguousarray(inst["x0"], dtype=dt).reshape(-1, prob.nx)
    state = None
    results, x0s = [], []
    for k in range(steps):
        if x0_seq is not None:
            x0 = np.ascontiguousarray(x0_seq[k], dtype=dt)
        x0s.append(x0.copy())
        if state is not None and reset_duals:  # quadrotor_tracking.cpp:92-93
            state["g"] = np.zeros_like(state["g"])
            state["y"] = np.zeros_like(state["y"])
        r = solve_fn(prob, settings, x0, inst["Xref"], inst.get("Uref"), state, state is None, tuple(state_names))
        results.append({k_: (None if v is None else np.array(v, copy=True)) for k_, v in r.items()})
        state = {n: r[n] for n in state_names}
        u0 = r["u"][:, 0, :].astype(np.float64)
        xn = x0.astype(np.float64) @ prob.A.astype(np.float64).T + u0 @ prob.B.astype(np.float64).T + prob.f.astype(np.float64)
        x0 = xn.astype(dt)
    return results, x0s


def load_golden(name):
    """-> (MPCProblem, Settings, inst, meta, steps[list of dict]) from tests/golden/<name>.npz"""
    d = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    dt = np.dtype(str(d["dtype"])).type
    kw = {k[5:]: d[k] for k in d.files if k.startswith("prob_")}
    prob = MPCProblem(nx=int(d["nx"]), nu=int(d["nu"]), N=int(d["N"]), dtype=dt, rho=float(d["rho"]), **kw)
    st = abi.Settings()
    for n, _ in abi.Settings._fields_:
        setattr(st, n, type(getattr(st, n))(d["set_" + n]))
    inst = dict(x0=d["x0_seq"][0], Xref=d["Xref"], Uref=d["Uref"] if "Uref" in d.files else None)
    names = [str(s) for s in d["state_names"]]
    steps = []
    for k in range(int(d["steps"])):
        steps.append({key: d[f"step{k}_{key}"] for key in OUT_KEYS + names})
    meta = dict(steps=int(d["steps"]), reset_duals=bool(int(d["reset_duals"])), state=names, x0_seq=d["x0_seq"])
    return prob, st, inst, meta, steps


def golden_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))
