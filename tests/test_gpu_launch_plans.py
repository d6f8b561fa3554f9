"""Launch geometry of every kernel family against a recorded table.

A grid of one-iteration solves (every compiled (nx, nu), fp32 / fp64, N in {10, 50, 100}, kernel AUTO / GPI / GPS / TPI,
batches from one instance to more than one full thread-per-instance wave, box constraints, cones and hyperplanes, with
and without the work->v / work->z outputs, the all-shared-memory GPI variant) runs on a fresh solver per case, and the
plan each solve reports through stats() (family, lanes, instances per CTA, CTAs, threads, shared / tensor memory,
workspace bytes, kernel launches) must match tests/golden/launch_plans_b200.json.gz.  The table belongs to one device:
the test fails on a card whose SM count or shared-memory opt-in differ from the ones it was recorded with.

    python tests/test_gpu_launch_plans.py --record out.json.gz   # regenerate the table (public Python API only)
"""
import argparse
import gzip
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import helpers as H  # noqa: E402
from tinympc_b200 import abi, workloads as wl  # noqa: E402
from tinympc_b200.problem import copy_settings  # noqa: E402
from tinympc_b200.solver import BatchedTinySolver, setup_problem  # noqa: E402

TABLE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "launch_plans_b200.json.gz")
DIMS = [(4, 1), (6, 3), (12, 4), (4, 2), (4, 4), (4, 8), (8, 2), (8, 4), (8, 8), (12, 2), (12, 8), (16, 2), (16, 4), (16, 8)]
DTYPES = {"f32": np.float32, "f64": np.float64}
HORIZONS = (10, 50, 100)
KERNELS = {"auto": abi.KERNEL_AUTO, "gpi": abi.KERNEL_GPI, "gps": abi.KERNEL_GPS, "tpi": abi.KERNEL_TPI}
BIG = 148 * 384 + 64  # just past the batch from which one thread per instance fills a 148-SM GPU
BATCHES = (1, 37, 4096, BIG)
PROBLEMS = [f"lti_{nx}_{nu}" for nx, nu in DIMS] + ["rocket", "quad_lin", "quad_tvlin"]
FIELDS = ("kernel_family", "lanes_per_instance", "instances_per_cta", "ctas", "threads_per_cta", "smem_bytes_per_cta",
          "tmem_cols_per_cta", "workspace_bytes", "kernel_launches", "gpi_instances")


def spec_of(problem, N):
    if problem == "rocket":
        return wl.rocket(N=N)
    if problem in ("quad_lin", "quad_tvlin"):
        return H.quad_linear_spec(tv=problem == "quad_tvlin", N=N)
    nx, nu = (int(v) for v in problem.split("_")[1:])
    return wl.random_lti(nx, nu, N, seed=nx + nu)


def cases(problem):
    """(N, kernel, B, variant) of one problem; variant: "" box / family constraints as the spec sets them, "vz" with
    work->v / work->z requested, "smem" with TINYMPC_GPI_TMEM=0, "host" through the host-pointer path"""
    lti = problem.startswith("lti")
    for N in HORIZONS:
        for kernel in KERNELS:
            for B in BATCHES:
                yield N, kernel, B, ""
                if kernel in ("auto", "gpi", "gps") and B in (37, 4096):
                    yield N, kernel, B, "vz"
                if lti and kernel == "gpi" and B in (37, BIG):
                    yield N, kernel, B, "smem"
                if lti and kernel in ("auto", "gpi") and B == BIG:
                    yield N, kernel, B, "host"


def key(problem, dt, N, kernel, B, variant):
    return f"{problem}/{dt}/N{N}/{kernel}/B{B}" + (f"/{variant}" if variant else "")


def run_case(prob, settings, inst, kernel, B, variant):
    """stats() after one solve on a fresh solver, or {"error": rc}"""
    import torch

    from tinympc_b200._lib import TinyMPCError

    if variant == "smem":
        os.environ["TINYMPC_GPI_TMEM"] = "0"
    try:
        solver = BatchedTinySolver(prob, settings, device=0, kernel=KERNELS[kernel])
        try:
            want = ("v", "z") if variant == "vz" else ()
            if variant == "host":
                solver.solve(inst["x0"], inst["Xref"], inst["Uref"], cold_start=True)
            else:
                batch, _ = solver.make_device_batch(inst["x0"], inst["Xref"], inst["Uref"], cold_start=True, want_state=want)
                solver.solve_device(batch)
                torch.cuda.synchronize()
            st = solver.stats()
            # workspace_bytes is compared on the device path only: a host-path solve of several chunks reports the plan
            # of its last chunk, while the handle's buffer was sized by the first
            return {f: int(st[f]) for f in FIELDS if not (variant == "host" and f == "workspace_bytes")}
        except TinyMPCError as e:
            return {"error": int(e.args[0])}
        finally:
            solver.close()
    finally:
        os.environ.pop("TINYMPC_GPI_TMEM", None)


def instances(problem, B, nx, N, dt):
    if problem == "rocket":
        return wl.rocket_instances(B, N=N, dtype=dt)
    return wl.random_instances(B, nx, N, seed=B + N, dtype=dt)


def run_problem(problem, dtname):
    dt = DTYPES[dtname]
    got = {}
    for N in HORIZONS:
        spec = spec_of(problem, N)
        prob = setup_problem(spec, dt)
        settings = copy_settings(spec.settings)
        settings.max_iter = 1
        insts = {}
        for N_, kernel, B, variant in cases(problem):
            if N_ != N:
                continue
            if B not in insts:
                insts[B] = instances(problem, B, spec.nx, N, dt)
            got[key(problem, dtname, N, kernel, B, variant)] = run_case(prob, settings, insts[B], kernel, B, variant)
    return got


def device():
    import torch

    p = torch.cuda.get_device_properties(0)
    return {"name": p.name, "sm_count": p.multi_processor_count, "smem_optin": p.shared_memory_per_block_optin}


@pytest.mark.gpu
@pytest.mark.parametrize("dtname", list(DTYPES))
@pytest.mark.parametrize("problem", PROBLEMS)
def test_launch_plans_match_table(problem, dtname):
    with gzip.open(TABLE, "rt") as fh:
        table = json.load(fh)
    here, rec = device(), table["device"]
    assert (here["sm_count"], here["smem_optin"]) == (rec["sm_count"], rec["smem_optin"]), \
        f"the table was recorded on {rec}, this device is {here}"
    want = {k: v for k, v in table["plans"].items() if k.startswith(f"{problem}/{dtname}/")}
    got = run_problem(problem, dtname)
    assert sorted(got) == sorted(want)
    bad = {k: (got[k], want[k]) for k in want if got[k] != want[k]}
    assert not bad, f"{len(bad)} of {len(want)} plans differ, e.g. {dict(list(bad.items())[:3])}"


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--record", required=True, metavar="OUT_JSON")
    a = ap.parse_args()
    plans = {}
    for problem in PROBLEMS:
        for dtname in DTYPES:
            plans.update(run_problem(problem, dtname))
            print(f"{problem} {dtname}: {len(plans)} plans", flush=True)
    rows = ",\n".join(f"{json.dumps(k)}: {json.dumps(plans[k], separators=(',', ':'))}" for k in sorted(plans))
    with (gzip.open if a.record.endswith(".gz") else open)(a.record, "wt") as fh:
        fh.write(f'{{"device": {json.dumps(device())},\n"plans": {{\n{rows}\n}}}}\n')
    print(f"{len(plans)} plans -> {a.record}")


if __name__ == "__main__":
    main()
