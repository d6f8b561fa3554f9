#!/usr/bin/env python3
"""Generate the golden fixtures from the UNMODIFIED reference (run in the build container only).

    python tests/golden/make_golden.py [closed_loop] [reference] [families]

closed_loop — for each parity case (tests/helpers.py:make_cases) this runs the reference — compiled with the pinned flags
into oracle/_ref/libtinympc_ref_{f64,f32}.so by oracle/Makefile — through a warm-started closed loop and stores,
per case, one compressed .npz with
  * the complete problem (model, the cache the reference's tiny_setup computed, bounds, cones, hyperplanes),
  * the settings, the inputs of every step (x0 sequence, Xref, Uref),
  * the reference's outputs of every step (solution, iter, solved, residuals, and every state array).
The fixtures pin the oracle restatement (tests/test_oracle_golden.py, runs anywhere) and the CUDA path
(tests/test_gpu_parity.py) to the reference bit-for-bit without /root/reference being present.

reference — tests/golden/reference/: the reference's outputs for the other tests that compare with it
  * lti_sweep_<dtype>.npz   cache and digests of the closed-loop outputs of the random-LTI sweep (tests/helpers.py:lti_sweep),
  * tiny_setup_<dtype>.npz  the cache tiny_setup computes for tests/helpers.py:precompute_models,
  * sensitivity_tables.npz  the tables tiny_initialize_sensitivity_matrices leaves,
  * examples/<name>.txt.gz  what the reference's example programs print (oracle/_ref/examples_ref, oracle/Makefile).

families — tests/golden/reference/families_<dtype>.npz: the cones / hyperplanes cases (tests/helpers.py:family_cases), in the
lti_sweep format: per case the cache tiny_setup computed, the x0 of every step, and the digests of every output and every one
of the 20 state arrays of a warm-started three-step loop.  Written on its own so that the other fixtures stay untouched.
"""
import ctypes as C
import gzip
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import helpers as H  # noqa: E402
from oracle import oracle  # noqa: E402
from tinympc_b200 import abi  # noqa: E402

PROBLEM_FIELDS = ["A", "B", "f", "Q", "R", "Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf", "x_min", "x_max", "u_min",
                  "u_max", "Acx", "qcx", "cx", "Acu", "qcu", "cu", "Alin_x", "blin_x", "Alin_u", "blin_u", "tv_Alin_x",
                  "tv_blin_x", "tv_Alin_u", "tv_blin_u"]


def _reference(prob, settings, x0, Xref, Uref, state, cold, want):
    return oracle.solve_batch(prob, settings, x0, Xref, Uref, state=state, cold_start=cold, want_state=want, impl="reference")


def _save(name, arrays):
    path = os.path.join(H.REF_DIR, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path)} bytes")


def reference_outputs():
    os.makedirs(os.path.join(H.REF_DIR, "examples"), exist_ok=True)
    for dt in (np.float32, np.float64):
        tag = np.dtype(dt).name
        out, digests = {}, {}
        for key, sp, inst in H.lti_sweep(dt):
            prob = H.problem_from_spec(sp, dt, oracle.ref_setup)
            res, x0s = H.closed_loop(prob, sp.settings, inst, 3, False, H.BOX_STATE, _reference)
            out.update({f"{key}_{f}": getattr(prob, f) for f in H.CACHE_FIELDS})
            digests[f"{key}_x0_seq"] = H.digest(np.stack(x0s))
            for k, r in enumerate(res):
                digests.update({f"{key}_step{k}_{n}": H.digest(r[n]) for n in H.OUT_KEYS + H.BOX_STATE})
        _save(f"lti_sweep_{tag}", dict(out, names=np.array(list(digests)), digests=np.array(list(digests.values()))))
        out = {}
        for nx, nu, specs in H.precompute_models():
            probs = [H.problem_from_spec(sp, dt, oracle.ref_setup) for sp in specs]
            out.update({f"{nx}_{nu}_{f}": np.stack([getattr(p, f) for p in probs]) for f in H.CACHE_FIELDS})
        _save(f"tiny_setup_{tag}", out)
    tables = [np.zeros(s, np.float64, order="F") for s in ((4, 12), (12, 12), (4, 4), (12, 12))]
    assert oracle.ref_lib(np.float64).tinympc_ref_sensitivity_tables(*[C.c_void_p(a.ctypes.data) for a in tables]) == 0
    _save("sensitivity_tables", dict(zip(("dKinf_drho", "dPinf_drho", "dC1_drho", "dC2_drho"), tables)))
    exe_dir = os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle", "_ref", "examples_ref")
    for name in H.EXAMPLES:
        r = subprocess.run([os.path.join(exe_dir, name)], capture_output=True, text=True, cwd=exe_dir, check=True, timeout=600)
        path = os.path.join(H.REF_DIR, "examples", name + ".txt.gz")
        with open(path, "wb") as fh, gzip.GzipFile(fileobj=fh, mode="wb", mtime=0) as gz:
            gz.write(r.stdout.encode())
        print(f"examples/{name}.txt.gz: {os.path.getsize(path)} bytes")


def family_outputs():
    for dt in (np.float32, np.float64):
        out, digests = {}, {}
        for key, sp, inst in H.family_cases(dt):
            prob = H.problem_from_spec(sp, dt, oracle.ref_setup)
            res, x0s = H.closed_loop(prob, sp.settings, inst, 3, False, H.ALL_STATE, _reference)
            out.update({f"{key}_{f}": getattr(prob, f) for f in H.CACHE_FIELDS})
            out[f"{key}_x0_seq"] = np.stack(x0s)
            for k, r in enumerate(res):
                digests.update({f"{key}_step{k}_{n}": H.digest(r[n]) for n in H.OUT_KEYS + H.ALL_STATE})
        _save(f"families_{np.dtype(dt).name}", dict(out, names=np.array(list(digests)), digests=np.array(list(digests.values()))))


def closed_loop_fixtures():
    cases = H.make_cases()
    for name in sorted(cases):
        c = cases[name]
        prob = H.problem_from_spec(c["spec"], c["dtype"], oracle.ref_setup)
        st = c["spec"].settings

        def fn(prob, settings, x0, Xref, Uref, state, cold, want):
            return oracle.solve_batch(prob, settings, x0, Xref, Uref, state=state, cold_start=cold, want_state=want,
                                      impl="reference")

        res, x0s = H.closed_loop(prob, st, c["inst"], c["steps"], c["reset_duals"], c["state"], fn)
        out = dict(nx=prob.nx, nu=prob.nu, N=prob.N, rho=prob.rho, dtype=np.dtype(prob.dtype).name, steps=c["steps"],
                   reset_duals=int(c["reset_duals"]), state_names=np.array(c["state"]))
        for f in PROBLEM_FIELDS:
            v = getattr(prob, f)
            if v is not None:
                out["prob_" + f] = v
        for n, _ in abi.Settings._fields_:
            out["set_" + n] = getattr(st, n)
        out["Xref"] = np.asarray(c["inst"]["Xref"], dtype=prob.dtype)
        if c["inst"].get("Uref") is not None:
            out["Uref"] = np.asarray(c["inst"]["Uref"], dtype=prob.dtype)
        out["x0_seq"] = np.stack(x0s)
        for k, r in enumerate(res):
            for key in H.OUT_KEYS + c["state"]:
                out[f"step{k}_{key}"] = r[key]
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: {os.path.getsize(path)} bytes, iters step0 {res[0]['iter'].tolist()}")


if __name__ == "__main__":
    for part in sys.argv[1:] or ["closed_loop", "reference", "families"]:
        {"closed_loop": closed_loop_fixtures, "reference": reference_outputs, "families": family_outputs}[part]()
