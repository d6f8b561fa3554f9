#!/usr/bin/env python3
"""bench.py — the contract benchmark of the batched TinyMPC solve path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[1], the configuration the metric is quoted on): quadrotor_hovering
(nx=12, nu=4, N=50, box constraints, quadrotor_20hz data), batch = 65536 identical instances per GPU, fp32,
cold start, max_iter=100, tolerances 1e-3.  One "step" = one batched tiny_solve() of the whole batch.
This instance does not converge in the reference either (SURVEY B.4): every instance runs the full 100 ADMM
iterations, so the metric "instances solved/s" is "instances terminated/s by the reference's rule", and
ADMM iterations/s/GPU is reported next to it.  Arithmetic mode: STRICT (bit-identical to the pinned reference).

value  : device-resident throughput, inputs already in HBM, CUDA events on the launch stream, per-step events,
         L2 flushed (256 MiB write) between timed steps, max over ranks.
e2e    : the same metric through the public host API (BatchedTinySolver.solve_prepared -> tinympc_b200_solve_host):
         pinned host inputs copied H2D and the complete solution copied D2H inside the timed region, every step.
configs: the other BASELINE configs, each timed the same way (device events, L2 flushed, max over ranks) with its own
         roofline and — at N=1 and in the reference arm — the reference's CPU figure for the same workload:
           C3  quadrotor_tracking, per-instance reference windows, to convergence (iteration histogram, solved fraction)
           C4  rocket_landing, second-order cones, N=100, fp64, per-instance references, 16384 instances per GPU
           C5  three corners of the random-LTI sweep at 2^20/8 = 131072 instances per GPU, fixed work (50 iterations)
         Under --gpus N every config runs sharded the same way (weak: fixed instances per GPU).
roofline, cpu_baseline, clocks: see DESIGN.md §7.

--impl reference times the reference's own CPU implementation (oracle/_ref = the unmodified reference compiled
here; falls back to the oracle port when the prebuilt library is absent) on the host cores, same metric/config:
a persistent pool of one TinySolver per thread (built once), threads = the cores this process may actually use
(affinity mask and cgroup quota, both reported), >= 256 instances per thread per step, warmed up; the 1-thread
figure and the per-core figure are reported next to it (BASELINE.md §3.3).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "quadrotor_hovering nx=12 nu=4 N=50 box batch=65536/GPU identical instances fp32 cold-start max_iter=100 (BASELINE configs[1])"
METRIC = "MPC instances solved/sec (terminated by the reference rule; ADMM iters/sec/GPU alongside)"
B_PER_GPU = 65536
N_HORIZON = 50
KERNEL_NAMES = {1: "tpi", 2: "gpi", 4: "gps"}
# `config` is the same dict in both arms (the driver compares them); arm-specific details go to `plan` / `arm`
CONFIG = {"workload": WORKLOAD, "instances_per_gpu": B_PER_GPU,
          "l2": "GPU arm: flushed (256 MiB write) between timed steps; CPU arm: every step re-solves the sample from cold state"}
# --dump-outputs: instances written per config; with every config dumped the files stay below 64 MB in all
DUMP_INSTANCES = 1024
DUMP_KEYS = ("sol_x", "sol_u", "iter", "solved", "residuals")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="strict", choices=["strict", "fast"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "tpi", "gpi", "gps"])
    ap.add_argument("--cpu-per-thread", type=int, default=256, help="instances per host thread per step in the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `configs` block (C3/C4/C5)")
    ap.add_argument("--extra-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed solve of each config returned as DIR/<config>_<name>.npy "
                         f"(float32/float64; at most {DUMP_INSTANCES} instances per config, a fixed seeded sample of larger batches)")
    args = ap.parse_args()
    if args.steps < 1 or args.extra_steps < 1:
        ap.error("--steps and --extra-steps must be >= 1")
    return args


# ---------------------------------------------------------------------------------------------------------
# workloads: the BASELINE configs as (model spec, dtype, instances per GPU, instance generator)
# ---------------------------------------------------------------------------------------------------------
def bytes_inst(nx, nu, N, es, per_x, per_u, warm=False):
    """Algorithmic bytes per instance, SURVEY §8(d)."""
    nN, mN = nx * N, nu * (N - 1)
    return es * nx + es * (nN * int(per_x) + mN * int(per_u)) + 2 * es * (nN + mN) * int(warm) + es * (nN + mN) + 4 * es + 8


def bytes_shared(nx, nu, N, es):
    nN, mN = nx * N, nu * (N - 1)
    return es * (1 + 2 * nx * nu + 3 * nx * nx + nu * nu + 3 * nx + 2 * nu + 2 * (nN + mN))


def flops_iter(nx, nu, N):
    """Box-only flop count of one ADMM iteration, SURVEY §8(d)."""
    return (N - 1) * (4 * nx * nx + 8 * nx * nu + 2 * nu * nu + 5 * nx + 4 * nu) + 2 * nx * nx + 15 * (nx * N + nu * (N - 1))


def make_case(name, B=None, seed=0):
    """-> dict(name, label, spec, dtype, B, inst) — identical for the GPU arm and the CPU arm (same generator, same seed)."""
    from tinympc_b200 import workloads as wl

    if name == "C2":
        spec, dt, B = wl.quadrotor(N=N_HORIZON), np.float32, B or B_PER_GPU
        inst = wl.hovering_instances(B, N=N_HORIZON, dtype=dt)
        label = WORKLOAD
    elif name == "C3":
        spec, dt, B = wl.quadrotor(N=N_HORIZON), np.float32, B or 65536
        inst = wl.tracking_instances(B, N=N_HORIZON, seed=seed, dtype=dt)
        label = ("quadrotor_tracking nx=12 nu=4 N=50 box, per-instance reference windows + x0 jitter, fp32, cold start, to convergence "
                 "(tol 1e-3, max_iter=100), batch=65536/GPU (BASELINE configs[2])")
    elif name == "C4":
        spec, dt, B = wl.rocket(N=100), np.float64, B or 16384
        inst = wl.rocket_instances(B, N=100, seed=seed, dtype=dt, per_instance_refs=True)
        label = ("rocket_landing nx=6 nu=3 N=100 box + one state cone + one input cone (dim 3), fp64, per-instance x0 (+-10%) and references, "
                 "cold start, max_iter=100 (never converges in the reference either: fixed work), batch=16384/GPU (BASELINE configs[3])")
    elif name.startswith("C5"):
        nx, nu, N = (int(v) for v in name.split("_")[1:])
        spec, dt, B = wl.random_lti(nx, nu, N, seed=1), np.float32, B or 131072
        spec.settings.abs_pri_tol = 0.0
        spec.settings.abs_dua_tol = 0.0
        spec.settings.max_iter = 50
        inst = wl.random_instances(B, nx, N, seed=2, dtype=dt)
        label = (f"random LTI nx={nx} nu={nu} N={N} box, fp32, cold start, fixed work (max_iter=50, tolerances 0), "
                 "batch=131072/GPU = 2^20/8 (BASELINE configs[4], one corner of the sweep)")
    else:
        raise ValueError(name)
    return dict(name=name, label=label, spec=spec, dtype=dt, B=B, inst=inst)


EXTRA_CASES = ["C3", "C4", "C5_4_2_10", "C5_12_4_50", "C5_16_8_100"]


# ---------------------------------------------------------------------------------------------------------
# host cores this process can really use
# ---------------------------------------------------------------------------------------------------------
def host_cores():
    """affinity mask, cgroup CPU quota (v2 cpu.max / v1 cfs_quota) -> threads the CPU arm uses."""
    info = {"cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except AttributeError:
        info["affinity"] = info["cpu_count"]
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except (OSError, ValueError):
        pass
    if quota is None:
        for base in ("/sys/fs/cgroup/cpu", "/sys/fs/cgroup/cpu,cpuacct"):
            try:
                q = int(open(base + "/cpu.cfs_quota_us").read())
                p = int(open(base + "/cpu.cfs_period_us").read())
                if q > 0 and p > 0:
                    quota = q / p
                break
            except (OSError, ValueError):
                continue
    info["cgroup_quota_cores"] = quota
    eff = info["affinity"]
    if quota is not None:
        eff = max(1, min(eff, int(math.ceil(quota))))
    info["effective"] = eff
    return info


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores (oracle/_ref), or the oracle port
# ---------------------------------------------------------------------------------------------------------
def cpu_case(case, steps, warmup, per_thread, cores):
    """Times the reference on a bounded sample (the first instances) of `case` -> dict(value inst/s, iters_per_s, one_thread, ...)."""
    from oracle import oracle
    from tinympc_b200.batch import HostBatch

    spec, dt, inst = case["spec"], case["dtype"], case["inst"]
    threads = cores["effective"]
    sample = min(case["B"], max(per_thread * threads, 1024))
    one_n = min(case["B"], per_thread)

    def sub(n):
        xr, ur = inst["Xref"], inst.get("Uref")
        return dict(x0=inst["x0"][:n], Xref=xr[:n] if np.ndim(xr) == 3 else xr, Uref=None if ur is None else (ur[:n] if np.ndim(ur) == 3 else ur))

    variants = [v for v in ("fast", "fastv3") if oracle.ref_available(dt, v)]
    res = {}
    if variants:
        kind = "reference"
        prob = oracle.ref_setup(spec.nx, spec.nu, spec.N, spec.rho, spec.A, spec.B, spec.f, spec.Qdiag, spec.Rdiag, dtype=dt,
                                variant=variants[0], **spec.constraints)
        s1 = sub(one_n)
        hb1 = HostBatch(prob, s1["x0"], s1["Xref"], s1["Uref"], cold_start=True)
        # the faster build of the reference (SSE2 vs AVX2+FMA), decided on one thread
        best, best_t = variants[0], 1e30
        for v in variants:
            pool = oracle.RefPool(prob, spec.settings, 1, variant=v)
            pool.solve(hb1, chunk=8)
            t = min(pool.solve(hb1, chunk=8) for _ in range(2))
            pool.close()
            if t < best_t:
                best, best_t = v, t
        variant = best
        res["one_thread"] = one_n / best_t
        res["one_thread_iters_per_s"] = float(hb1.iter.sum()) / best_t
        sN = sub(sample)
        hbN = HostBatch(prob, sN["x0"], sN["Xref"], sN["Uref"], cold_start=True)
        pool = oracle.RefPool(prob, spec.settings, threads, variant=variant)
        chunk = max(1, min(16, sample // (threads * 8)))
        for _ in range(max(1, warmup)):
            pool.solve(hbN, chunk=chunk)
        secs = [pool.solve(hbN, chunk=chunk) for _ in range(steps)]
        pool.close()
        iters_step = int(hbN.iter.sum())
        solved_step = int(hbN.solved.sum())
    else:
        kind, variant = "port", "oracle/tinympc_oracle.c -O2 -ffp-contract=off"
        prob = oracle.port_setup(spec.nx, spec.nu, spec.N, spec.rho, spec.A, spec.B, spec.f, spec.Qdiag, spec.Rdiag, dtype=dt,
                                 **spec.constraints)

        def run(n, nth):
            s_ = sub(n)
            t0 = time.perf_counter()
            r = oracle.solve_batch(prob, spec.settings, s_["x0"], s_["Xref"], s_["Uref"], cold_start=True, impl="port", nthreads=nth)
            return time.perf_counter() - t0, r
        run(one_n, 1)
        t1, r1 = run(one_n, 1)
        res["one_thread"] = one_n / t1
        res["one_thread_iters_per_s"] = float(r1["iter"].sum()) / t1
        for _ in range(max(1, warmup)):
            run(sample, threads)
        secs, r = [], None
        for _ in range(steps):
            t, r = run(sample, threads)
            secs.append(t)
        iters_step, solved_step = int(r["iter"].sum()), int(r["solved"].sum())
    tot = float(sum(secs))
    value = sample * steps / tot
    res.update(value=value, iters_per_s=iters_step * steps / tot, kind=kind, variant=variant, threads=threads,
               per_core=value / threads, parallel_speedup=value / res["one_thread"], ms_per_step=tot / steps * 1e3,
               solved_fraction=solved_step / sample, mean_iters=iters_step / sample, sample_instances=sample,
               sample=f"{sample} instances per step ({iters_step} ADMM iterations), {steps} timed step(s) after {max(1, warmup)} warm-up, "
                      f"{threads} pooled host threads (one TinySolver each, built once), {np.dtype(dt).name} build '{variant}'; "
                      f"1-thread figure on {one_n} instances",
               unit="instances/s")
    return res


def cpu_summary(c, cores):
    return {"value": c["value"], "unit": "instances/s", "cores": c["threads"], "kind": c["kind"], "sample": c["sample"],
            "admm_iters_per_s": c["iters_per_s"], "per_core": c["per_core"], "one_thread": c["one_thread"],
            "one_thread_admm_iters_per_s": c["one_thread_iters_per_s"], "parallel_speedup": c["parallel_speedup"],
            "solved_fraction": c["solved_fraction"], "mean_iters": c["mean_iters"],
            "host": {"cpu_count": cores["cpu_count"], "affinity": cores["affinity"], "cgroup_quota_cores": cores["cgroup_quota_cores"]}}


def reference_main(args, rank, world):
    if rank != 0:
        return
    cores = host_cores()
    W = max(1, args.warmup)
    c2 = cpu_case(make_case("C2"), args.steps, W, args.cpu_per_thread, cores)
    cb = cpu_summary(c2, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": c2["value"], "unit": "instances/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": W, "ms_per_step": c2["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(CONFIG), "arm": "reference CPU implementation on the host cores (bounded sample per step)",
        "admm_iters_per_s": c2["iters_per_s"],
        "cpu_baseline": cb,
        "e2e": {"value": c2["value"], "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_extras:
        cfgs = {}
        for name in EXTRA_CASES:
            try:
                case = make_case(name)  # the GPU arm's batch (same generator, same seed): the sample is its first instances
                c = cpu_case(case, 2, 1, args.cpu_per_thread, cores)
                cfgs[name] = {"workload": case["label"], "dtype": np.dtype(case["dtype"]).name, "ms_per_step": c["ms_per_step"],
                              "cpu_reference": cpu_summary(c, cores), "value": c["value"], "unit": "instances/s"}
            except Exception as e:
                cfgs[name] = {"error": str(e)[:200]}
        line["configs"] = cfgs
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, the recipe's query)
# ---------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.rows:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                if t0 - 0.05 <= t <= t1 + 0.05:
                    sm.append(float(p[1]))
                    power.append(float(p[3]))
                    for n, v in zip(names, p[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
                smax = float(p[2])
            except ValueError:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------------------
# NUMA: run this rank's host threads (and first-touch its pinned buffers) next to its GPU
# ---------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(local):
    try:
        import torch

        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"numa_node": None}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus_bound": len(allowed)}
    except Exception as e:  # best effort: topology files may be absent in a container
        return {"numa_node": None, "note": str(e)[:80]}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
class Gpu:
    def __init__(self, args, local, world):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.args, self.local, self.world = args, local, world
        self.dev = torch.device("cuda", local)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.stream = torch.cuda.current_stream(self.dev)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, xs):
        if self.world == 1:
            return [float(x) for x in xs]
        t = self.torch.tensor([float(x) for x in xs], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().tolist()

    def device_arm(self, solver, case, K, W):
        """W warm-up + K timed batched solves, device-resident inputs, per-step CUDA events, L2 flushed between steps."""
        torch = self.torch
        inst = case["inst"]
        batch, out = solver.make_device_batch(inst["x0"], inst["Xref"], inst.get("Uref"), cold_start=True)
        for _ in range(W):
            solver.solve_device(batch, self.stream)
        torch.cuda.synchronize(self.dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        self.barrier()
        for i in range(K):
            self.flush.zero_()
            ev[i][0].record(self.stream)
            solver.solve_device(batch, self.stream)
            ev[i][1].record(self.stream)
        self.barrier()
        step_ms = [a.elapsed_time(b) for a, b in ev]
        return batch, out, step_ms

    def e2e_arm(self, solver, prob, case, K, W):
        """Public host API on pinned host buffers: H2D of the inputs and D2H of the complete solution inside the timed region."""
        from tinympc_b200.batch import HostBatch

        torch = self.torch
        inst = case["inst"]
        hb = HostBatch(prob, inst["x0"], inst["Xref"], inst.get("Uref"), cold_start=True)
        pins = {}
        for name in ("x0", "Xref", "Uref", "sol_x", "sol_u", "iter", "solved", "residuals"):
            a = getattr(hb, name)
            if a is None:
                continue
            tpin = torch.from_numpy(np.array(a, copy=True)).pin_memory()
            pins[name] = tpin
            setattr(hb, name, tpin.numpy())
        cb = hb.to_c()
        for _ in range(W):
            solver.solve_prepared(hb, cb)
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            solver.solve_prepared(hb, cb)
        torch.cuda.synchronize(self.dev)
        ms = self.max_over_ranks((time.perf_counter() - t0) * 1e3)
        h2d = int(hb.x0.nbytes + hb.Xref.nbytes + (0 if hb.Uref is None else hb.Uref.nbytes))
        d2h = int(hb.sol_x.nbytes + hb.sol_u.nbytes + hb.iter.nbytes + hb.solved.nbytes + hb.residuals.nbytes)
        hb._pins = pins
        return hb, ms, h2d, d2h


def roofline(case, st, k_ms, iters_per_launch, peak, peak_src):
    spec, es = case["spec"], np.dtype(case["dtype"]).itemsize
    inst = case["inst"]
    per_x = np.ndim(inst["Xref"]) == 3
    per_u = inst.get("Uref") is not None and np.ndim(inst["Uref"]) == 3
    # SURVEY §8(d): one "per-instance refs" switch for Xref and Uref together (C3 = 6 440 B, C4 = 14 440 B); the bytes a
    # launch really has to move are fewer when Uref is NULL or shared (reported next to it)
    bi = bytes_inst(spec.nx, spec.nu, spec.N, es, per_x, per_x or per_u)
    bi_moved = bytes_inst(spec.nx, spec.nu, spec.N, es, per_x, per_u)
    alg = case["B"] * bi + st["ctas"] * bytes_shared(spec.nx, spec.nu, spec.N, es)
    achieved = alg / (k_ms * 1e-3) / 1e9
    fl = iters_per_launch * flops_iter(spec.nx, spec.nu, spec.N) / (k_ms * 1e-3)
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "bytes_per_instance": bi, "bytes_per_instance_moved": bi_moved, "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms,
            "flops_achieved_tflops": fl / 1e12, "workspace_bytes": st["workspace_bytes"]}


def plan_of(st):
    return {"kernel": KERNEL_NAMES.get(st["kernel_family"], str(st["kernel_family"])), "lanes_per_instance": st["lanes_per_instance"],
            "ctas": st["ctas"], "threads_per_cta": st["threads_per_cta"], "smem_bytes_per_cta": st["smem_bytes_per_cta"],
            "tmem_cols_per_cta": st["tmem_cols_per_cta"], "instances_per_cta": st["instances_per_cta"]}


def dump_outputs(dirname, name, out):
    """Writes the arrays a caller of the timed path receives (`out` of the last timed solve) as float32/float64 .npy files,
    restricted to a fixed seeded sample of DUMP_INSTANCES instances when the batch is larger, so that two builds run with the
    same arguments can be compared output for output."""
    import torch

    B = int(out["iter"].shape[0])
    idx = np.arange(B) if B <= DUMP_INSTANCES else np.sort(np.random.default_rng(0).choice(B, DUMP_INSTANCES, replace=False))
    os.makedirs(dirname, exist_ok=True)
    for key in DUMP_KEYS:
        a = out[key].index_select(0, torch.as_tensor(idx, device=out[key].device)).cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)  # iter, solved: int32, exact in float64
        np.save(os.path.join(dirname, f"{name}_{key}.npy"), a)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_main(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from tinympc_b200 import abi
    from tinympc_b200.parallel import reduce_stats
    from tinympc_b200.solver import BatchedTinySolver, setup_problem

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cores_before = host_cores()
    numa = bind_to_gpu_numa(local) if world > 1 else {"numa_node": None, "note": "single rank: not bound"}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    g = Gpu(args, local, world)

    K, W = args.steps, max(3, args.warmup)
    mode = abi.MODE_STRICT if args.mode == "strict" else abi.MODE_FAST
    kern = dict(auto=abi.KERNEL_AUTO, tpi=abi.KERNEL_TPI, gpi=abi.KERNEL_GPI, gps=abi.KERNEL_GPS)[args.kernel]
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    # ---- headline: C2 ----
    case = make_case("C2")
    B = case["B"]
    prob = setup_problem(case["spec"], case["dtype"])
    solver = BatchedTinySolver(prob, case["spec"].settings, device=local, mode=mode, kernel=kern)
    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.25)
    t_wall0 = time.perf_counter()
    batch, out, step_ms = g.device_arm(solver, case, K, W)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "C2", out)
    total_ms = float(sum(step_ms))
    st = solver.stats()
    iters_step = int(out["iter"].sum().item())
    solved_step = int(out["solved"].sum().item())
    res_max = out["residuals"].max(dim=0).values.double().cpu().tolist()
    red = reduce_stats(dict(instances=B * K, solved=solved_step * K, iters=iters_step * K, res_max=res_max, ms=total_ms),
                       device=dev if world > 1 else None)
    launches = K * st["kernel_launches"]
    hb, e2e_ms, h2d, d2h = g.e2e_arm(solver, prob, case, K, W)
    e2e_launches = solver.stats()["kernel_launches"]
    clk = clocks.stop(t_wall0, time.perf_counter())
    e2e_ok = bool(np.array_equal(hb.sol_u.view(np.uint8), out["sol_u"].cpu().numpy().view(np.uint8)))
    k_ms = float(np.mean(step_ms))  # one launch per step: the step IS the kernel
    roof = roofline(case, st, k_ms, iters_step, peak, peak_src)
    traffic_table = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic_table = json.load(open(tpath))  # DRAM bytes per launch from the committed ncu captures
        except Exception:
            traffic_table = {}
    roof["traffic"] = traffic_table.get(f"family{st['kernel_family']}_{args.mode}")
    roof["note"] = ("compute-bound by construction (SURVEY §8d: ~2000 flop per compulsory byte); the fp32-pipe / issue-slot "
                    "utilisation from ncu is the quality figure (profiles/r02_ncu_summary.md)")
    roof["flops_frac_of_74.5_tflops_fp32"] = roof["flops_achieved_tflops"] / 74.5
    del batch, out, hb
    solver.close()
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs ----
    cfgs = {}
    extra_launches = 0
    if not args.no_extras:
        Kx = max(1, min(K, args.extra_steps))
        for name in EXTRA_CASES:
            c = make_case(name, seed=rank)  # a different shard of the instance stream per rank
            p = setup_problem(c["spec"], c["dtype"])
            s = BatchedTinySolver(p, c["spec"].settings, device=local, mode=mode, kernel=abi.KERNEL_AUTO)
            b_, o_, ms_ = g.device_arm(s, c, Kx, W)
            if args.dump_outputs and rank == 0:
                dump_outputs(args.dump_outputs, name, o_)
            sx = s.stats()
            it = o_["iter"]
            iters_x, solved_x = int(it.sum().item()), int(o_["solved"].sum().item())
            hist = torch.bincount(it.clamp(min=0), minlength=1).cpu().tolist()
            tot = g.max_over_ranks(float(sum(ms_)))
            s_iters, s_solved = g.sum_over_ranks([iters_x, solved_x])
            kx = float(np.mean(ms_))
            entry = {"workload": c["label"], "dtype": np.dtype(c["dtype"]).name, "instances_per_gpu": c["B"], "steps": Kx,
                     "ms_per_step": tot / Kx, "value": world * c["B"] * Kx / (tot * 1e-3), "unit": "instances/s",
                     "admm_iters_per_s_per_gpu": s_iters / world * Kx / (tot * 1e-3), "solved_fraction": s_solved / (world * c["B"]),
                     "mean_iters": s_iters / (world * c["B"]),
                     "iter_histogram_rank0": {str(i): n for i, n in enumerate(hist) if n},
                     "plan": plan_of(sx), "gpu_launches": Kx * sx["kernel_launches"],
                     "roofline": roofline(c, sx, kx, iters_x, peak, peak_src)}
            entry["roofline"]["traffic"] = traffic_table.get(f"{name.split('_')[0].lower()}_family{sx['kernel_family']}_{args.mode}")
            extra_launches += Kx * sx["kernel_launches"]
            del b_, o_
            if name in ("C3", "C4"):
                hbx, ems, h2dx, d2hx = g.e2e_arm(s, p, c, Kx, 2)
                entry["e2e"] = {"value": world * c["B"] * Kx / (ems * 1e-3), "unit": "instances/s", "ms_per_step": ems / Kx,
                                "h2d_bytes_per_step": h2dx, "d2h_bytes_per_step": d2hx}
                del hbx
            s.close()
            torch.cuda.empty_cache()
            cfgs[name] = entry

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": world * B * K / (red["ms"] * 1e-3), "unit": "instances/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": red["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": dict(CONFIG),
        "plan": dict({"mode": args.mode, "parallelism": f"batch-sharded x{world}, no data-path collective", "gpi_instances": st["gpi_instances"],
                      "numa": numa}, **plan_of(st)),
        "admm_iters_per_s_per_gpu": red["iters"] / world / (red["ms"] * 1e-3),
        "solved_fraction": red["solved"] / red["instances"],
        "residual_max": red["res_max"],
        "gpu_launches": launches,
        "e2e": {"value": world * B * K / (e2e_ms * 1e-3), "unit": "instances/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / K, "kernel_launches_per_step": e2e_launches, "matches_device_arm": e2e_ok},
        "roofline": roof,
        "clocks": clk,
    }
    if cfgs:
        line["configs"] = cfgs
        line["gpu_launches_configs"] = extra_launches
    if not args.no_cpu_baseline and world == 1:
        try:
            cores = cores_before
            pt = args.cpu_per_thread
            c2 = cpu_case(make_case("C2"), 2, 1, pt, cores)
            line["cpu_baseline"] = cpu_summary(c2, cores)
            for name in cfgs:
                cc = cpu_case(make_case(name), 1, 1, pt, cores)
                cfgs[name]["cpu_reference"] = cpu_summary(cc, cores)
        except Exception as e:  # the checker libraries are optional for the product arm
            line["cpu_baseline"] = {"value": None, "unit": "instances/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": str(e)[:200]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
