"""bench.py contract pieces: without a GPU, the algorithmic byte / flop counts of SURVEY §8(d), the host-core probe and the
reference arm's JSON line (run on a tiny sample); on the GPU, the arrays --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_survey_byte_and_flop_counts():
    assert bench.bytes_inst(12, 4, 50, 4, False, False) == 3256    # C2: identical instances, cold, fp32
    assert bench.bytes_inst(12, 4, 50, 4, True, True) == 6440      # C3: per-instance references
    assert bench.bytes_inst(6, 3, 100, 8, True, True) == 14440     # C4: fp64, per-instance references
    assert bench.bytes_inst(4, 1, 10, 8, True, True) == 856        # C1
    assert bench.flops_iter(12, 4, 50) == 64560
    assert bench.flops_iter(4, 1, 10) == 1865
    assert bench.flops_iter(16, 8, 100) == 262904


def test_host_core_probe():
    c = bench.host_cores()
    assert 1 <= c["effective"] <= c["affinity"] <= c["cpu_count"]
    assert c["cgroup_quota_cores"] is None or c["cgroup_quota_cores"] > 0


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--no-extras",
                        "--cpu-per-thread", "16"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["config"] == bench.CONFIG
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["one_thread"] > 0 and cb["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dump_outputs_writes_the_timed_solution(tmp_path):
    """--dump-outputs writes, after the timed steps, the headline solve's arrays (a fixed sample of its instances) as
    float32/float64 .npy files; they equal the oracle's solve of the same instances bit for bit."""
    import numpy as np

    from oracle import oracle
    from tinympc_b200.solver import setup_problem

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extras", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    got = {k: np.load(tmp_path / f"C2_{k}.npy") for k in bench.DUMP_KEYS}
    assert sorted(os.listdir(tmp_path)) == sorted(f"C2_{k}.npy" for k in bench.DUMP_KEYS)
    assert all(a.dtype in (np.float32, np.float64) and a.shape[0] == bench.DUMP_INSTANCES for a in got.values())
    case = bench.make_case("C2", B=bench.DUMP_INSTANCES)  # identical instances: any sample of the batch is this batch
    prob = setup_problem(case["spec"], case["dtype"])
    ref = oracle.solve_batch(prob, case["spec"].settings, case["inst"]["x0"], case["inst"]["Xref"], None, cold_start=True, nthreads=4)
    for k in bench.DUMP_KEYS:
        assert np.array_equal(got[k], ref[k].astype(got[k].dtype)), k
