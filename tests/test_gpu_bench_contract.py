"""-m gpu: bench.py honours the driver's JSON contract (keys, types, roofline / e2e / cpu_baseline objects) for every workload
and for the reference arm.  Small sizes so that the whole file runs in well under a minute."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
             "config", "e2e", "gpu_launches"}


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def check_common(d):
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert isinstance(d["config"], dict) and "workload" in d["config"] and "model" not in d["config"]
    if d.get("impl") != "reference":
        assert d["config"]["launch_mode"].startswith(("CUDA graph", "eager"))
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e) and e["value"] > 0


def test_default_workload_line():
    d = run_bench("--steps", "5", "--warmup", "3", "--samples", "262144", "--cpu-samples", "256", "--gram-samples", "300000")
    check_common(d)
    assert d["metric"] == "rnea_samples_per_s" and d["unit"] == "samples/s" and d["dtype"] == "f64" and d["n_gpus"] == 1
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert r["algorithmic_bytes_per_launch"] == 192 * 262144
    assert d["gpu_launches"] == 5
    # headline e2e = the SoA host entry: only the 15 live rows are uploaded (the kernel never reads the three gantry positions)
    assert r["live_input_rows"] == 15 and r["bytes_moved_per_launch"] == 168 * 262144 and abs(r["frac_moved"] - r["frac"] * 168 / 192) < 1e-12
    assert d["e2e"]["h2d_bytes_per_step"] == 120 * 262144 and d["e2e"]["d2h_bytes_per_step"] == 48 * 262144
    assert d["e2e"]["value"] < d["value"]  # host copies are inside the e2e timed region
    v = d["e2e"]["variants"]
    assert v["aos_host"]["h2d_bytes_per_step"] == 144 * 262144 and v["planned_host"]["h2d_bytes_per_step"] == 0 and v["planned_host"]["value"] > 0
    # the other BASELINE configs ride on the same line
    x = d["extra"]
    for dt_ in ("f64", "f32"):
        gx = x["gram"][dt_]
        assert gx["samples_per_gpu"] == 300_000 and gx["value"] > 0 and gx["pack_n_ok"] is True and 0 < gx["frac"] < 2
    assert x["linearize"]["value"] > 0 and x["rnea_f32"]["value"] > 0
    gen = x["rnea_generic"]
    assert gen["f64"]["kernel_path"] == "generic" and gen["f64"]["value"] > 0 and gen["f32"]["value"] > 0
    assert gen["f64"]["bound"] == "fp64 pipe" and 0 < gen["f64"]["frac_of_fp64_ceiling"] < 1
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    k = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(k)
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(k["reasons"]))


@pytest.mark.parametrize("extra", [("--dtype", "f32"), ("--workload", "gram", "--samples", "262144"), ("--workload", "gram", "--dtype", "f32", "--samples", "262144"),
                                   ("--workload", "linearize", "--samples", "65536")])
def test_other_workloads(extra):
    d = run_bench("--steps", "3", "--warmup", "3", "--no-cpu", "--no-extra", *extra)
    check_common(d)
    assert 0 < d["roofline"]["frac"] < 2


def test_dump_outputs(tmp_path):
    """--dump-outputs writes what the last timed step returned: the same in graph-replay and eager mode, equal to the oracle on that
    step's inputs, identical from run to run, and cut to a seeded subset of the samples when the outputs exceed 64 MB."""
    import numpy as np

    import bench
    from oracle import rnea_vec as rv

    n = 262144
    common = ("--steps", "1", "--warmup", "2", "--no-cpu", "--no-extra", "--samples", str(n))
    d = run_bench(*common, "--dump-outputs", str(tmp_path / "graph"))
    assert d["steps"] == 1 and d["config"]["launch_mode"].startswith("CUDA graph") and d["outputs"]["samples_kept"] == "all"
    run_bench(*common, "--eager", "--dump-outputs", str(tmp_path / "eager"))
    tau = np.load(tmp_path / "graph" / "tau.npy")
    assert tau.dtype == np.float64 and tau.shape == (6, n)
    assert np.array_equal(tau, np.load(tmp_path / "eager" / "tau.npy"))
    traj = bench.sample_states(np.random.default_rng(1000), n)[::997]  # the first input set is the one the single timed step reads
    c = bench.load_constants()
    ref = rv.inverse_batched(traj, c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0)["tau"]
    assert np.abs(tau[:, ::997].T - ref).max() < 1e-9 * np.abs(ref).max()

    lin = ("--workload", "linearize", "--samples", "65536", "--steps", "2", "--warmup", "1", "--no-cpu", "--no-extra")  # 113 MB of A, B
    d = run_bench(*lin, "--dump-outputs", str(tmp_path / "lin1"))
    run_bench(*lin, "--dump-outputs", str(tmp_path / "lin2"))
    k = d["outputs"]["samples_kept"]
    assert 0 < k < 65536
    for name, shape in (("A", (k, 12, 12)), ("B", (k, 12, 6))):
        a, b = np.load(tmp_path / "lin1" / f"{name}.npy"), np.load(tmp_path / "lin2" / f"{name}.npy")
        assert a.shape == shape and a.dtype == np.float64 and np.isfinite(a).all() and np.array_equal(a, b)
    assert sum(os.path.getsize(tmp_path / "lin1" / f) for f in os.listdir(tmp_path / "lin1")) <= bench.DUMP_BYTES + 1024


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-samples", "128")
    check_common(d)
    assert d["impl"] == "reference" and d["metric"] == "rnea_samples_per_s" and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] == "port"
