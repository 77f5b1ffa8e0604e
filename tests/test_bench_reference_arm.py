"""`not gpu`: the reference arm of bench.py (`--impl reference`) needs no device -- it times the per-sample CPU port of the reference's
dynamics.inverse on the host cores -- so its contract is checked here too: one JSON line from rank 0 with the base keys, `impl`,
`cpu_baseline`, a zero-copy `e2e`, no GPU launches; every other rank of a torchrun launch exits 0 without output."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"}


def run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-samples", "64", *args],
                          capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)


def test_reference_arm_prints_one_contract_line_without_a_gpu():
    out = run({"CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["metric"] == "rnea_samples_per_s" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] == d["value"] and "sample" in c
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_rejects_zero_steps_and_a_dump_of_the_reference_arm(tmp_path):
    for extra in (("--steps", "0"), ("--dump-outputs", str(tmp_path))):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *extra], capture_output=True, text=True,
                             timeout=600, cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        assert out.returncode == 2 and extra[0] in out.stderr, out.stderr[-2000:]
        assert not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_other_ranks_exit_quietly():
    out = run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "CUDA_VISIBLE_DEVICES": ""}, "--gpus", "2")
    assert out.returncode == 0, out.stderr[-2000:]
    assert not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
