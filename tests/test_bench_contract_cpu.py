"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (the CPU oracle port) prints one JSON
line with the keys the driver reads, and the product arm refuses to run without a B200 (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, timeout=600):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT, env=env)


def test_reference_arm_prints_the_contract_line():
    r = run("--impl", "reference", "--workload", "c1", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "points/s"
    assert line["steps"] == 2
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["gpu_launches"] == 0 and line["value"] > 0


def test_product_arm_refuses_to_run_without_a_gpu():
    r = run("--steps", "1", "--warmup", "1", "--workload", "c4cmps", timeout=900)
    assert r.returncode != 0
    assert "B200" in (r.stderr + r.stdout)
