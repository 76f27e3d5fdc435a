"""CPU test of the bench.py driver contract on the arm that needs no GPU (`--impl reference`): exactly one JSON line with the
keys the driver reads, the tier-specific objects (`cpu_baseline`, `e2e` with zero copy bytes), and sane values."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0", "--n", "1536"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "TFLOP/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"]


def test_bench_rejects_zero_steps_and_dumps_outside_the_gpu_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "dump"], ["--gpus", "2", "--dump-outputs", "dump"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                             cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ)
    env["RANK"] = "1"; env["WORLD_SIZE"] = "2"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]
