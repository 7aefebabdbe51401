"""CPU: the reference arm of bench.py (the oracle port of learn() on the host cores -- the one leg of bench.py that may execute
oracle/) runs without a GPU and prints the JSON line the driver parses."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "ppo_update_samples_per_s" and line["unit"] == "samples/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1 and line["value"] > 0
    assert line["config"]["workload"].startswith("synthetic scale")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bad_arguments_are_refused_before_any_work():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr and out.stdout == "", (extra, out.stderr[-500:])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
