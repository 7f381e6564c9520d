"""`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) on the smallest workload: the line's contract, the
same-work fields, and the N > 1 launch in which only rank 0 works.  No GPU needed; the GPU arm of bench.py is exercised on the B200."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ); env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "real", "--steps", "2", "--warmup", "0",
                           "--single-rounds", "1", *args], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)


def test_reference_arm_line_contract(oracle):
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                   # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ICP iterations/sec (corr+LM)" and d["unit"] == "iter/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3
    assert "18 real Bunny_RealData frames" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if oracle.ref_lib() is not None else "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "rounds 0..1" in cb["sample"]
    assert cb["single_thread"]["cores"] == 1 and cb["single_thread"]["same_counts_as_all_core"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    assert len(d["inliers_per_round"]) == 2 and len(d["lm_iterations_per_round"]) == 2 and d["lm_iterations_per_round"][0] == 8
    assert d["inliers_per_round"][0] == 414972               # round 0 of the reference's default workload (tests/golden/bunny18.npz)
    assert len(d["pose_sha"]) == 64


def test_reference_arm_under_torchrun_only_rank0_works():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29999"}, ("--gpus", "2"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]      # ranks other than 0 exit without work
