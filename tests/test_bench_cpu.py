"""bench.py's CPU arm (`--impl reference`) end to end on a tiny budget: one JSON line with the contract's keys, the
true sizes of what was run, an explicit thread count, per-stage seconds.  No GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports: the CPU arm must ignore it
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-budget", "3", *extra], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_reference_arm_line_small_workload():
    j = _run("--workload", "small")
    assert j["impl"] == "reference" and j["unit"] == "evals/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == j["value"]
    assert cb["cores"] == max(1, len(os.sched_getaffinity(0)))            # not torchrun's OMP_NUM_THREADS=1
    assert set(cb["stage_s"]) == {"graph_s", "build_s", "cycle_s", "pgd_s", "gcw_s"}
    cfg = j["config"]
    assert cfg["m_cycle"] > 0 and cfg["n"] <= 2000 and isinstance(cfg["same_config"], bool)
    if not cfg["same_config"]:
        assert "reduced member" in cfg["workload"] and ("n=%d" % cfg["n"]) in cfg["workload"]


def test_reference_arm_ring_workload_has_no_gcw_stage():
    j = _run("--workload", "cfg5")
    assert "DESC_PGD" in j["metric"] and j["cpu_baseline"]["stage_s"]["gcw_s"] == 0.0
    assert j["config"]["same_config"] is False and j["config"]["n"] < 50000


def test_step_counts_below_one_are_rejected():
    for steps in ("0", "-1"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", steps],
                           capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""


def test_other_ranks_of_a_torchrun_launch_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""
