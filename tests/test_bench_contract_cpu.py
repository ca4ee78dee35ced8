"""CPU: the reference arm of bench.py (`--impl reference`: the CPU restatement on the host cores) prints exactly one
JSON line with the keys of the measurement contract."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "60",
                          "--warmup", "3", "--burnin", "40", "--cpu-budget", "1.5"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "agent-env-steps/sec" and d["unit"] == "agent-env-steps/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["data"] == "synthetic" and d["value"] > 0
    assert "workload" in d["config"] and "MA2C" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "replicas" in cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def test_reference_arm_covers_the_learner_and_the_monaco_scenario():
    """The reference arm times the same work as our arm (control step + policy forward + n-step update), says so in
    `sample`, and the configs[3] scenario (Monaco, 28 agents, n_step 40) runs through the same contract."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scenario", "real_net",
                          "--steps", "20", "--warmup", "3", "--burnin", "20", "--cpu-budget", "1.0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][0])
    assert "Monaco" in d["config"]["workload"] and "configs[3]" in d["config"]["workload"]
    s = d["cpu_baseline"]["sample"]
    assert "policy forward" in s and "A2C update" in s and "tsc_sim_ref.c" in s
    assert d["cpu_baseline"]["sim_only_value"] > d["value"] > 0
    assert d["cpu_baseline"]["cores"] <= len(os.sched_getaffinity(0))


def test_reference_arm_times_the_steps_it_reports():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "7",
                          "--warmup", "3", "--burnin", "20", "--cpu-budget", "1.0", "--mode", "sim"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][0])
    cb = d["cpu_baseline"]
    assert d["steps"] == cb["steps"] == 7 and " x 7 control steps after 20 burn-in steps" in cb["sample"]


def test_arguments_that_would_time_or_dump_nothing_are_rejected(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                  ["--impl", "reference", "--burnin", "240", "--steps", "481"]):     # 721 steps: past the 720-step episode
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr and not out.stdout.strip(), extra
    assert not os.listdir(tmp_path)
