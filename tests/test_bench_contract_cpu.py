"""bench.py's reference arm (the reference's own scripts from oracle/_ref on the host cores -- the oracle port only when that copy is
absent) runs without a GPU: check the JSON line the driver parses -- one line on stdout, the base-contract keys, the tier's `cpu_baseline` /
`e2e` objects, `"impl": "reference"`, and that `steps` / `warmup` say what was actually run."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "7", "--warmup", "2",
                          "--batch", "2"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train clips/sec" and d["unit"] == "clips/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "causal_anomaly_detection.py" in d["config"]["workload"]
    # the M-A reference step is seconds of CPU work: at most 3 timed steps + 1 warm-up are run, and the line reports THAT, not the request
    assert d["steps"] == 3 and d["warmup"] == 1 and d["requested"] == {"steps": 7, "warmup": 2}
    cb = d["cpu_baseline"]
    from oracle.ref_harness import reference_dir
    assert cb["kind"] == ("reference" if reference_dir() is not None else "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_of_the_other_workloads():
    """--workload mc_infer (BASELINE.json configs[0], the reference's own CPU-runnable case): frames/s of SimpleVideoAnomalyDetector.forward."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "mc_infer", "--steps", "3", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip())
    assert d["impl"] == "reference" and d["metric"] == "inference frames/sec" and d["unit"] == "frames/s" and d["steps"] == 3 and d["value"] > 0
    assert d["config"]["name"] == "mc_infer" and "minicausal_vad_complete3.py" in d["config"]["workload"]
