"""bench.py --dump-outputs on the GPU: the arrays written are what the timed path returned in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_step(dev, gold, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "mc_infer", "--steps", "5", "--warmup", "1", "--no-cpu",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip())
    assert d["steps"] == 5 and d["self_check"]["ok"]
    assert sorted(os.listdir(tmp_path)) == ["scores_T16.npy"]
    got = np.load(tmp_path / "scores_T16.npy")
    assert got.dtype == np.float32 and got.shape == (4, 1)
    # inference on fixed weights and a seeded batch: every step returns the scores of the unmodified reference on that batch
    want = next(c for c in gold("mc.pt")["eval"] if c["weights"] == "synth" and (c["B"], c["T"], c["seed"]) == (4, 16, 1234))["scores"].numpy()
    assert float(np.abs(got - want).max() / np.abs(want).max()) < 1e-5
