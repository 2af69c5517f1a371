"""bench.py --dump-outputs on the device: the dump holds the trained head after exactly --steps timed steps and the
loss record the JSON line reports for the last of them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_the_timed_steps(tmp_path):
    out_dir = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg2", "--steps", "4", "--warmup", "3",
                          "--cpu-seconds", "1", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 4
    assert sorted(os.listdir(out_dir)) == ["head.weight.npy", "image_loss.npy", "img_acc.npy", "text_acc.npy", "text_loss.npy"]
    w = np.load(out_dir / "head.weight.npy")
    assert w.dtype == np.float32 and w.shape == (1000, 512) and np.isfinite(w).all()
    for k, v in line["final_losses"].items():
        got = np.load(out_dir / f"{k}.npy")
        assert got.dtype == np.float64 and float(got) == v, k
