"""bench.py's reference arm runs without a GPU; check the JSON line it prints against the driver's contract."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg2", "--steps", "3",
                          "--warmup", "3"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 3 and line["gpu_launches"] == 0 and line["vs_baseline"] is None
    cb, e2e = line["cpu_baseline"], line["e2e"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert e2e == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_dump_outputs_writes_parameters_and_the_step_record(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from uml_b200.engine.models.head import UML

    model = UML("synthetic:16", 8, 5, learnable_temp=True)  # img_proj 8 x 16, head 5 x 8, two scales
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 100)
    stats = {"image_loss": 1.25, "text_loss": 0.5, "img_acc": 0.25, "text_acc": 1.0}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), model, stats)
    names = {"img_proj.weight", "head.weight", "img_scale", "txt_scale", *stats}
    assert {f[:-4] for f in os.listdir(tmp_path / "a")} == names
    for n in names:
        a, b = np.load(tmp_path / "a" / f"{n}.npy"), np.load(tmp_path / "b" / f"{n}.npy")
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n  # the sample is the same in every run
    assert np.array_equal(np.load(tmp_path / "a" / "head.weight.npy"), model.head.weight.numpy())
    proj = np.load(tmp_path / "a" / "img_proj.weight.npy")
    assert proj.shape == (100,) and np.isin(proj, model.img_proj.weight.numpy()).all()
    assert float(np.load(tmp_path / "a" / "image_loss.npy")) == 1.25


def test_bench_rejects_what_it_cannot_do():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"],
                  ["--workload", "cfg2_sweep", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-2000:])
    assert not os.path.exists(os.path.join(ROOT, "unused"))


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "cfg2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
