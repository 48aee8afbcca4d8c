"""The reference arm of bench.py (`--impl reference`) runs on the host CPU and must keep the JSON contract the driver
parses: one line, the candidate arm's metric / unit / config naming, `impl`, `cpu_baseline`, a zero-copy `e2e`."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--image-size", "224"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec at 224x224 bf16" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                              "--warmup", "0", "--image-size", "224", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(tmp_path / run)) == ["attention.npy", "confidence.npy", "depth.npy"]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("depth", "confidence", "attention")})
    a, b = dumps
    assert a["depth"].shape == a["confidence"].shape == (2, 1) and a["attention"].shape == (2, 256)
    for n in a:
        assert a[n].dtype == np.float32 and np.isfinite(a[n]).all()
        assert np.array_equal(a[n], b[n]), n


def test_dump_outputs_samples_what_exceeds_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 64 * 1024)
    big = {"a": torch.arange(40000, dtype=torch.float64), "b": torch.ones(3, 2)}
    bench.dump_outputs(str(tmp_path / "x"), big)
    bench.dump_outputs(str(tmp_path / "y"), big)
    sizes = sum(os.path.getsize(tmp_path / "x" / f) for f in os.listdir(tmp_path / "x"))
    assert sizes <= 64 * 1024
    a = np.load(tmp_path / "x" / "a.npy")
    assert a.dtype == np.float32 and 0 < a.size < 40000 and (np.diff(a) > 0).all()   # a sorted subset of the elements
    assert np.array_equal(a, np.load(tmp_path / "y" / "a.npy"))                        # ... the same one every time
    small = {"c": torch.ones(4, 5)}
    bench.dump_outputs(str(tmp_path / "z"), small)
    assert np.load(tmp_path / "z" / "c.npy").shape == (4, 5)                         # under the limit: whole


def test_candidate_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
