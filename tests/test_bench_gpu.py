"""bench.py --dump-outputs on the CUDA path: the arrays it writes are what the last timed step returned, checked against
the oracle on the same seeded weights and inputs (bench.py seeds both, so a dump identifies a build's results)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_are_the_last_timed_step(cuda_device, tmp_path):
    B, S, steps = 2, 224, 5
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                          "--batch", str(B), "--image-size", str(S), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("depth", "confidence", "attention")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["depth"].shape == got["confidence"].shape == (B, 1) and got["attention"].shape == (B, (S // 14) ** 2)
    # the last timed step i: instruction i % 9 on resident input batch i % 3 (bench.run_candidate, rank 0)
    i = steps - 1
    sd, x, ex = orc.build_state_dict(0), orc.synthetic_images(B, S, seed=1234 + i % 3), orc.synthetic_exif(B, seed=1236)
    torch.manual_seed(11)  # after build_state_dict, which seeds and draws from the same generator
    ref = orc.forward_with_guidance(sd, x, ex, bench.INSTRUCTIONS[i % 9], update_history=False)
    assert (np.abs(got["depth"] - ref["depth"].numpy()) / ref["depth"].numpy()).max() <= 1e-2
    assert np.abs(got["confidence"] - ref["confidence"].numpy()).max() <= 1e-2
    assert np.abs(got["attention"] - ref["heatmap"].numpy()).max() <= 1e-2
