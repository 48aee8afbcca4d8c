"""Instruction sweep against the calls it replaces: one `forward_with_guidance_sweep` over the nine instructions of
demo_results/ against nine `forward_with_guidance` calls, alternating in one process.

    python tools/bench_sweep.py [--steps 30] [--warmup 5] [--shapes 1x224,32x518]

Timing: CUDA events on the calling stream around each arm (a sweep, or the nine calls), after warm-up of both arms at
every shape.  The images rotate through a set larger than the 126 MB L2 so that no arm reads its input from the cache
the other arm left.  Prints one JSON line with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cognitive_aim_depth_estimation_b200.model import create_model  # noqa: E402

INSTRUCTIONS = ["center", "left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right"]
CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
L2_BYTES = 126 * 2 ** 20


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout
        power, clock = (v.strip() for v in out.strip().split(","))
        info.update(power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except (FileNotFoundError, ValueError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, max_sm_clock_mhz=None)
    return info


def bench(model, B: int, S: int, steps: int, warmup: int):
    dev = torch.device("cuda:0")
    per_input = B * 3 * S * S * 4
    n_inputs = max(3, math.ceil(1.5 * L2_BYTES / per_input))
    gen = torch.Generator(device=dev).manual_seed(B * 10000 + S)
    xs = [torch.randn(B, 3, S, S, device=dev, generator=gen) for _ in range(n_inputs)]
    ex = {"focal_length": torch.full((B,), 50.0, device=dev), "aperture": torch.full((B,), 2.8, device=dev),
          "iso": torch.full((B,), 100.0, device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}

    def calls(x):
        for ins in INSTRUCTIONS:
            model.forward_with_guidance(x, ex, ins)

    def sweep(x):
        model.forward_with_guidance_sweep(x, ex, INSTRUCTIONS)

    arms = {"calls": calls, "sweep": sweep}
    i = 0
    for _ in range(warmup):  # first call eager, second capture, then replays: warm every graph of both arms
        for fn in arms.values():
            fn(xs[i % n_inputs])
            i += 1
    torch.cuda.synchronize()
    events = {name: [] for name in arms}
    for step in range(steps):
        order = ("calls", "sweep") if step % 2 == 0 else ("sweep", "calls")
        for name in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            arms[name](xs[i % n_inputs])
            e1.record()
            i += 1
            events[name].append((e0, e1))
    torch.cuda.synchronize()
    ms = {name: [a.elapsed_time(b) for a, b in ev] for name, ev in events.items()}
    res = {"B": B, "S": S, "K": len(INSTRUCTIONS), "rotating_inputs": n_inputs,
           "rotating_input_mb": round(n_inputs * per_input / 2 ** 20, 1)}
    for name, v in ms.items():
        res[f"{name}_ms_median"] = round(statistics.median(v), 4)
        res[f"{name}_ms_min"] = round(min(v), 4)
        res[f"{name}_ms_max"] = round(max(v), 4)
    res["speedup_median"] = round(res["calls_ms_median"] / res["sweep_ms_median"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shapes", default="1x224,32x518", help="comma-separated BxS")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sweep.py measures on a B200: no CUDA device is visible")
    torch.manual_seed(0)
    model = create_model(CFG, {"num_cameras": 71}, device="cuda:0")
    out = {"workload": "instruction sweep (K = 9) vs nine forward_with_guidance calls", **gpu_info(),
           "steps": args.steps, "warmup": args.warmup, "results": []}
    for shape in args.shapes.split(","):
        B, S = (int(v) for v in shape.lower().split("x"))
        out["results"].append(bench(model, B, S, args.steps, args.warmup))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
