"""`guide_many` over m scenes against the loop of m `guide` calls it replaces, alternating in one process.

    python tools/bench_guide_many.py [--steps 30] [--warmup 3] [--cases 8x1x224,32x1x224,8x1x518,32x1x518,4x8x518,1x1x518]
                                     [--out profiles/bench_guide_many.json]

A case mxBxS is m scenes of B images at S x S, each encoded once from its own images (what a server holding many users'
photographs keeps); every step answers one instruction per scene.  Both front ends are timed: the Python model
(`guide_many` vs a loop of `guide`) and the handle (`NativeModel.guide_many` vs a loop of `NativeModel.guide`, i.e.
ca_guide_many vs ca_guide).  `draws_ms` times, in the same run, the host draws every arm makes per step: per call
randn(B, 192), randn(B, 768) and a fresh nn.Linear(768, 64), the reference's generator contract.  Timing: the host
clock around the call plus a device synchronise (what the waiting users see) and CUDA events on the calling stream.  The m scenes' tokens (m * B * 4.2 MB at
518^2) are read where the scenes keep them; at m * B = 32, 518^2 that is 135 MB, more than the 126 MB L2.
Writes one JSON object (GPU name and power limit read in the same run) to --out and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cognitive_aim_depth_estimation_b200.model import create_model  # noqa: E402
from cognitive_aim_depth_estimation_b200.native import NativeModel  # noqa: E402
from tools.bench_sweep import CFG, INSTRUCTIONS, gpu_info  # noqa: E402


def _stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}


def bench_case(model, nat, m: int, B: int, S: int, steps: int, warmup: int):
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(m * 1000 + B * 10 + S)
    ex = {"focal_length": torch.full((B,), 50.0, device=dev), "aperture": torch.full((B,), 2.8, device=dev),
          "iso": torch.full((B,), 100.0, device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}
    xs = [torch.randn(B, 3, S, S, device=dev, generator=gen) for _ in range(m)]
    scenes = [model.encode(x, ex) for x in xs]
    nscenes = [nat.encode(x, ex) for x in xs]
    state = {"k": 0}

    def instructions():
        state["k"] += 1
        return [INSTRUCTIONS[(state["k"] + j) % len(INSTRUCTIONS)] for j in range(m)]

    def loop():
        for scene, ins in zip(scenes, instructions()):
            model.guide(scene, ins)

    def native_loop():
        for scene, ins in zip(nscenes, instructions()):
            nat.guide(scene, ins)

    def draws():
        for _ in range(m):
            model._sweep_draws(B, 1)

    arms = {"guide_loop": loop, "guide_many": lambda: model.guide_many(scenes, instructions()),
            "native_guide_loop": native_loop, "native_guide_many": lambda: nat.guide_many(nscenes, instructions()),
            "draws": draws}
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    wall = {n: [] for n in arms}
    devt = {n: [] for n in arms}
    names = list(arms)
    for step in range(steps):
        for name in names[step % len(names):] + names[:step % len(names)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            arms[name]()
            e1.record()
            torch.cuda.synchronize()
            wall[name].append((time.perf_counter() - t0) * 1e3)
            devt[name].append(e0.elapsed_time(e1))
    res = {"m": m, "B": B, "S": S, "rows": m * B}
    for name in arms:
        res[f"{name}_wall_ms"] = _stats(wall[name])
        res[f"{name}_device_ms"] = _stats(devt[name])
    res["speedup_wall_median"] = round(res["guide_loop_wall_ms"]["median"] / res["guide_many_wall_ms"]["median"], 2)
    res["native_speedup_wall_median"] = round(res["native_guide_loop_wall_ms"]["median"] /
                                              res["native_guide_many_wall_ms"]["median"], 2)
    for s in nscenes:
        s.close()
    del scenes
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cases", default="8x1x224,32x1x224,8x1x518,32x1x518,4x8x518,1x1x518", help="comma-separated mxBxS")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_guide_many.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_guide_many.py measures on a B200: no CUDA device is visible")
    torch.manual_seed(0)
    model = create_model(CFG, {"num_cameras": 71}, device="cuda:0")
    nat = NativeModel(model.state_dict(), device="cuda:0")
    out = {"workload": "one instruction for each of m scenes: guide_many vs a loop of guide calls (model.py and handle)",
           **gpu_info(), "steps": args.steps, "warmup": args.warmup, "results": []}
    for case in args.cases.split(","):
        m, B, S = (int(v) for v in case.lower().split("x"))
        with torch.cuda.stream(torch.cuda.Stream()):  # the handle captures its graphs on a non-default stream
            out["results"].append(bench_case(model, nat, m, B, S, args.steps, args.warmup))
    nat.close()
    text = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
