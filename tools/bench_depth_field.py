"""Depth fields against the guide calls they replace, on one encoded scene per shape.

    python tools/bench_depth_field.py [--steps 30] [--warmup 5] [--out profiles/bench_depth_field.json]

  * B = 1 at 224^2 and 518^2: `depth_field` against `guide` looped over every cell with that cell's focus mask (one
    full loop, host clock around it plus a device synchronise), and the largest |field - guide| over all cells (each
    guide call from the field's seed and ring state).
  * B = 32 at 518^2 and B = 8 at 1036^2: `depth_field` against a timed sample of guide calls, scaled per call to the N
    calls of a full loop (an estimate, labelled as such).
  * token_project alone (CUDA events over back-to-back launches), with its bytes and FLOP from shapes: the tokens read
    once, P written once, 2 * B * N * 768 * 64 FLOP.
  * per-kernel device time of a depth_field call with torch.profiler, in a separate pass after the timed ones.
`depth_field` is timed with CUDA events around the call (graph replay after its second call) and with the host clock
plus a synchronise.  Writes one JSON object (GPU name and power limit read in the same run) to --out and prints it.
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

from cognitive_aim_depth_estimation_b200 import ops, tables  # noqa: E402
from cognitive_aim_depth_estimation_b200.model import create_model  # noqa: E402
from tools.bench_sweep import CFG, gpu_info  # noqa: E402

GUIDE_SAMPLE = 64  # guide calls timed for the shapes where a full loop over the cells takes minutes


def _stats(v, scale=1.0):
    return {"median": round(statistics.median(v) * scale, 4), "min": round(min(v) * scale, 4),
            "max": round(max(v) * scale, 4)}


def _exif(B, dev):
    return {"focal_length": torch.full((B,), 50.0, device=dev), "aperture": torch.full((B,), 2.8, device=dev),
            "iso": torch.full((B,), 100.0, device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}


def _ring(m):
    cm = m.curiosity_module
    return cm.exploration_history.clone(), cm.history_pointer.clone()


def _set_ring(m, ring):
    m.curiosity_module.exploration_history.copy_(ring[0])
    m.curiosity_module.history_pointer.copy_(ring[1])


def _time_field(model, scene, steps, warmup):
    ev, host = [], []
    for i in range(warmup + steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        model.depth_field(scene)
        e1.record()
        torch.cuda.synchronize()
        if i >= warmup:
            host.append(time.perf_counter() - t0)
            ev.append(e0.elapsed_time(e1))
    return {"field_event_ms": _stats(ev), "field_host_ms": _stats(host, 1e3)}


def _time_projection(model, scene, reps=50):
    B, g = scene.B, scene.S // 14
    N, T = g * g, g * g + 1
    P = torch.empty(B, N, 64, device=scene.tokens.device)
    w = torch.randn(64, 768, device=scene.tokens.device)
    ops.token_project(scene.tokens, T * 768, 1, w, P, B, N)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.token_project(scene.tokens, T * 768, 1, w, P, B, N)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = B * N * 768 * 4 + B * N * 64 * 4 + 64 * 768 * 4
    flop = 2 * B * N * 768 * 64
    return {"token_project_us": round(us, 3), "token_project_bytes": nbytes, "token_project_flop": flop,
            "token_project_gb_per_s": round(nbytes / us / 1e3, 1), "token_project_tflop_per_s": round(flop / us / 1e6, 2),
            "token_project_note": "back-to-back launches on one scene: the tokens of B <= 32 at 518^2 (135 MB) are "
                                  "partly L2-resident between repetitions"}


def bench_shape(model, B, S, steps, warmup, full_loop):
    dev = torch.device("cuda:0")
    g = S // 14
    N = g * g
    x = torch.randn(B, 3, S, S, device=dev, generator=torch.Generator(device=dev).manual_seed(B * 10000 + S))
    scene = model.encode(x, _exif(B, dev))
    ring = _ring(model)
    out = {"B": B, "S": S, "grid": g, "cells": N}
    out.update(_time_field(model, scene, steps, warmup))
    out.update(_time_projection(model, scene))
    _set_ring(model, ring)
    torch.manual_seed(5)
    fd, fc = (t.flatten(1) for t in model.depth_field(scene))
    cells = list(range(N)) if full_loop else torch.randperm(N, generator=torch.Generator().manual_seed(S))[:GUIDE_SAMPLE].tolist()
    masks = [tables.focus_mask(c // g, c % g, g).to(dev) for c in cells]
    for m in masks[:3]:  # warm the guide path (eager, capture, replay)
        model.guide(scene, m)
    dmax = cmax = 0.0
    per_call = []
    torch.cuda.synchronize()
    t_loop = time.perf_counter()
    for c, m in zip(cells, masks):
        _set_ring(model, ring)
        torch.manual_seed(5)
        t0 = time.perf_counter()
        d, cf = model.guide(scene, m)
        torch.cuda.synchronize()
        per_call.append(time.perf_counter() - t0)
        dmax = max(dmax, (d[:, 0] - fd[:, c]).abs().max().item())
        cmax = max(cmax, (cf[:, 0] - fc[:, c]).abs().max().item())
    loop_s = time.perf_counter() - t_loop
    out["max_abs_delta"] = {"depth": dmax, "confidence": cmax, "cells_compared": len(cells)}
    field_ms = out["field_host_ms"]["median"]
    if full_loop:
        out["guide_loop_all_cells_ms"] = round(loop_s * 1e3, 2)
        out["speedup_vs_guide_loop"] = round(loop_s * 1e3 / field_ms, 1)
    else:
        est = statistics.median(per_call) * N * 1e3
        out["guide_call_host_ms"] = _stats(per_call, 1e3)
        out["guide_loop_all_cells_ms_estimated"] = round(est, 1)
        out["speedup_vs_guide_loop_estimated"] = round(est / field_ms, 1)
    out["token_traffic_bytes"] = {"depth_field": B * N * 768 * 4, "guide_loop": N * B * N * 768 * 4}
    return out, scene


def profile_kernels(model, scene, reps=10):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        model.depth_field(scene)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            model.depth_field(scene)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            name = e.key
            for short in ("token_project", "field_const", "depth_field_cells", "curiosity", "fetch_pinned"):
                if short in name:
                    name = short
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            per[name] = round(per.get(name, 0.0) + t / reps, 3)
    return {"B": scene.B, "S": scene.S, "us_per_call_by_kernel": per}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_depth_field.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_depth_field.py measures on a B200: no CUDA device is visible")
    torch.manual_seed(0)
    model = create_model(CFG, {"num_cameras": 71}, device="cuda:0")
    out = {"workload": "depth_field (guided depth with the focus on every grid cell) vs guide looped over the cells",
           **gpu_info(), "steps": args.steps, "warmup": args.warmup, "results": [], "profile": []}
    scenes = []
    for B, S, full in ((1, 224, True), (1, 518, True), (32, 518, False), (8, 1036, False)):
        res, scene = bench_shape(model, B, S, args.steps, args.warmup, full)
        out["results"].append(res)
        scenes.append(scene)
        print(json.dumps(res), flush=True)
    for scene in scenes:  # profiler pass after every timed pass
        out["profile"].append(profile_kernels(model, scene))
    text = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
