"""Scenes against the calls they replace, alternating in one process: `encode`, one `guide` call on an encoded scene,
one `forward_with_guidance` call, and the fused tail kernel (`ops.guide_tail`) against the guided_softmax ->
weighted_pool -> heads chain on the same scene.

    python tools/bench_scene.py [--steps 50] [--warmup 5] [--shapes 1x224,1x518,32x518] [--out profiles/bench_scene.json]

Timing:
  * encode / guide / forward_with_guidance: CUDA events on the calling stream around each call (device time from the
    call's first enqueued work to its last), and the host clock around the call plus a device synchronise (what an
    interactive caller waits).  encode and forward_with_guidance rotate through images larger in total than the 126 MB
    L2; guide runs on one scene, as an interactive front end does with the photograph on screen.
  * tail vs chain: each captured into a CUDA graph of 20 back-to-back repetitions (the guide call replays its tail from
    a graph too) and timed with events around a replay, alternating; per-repetition time is reported.
Writes one JSON object (GPU name and power limit read in the same run) to --out and prints it.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cognitive_aim_depth_estimation_b200 import ops  # noqa: E402
from cognitive_aim_depth_estimation_b200.model import _POOL_SPLITS, create_model  # noqa: E402
from tools.bench_sweep import CFG, INSTRUCTIONS, L2_BYTES, gpu_info  # noqa: E402

TAIL_REPS = 20


def _stats(v, scale=1.0):
    return {"median": round(statistics.median(v) * scale, 4), "min": round(min(v) * scale, 4),
            "max": round(max(v) * scale, 4)}


def bench_calls(model, B: int, S: int, steps: int, warmup: int):
    dev = torch.device("cuda:0")
    per_input = B * 3 * S * S * 4
    n_inputs = max(3, math.ceil(1.5 * L2_BYTES / per_input))
    gen = torch.Generator(device=dev).manual_seed(B * 10000 + S)
    xs = [torch.randn(B, 3, S, S, device=dev, generator=gen) for _ in range(n_inputs)]
    ex = {"focal_length": torch.full((B,), 50.0, device=dev), "aperture": torch.full((B,), 2.8, device=dev),
          "iso": torch.full((B,), 100.0, device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}
    scene = model.encode(xs[0], ex)
    state = {"i": 0, "k": 0}

    def nxt():
        state["i"] += 1
        return xs[state["i"] % n_inputs]

    def ins():
        state["k"] += 1
        return INSTRUCTIONS[state["k"] % len(INSTRUCTIONS)]

    arms = {"encode": lambda: model.encode(nxt(), ex),
            "guide": lambda: model.guide(scene, ins()),
            "forward_with_guidance": lambda: model.forward_with_guidance(nxt(), ex, ins())}
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    dev_ms = {n: [] for n in arms}
    wall_ms = {n: [] for n in arms}
    names = list(arms)
    for step in range(steps):
        for name in names[step % 3:] + names[:step % 3]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            arms[name]()
            e1.record()
            torch.cuda.synchronize()
            wall_ms[name].append((time.perf_counter() - t0) * 1e3)
            dev_ms[name].append(e0.elapsed_time(e1))
    res = {"B": B, "S": S, "rotating_inputs": n_inputs, "rotating_input_mb": round(n_inputs * per_input / 2 ** 20, 1)}
    for name in arms:
        res[f"{name}_device_ms"] = _stats(dev_ms[name])
        res[f"{name}_wall_ms"] = _stats(wall_ms[name])
    res["guide_speedup_device_median"] = round(res["forward_with_guidance_device_ms"]["median"] /
                                               res["guide_device_ms"]["median"], 2)
    res["guide_speedup_wall_median"] = round(res["forward_with_guidance_wall_ms"]["median"] /
                                             res["guide_wall_ms"]["median"], 2)
    res.update(bench_tail(model, scene, steps, warmup))
    return res


def bench_tail(model, scene, steps: int, warmup: int):
    """The fused tail against the three-kernel chain on the scene's tokens and base attention."""
    B, S = scene.B, scene.S
    g = S // 14
    N, T, D = g * g, g * g + 1, 768
    pk = model._pack()
    dev = scene.device
    mask = model._mask("top-left", g).expand(B, N).contiguous()
    proj = torch.nn.Linear(D, 64)
    tmp_w, tmp_b = proj.weight.detach().to(dev).contiguous(), proj.bias.detach().to(dev).contiguous()
    fault = model._fault_word().data_ptr()
    bufs = [{"heat": torch.empty(B, N, device=dev), "arg": torch.empty(B, device=dev, dtype=torch.int32),
             "pool": torch.empty(B, _POOL_SPLITS, D, device=dev), "depth": torch.empty(B, device=dev),
             "conf": torch.empty(B, device=dev)} for _ in range(2)]
    ticket = torch.zeros(B, device=dev, dtype=torch.int32)
    heads_kw = dict(exif=scene.exif, camera_idx=scene.camera_idx, num_cameras=model.cfg.num_cameras, fault_ptr=fault)

    def chain(b=bufs[0]):
        ops.guided_softmax(scene.base, mask, b["heat"], b["arg"], B, N)
        ops.weighted_pool(scene.tokens, T * D, 1, b["heat"], None, b["pool"], B, N, D, _POOL_SPLITS)
        ops.heads(pk["heads"], tokens=scene.tokens, tokens_per_img=T, depth=b["depth"], conf=b["conf"], B=B,
                  pool_partial=b["pool"], pool_splits=_POOL_SPLITS, tmp_w=tmp_w, tmp_b=tmp_b, **heads_kw)

    def tail(b=bufs[1]):
        ops.guide_tail(pk["heads"], base=scene.base, mask=mask, heat=b["heat"], argmax=b["arg"], ticket=ticket,
                       tokens=scene.tokens, depth=b["depth"], conf=b["conf"], B=B, N=N, pool_partial=b["pool"],
                       tmp_w=tmp_w, tmp_b=tmp_b, **heads_kw)

    graphs = {}
    for name, fn in (("chain", chain), ("tail", tail)):
        fn()  # eager first: one-time library set-up is not capturable
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(TAIL_REPS):
                fn()
        graphs[name] = gr
    torch.cuda.synchronize()
    same = all(torch.equal(bufs[0][k], bufs[1][k]) for k in ("heat", "arg", "depth", "conf"))
    for _ in range(warmup):
        for gr in graphs.values():
            gr.replay()
    torch.cuda.synchronize()
    us = {n: [] for n in graphs}
    for step in range(steps):
        for name in (("chain", "tail") if step % 2 == 0 else ("tail", "chain")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs[name].replay()
            e1.record()
            us[name].append((e0, e1))
    torch.cuda.synchronize()
    out = {"tail_outputs_equal_chain": same}
    for name, ev in us.items():
        out[f"{name}_us_per_call"] = _stats([a.elapsed_time(b) for a, b in ev], 1e3 / TAIL_REPS)
    out["tail_speedup_median"] = round(out["chain_us_per_call"]["median"] / out["tail_us_per_call"]["median"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shapes", default="1x224,1x518,32x518", help="comma-separated BxS")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_scene.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene.py measures on a B200: no CUDA device is visible")
    torch.manual_seed(0)
    model = create_model(CFG, {"num_cameras": 71}, device="cuda:0")
    out = {"workload": "encode once + guide per instruction vs forward_with_guidance; fused tail vs three-kernel chain",
           **gpu_info(), "steps": args.steps, "warmup": args.warmup, "tail_graph_reps": TAIL_REPS, "results": []}
    for shape in args.shapes.split(","):
        B, S = (int(v) for v in shape.lower().split("x"))
        out["results"].append(bench_calls(model, B, S, args.steps, args.warmup))
    text = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
