"""Ingest of differently sized photographs: today's grouped route against the list route, alternating in one process.

    python tools/bench_ragged_ingest.py [--steps 20] [--warmup 3] [--out profiles/bench_ragged_ingest.json]

Routes, both ending in one guided `forward_with_guidance` at the model resolution S:
  (a) grouped: `model.preprocess` per distinct source size (resize + five torch ops) -> fp32 [B, 3, S, S] -> forward
  (b) list:    the list of uint8 [H_i, W_i, 3] photographs -> forward (one ragged resize, the fused uint8 preprocess)
Workloads: B = 32 at S = 518 with eight source sizes from 640x480 to 4032x3024 (device-resident uint8, as nvJPEG leaves
them; more than the 126 MB of L2), B = 1 with one 4032x3024 photograph at S = 224, and the uniform case, a
[32, 1080, 1920, 3] tensor through `forward`.  Timing: CUDA events around each arm after warm-up of every arm.

The resize passes on their own: a torch.profiler run after the timed section, CUDA kernel time of `resize_h_kernel` and
`resize_v_kernel` at the first workload.  The horizontal pass's rate counts the source bytes it reads plus the
intermediate bytes it writes, over its kernel time, against the 7.7 TB/s of the HGX B200 data sheet.
Writes one JSON file with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cognitive_aim_depth_estimation_b200.model import create_model  # noqa: E402
from tools.bench_sweep import CFG, gpu_info  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
# (H, W) of the eight source sizes of the B = 32 workload, four photographs each
MIXED = [(480, 640), (768, 1024), (1080, 1920), (1200, 1600), (1536, 2048), (2448, 3264), (3000, 4000), (3024, 4032)]


def _exif(B, dev):
    return {"focal_length": torch.full((B,), 50.0, device=dev), "aperture": torch.full((B,), 2.8, device=dev),
            "iso": torch.full((B,), 100.0, device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}


def _groups(sizes, per_size, dev, seed):
    """One [k, H, W, 3] block per size (what ops.jpeg_decode_batch(return_groups=True) leaves) and the list of slices."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    blocks, imgs = [], []
    for i, (h, w) in enumerate(sizes):
        block = torch.randint(0, 256, (per_size, h, w, 3), generator=gen, device=dev, dtype=torch.uint8)
        blocks.append((block, list(range(i * per_size, (i + 1) * per_size))))
        imgs += list(block)
    return blocks, imgs


def _time(arms, steps, warmup):
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    events = {name: [] for name in arms}
    names = list(arms)
    for step in range(steps):
        for name in (names if step % 2 == 0 else names[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            arms[name]()
            e1.record()
            events[name].append((e0, e1))
    torch.cuda.synchronize()
    res = {}
    for name, ev in events.items():
        v = [a.elapsed_time(b) for a, b in ev]
        res[f"{name}_ms_median"] = round(statistics.median(v), 4)
        res[f"{name}_ms_min"] = round(min(v), 4)
        res[f"{name}_ms_max"] = round(max(v), 4)
    return res


def mixed_workload(model, sizes, per_size, S, steps, warmup, seed):
    dev = torch.device("cuda:0")
    blocks, imgs = _groups(sizes, per_size, dev, seed)
    B = len(imgs)
    ex = _exif(B, dev)
    model.input_size = S

    def grouped():
        x = torch.empty(B, 3, S, S, device=dev)
        for block, idx in blocks:
            x[idx] = model.preprocess(block, S)
        model.forward_with_guidance(x, ex, "center")

    def listed():
        model.forward_with_guidance(imgs, ex, "center")

    res = {"B": B, "S": S, "source_sizes_hw": sorted(set(sizes)),
           "source_mb": round(sum(t.numel() for t in imgs) / 2 ** 20, 1),
           **_time({"grouped": grouped, "list": listed}, steps, warmup)}
    res["grouped_over_list_median"] = round(res["grouped_ms_median"] / res["list_ms_median"], 3)
    return res, imgs


def uniform_workload(model, steps, warmup):
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(7)
    x = torch.randint(0, 256, (32, 1080, 1920, 3), generator=gen, device=dev, dtype=torch.uint8)
    ex = _exif(32, dev)
    model.input_size = 518
    res = {"B": 32, "S": 518, "source_hw": [1080, 1920], "source_mb": round(x.numel() / 2 ** 20, 1),
           **_time({"forward": lambda: model.forward(x, ex)}, steps, warmup)}
    return res


def resize_kernels(imgs, S):
    """Kernel time of the two resize passes over `imgs` (torch.profiler, CUDA activity), bytes they move."""
    from torch.profiler import ProfilerActivity, profile

    from cognitive_aim_depth_estimation_b200 import ops
    reps = 10
    ops.resize_u8_list(imgs, S, S)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ops.resize_u8_list(imgs, S, S)
        torch.cuda.synchronize()
    us = {"resize_h_kernel": 0.0, "resize_v_kernel": 0.0}
    for e in prof.key_averages():
        for k in us:
            if k in e.key:
                us[k] += e.device_time_total / reps  # microseconds per call
    src = sum(t.numel() for t in imgs)
    # the horizontal pass writes the source rows the vertical pass reads (all of them when downscaling), S columns each
    inter = sum(t.shape[0] * S * 3 for t in imgs)
    h_s = us["resize_h_kernel"] * 1e-6
    return {"S": S, "resize_h_us": round(us["resize_h_kernel"], 1), "resize_v_us": round(us["resize_v_kernel"], 1),
            "h_bytes_mb": round((src + inter) / 2 ** 20, 1),
            "h_tb_per_s": round((src + inter) / h_s / 1e12, 3) if h_s else None,
            "h_share_of_7p7_tb_per_s": round((src + inter) / h_s / HBM_BYTES_PER_S, 3) if h_s else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_ragged_ingest.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged_ingest.py measures on a B200: no CUDA device is visible")
    torch.manual_seed(0)
    model = create_model(CFG, {"num_cameras": 71}, device="cuda:0")
    out = {"workload": "mixed-size photographs: grouped preprocess -> fp32 -> forward_with_guidance vs list -> "
                       "forward_with_guidance", **gpu_info(), "steps": args.steps, "warmup": args.warmup}
    out["b32_s518_mixed"], imgs = mixed_workload(model, MIXED, 4, 518, args.steps, args.warmup, seed=1)
    out["b1_s224_4032x3024"], _ = mixed_workload(model, [(3024, 4032)], 1, 224, args.steps, args.warmup, seed=2)
    out["uniform_b32_1080x1920_forward"] = uniform_workload(model, args.steps, args.warmup)
    out["resize_passes_b32_s518_mixed"] = resize_kernels(imgs, 518)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f)
        f.write("\n")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
