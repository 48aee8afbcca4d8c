"""Benchmark of the Cognitive-Aim guided forward (BASELINE.json metric: images/sec at 518x518, bf16 tensor-core
operands) on N B200s of one node, plus the CPU reference arm.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # candidate (this repo's CUDA path)
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # reference algorithm on the host CPU cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...             # N > 1: one rank per GPU, batch-sharded
    python bench.py ... --dump-outputs DIR                            # + the last timed step's outputs as DIR/*.npy

A step = one `forward_with_guidance` call over one batch of 32 synthetic 518x518 images per GPU
(BASELINE.json configs[1]), cycling through the 9 instructions.  Prints ONE JSON line on rank 0.

Weights and inputs are seeded, so two runs with the same arguments see the same inputs: `--dump-outputs` lets two
builds of the project be compared output for output (rank 0's shard when N > 1).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

S = 518  # overridden by --image-size (parity / sweep configs; the headline is 518)
BATCH_PER_GPU = 32
CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
INSTRUCTIONS = ["center", "left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right"]
# SURVEY.md §8(d): algorithmic FLOPs per image (backbone + focal Q|K projection and one QK^T x3)
ALGO_GFLOP_BY_SIZE = {224: 48.4, 518: 321.5, 1036: 2218.0}
ALGO_GFLOP_BACKBONE = {224: 46.32, 518: 303.15, 1036: 2041.0}  # --workload backbone (BASELINE.json configs[2])
ALGO_GFLOP_PER_IMAGE = 321.5
METRIC = "images/sec at 518x518 bf16"
DUMP_MAX_BYTES = 64 * 10**6  # --dump-outputs: all .npy files together


def dump_outputs(out_dir: str, arrays: dict):
    """Write each tensor as `out_dir/<name>.npy` in float32.  When together they would exceed DUMP_MAX_BYTES, each is
    replaced by the same share of its (flattened) elements, picked by a fixed seed, so runs stay comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_MAX_BYTES - 1024 * len(arrays)  # room for the .npy headers
    for name, a in arrays.items():
        if total > budget:
            keep = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops_sustained", 1393.6), "hbm_gbs": d.get("hbm_gbs", 6539.9),
                "source": "MEASURED_PEAKS.json (sustained bf16 GEMM / copy bandwidth, measured)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback of B200_PROFILING.md (file absent)"}


def _profiled_traffic():
    """DRAM bytes per dense-GEMM launch from the newest committed ncu capture (profiles/*_traffic.json), or None."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    return d.get("dense_gemm_mean_bytes_per_launch"), os.path.basename(files[-1])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def _dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------------
# CPU reference arm / baseline (oracle port of the reference algorithm; the pure-Python reference cannot travel)
# ------------------------------------------------------------------------------------------------------
def cpu_reference(steps: int, warmup: int, images_per_step: int):
    from oracle import cogaim_oracle as orc
    torch.set_num_threads(os.cpu_count() or 1)
    sd = orc.build_state_dict(0)
    x = orc.synthetic_images(images_per_step, S)
    ex = orc.synthetic_exif(images_per_step)
    times = []
    for i in range(warmup + steps):
        torch.manual_seed(11)
        t0 = time.perf_counter()
        out = orc.forward_with_guidance(sd, x, ex, INSTRUCTIONS[i % 9], update_history=False)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": images_per_step * len(times) / total, "ms_per_step": 1e3 * total / len(times),
            "cores": torch.get_num_threads(), "images_per_step": images_per_step,
            "outputs": {"depth": out["depth"], "confidence": out["confidence"], "attention": out["heatmap"]}}


def run_reference(args):
    rank, _, world = _dist_env()
    if rank != 0:
        return
    ips = 2
    r = cpu_reference(args.steps, args.warmup, ips)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["outputs"])
    sample = f"{ips} synthetic 518x518 images per step, oracle port of reference forward_with_guidance, fp32, {r['cores']} threads"
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: full cognitive model, guided forward, 518x518, 9 instructions cycled",
                       "images_per_step": ips},
            "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": sample},
            "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# The other BASELINE.json configurations, measured after the headline region on the same box (N = 1 only)
# ------------------------------------------------------------------------------------------------------
def _timed_region(fn, dev_index: int, target_s: float = 0.8):
    """warm-up (3 calls, the first captures the CUDA graph), then K calls timed with CUDA events on the launching stream,
    K chosen so the region lasts ~target_s (at least two 200 ms clock samples).  -> (ms per call, K, clocks)"""
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn(3)
    e1.record()
    torch.cuda.synchronize()
    k = int(min(80, max(6, target_s * 1e3 / max(e0.elapsed_time(e1), 1e-3) + 1)))
    sampler = ClockSampler(dev_index)
    sampler.start()
    torch.cuda.synchronize()
    e0.record()
    for i in range(k):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k, k, sampler.stop()


def other_configs(model, dev, local_rank: int, ex_fn, img_fn):
    """configs[2] (backbone only), configs[3]'s per-GPU shape (64 images), configs[4] (1036 x 1036), the un-guided
    `forward`, and the demo-shaped uint8 flow end to end — each its own timed region with its own clock record.
    Inputs are device-resident (three rotating batches, larger than L2 together with the activations) except for the
    uint8 flow, which is timed on the wall clock with the H2D / D2H copies inside."""
    out = {}

    def entry(name, workload, B, S_, ms, k, clocks, gflop_per_image=None, **extra):
        d = {"workload": workload, "batch_per_gpu": B, "image_size": S_, "ms_per_step": ms, "steps": k,
             "value": B / (ms / 1e3), "unit": "images/s", "clocks": clocks}
        if gflop_per_image:
            d["whole_step_tflops"] = gflop_per_image * d["value"] / 1e3
        d.update(extra)
        out[name] = d

    # configs[2]: backbone only, 518 x 518, 32 images
    B, S_ = 32, 518
    imgs = [img_fn(B, S_, 100 + i).to(dev) for i in range(3)]
    ms, k, ck = _timed_region(lambda i: model.backbone_tokens(imgs[i % 3]), local_rank)
    entry("configs[2] backbone only", "Dinov2Model last_hidden_state (eval_configs/baseline_dinov2_config.yaml)", B, S_, ms,
          k, ck, ALGO_GFLOP_BACKBONE[518])
    # un-guided forward (src/model.py:1064), same inputs
    ex = {kk: v.to(dev) for kk, v in ex_fn(B, 300).items()}
    ms, k, ck = _timed_region(lambda i: model(imgs[i % 3], ex, return_attention=True), local_rank)
    entry("un-guided forward", "CognitiveAimModel.forward(images, exif, return_attention=True)", B, S_, ms, k, ck)
    # demo-shaped flow end to end: pinned uint8 HWC on the host -> H2D (25.8 MB / step) -> fused normalise + patchify ->
    # guided forward -> depth / confidence / heat-map back to pinned host memory; wall clock
    g = torch.Generator().manual_seed(1235)
    host_u8 = [torch.randint(0, 256, (B, S_, S_, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(3)]
    stage = [torch.empty(B, S_, S_, 3, dtype=torch.uint8, device=dev) for _ in range(2)]
    outs = [torch.empty(B, 1).pin_memory(), torch.empty(B, 1).pin_memory(), torch.empty(B, (S_ // 14) ** 2).pin_memory()]
    copy_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def u8_loop(n):
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        with torch.cuda.stream(copy_stream):
            stage[0].copy_(host_u8[0], non_blocking=True)
            ready[0].record()
        for i in range(n):
            cur = i % 2
            torch.cuda.current_stream().wait_event(ready[cur])
            if i + 1 < n:
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(done[1 - cur])
                    stage[1 - cur].copy_(host_u8[(i + 1) % 3], non_blocking=True)
                    ready[1 - cur].record()
            torch.manual_seed(11)
            res = model.forward_with_guidance(stage[cur], ex, INSTRUCTIONS[i % 9], return_attention=True)
            done[cur].record()
            d2h_stream.wait_event(done[cur])
            with torch.cuda.stream(d2h_stream):
                for dst, src in zip(outs, res):
                    dst.copy_(src, non_blocking=True)
                    src.record_stream(d2h_stream)
        torch.cuda.synchronize()

    u8_loop(4)
    sampler = ClockSampler(local_rank)
    sampler.start()
    n = 40
    t0 = time.perf_counter()
    u8_loop(n)
    wall = time.perf_counter() - t0
    entry("uint8 end to end", "pinned uint8 [B,518,518,3] on the host -> H2D -> normalise+patchify -> guided forward -> "
          "outputs D2H (demo.py:312-346 flow), wall clock", B, S_, wall / n * 1e3, n, sampler.stop(),
          h2d_bytes_per_step=B * S_ * S_ * 3 + 64 * 768 * 4 + 64 * 4, d2h_bytes_per_step=B * (2 + (S_ // 14) ** 2) * 4)
    del imgs, host_u8, stage
    # configs[3]'s per-GPU shape: 64 images per call
    B = 64
    imgs = [img_fn(B, S_, 200 + i).to(dev) for i in range(3)]
    ex = {kk: v.to(dev) for kk, v in ex_fn(B, 301).items()}

    def guided(i):
        torch.manual_seed(11)
        return model.forward_with_guidance(imgs[i % 3], ex, INSTRUCTIONS[i % 9], return_attention=True)

    ms, k, ck = _timed_region(guided, local_rank)
    entry("configs[3] per-GPU shape", "full cognitive model + EXIF, guided forward, 64 images per call", B, S_, ms, k, ck,
          ALGO_GFLOP_BY_SIZE[518])
    # the same shape through the handle-level C-ABI (one native call per forward: csrc/launcher.cu), and the single-image
    # latency of configs[0]'s shape through both front ends
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    nat = NativeModel({k: v.detach() for k, v in model.state_dict().items()}, device=dev)
    side = torch.cuda.Stream(device=dev)

    def native_guided(i):
        with torch.cuda.stream(side):
            torch.manual_seed(11)
            return nat.forward_with_guidance(imgs[i % 3], ex, INSTRUCTIONS[i % 9])

    def on_side(fn):
        def run(i):
            with torch.cuda.stream(side):
                return fn(i)
        return run

    def timed_on_side(fn):
        side.wait_stream(torch.cuda.current_stream())
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k = 20
        sampler = ClockSampler(local_rank)
        sampler.start()
        with torch.cuda.stream(side):
            e0.record()
        for i in range(k):
            fn(i)
        with torch.cuda.stream(side):
            e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k, k, sampler.stop()

    ms, k, ck = timed_on_side(native_guided)
    entry("handle-level C-ABI, 64 images", "ca_forward_guided (one native call per forward), same inputs", B, S_, ms, k, ck,
          ALGO_GFLOP_BY_SIZE[518], gpu_launches_per_call=nat.launch_count())
    one = imgs[0][:1].contiguous()
    ex1 = {kk: v[:1].contiguous() for kk, v in ex.items()}

    def py_one(i):
        torch.manual_seed(11)
        return model.forward_with_guidance(one, ex1, INSTRUCTIONS[i % 9], return_attention=True)

    def nat_one(i):
        with torch.cuda.stream(side):
            torch.manual_seed(11)
            return nat.forward_with_guidance(one, ex1, INSTRUCTIONS[i % 9])

    for name, fn in (("single image, Python front end", py_one), ("single image, handle-level C-ABI", nat_one)):
        side.wait_stream(torch.cuda.current_stream())
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(200):
            fn(i)
        torch.cuda.synchronize()
        entry(name, "configs[0] shape: one 518 x 518 image per call, wall clock per call (device-bound: ~110 dependent "
              "launches of 5-20 us each in one CUDA graph)", 1, S_, (time.perf_counter() - t0) / 200 * 1e3, 200, None)
    nat.close()
    del imgs
    # configs[4]: 1036 x 1036 (4x tokens), 8 images per call
    B, S_ = 8, 1036
    imgs = [img_fn(B, S_, 400 + i).to(dev) for i in range(3)]
    ex = {kk: v.to(dev) for kk, v in ex_fn(B, 302).items()}
    ms, k, ck = _timed_region(guided, local_rank)
    entry("configs[4] 1036x1036", "full cognitive model, guided forward, 5477 tokens per image", B, S_, ms, k, ck,
          ALGO_GFLOP_BY_SIZE[1036])
    return out


# ------------------------------------------------------------------------------------------------------
# Candidate arm
# ------------------------------------------------------------------------------------------------------
def run_candidate(args):
    from cognitive_aim_depth_estimation_b200 import ops
    from cognitive_aim_depth_estimation_b200.model import create_model
    from oracle import cogaim_oracle as orc  # weights / synthetic inputs + cpu_baseline leg only

    rank, local_rank, world = _dist_env()
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # rank 0 must print exactly ONE line on stdout: NCCL writes its version banner to the C stdout when the first
        # communicator is created (NCCL_DEBUG=VERSION/WARN on these boxes), so fd 1 points at /dev/null until then
        sys.stdout.flush()
        saved_fd, null_fd = os.dup(1), os.open(os.devnull, os.O_WRONLY)
        os.dup2(null_fd, 1)
        try:
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
            os.close(null_fd)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch
    torch.manual_seed(0)  # the reference's random init (create_model replays its construction order: init.py)
    model = create_model(CFG, {"num_cameras": 71}, device=dev)
    # default API path: input validation stays ON (the camera_idx range check runs inside the heads kernel, no sync)
    # three distinct resident input batches (3 x 103 MB fp32) rotate so no step re-reads an L2-resident input;
    # per-step activations (~1 GB) exceed the 126 MB L2 on their own
    n_sets = 3
    host = [orc.synthetic_images(B, S, seed=1234 + 17 * rank + i).pin_memory() for i in range(n_sets)]
    dev_imgs = [h.to(dev) for h in host]
    ex = {k: v.to(dev) for k, v in orc.synthetic_exif(B, seed=1236 + rank).items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    backbone_only = args.workload == "backbone"

    def step(i, imgs):
        if backbone_only:
            # BASELINE.json configs[2] (eval_configs/baseline_dinov2_config.yaml): the reference has no functional
            # backbone-only depth path (SURVEY.md §0 quirk 5), so this is `Dinov2Model(images).last_hidden_state`;
            # the per-image result handed back is the CLS row
            cls = model.backbone_tokens(imgs)[:, 0]
            return cls, cls[:, :1], cls[:, :1]
        torch.manual_seed(11)
        return model.forward_with_guidance(imgs, ex, INSTRUCTIONS[i % 9], return_attention=True)

    # ---- device-resident throughput (`value`): the forward as a user gets it (CUDA-graph replay of the launch sequence) ----
    for i in range(args.warmup):
        step(i, dev_imgs[i % n_sets])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.trace_start(with_events=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        out = step(i, dev_imgs[i % n_sets])
    e1.record()
    barrier()
    launches, _ = ops.trace_stop()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        # written before the next pass: the backbone's CLS rows are a view of a workspace that it overwrites
        names = ("cls_tokens",) if backbone_only else ("depth", "confidence", "attention")
        dump_outputs(args.dump_outputs, dict(zip(names, out)))

    # ---- per-kernel device times: a second pass of the same K steps, launched eagerly with a CUDA-event pair around
    # every launch on the launching stream (graph replay hides individual launches from events) ----
    ops.trace_start(with_events=True)
    barrier()
    for i in range(args.steps):
        step(i, dev_imgs[i % n_sets])
    barrier()
    _, events = ops.trace_stop()
    per_kernel = {}
    ms_events = 0.0
    for name, work, a, b in events:
        t, w, n = per_kernel.get(name, (0.0, 0.0, 0))
        dt = a.elapsed_time(b)
        ms_events += dt
        per_kernel[name] = (t + dt, w + work, n + 1)

    # ---- end to end through the public API with HOST buffers (pinned fp32 images in, outputs back to host) ----
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty_like(dev_imgs[0]) for _ in range(2)]
    out_host = [torch.empty(B, 768 if backbone_only else 1).pin_memory(), torch.empty(B, 1).pin_memory(),
                torch.empty(B, 1 if backbone_only else (S // 14) ** 2).pin_memory()]

    def e2e_loop(n):
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        with torch.cuda.stream(copy_stream):
            stage[0].copy_(host[0], non_blocking=True)
            ready[0].record()
        for i in range(n):
            cur = i % 2
            torch.cuda.current_stream().wait_event(ready[cur])
            if i + 1 < n:  # prefetch the next batch while this one computes
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(done[1 - cur])
                    stage[1 - cur].copy_(host[(i + 1) % n_sets], non_blocking=True)
                    ready[1 - cur].record()
            d, c, h = step(i, stage[cur])
            done[cur].record()
            # results go home on their own stream: three small D2H copies on the compute stream would hold back the
            # next step's first kernels for the copy engine's latency each
            d2h_stream.wait_event(done[cur])
            with torch.cuda.stream(d2h_stream):
                for dst, src in zip(out_host, (d, c, h)):
                    dst.copy_(src, non_blocking=True)
                    src.record_stream(d2h_stream)
        torch.cuda.synchronize()

    e2e_loop(max(2, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0

    if world > 1:
        t = torch.tensor([ms, e2e_s * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = t[0].item(), t[1].item() / 1e3
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = _peaks()
    imgs = B * world * args.steps
    value = imgs / (ms / 1e3)
    g_t, g_w, g_n = per_kernel.get("gemm", (0.0, 0.0, 1))
    a_t, a_w, a_n = per_kernel.get("attention", (0.0, 0.0, 1))
    gemm_tflops = g_w / (g_t * 1e-3) / 1e12 if g_t else 0.0
    attn_tflops = a_w / (a_t * 1e-3) / 1e12 if a_t else 0.0
    breakdown = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[2] / args.steps,
                     "share": v[0] / ms_events} for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1][0])}
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": (f"configs[2]: baseline_dinov2 backbone only (DINOv2 ViT-B/14 last_hidden_state), {S}x{S}, "
                                f"batch {B}/GPU, random-init weights (seed 0)") if backbone_only else
                               (f"configs[1]: experiment_B full cognitive model, guided forward, {S}x{S}, "
                                f"batch {B}/GPU, 9 instructions cycled, random-init weights (seed 0)"),
                   "batch_per_gpu": B, "global_batch": B * world, "image_size": S, "parallelism": f"batch-shard x{world}",
                   "l2": f"{n_sets} rotating resident input batches (3 x {B * 3 * S * S * 4 / 1e6:.0f} MB) + ~1 GB of "
                         "activations per step: working set > 126 MB L2"},
        "e2e": {"value": B * world * args.steps / e2e_s, "unit": "images/s",
                "h2d_bytes_per_step": B * 3 * S * S * 4 + (0 if backbone_only else 64 * 768 * 4 + 64 * 4),
                "d2h_bytes_per_step": B * (770 if backbone_only else 2 + (S // 14) ** 2) * 4,
                "note": "pinned fp32 host images -> H2D on a copy stream (double-buffered) -> %s D2H, wall clock incl. all "
                        "copies" % ("backbone_tokens -> CLS rows" if backbone_only else
                                    "forward_with_guidance -> depth/conf/heatmap")},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": gemm_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / peaks["bf16_tflops"], "traffic": _profiled_traffic()[0],
                     "traffic_note": "mean DRAM read+write bytes per dense-GEMM launch, ncu capture %s (the captured "
                                     "launches cover the QKV / proj / fc1 / fc2 shapes)" % _profiled_traffic()[1],
                     "kernel": "gemm_tcgen05_kernel (all dense epilogues)", "launches_per_step": g_n / args.steps,
                     "peak_source": peaks["source"],
                     "algorithmic_flops_per_launch_avg": g_w / max(g_n, 1)},
        "roofline_attention": {"bound": "tensor", "achieved": attn_tflops, "peak": peaks["bf16_tflops"],
                               "unit": "TFLOP/s", "frac": attn_tflops / peaks["bf16_tflops"]},
        "whole_step_tflops": ALGO_GFLOP_PER_IMAGE * value / 1e3,
        "whole_step_frac_of_peak": ALGO_GFLOP_PER_IMAGE * value / 1e3 / peaks["bf16_tflops"],
        "kernel_breakdown": breakdown,
        "kernel_breakdown_note": "second pass of the same steps launched eagerly with per-launch CUDA events; `value` is "
                                 "the CUDA-graph replay of the same launch sequence (use_cuda_graphs=%s)" % model.use_cuda_graphs,
    }
    if world == 1 and not args.no_other_configs and not backbone_only and B == BATCH_PER_GPU and S == 518:
        del dev_imgs, stage
        torch.cuda.empty_cache()
        line["other_configs"] = other_configs(model, dev, local_rank, lambda b, seed: orc.synthetic_exif(b, seed=seed),
                                              lambda b, s_, seed: orc.synthetic_images(b, s_, seed=seed))
    if world == 1 and not args.no_cpu_baseline and not backbone_only:
        r = cpu_reference(steps=3, warmup=1, images_per_step=2)
        line["cpu_baseline"] = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                                "sample": "3 timed + 1 warm-up guided forwards of 2 synthetic 518x518 images (oracle "
                                          "port of the reference forward, fp32, all host threads)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=18)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="candidate", choices=["candidate", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the extra timed regions (configs[2..4], un-guided forward, uint8 end to end) after the headline")
    ap.add_argument("--image-size", type=int, default=518, choices=sorted(ALGO_GFLOP_BY_SIZE),
                    help="sweep configs of BASELINE.json (224 / 1036); the headline metric is quoted at 518")
    ap.add_argument("--workload", default="guided", choices=["guided", "backbone"],
                    help="guided = configs[1] (default, the headline); backbone = configs[2] (DINOv2 tokens only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    global S, ALGO_GFLOP_PER_IMAGE, METRIC
    S = args.image_size
    ALGO_GFLOP_PER_IMAGE = (ALGO_GFLOP_BACKBONE if args.workload == "backbone" else ALGO_GFLOP_BY_SIZE)[S]
    METRIC = f"images/sec at {S}x{S} bf16"
    args.warmup = max(args.warmup, 3) if args.impl == "candidate" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the candidate arm has no CPU fallback (use --impl reference)")
        run_candidate(args)


if __name__ == "__main__":
    main()
