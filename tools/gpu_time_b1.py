"""Device time of ONE graph replay of the guided forward at B = 1 (is config[0] latency host-bound or node-bound?)"""
import sys, time
import torch
sys.path.insert(0, '/root/repo')
from cognitive_aim_depth_estimation_b200.model import create_model
dev = torch.device('cuda:0')
CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
torch.manual_seed(0)
model = create_model(CFG, {"num_cameras": 71}, device=dev)
for B, S in ((1, 518), (1, 224), (8, 518)):
    x = torch.randn(B, 3, S, S, device=dev)
    ex = {"focal_length": torch.full((B,), 50., device=dev), "aperture": torch.full((B,), 2.8, device=dev),
          "iso": torch.full((B,), 100., device=dev), "camera_idx": torch.zeros(B, dtype=torch.long, device=dev)}
    for _ in range(5):
        model.forward_with_guidance(x, ex, "center", return_attention=True)
    torch.cuda.synchronize()
    ws = model._workspace(B, S)
    (graph, n), = [v for k, v in ws["graphs"].items() if k[:2] == ("sweep", 1)]  # a guided call is a sweep of one
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        graph.replay()
    e1.record(); torch.cuda.synchronize()
    n_it = 300
    t0 = time.perf_counter()
    for _ in range(n_it):
        model.forward_with_guidance(x, ex, "center", return_attention=True)
    t_host = (time.perf_counter() - t0) / n_it
    torch.cuda.synchronize()
    t_all = (time.perf_counter() - t0) / n_it
    print(f"B={B} S={S}: graph of {n} launches: {e0.elapsed_time(e1) / 50:.3f} ms device time per replay; "
          f"host enqueue {t_host * 1e3:.3f} ms, wall {t_all * 1e3:.3f} ms per call")
