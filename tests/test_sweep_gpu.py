"""Instruction sweeps (`forward_with_guidance_sweep`, `ca_forward_guided_sweep`): K guided calls over one batch in one
pass must equal K successive `forward_with_guidance` calls bit for bit — outputs, global generator state, the
CuriosityModule ring buffer and the `_last_*` state — and match the CPU oracle at the usual tolerances."""
import importlib.util
import io
import os

import pytest
import torch

from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
CFG_GUIDED = dict(CFG, curiosity_guided_attention={"enabled": True})
SWEEP_MAX_K = 16


@pytest.fixture(scope="module")
def sd():
    return orc.build_state_dict(0)


def _model(cuda_device, cfg, sd):
    from cognitive_aim_depth_estimation_b200.model import create_model
    m = create_model(cfg, {"num_cameras": 71}, device=cuda_device)
    m.load_state_dict(sd)
    return m


@pytest.fixture(scope="module")
def model(cuda_device, sd):
    return _model(cuda_device, CFG, sd)


def _exif(ex):
    return {k: v.cuda() for k, v in ex.items()}


def _ring(m):
    cm = m.curiosity_module
    return cm.exploration_history.clone(), cm.history_pointer.clone()


def _set_ring(m, ring):
    m.curiosity_module.exploration_history.copy_(ring[0])
    m.curiosity_module.history_pointer.copy_(ring[1])


def _sweep_argmax(m, B, S, K):
    return m._ws[(B, S)]["sweeps"][K]["argmax"]


def _assert_sweep_equals_calls(m, x, ex, guidances, seed=11):
    """K forward_with_guidance calls, then the sweep from the same generator and ring-buffer state: every observable
    result and side effect must be identical."""
    K, B, S = len(guidances), x.shape[0], x.shape[-1]
    ring0 = _ring(m)
    torch.manual_seed(seed)
    outs, argmax = [], []
    for gd in guidances:
        outs.append([t.clone() for t in m.forward_with_guidance(x, ex, gd, return_attention=True)])
        argmax.append(m._last_argmax.clone())
    want = [torch.stack([o[i] for o in outs]) for i in range(3)] + [torch.stack(argmax)]
    want_last = (m._last_attention_weights.clone(), m._last_argmax.clone(), m._last_curiosity.clone())
    want_rng, want_ring = torch.get_rng_state(), _ring(m)

    _set_ring(m, ring0)
    torch.manual_seed(seed)
    depth, conf, heat = m.forward_with_guidance_sweep(x, ex, guidances, return_attention=True)
    torch.cuda.synchronize()
    assert depth.shape == (K, B, 1) and conf.shape == (K, B, 1) and heat.shape == want[2].shape
    for name, a, b in (("depth", depth, want[0]), ("conf", conf, want[1]), ("heat", heat, want[2]),
                       ("argmax", _sweep_argmax(m, B, S, K), want[3])):
        assert torch.equal(a, b), name
    assert torch.equal(m._last_attention_weights, want_last[0])
    assert torch.equal(m._last_argmax, want_last[1])
    assert torch.equal(m._last_curiosity, want_last[2])
    assert torch.equal(torch.get_rng_state(), want_rng)
    ring = _ring(m)
    assert torch.equal(ring[1], want_ring[1]) and torch.equal(ring[0], want_ring[0])
    return depth, conf, heat


@pytest.mark.parametrize("S,B", [(224, 1), (518, 4)])
def test_sweep_of_nine_instructions_equals_nine_calls(model, S, B):
    """The nine instructions of demo_results/, three times in a row: eager first call, graph capture, graph replay."""
    x = orc.synthetic_images(B, S).cuda()
    ex = _exif(orc.synthetic_exif(B))
    for _ in range(3):
        _assert_sweep_equals_calls(model, x, ex, list(orc.INSTRUCTIONS))


def test_sweep_ring_buffer_wraps_like_calls(model):
    """K runs of B rewards cross the end of the 1000-entry exploration ring buffer in call order."""
    x = orc.synthetic_images(4, 224, seed=3).cuda()
    ex = _exif(orc.synthetic_exif(4, seed=4))
    model.curiosity_module.history_pointer.fill_(990)
    _assert_sweep_equals_calls(model, x, ex, list(orc.INSTRUCTIONS))
    assert int(model.curiosity_module.history_pointer) == (990 + 9 * 4) % 1000


def test_sweep_of_mixed_guidance_entries(model):
    """An alias, a guidance tensor of another grid size (resized like the reference) and a per-image list, in one sweep."""
    B = 3
    x = orc.synthetic_images(B, 224, seed=8).cuda()
    ex = _exif(orc.synthetic_exif(B, seed=9))
    guide = torch.rand(20 * 20, generator=torch.Generator().manual_seed(3)) * 3
    for _ in range(2):
        _assert_sweep_equals_calls(model, x, ex, ["bottomright", guide, ["left", "top", "center"], "Top-Left"])


def test_sweep_in_curiosity_guided_configuration(cuda_device):
    """curiosity_guided_attention enabled: each call's focal attention depends on its own curiosity score, so the focal
    iterations run once per instruction — still equal to K calls."""
    m = _model(cuda_device, CFG_GUIDED, orc.build_state_dict(0, curiosity_guided=True))
    x = orc.synthetic_images(2, 224).cuda()
    ex = _exif(orc.synthetic_exif(2))
    for _ in range(3):
        _, _, heat = _assert_sweep_equals_calls(m, x, ex, ["top-left", "right", "center"])
    # each call's draws give it its own curiosity score: the per-call base attentions differ
    _assert_sweep_equals_calls(m, x, ex, ["left", "left"])
    base = m._ws[(2, 224)]["sweeps"][2]["base"]
    assert not torch.equal(base[0], base[1])


def _assert_parity(depth, conf, heat, ref, what):
    depth, conf, heat = depth.cpu(), conf.cpu(), heat.cpu()
    assert ((depth - ref["depth"]).abs() / ref["depth"].abs()).max().item() <= 1e-2, what
    assert (conf - ref["confidence"]).abs().max().item() <= 1e-2, what
    assert (heat - ref["heatmap"]).abs().max().item() <= 1e-2, what
    assert torch.equal(heat.argmax(-1), ref["heatmap"].argmax(-1)), what


def test_sweep_matches_the_oracle(model, sd):
    """One sweep against K successive oracle calls (depth abs-rel 1e-2, confidence / heat map 1e-2, argmax exact)."""
    B, S = 2, 224
    x, ex = orc.synthetic_images(B, S, seed=21), orc.synthetic_exif(B, seed=22)
    tokens = orc.dinov2_tokens(sd, x)
    torch.manual_seed(11)
    refs = [orc.forward_with_guidance(sd, None, ex, ins, tokens=tokens, update_history=False) for ins in orc.INSTRUCTIONS]
    torch.manual_seed(11)
    depth, conf, heat = model.forward_with_guidance_sweep(x.cuda(), _exif(ex), list(orc.INSTRUCTIONS),
                                                          return_attention=True)
    for k, (ins, ref) in enumerate(zip(orc.INSTRUCTIONS, refs)):
        _assert_parity(depth[k], conf[k], heat[k], ref, ins)


@pytest.mark.parametrize("K", [1, 9, SWEEP_MAX_K])
def test_sweep_kernels_equal_single_launches(cuda_device, K):
    """ca_weighted_pool_sweep == K ca_weighted_pool launches and ca_guided_softmax_sweep == K ca_guided_softmax launches,
    bit for bit: random tokens, g = 19 (361 rows: a ragged last split and a ragged last batch of 8)."""
    from cognitive_aim_depth_estimation_b200 import ops
    B, g, D, splits = 3, 19, 768, 32
    N, T = g * g, g * g + 1
    gen = torch.Generator().manual_seed(K)
    tokens = torch.randn(B, T, D, generator=gen).cuda()
    w = torch.rand(K, B, N, generator=gen).cuda()
    w /= w.sum(-1, keepdim=True)
    got = torch.full((K * B, splits, D), float("nan"), device="cuda")
    ops.weighted_pool_sweep(tokens, T * D, 1, w, got, K, B, N, D, splits)
    for k in range(K):
        one = torch.full((B, splits, D), float("nan"), device="cuda")
        ops.weighted_pool(tokens, T * D, 1, w[k], None, one, B, N, D, splits)
        assert torch.equal(got[k * B:(k + 1) * B], one), k
    mask = (torch.rand(K, B, N, generator=gen) * 5).cuda()
    for shared in (True, False):
        base = torch.rand(1 if shared else K, B, N, generator=gen).cuda()
        heat = torch.empty(K, B, N, device="cuda")
        arg = torch.empty(K, B, device="cuda", dtype=torch.int32)
        ops.guided_softmax_sweep(base, 0 if shared else B * N, mask, heat, arg, K, B, N)
        for k in range(K):
            h1 = torch.empty(B, N, device="cuda")
            a1 = torch.empty(B, device="cuda", dtype=torch.int32)
            ops.guided_softmax(base[0 if shared else k], mask[k].contiguous(), h1, a1, B, N)
            assert torch.equal(heat[k], h1) and torch.equal(arg[k], a1), (shared, k)


def test_sweep_kernels_refuse_more_than_the_cap(cuda_device):
    from cognitive_aim_depth_estimation_b200 import ops
    from cognitive_aim_depth_estimation_b200._lib import SWEEP_MAX_K as cap, CogAimError
    assert cap == SWEEP_MAX_K
    B, N, D, K = 1, 16, 768, SWEEP_MAX_K + 1
    tokens = torch.zeros(B, N + 1, D, device="cuda")
    with pytest.raises(CogAimError):
        ops.weighted_pool_sweep(tokens, (N + 1) * D, 1, torch.zeros(K, B, N, device="cuda"),
                                torch.empty(K * B, 32, D, device="cuda"), K, B, N, D, 32)


def test_native_sweep_equals_native_calls(cuda_device, sd):
    """NativeModel.forward_with_guidance_sweep (one ca_forward_guided_sweep call) == K NativeModel.forward_with_guidance
    calls, eagerly and through graph capture / replay, ring buffer included; instruction strings and a mask set."""
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    nat = NativeModel(sd, device=cuda_device)
    try:
        B, S = 2, 224
        x, ex = orc.synthetic_images(B, S).cuda(), _exif(orc.synthetic_exif(B))
        N = (S // 14) ** 2
        guides = [torch.rand(N, generator=torch.Generator().manual_seed(i)) * 3 for i in range(3)]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        nat.history_pointer.fill_(995)
        for guidances in (list(orc.INSTRUCTIONS), guides):
            for _ in range(3):  # eager, capture, replay
                with torch.cuda.stream(side):
                    ring0 = (nat.exploration_history.clone(), nat.history_pointer.clone())
                    torch.manual_seed(11)
                    calls = [nat.forward_with_guidance(x, ex, gd) for gd in guidances]
                    want = [torch.stack([c[i] for c in calls]) for i in range(4)]
                    want_ring = (nat.exploration_history.clone(), nat.history_pointer.clone())
                    want_rng = torch.get_rng_state()
                    nat.exploration_history.copy_(ring0[0])
                    nat.history_pointer.copy_(ring0[1])
                    torch.manual_seed(11)
                    got = nat.forward_with_guidance_sweep(x, ex, guidances)
                    torch.cuda.synchronize()
                for i in range(4):
                    assert torch.equal(got[i], want[i]), i
                assert torch.equal(torch.get_rng_state(), want_rng)
                assert torch.equal(nat.history_pointer, want_ring[1])
                assert torch.equal(nat.exploration_history, want_ring[0])
        with pytest.raises(ValueError):
            nat.forward_with_guidance_sweep(x, ex, [])
    finally:
        nat.close()


def test_predict_all_equals_predict_calls(cuda_device, sd):
    """examples/predict_like_demo.py: Predictor.predict_all (one sweep) == nine Predictor.predict calls."""
    import numpy as np
    from PIL import Image
    spec = importlib.util.spec_from_file_location(
        "predict_like_demo", os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "predict_like_demo.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    p = mod.Predictor(sd, image_size=224)
    buf = io.BytesIO()
    Image.fromarray(np.random.default_rng(7).integers(0, 256, (240, 320, 3), dtype=np.uint8)).save(buf, format="JPEG")
    data = buf.getvalue()
    ring0 = _ring(p.model)
    torch.manual_seed(0)
    want = [p.predict(data, ins, overlay_size=(48, 64)) for ins in mod.INSTRUCTIONS]
    want_rng, want_ring = torch.get_rng_state(), _ring(p.model)
    _set_ring(p.model, ring0)
    torch.manual_seed(0)
    got = p.predict_all(data, mod.INSTRUCTIONS, overlay_size=(48, 64))
    assert torch.equal(torch.get_rng_state(), want_rng)
    assert torch.equal(_ring(p.model)[0], want_ring[0]) and torch.equal(_ring(p.model)[1], want_ring[1])
    for (d0, c0, m0), (d1, c1, m1) in zip(want, got):
        assert d0 == d1 and c0 == c1
        assert m0["attention_cell"] == m1["attention_cell"] and m0["instruction"] == m1["instruction"]
        assert torch.equal(m0["overlay"], m1["overlay"])


def test_sweep_argument_errors(model, cuda_device, sd):
    x = orc.synthetic_images(2, 224).cuda()
    ex = _exif(orc.synthetic_exif(2))
    for bad in ([], ["center"] * (SWEEP_MAX_K + 1), ["center", None], ["left", ["top", "left", "right"]]):
        with pytest.raises(ValueError):
            model.forward_with_guidance_sweep(x, ex, bad)
    with pytest.raises(ValueError):
        model.forward_with_guidance_sweep(x, None, ["center"])
    from cognitive_aim_depth_estimation_b200.model import create_model
    no_exif = create_model({"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream"]}},
                           {"num_cameras": 71}, device=cuda_device)
    with pytest.raises(ValueError):
        no_exif.forward_with_guidance_sweep(x, ex, ["center"])
    # the cap itself is accepted
    d, c = model.forward_with_guidance_sweep(x, ex, ["center"] * SWEEP_MAX_K)
    assert d.shape == (SWEEP_MAX_K, 2, 1)
