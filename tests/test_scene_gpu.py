"""Scenes (`encode` once, then `guide` / `guide_sweep` per instruction) must equal `forward_with_guidance` /
`forward_with_guidance_sweep` on the encoded images bit for bit — outputs, global generator state, the CuriosityModule
ring buffer and pointer, and the `_last_*` state — and the fused tail kernel `ops.guide_tail` must equal the
guided_softmax -> weighted_pool -> heads chain it replaces."""
import gc

import pytest
import torch

from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
CFG_GUIDED = dict(CFG, curiosity_guided_attention={"enabled": True})


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


def _state(m):
    return (torch.get_rng_state(), _ring(m), m._last_attention_weights.clone(), m._last_argmax.clone(),
            m._last_curiosity.clone())


def _assert_same_state(a, b):
    assert torch.equal(a[0], b[0]), "generator state"
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[1][1], b[1][1]), "ring buffer"
    for name, x, y in zip(("_last_attention_weights", "_last_argmax", "_last_curiosity"), a[2:], b[2:]):
        assert torch.equal(x, y), name


def _assert_outputs(got, want):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        for j, (x, y) in enumerate(zip(a, b)):
            assert torch.equal(x, y), (i, j)


def _assert_guides_equal_calls(m, x, ex, guidances, seed=11):
    """len(guidances) forward_with_guidance calls, then encode + the same number of guide calls from the same
    generator and ring state: identical in everything observable.  The guide calls run eagerly, then capture a graph
    on the scene, then replay it."""
    ring0 = _ring(m)
    torch.manual_seed(seed)
    want = [[t.clone() for t in m.forward_with_guidance(x, ex, gd, return_attention=True)] for gd in guidances]
    want_state = _state(m)
    _set_ring(m, ring0)
    torch.manual_seed(seed)
    scene = m.encode(x, ex)
    got = [[t.clone() for t in m.guide(scene, gd, return_attention=True)] for gd in guidances]
    torch.cuda.synchronize()
    _assert_outputs(got, want)
    _assert_same_state(_state(m), want_state)
    return scene


@pytest.mark.parametrize("S,B,form", [(224, 1, "f32"), (518, 1, "f32"), (1036, 1, "f32"), (518, 32, "f32"),
                                      (224, 2, "u8"), (224, 3, "list")])
def test_nine_guides_equal_nine_calls(model, S, B, form):
    """The nine instructions of demo_results/, the ring pointer starting near the end so that it wraps around."""
    if form == "f32":
        x = orc.synthetic_images(B, S).cuda()
    else:
        gen = torch.Generator().manual_seed(S + B)
        sizes = [(S, S)] * B if form == "u8" else [(240, 320), (S, S), (600, 410)][:B]
        imgs = [torch.randint(0, 256, (h, w, 3), generator=gen, dtype=torch.uint8).cuda() for h, w in sizes]
        x = torch.stack(imgs) if form == "u8" else imgs
        model.input_size = S
    try:
        ex = _exif(orc.synthetic_exif(B))
        model.curiosity_module.history_pointer.fill_(1000 - 4 * B)
        _assert_guides_equal_calls(model, x, ex, list(orc.INSTRUCTIONS))
    finally:
        model.input_size = None


def test_mixed_guidance_entries(model):
    """An alias, a guidance tensor of another grid size, per-image lists and an upper-case spelling."""
    B = 3
    x = orc.synthetic_images(B, 224, seed=8).cuda()
    ex = _exif(orc.synthetic_exif(B, seed=9))
    guide = torch.rand(20 * 20, generator=torch.Generator().manual_seed(3)) * 3
    _assert_guides_equal_calls(model, x, ex, ["bottomright", guide, ["left", "top", "center"], "Top-Left",
                                              ["right"] * 3, guide])


def test_guides_with_other_forwards_in_between(model):
    """forward, forward_with_guidance on other images and a sweep between guide calls (same batch shape, so they
    overwrite the workspace the guide calls share): still the calls' results and state."""
    B, S = 2, 224
    x, ex = orc.synthetic_images(B, S, seed=1).cuda(), _exif(orc.synthetic_exif(B, seed=2))
    y, ey = orc.synthetic_images(B, S, seed=3).cuda(), _exif(orc.synthetic_exif(B, seed=4))

    def run(first, then):
        out = [first("center")]
        for gd in ("left", "top-right", "bottom", "center"):
            model.forward(y, ey, return_attention=True)
            model.forward_with_guidance(y, ey, "right")
            model.forward_with_guidance_sweep(y, ey, ["left", "top"])
            out.append(then(gd))
        return [[t.clone() for t in o] for o in out]

    ring0 = _ring(model)
    torch.manual_seed(5)
    fwg = lambda gd: model.forward_with_guidance(x, ex, gd, return_attention=True)  # noqa: E731
    want = run(fwg, fwg)
    want_state = _state(model)
    _set_ring(model, ring0)
    torch.manual_seed(5)
    scene = model.encode(x, ex)
    g = lambda gd: model.guide(scene, gd, return_attention=True)  # noqa: E731
    got = run(g, g)
    _assert_outputs(got, want)
    _assert_same_state(_state(model), want_state)


def test_two_scenes_of_one_shape_keep_their_own_results(model):
    """Two scenes of the same (B, S), guided alternately through their own captured graphs."""
    B, S = 2, 224
    xs = [orc.synthetic_images(B, S, seed=s).cuda() for s in (30, 31)]
    exs = [_exif(orc.synthetic_exif(B, seed=s)) for s in (32, 33)]
    order = [0, 1, 0, 1, 1, 0, 0, 1]
    ring0 = _ring(model)
    torch.manual_seed(2)
    want = [[t.clone() for t in model.forward_with_guidance(xs[i], exs[i], "top", return_attention=True)] for i in order]
    want_state = _state(model)
    _set_ring(model, ring0)
    torch.manual_seed(2)
    scenes = [model.encode(x, e) for x, e in zip(xs, exs)]
    got = [[t.clone() for t in model.guide(scenes[i], "top", return_attention=True)] for i in order]
    _assert_outputs(got, want)
    _assert_same_state(_state(model), want_state)
    assert all(len(s._graphs) == 1 for s in scenes)


def test_graphs_off_equal_graphs_on(model):
    x, ex = orc.synthetic_images(1, 224, seed=40).cuda(), _exif(orc.synthetic_exif(1, seed=41))
    ring0 = _ring(model)
    torch.manual_seed(3)
    s = model.encode(x, ex)
    want = [[t.clone() for t in model.guide(s, gd, return_attention=True)] for gd in ("left", "top", "center")]
    _set_ring(model, ring0)
    model.use_cuda_graphs = False
    try:
        torch.manual_seed(3)
        s = model.encode(x, ex)
        got = [[t.clone() for t in model.guide(s, gd, return_attention=True)] for gd in ("left", "top", "center")]
    finally:
        model.use_cuda_graphs = True
    _assert_outputs(got, want)


def _assert_guide_sweep_equals_sweep(m, x, ex, guidances, seed=11):
    ring0 = _ring(m)
    torch.manual_seed(seed)
    want = [t.clone() for t in m.forward_with_guidance_sweep(x, ex, guidances, return_attention=True)]
    want_state = _state(m)
    _set_ring(m, ring0)
    torch.manual_seed(seed)
    scene = m.encode(x, ex)
    for _ in range(3):  # eager, capture, replay: each equal to its own sweep
        ring1 = _ring(m)
        rng1 = torch.get_rng_state()
        got = [t.clone() for t in m.guide_sweep(scene, guidances, return_attention=True)]
        _assert_outputs([got], [want])
        _assert_same_state(_state(m), want_state)
        _set_ring(m, ring1)
        torch.set_rng_state(rng1)


def test_guide_sweep_equals_sweep(model):
    x, ex = orc.synthetic_images(3, 518, seed=5).cuda(), _exif(orc.synthetic_exif(3, seed=6))
    guide = torch.rand(20 * 20, generator=torch.Generator().manual_seed(3)) * 3
    _assert_guide_sweep_equals_sweep(model, x, ex, list(orc.INSTRUCTIONS))
    _assert_guide_sweep_equals_sweep(model, x, ex, ["left", guide, ["top", "left", "right"]])


def test_curiosity_guided_configuration(cuda_device):
    """Each call's focal attention depends on its own curiosity score: the scene keeps the tokens only, and every
    guide call reruns the focal iterations with its own modulation."""
    m = _model(cuda_device, CFG_GUIDED, orc.build_state_dict(0, curiosity_guided=True))
    x = orc.synthetic_images(2, 224).cuda()
    ex = _exif(orc.synthetic_exif(2))
    scene = _assert_guides_equal_calls(m, x, ex, ["top-left", "right", "center", "left"])
    assert scene.base is None
    _assert_guide_sweep_equals_sweep(m, x, ex, ["top-left", "right", "center"])


def test_guide_matches_the_oracle(model, sd):
    """Nine guide calls against nine oracle calls at 224^2 (README bar: depth abs-rel 1e-2, confidence / heat map 1e-2,
    argmax exact)."""
    B, S = 2, 224
    x, ex = orc.synthetic_images(B, S, seed=21), orc.synthetic_exif(B, seed=22)
    tokens = orc.dinov2_tokens(sd, x)
    torch.manual_seed(11)
    refs = [orc.forward_with_guidance(sd, None, ex, ins, tokens=tokens, update_history=False) for ins in orc.INSTRUCTIONS]
    torch.manual_seed(11)
    scene = model.encode(x.cuda(), _exif(ex))
    for ins, ref in zip(orc.INSTRUCTIONS, refs):
        depth, conf, heat = (t.cpu() for t in model.guide(scene, ins, return_attention=True))
        assert ((depth - ref["depth"]).abs() / ref["depth"].abs()).max().item() <= 1e-2, ins
        assert (conf - ref["confidence"]).abs().max().item() <= 1e-2, ins
        assert (heat - ref["heatmap"]).abs().max().item() <= 1e-2, ins
        assert torch.equal(heat.argmax(-1), ref["heatmap"].argmax(-1)), ins


@pytest.mark.parametrize("g", [16, 37, 74])
@pytest.mark.parametrize("B", [1, 32])
def test_guide_tail_equals_the_chain(model, g, B):
    """ops.guide_tail == guided_softmax -> weighted_pool -> heads bit for bit (heat, argmax, depth, confidence, pooled
    vector) at N = 256, 1369 and 5476, for a batch-wide and a per-image mask, with NaN-filled scratch buffers; twice in a
    row, since the per-image tickets must re-arm themselves."""
    from cognitive_aim_depth_estimation_b200 import ops
    pk = model._pack()
    N, T, D, splits = g * g, g * g + 1, 768, 32
    gen = torch.Generator().manual_seed(g * 100 + B)
    tokens = torch.randn(B, T, D, generator=gen).cuda()
    base = torch.rand(B, N, generator=gen).cuda()
    base /= base.sum(-1, keepdim=True)
    tmp_w, tmp_b = (torch.randn(64, D, generator=gen) * 0.03).cuda(), (torch.randn(64, generator=gen) * 0.03).cuda()
    ex = _exif(orc.synthetic_exif(B, seed=g))
    exif = torch.stack([ex["focal_length"], ex["aperture"], ex["iso"]], 1).float().contiguous()
    cam = ex["camera_idx"].long().contiguous()
    fault = model._fault_word().data_ptr()
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")  # noqa: E731
    ticket = torch.zeros(B, device="cuda", dtype=torch.int32)
    for mask in ((torch.rand(N, generator=gen) * 3).cuda(), (torch.rand(B, N, generator=gen) * 3).cuda()):
        heat1, pool1, pooled1, d1, c1 = nan(B, N), nan(B, splits, D), nan(B, D), nan(B), nan(B)
        arg1 = torch.full((B,), -1, device="cuda", dtype=torch.int32)
        ops.guided_softmax(base, mask, heat1, arg1, B, N)
        ops.weighted_pool(tokens, T * D, 1, heat1, None, pool1, B, N, D, splits)
        ops.heads(pk["heads"], tokens=tokens, tokens_per_img=T, depth=d1, conf=c1, B=B, pool_partial=pool1,
                  pool_splits=splits, tmp_w=tmp_w, tmp_b=tmp_b, pooled_out=pooled1, exif=exif, camera_idx=cam,
                  num_cameras=71, fault_ptr=fault)
        for _ in range(2):
            heat2, pool2, pooled2, d2, c2 = nan(B, N), nan(B, splits, D), nan(B, D), nan(B), nan(B)
            arg2 = torch.full((B,), -1, device="cuda", dtype=torch.int32)
            ops.guide_tail(pk["heads"], base=base, mask=mask, heat=heat2, argmax=arg2, ticket=ticket, tokens=tokens,
                           depth=d2, conf=c2, B=B, N=N, pool_partial=pool2, tmp_w=tmp_w, tmp_b=tmp_b, exif=exif,
                           camera_idx=cam, num_cameras=71, fault_ptr=fault, pooled_out=pooled2)
            torch.cuda.synchronize()
            for name, a, b in (("heat", heat2, heat1), ("argmax", arg2, arg1), ("pool", pool2, pool1),
                               ("pooled", pooled2, pooled1), ("depth", d2, d1), ("conf", c2, c1)):
                assert torch.equal(a, b), name
            assert not torch.isnan(d2).any()
            assert int(ticket.abs().sum()) == 0


def test_stale_scene_raises(cuda_device, sd):
    m = _model(cuda_device, CFG, sd)
    x, ex = orc.synthetic_images(1, 224).cuda(), _exif(orc.synthetic_exif(1))
    scene = m.encode(x, ex)
    m.guide(scene, "center")
    m.load_state_dict(sd)
    with pytest.raises(ValueError, match="stale"):
        m.guide(scene, "center")
    with pytest.raises(ValueError, match="stale"):
        m.guide_sweep(scene, ["center"])
    other = _model(cuda_device, CFG, sd)
    with pytest.raises(ValueError, match="another model"):
        other.guide(m.encode(x, ex), "center")


def test_encode_draws_nothing_and_leaves_state(model):
    x, ex = orc.synthetic_images(2, 224, seed=50).cuda(), _exif(orc.synthetic_exif(2, seed=51))
    model.forward_with_guidance(x, ex, "left")
    torch.manual_seed(4)
    before = _state(model)
    model.encode(orc.synthetic_images(2, 224, seed=52).cuda(), ex)
    torch.cuda.synchronize()
    _assert_same_state(_state(model), before)


def test_scene_memory_is_released(model):
    """The scene's tokens, attention, EXIF and graphs go back to the allocator when the scene is dropped."""
    B, S = 4, 518
    x, ex = orc.synthetic_images(B, S, seed=60).cuda(), _exif(orc.synthetic_exif(B, seed=61))
    scene = model.encode(x, ex)
    for gd in ("left", "top", "center"):
        model.guide(scene, gd)
    del scene
    gc.collect()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    scene = model.encode(x, ex)
    for gd in ("left", "top", "center"):
        model.guide(scene, gd)
    torch.cuda.synchronize()
    T = (S // 14) ** 2 + 1
    assert torch.cuda.memory_allocated() - base >= B * T * 768 * 4
    del scene
    gc.collect()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == base


def _demo_module():
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "predict_like_demo.py")
    spec = importlib.util.spec_from_file_location("predict_like_demo", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, path


def _jpeg(tmp_path):
    import numpy as np
    from PIL import Image
    path = tmp_path / "photo.jpg"
    Image.fromarray(np.random.default_rng(7).integers(0, 256, (240, 320, 3), dtype=np.uint8)).save(path, format="JPEG")
    return path


def test_interactive_example_prints_the_predict_lines(cuda_device, tmp_path):
    """`predict_like_demo.py IMAGE --interactive` with three instructions on stdin prints the lines of three
    successive `predict` calls of a fresh session (seed 0, random init), and predict_scene equals predict."""
    import subprocess
    import sys
    mod, script = _demo_module()
    path = _jpeg(tmp_path)
    data = path.read_bytes()
    three = ["top-left", "center", "bottom-right"]
    torch.manual_seed(0)
    p = mod.Predictor(None, image_size=224)
    want = [mod.result_line(ins, *p.predict(data, ins)) for ins in three]
    torch.manual_seed(0)
    q = mod.Predictor(None, image_size=224)
    scene = q.encode(data)
    got = [mod.result_line(ins, *q.predict_scene(scene, ins)) for ins in three]
    assert got == want
    env = {k: v for k, v in __import__("os").environ.items()}
    env["PYTHONNOUSERSITE"] = "1"
    out = subprocess.run([sys.executable, script, str(path), "--interactive"], input="\n".join(three) + "\n",
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr
    assert out.stdout.splitlines() == want


def test_native_scene_equals_native_calls(cuda_device, sd):
    """NativeModel.encode / guide / guide_sweep (ca_encode, ca_guide, ca_guide_sweep) == NativeModel.forward_with_guidance
    / forward_with_guidance_sweep from the same seed and ring state: eager, captured and replayed; instruction strings and
    guidance tensors."""
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    nat = NativeModel(sd, device=cuda_device)
    try:
        B, S = 2, 224
        x, ex = orc.synthetic_images(B, S, seed=70).cuda(), _exif(orc.synthetic_exif(B, seed=71))
        N = (S // 14) ** 2
        guides = [torch.rand(N, generator=torch.Generator().manual_seed(i)) * 3 for i in range(2)]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        nat.history_pointer.fill_(996)
        with torch.cuda.stream(side):
            seq = ["top-left", guides[0], "center", "bottom", guides[1], "left"]
            ring0 = (nat.exploration_history.clone(), nat.history_pointer.clone())
            torch.manual_seed(11)
            want = [[t.clone() for t in nat.forward_with_guidance(x, ex, gd)] for gd in seq]
            want_sweep = [t.clone() for t in nat.forward_with_guidance_sweep(x, ex, list(orc.INSTRUCTIONS))]
            want_ring = (nat.exploration_history.clone(), nat.history_pointer.clone())
            want_rng = torch.get_rng_state()
            nat.exploration_history.copy_(ring0[0])
            nat.history_pointer.copy_(ring0[1])
            torch.manual_seed(11)
            scene = nat.encode(x, ex)
            got = [[t.clone() for t in nat.guide(scene, gd)] for gd in seq]
            got_sweep = [t.clone() for t in nat.guide_sweep(scene, list(orc.INSTRUCTIONS))]
            torch.cuda.synchronize()
        _assert_outputs(got, want)
        _assert_outputs([got_sweep], [want_sweep])
        assert torch.equal(torch.get_rng_state(), want_rng)
        assert torch.equal(nat.history_pointer, want_ring[1])
        assert torch.equal(nat.exploration_history, want_ring[0])
        # three more sweeps: eager once, then captured and replayed on the scene
        for _ in range(2):
            nat.guide_sweep(scene, ["left", "right"])
        torch.cuda.synchronize()
        scene.close()
    finally:
        nat.close()


def test_native_destroyed_scene_or_handle_is_refused(cuda_device, sd):
    import ctypes as C
    from cognitive_aim_depth_estimation_b200._lib import CogAimError
    from cognitive_aim_depth_estimation_b200.native import NativeModel, NativeScene
    nat = NativeModel(sd, device=cuda_device)
    x, ex = orc.synthetic_images(1, 224, seed=72).cuda(), _exif(orc.synthetic_exif(1, seed=73))
    scene = nat.encode(x, ex)
    nat.guide(scene, "center")
    stale = NativeScene(nat.lib, C.c_void_p(scene.ptr.value), scene.B, scene.S, scene.device)
    scene.close()
    try:
        with pytest.raises(CogAimError):
            nat.guide(stale, "center")
        with pytest.raises(CogAimError):
            nat.guide_sweep(stale, ["center"])
        with pytest.raises(CogAimError):
            stale.close()  # already destroyed
    finally:
        stale.ptr = None
    other = nat.encode(x, ex)
    nat2 = NativeModel(sd, device=cuda_device)
    try:
        with pytest.raises(CogAimError):  # a scene of another handle
            nat2.guide(other, "center")
        h = nat._h
        nat.close()
        nat._h = h  # the destroyed handle's address: its scenes are refused, not dereferenced
        with pytest.raises(CogAimError):
            nat.guide(other, "center")
        nat._h = None
        other.close()  # a scene outlives its handle and is still released
    finally:
        nat2.close()


def test_guide_with_the_three_kernel_tail(model, monkeypatch):
    """Batches above the fused tail's size limit run guided_softmax -> weighted_pool -> heads: the same results."""
    import cognitive_aim_depth_estimation_b200.model as mod
    monkeypatch.setattr(mod, "_GUIDE_TAIL_MAX_B", 0)
    x, ex = orc.synthetic_images(3, 224, seed=80).cuda(), _exif(orc.synthetic_exif(3, seed=81))
    _assert_guides_equal_calls(model, x, ex, ["center", "left", ["top", "right", "bottom"], "top-left"])
