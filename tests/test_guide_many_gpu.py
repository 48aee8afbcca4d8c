"""`guide_many(scenes, guidances)` must equal the loop `[guide(s, g) for s, g in zip(scenes, guidances)]` bit for bit —
outputs, heat maps, argmax, global generator state, the CuriosityModule ring buffer and pointer, and the `_last_*`
state — whatever the scenes' batch sizes, input forms and guidance forms, through eager, captured and replayed calls.
Its new kernels (the row-table gather and pool, the heads' per-row projection) must equal the kernels they stand in for."""
import gc

import pytest
import torch

from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
CFG_GUIDED = dict(CFG, curiosity_guided_attention={"enabled": True})
MAX_CALLS, MAX_ROWS = 64, 256


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
        assert len(a) == len(b)
        for j, (x, y) in enumerate(zip(a, b)):
            assert torch.equal(x, y), (i, j)


def _clone(outs):
    return [[t.clone() for t in o] for o in outs]


def _assert_many_equals_loop(m, scenes, guidances, seed=11, reps=3, pointer=None):
    """guide_many against the loop of guide calls from the same generator and ring state, `reps` times (eager, captured,
    replayed).  `pointer`: the ring pointer each repetition starts from."""
    for rep in range(reps):
        if pointer is not None:
            m.curiosity_module.history_pointer.fill_(pointer)
        ring0 = _ring(m)
        torch.manual_seed(seed + rep)
        want = _clone(m.guide(s, gd, return_attention=True) for s, gd in zip(scenes, guidances))
        want_state = _state(m)
        _set_ring(m, ring0)
        torch.manual_seed(seed + rep)
        got = _clone(m.guide_many(scenes, guidances, return_attention=True))
        torch.cuda.synchronize()
        _assert_outputs(got, want)
        _assert_same_state(_state(m), want_state)


def _encode(m, B, S, form, seed):
    ex = _exif(orc.synthetic_exif(B, seed=seed + 1))
    if form == "f32":
        return m.encode(orc.synthetic_images(B, S, seed=seed).cuda(), ex)
    gen = torch.Generator().manual_seed(seed)
    sizes = [(S, S)] * B if form == "u8" else [((240, 320), (S, S), (600, 410))[i % 3] for i in range(B)]
    imgs = [torch.randint(0, 256, (h, w, 3), generator=gen, dtype=torch.uint8).cuda() for h, w in sizes]
    m.input_size = S
    try:
        return m.encode(torch.stack(imgs) if form == "u8" else imgs, ex)
    finally:
        m.input_size = None


def _guidances(sizes, g):
    """One of every guidance form `guide` takes, cycled over the calls."""
    gen = torch.Generator().manual_seed(g)
    forms = [lambda B: "top-left", lambda B: "bottomright", lambda B: torch.rand(20 * 20, generator=gen) * 3,
             lambda B: [(torch.rand(g * g, generator=gen) * 3).cuda() for _ in range(B)],
             lambda B: [orc.INSTRUCTIONS[i % 9] for i in range(B)], lambda B: "Center"]
    return [forms[j % len(forms)](B) for j, B in enumerate(sizes)]


@pytest.mark.parametrize("S", [224, 518, 1036])
@pytest.mark.parametrize("sizes", [(1, 1, 1), (1, 3, 32, 1)])
def test_guide_many_equals_the_guide_loop(model, S, sizes):
    """Scenes encoded from fp32, uint8 and ragged-list input, every guidance form, a ring pointer that wraps during the
    call; eager, captured and replayed."""
    forms = ("f32", "u8", "list")
    scenes = [_encode(model, B, S, forms[j % 3], seed=100 * S + j) for j, B in enumerate(sizes)]
    R = sum(sizes)
    _assert_many_equals_loop(model, scenes, _guidances(sizes, S // 14), pointer=1000 - R // 2)


def test_repeated_scene_and_no_attention(model):
    a, b = _encode(model, 2, 224, "f32", 1), _encode(model, 1, 224, "f32", 2)
    scenes = [a, b, a, a]
    _assert_many_equals_loop(model, scenes, ["left", "top", ["right", "center"], "left"], reps=2)
    torch.manual_seed(3)
    outs = model.guide_many(scenes, ["left"] * 4)
    assert [tuple(t.shape for t in o) for o in outs] == [((2, 1), (2, 1)), ((1, 1), (1, 1)), ((2, 1), (2, 1)),
                                                         ((2, 1), (2, 1))]


def test_replay_with_other_scenes(model):
    """The graph captured at the second call replays for other scenes of the same row layout, after the scenes it was
    captured with were dropped: the row table is data."""
    first = [_encode(model, B, 518, "f32", 10 + j) for j, B in enumerate((1, 3))]
    for _ in range(2):
        model.guide_many(first, ["left", "top"])
    other = [_encode(model, B, 518, "f32", 20 + j) for j, B in enumerate((1, 3))]  # drops the call's keep-alive
    del first
    gc.collect()
    torch.cuda.synchronize()
    graphs = dict(model._many[518]["graphs"])
    _assert_many_equals_loop(model, other, ["center", ["top", "left", "right"]], reps=2)
    assert model._many[518]["graphs"] == graphs  # replayed, not captured again


def test_interleaved_with_forward_and_guide(model):
    """forward, forward_with_guidance and guide calls between guide_many calls: each guide_many still equals its loop."""
    S = 224
    scenes = [_encode(model, B, S, "f32", 30 + j) for j, B in enumerate((1, 2, 1))]
    y, ey = orc.synthetic_images(2, S, seed=40).cuda(), _exif(orc.synthetic_exif(2, seed=41))
    gds = ["top", "left", "right", "bottom"]

    def run(many):
        out = []
        for i in range(4):
            out += many((gds[i:] + gds[:i])[:3])
            out.append(model.forward(y, ey, return_attention=True))
            out.append(model.guide(scenes[1], "center", return_attention=True))
            out.append(model.forward_with_guidance(y, ey, "right", return_attention=True))
        return _clone(out)

    ring0 = _ring(model)
    torch.manual_seed(5)
    want = run(lambda g: [model.guide(s, gd, return_attention=True) for s, gd in zip(scenes, g)])
    want_state = _state(model)
    _set_ring(model, ring0)
    torch.manual_seed(5)
    got = run(lambda g: model.guide_many(scenes, g, return_attention=True))
    _assert_outputs(got, want)
    _assert_same_state(_state(model), want_state)


def test_curiosity_guided_configuration(cuda_device):
    m = _model(cuda_device, CFG_GUIDED, orc.build_state_dict(0, curiosity_guided=True))
    scenes = [_encode(m, B, 224, "f32", 50 + j) for j, B in enumerate((2, 1, 3))]
    _assert_many_equals_loop(m, scenes, ["top-left", "right", ["center", "left", "bottom"]], reps=2,
                             pointer=998)


def test_guide_many_matches_the_oracle(model, sd):
    """Two scenes against the oracle's forward_with_guidance calls in the same order (README bar: depth abs-rel 1e-2,
    confidence / heat map 1e-2, argmax exact)."""
    S, sizes, ins = 224, (2, 1), ["top-right", "left"]
    xs = [orc.synthetic_images(B, S, seed=60 + j) for j, B in enumerate(sizes)]
    exs = [orc.synthetic_exif(B, seed=70 + j) for j, B in enumerate(sizes)]
    torch.manual_seed(11)
    refs = [orc.forward_with_guidance(sd, None, ex, gd, tokens=orc.dinov2_tokens(sd, x), update_history=False)
            for x, ex, gd in zip(xs, exs, ins)]
    scenes = [model.encode(x.cuda(), _exif(ex)) for x, ex in zip(xs, exs)]
    torch.manual_seed(11)
    for (depth, conf, heat), ref in zip(model.guide_many(scenes, ins, return_attention=True), refs):
        depth, conf, heat = depth.cpu(), conf.cpu(), heat.cpu()
        assert ((depth - ref["depth"]).abs() / ref["depth"].abs()).max().item() <= 1e-2
        assert (conf - ref["confidence"]).abs().max().item() <= 1e-2
        assert (heat - ref["heatmap"]).abs().max().item() <= 1e-2
        assert torch.equal(heat.argmax(-1), ref["heatmap"].argmax(-1))


def _table(images, bases, exif, cam, calls):
    """ca_guide_many_row [R] (int64 words, on the device) for rows given as per-row tensors."""
    words = []
    for t, b, e, c, j in zip(images, bases, exif, cam, calls):
        words += [t.data_ptr(), b.data_ptr(), e.data_ptr(), c.data_ptr(), 0, j]
    return torch.tensor(words, dtype=torch.int64).cuda()


@pytest.mark.parametrize("g", [16, 37, 74])
def test_row_pool_and_gather_equal_the_per_image_kernels(g):
    """ops.weighted_pool_rows == ops.weighted_pool on each image alone, bit for bit, with the images in separate
    allocations; ops.gather_rows copies exactly.  NaN-filled outputs (CA_POISON_WS=1 is the suite's default)."""
    from cognitive_aim_depth_estimation_b200 import ops
    assert __import__("os").environ.get("CA_POISON_WS") == "1"
    N, T, D, splits, R = g * g, g * g + 1, 768, 32, 5
    gen = torch.Generator().manual_seed(g)
    images = [torch.randn(T, D, generator=gen).cuda() for _ in range(R)]
    bases = [torch.rand(N, generator=gen).cuda() for _ in range(R)]
    exif = [torch.rand(3, generator=gen).cuda() for _ in range(R)]
    cam = [torch.tensor([i * 7], dtype=torch.int64).cuda() for i in range(R)]
    calls = [0, 0, 1, 2, 2]
    rows = _table(images, bases, exif, cam, calls)
    w = torch.rand(R, N, generator=gen).cuda()
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")  # noqa: E731
    part = nan(R, splits, D)
    ops.weighted_pool_rows(rows, w, part, R, N, D, splits)
    cls, base, ex = nan(R, D), nan(R, N), nan(R, 3)
    cm = torch.full((R,), -1, device="cuda", dtype=torch.int64)
    cr = torch.full((R,), -1, device="cuda", dtype=torch.int32)
    ops.gather_rows(rows, R, N, cls, base, ex, cm, cr)
    for r in range(R):
        want = nan(1, splits, D)
        ops.weighted_pool(images[r].unsqueeze(0), T * D, 1, w[r:r + 1].contiguous(), None, want, 1, N, D, splits)
        assert torch.equal(part[r], want[0]), r
        assert torch.equal(cls[r], images[r][0]) and torch.equal(base[r], bases[r]) and torch.equal(ex[r], exif[r])
    assert cm.tolist() == [i * 7 for i in range(R)] and cr.tolist() == calls


def test_heads_call_of_row_equal_the_sweep_heads(model):
    """ops.heads with call_of_row over gathered CLS rows == the sweep heads (sweep_images = B) row for row."""
    from cognitive_aim_depth_estimation_b200 import ops
    pk = model._pack()
    K, B, N, D, splits = 3, 4, 256, 768, 32
    T = N + 1
    gen = torch.Generator().manual_seed(5)
    tokens = torch.randn(B, T, D, generator=gen).cuda()
    pool = torch.randn(K * B, splits, D, generator=gen).cuda()
    tmp_w, tmp_b = (torch.randn(K, 64, D, generator=gen) * 0.03).cuda(), (torch.randn(K, 64, generator=gen) * 0.03).cuda()
    ex = _exif(orc.synthetic_exif(B, seed=6))
    exif = torch.stack([ex["focal_length"], ex["aperture"], ex["iso"]], 1).float().contiguous()
    cam = ex["camera_idx"].long().contiguous()
    fault = model._fault_word().data_ptr()
    d1, c1 = torch.empty(K * B, device="cuda"), torch.empty(K * B, device="cuda")
    ops.heads(pk["heads"], tokens=tokens, tokens_per_img=T, depth=d1, conf=c1, B=K * B, pool_partial=pool,
              pool_splits=splits, tmp_w=tmp_w, tmp_b=tmp_b, exif=exif, camera_idx=cam, num_cameras=71, fault_ptr=fault,
              sweep_images=B)
    cls = tokens[:, 0].repeat(K, 1).contiguous()
    call = torch.arange(K, dtype=torch.int32).repeat_interleave(B).cuda()
    d2, c2 = torch.empty(K * B, device="cuda"), torch.empty(K * B, device="cuda")
    ops.heads(pk["heads"], tokens=cls, tokens_per_img=1, depth=d2, conf=c2, B=K * B, pool_partial=pool,
              pool_splits=splits, tmp_w=tmp_w, tmp_b=tmp_b, exif=exif.repeat(K, 1).contiguous(),
              camera_idx=cam.repeat(K).contiguous(), num_cameras=71, fault_ptr=fault, call_of_row=call)
    torch.cuda.synchronize()
    assert torch.equal(d1, d2) and torch.equal(c1, c2)


def test_refusals_come_before_any_draw(cuda_device, model, sd):
    a, b = _encode(model, 2, 224, "f32", 80), _encode(model, 1, 224, "f32", 81)
    wide = _encode(model, 1, 518, "f32", 82)
    foreign = _model(cuda_device, CFG, sd).encode(orc.synthetic_images(1, 224).cuda(), _exif(orc.synthetic_exif(1)))
    big = _encode(model, 32, 224, "f32", 83)
    cases = [
        (a, ["left"], "list"), ([a], "left", "list"), ([], [], "m >= 1"), ([a, b], ["left"], "one guidance"),
        ([a, None], ["left", "top"], "Scene"), ([a, b], ["left", None], "None"),
        ([a, foreign], ["left", "top"], "another model"), ([a, wide], ["left", "top"], "share the image side"),
        ([a, b], [["left"], "top"], "per-image"), ([a, b], ["left", "sideways"], "unknown instruction"),
        ([a, b], [["left", "nowhere"], "top"], "unknown instruction"),
        ([b] * (MAX_CALLS + 1), ["left"] * (MAX_CALLS + 1), "at most"),
        ([big] * (MAX_ROWS // 32 + 1), ["left"] * (MAX_ROWS // 32 + 1), "at most"),
        ([a, b], [[torch.rand(256)] * 3, "top"], "per-image"),
        # `guide` takes a per-image list of [N] tensors, not a [B, N] tensor: neither does guide_many
        ([a, b], [torch.rand(2, 256).cuda(), "top"], "1-D tensor"),
    ]
    torch.manual_seed(9)
    before = _ring(model)
    for scenes, gds, msg in cases:
        rng = torch.get_rng_state()
        with pytest.raises(ValueError, match=msg):
            model.guide_many(scenes, gds)
        assert torch.equal(torch.get_rng_state(), rng), msg
    torch.cuda.synchronize()
    after = _ring(model)
    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])
    with pytest.raises(ValueError, match="1-D tensor"):
        model.guide(a, torch.rand(2, 256).cuda())
    model.load_state_dict(sd)  # the same weights, re-packed: every scene encoded before is stale
    rng = torch.get_rng_state()
    with pytest.raises(ValueError, match="stale"):
        model.guide_many([b, a], ["left", "top"])
    assert torch.equal(torch.get_rng_state(), rng)


def test_bad_camera_index_in_one_scene_is_reported(model):
    good = _encode(model, 1, 224, "f32", 90)
    ex = _exif(orc.synthetic_exif(2, seed=91))
    ex["camera_idx"] = torch.tensor([3, 500], device="cuda")  # on the device: checked by the heads kernel
    bad = model.encode(orc.synthetic_images(2, 224, seed=92).cuda(), ex)
    model.guide_many([good, bad], ["left", "top"])
    with pytest.raises(ValueError, match="camera_idx"):
        model.check_inputs(sync=True)
    model.guide_many([good, good], ["left", "top"])
    model.check_inputs(sync=True)  # the fault word was cleared: later calls are clean


def test_one_batched_pass_whatever_m(model):
    """The launches of a guide_many call do not grow with the number of scenes: one pass, not m chains."""
    from cognitive_aim_depth_estimation_b200 import ops
    scenes = [_encode(model, 1, 224, "f32", 100 + j) for j in range(32)]
    counts = []
    for m in (2, 32):
        for _ in range(2):  # eager, then captured: the third call replays
            model.guide_many(scenes[:m], ["left"] * m)
        n0 = ops.launch_count()
        model.guide_many(scenes[:m], ["left"] * m)
        counts.append(ops.launch_count() - n0)
    assert counts[0] == counts[1], counts


def _native_many_vs_guides(nat, scenes, guidances, reps=3):
    """NativeModel.guide_many against successive NativeModel.guide calls from the same generator and ring state."""
    for rep in range(reps):
        ring0 = (nat.exploration_history.clone(), nat.history_pointer.clone())
        torch.manual_seed(20 + rep)
        want = _clone(nat.guide(s, gd) for s, gd in zip(scenes, guidances))
        want_ring = (nat.exploration_history.clone(), nat.history_pointer.clone())
        want_rng = torch.get_rng_state()
        nat.exploration_history.copy_(ring0[0])
        nat.history_pointer.copy_(ring0[1])
        torch.manual_seed(20 + rep)
        got = _clone(nat.guide_many(scenes, guidances))
        torch.cuda.synchronize()
        _assert_outputs(got, want)
        assert torch.equal(torch.get_rng_state(), want_rng)
        assert torch.equal(nat.history_pointer, want_ring[1]) and torch.equal(nat.exploration_history, want_ring[0])


def test_native_guide_many_equals_native_guides(cuda_device, sd):
    """ca_guide_many (NativeModel.guide_many) == successive ca_guide calls: eager, captured and replayed, instruction
    strings and guidance tensors, a ring that wraps; and its launch count does not grow with m."""
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    nat = NativeModel(sd, device=cuda_device)
    try:
        S = 518
        N = (S // 14) ** 2
        scenes = [nat.encode(orc.synthetic_images(B, S, seed=110 + j).cuda(), _exif(orc.synthetic_exif(B, seed=120 + j)))
                  for j, B in enumerate((1, 3, 2))]
        side = torch.cuda.Stream()  # graphs are captured on a non-default stream
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            nat.history_pointer.fill_(997)
            _native_many_vs_guides(nat, scenes + [scenes[1]], ["top-left", "Center", "bottomright", "left"])
            gen = torch.Generator().manual_seed(3)
            tens = [torch.rand(N, generator=gen) * 3, (torch.rand(3, N, generator=gen) * 3).cuda(),
                    torch.rand(N, generator=gen) * 3]
            _native_many_vs_guides(nat, scenes, tens)
            ones = [nat.encode(orc.synthetic_images(1, 224, seed=130 + j).cuda(), _exif(orc.synthetic_exif(1, seed=j)))
                    for j in range(32)]
            counts = []
            for m in (2, 32):
                for _ in range(3):
                    nat.guide_many(ones[:m], ["left"] * m)
                counts.append(nat.launch_count())
            torch.cuda.synchronize()
        assert counts[0] == counts[1], counts
        for s in scenes + ones:
            s.close()
    finally:
        nat.close()


def test_native_guide_many_refusals(cuda_device, sd):
    """A destroyed scene, a scene of another handle, a scene whose handle is gone: CA_STATUS_INVALID, nothing launched."""
    import ctypes as C
    from cognitive_aim_depth_estimation_b200._lib import CogAimError
    from cognitive_aim_depth_estimation_b200.native import NativeModel, NativeScene
    nat, nat2 = NativeModel(sd, device=cuda_device), NativeModel(sd, device=cuda_device)
    x, ex = orc.synthetic_images(1, 224, seed=140).cuda(), _exif(orc.synthetic_exif(1, seed=141))
    try:
        good = nat.encode(x, ex)
        gone = nat.encode(x, ex)
        stale = NativeScene(nat.lib, C.c_void_p(gone.ptr.value), gone.B, gone.S, gone.device)
        gone.close()
        other = nat2.encode(x, ex)
        ring = (nat.exploration_history.clone(), nat.history_pointer.clone())
        for bad in (stale, other):
            with pytest.raises(CogAimError):
                nat.guide_many([good, bad], ["left", "top"])
        stale.ptr = None
        with pytest.raises(CogAimError):
            nat.guide_many([good, good], ["left", "sideways"])
        torch.cuda.synchronize()
        assert torch.equal(nat.exploration_history, ring[0]) and torch.equal(nat.history_pointer, ring[1])
        h = nat2._h
        nat2.close()
        nat2._h = h  # the destroyed handle's address: its scenes are refused, not dereferenced
        with pytest.raises(CogAimError):
            nat2.guide_many([other], ["left"])
        nat2._h = None
        other.close()
        good.close()
    finally:
        nat.close()
        nat2.close()


def test_native_bad_camera_index_reported_in_its_scene(cuda_device, sd):
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    nat = NativeModel(sd, device=cuda_device)
    try:
        good = nat.encode(orc.synthetic_images(1, 224, seed=150).cuda(), _exif(orc.synthetic_exif(1, seed=151)))
        ex = _exif(orc.synthetic_exif(2, seed=152))
        ex["camera_idx"] = torch.tensor([3, 500], device="cuda")
        fault = torch.zeros(1, dtype=torch.int32).pin_memory()
        bad = nat.encode(orc.synthetic_images(2, 224, seed=153).cuda(), ex, fault=fault)
        nat.guide_many([good, good], ["left", "top"])
        torch.cuda.synchronize()
        assert int(fault[0]) == 0
        nat.guide_many([good, bad], ["left", "top"])
        torch.cuda.synchronize()
        assert int(fault[0]) & 1  # scene `bad`'s own fault word
        good.close()
        bad.close()
    finally:
        nat.close()


def test_interactive_example_with_several_photographs(cuda_device, tmp_path):
    """`predict_like_demo.py A B --interactive`: one line per step with one instruction per photograph ('-' skips one),
    each line answered by one guide_many call; the printed lines are those of successive `predict` calls."""
    import importlib.util
    import os
    import subprocess
    import sys
    import numpy as np
    from PIL import Image
    script = os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "predict_like_demo.py")
    spec = importlib.util.spec_from_file_location("predict_like_demo", script)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    paths = []
    for i, (h, w) in enumerate(((240, 320), (300, 200))):
        path = tmp_path / f"photo{i}.jpg"
        Image.fromarray(np.random.default_rng(i).integers(0, 256, (h, w, 3), dtype=np.uint8)).save(path, format="JPEG")
        paths.append(path)
    datas = [p.read_bytes() for p in paths]
    lines = [["top-left", "center"], ["-", "bottom-right"], ["left", "-"]]
    torch.manual_seed(0)
    p = mod.Predictor(None, image_size=224)
    want = [f"{paths[j].name}: " + mod.result_line(ins, *p.predict(datas[j], ins))
            for words in lines for j, ins in enumerate(words) if ins != "-"]
    env = dict(os.environ, PYTHONNOUSERSITE="1")
    out = subprocess.run([sys.executable, script, *map(str, paths), "--interactive"],
                         input="\n".join(" ".join(w) for w in lines) + "\n", capture_output=True, text=True, timeout=600,
                         env=env)
    assert out.returncode == 0, out.stderr
    assert out.stdout.splitlines() == want
