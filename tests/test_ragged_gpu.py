"""Batches of differently sized photographs (demo.py:406-432 `predict_batch` over a folder): the ragged exact-Pillow resize
(`ops.resize_u8_list`, `ca_resize_u8_list`) against Pillow bit for bit, and every forward entry point of the module and of
the handle given a list of uint8 [H_i, W_i, 3] images against the uniform uint8 path on the per-image resized stack."""
import ctypes
import importlib.util
import io
import os

import numpy as np
import pytest
import torch

from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
MAX_SIDE = 16384
# (H, W): landscape and portrait photographs, the identity at S = 518, one axis only, upscaling, a tiny image and a
# strip as wide as the resize accepts
SIZES = [(480, 640), (1080, 1920), (4032, 3024), (518, 518), (518, 300), (300, 518), (100, 77), (41, 37),
         (24, MAX_SIDE)]


@pytest.fixture(scope="module")
def sd():
    return orc.build_state_dict(0)


@pytest.fixture(scope="module")
def model(cuda_device, sd):
    from cognitive_aim_depth_estimation_b200.model import create_model
    m = create_model(CFG, {"num_cameras": 71}, device=cuda_device)
    m.load_state_dict(sd)
    return m


def _photos(sizes, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for i, (h, w) in enumerate(sizes):
        a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if i % 2 == 0:
            a[: h // 2] = 255  # saturated region: exercises the 8-bit clamp
        out.append(a)
    return out


def _exif(B, seed=0):
    return {k: v.cuda() for k, v in orc.synthetic_exif(B, seed=seed).items()}


def _ring(m):
    cm = m.curiosity_module
    return cm.exploration_history.clone(), cm.history_pointer.clone()


def _set_ring(m, ring):
    m.curiosity_module.exploration_history.copy_(ring[0])
    m.curiosity_module.history_pointer.copy_(ring[1])


def _stack_resized(imgs, S):
    """The reference input: each photograph resized on its own by the uniform resize, stacked [B, S, S, 3]."""
    from cognitive_aim_depth_estimation_b200 import ops
    return torch.cat([ops.resize_u8(t.cuda()[None].contiguous(), S, S) for t in imgs])


@pytest.mark.parametrize("S", [224, 518, 70])
def test_resize_list_matches_pillow(cuda_device, S):
    from PIL import Image
    from cognitive_aim_depth_estimation_b200 import ops
    arrs = _photos(SIZES, seed=S)
    want = np.stack([np.asarray(Image.fromarray(a).resize((S, S), Image.BILINEAR)) for a in arrs])
    imgs = [torch.from_numpy(a).to(cuda_device) for a in arrs]
    n0 = ops.launch_count()
    got = ops.resize_u8_list(imgs, S, S)
    assert ops.launch_count() - n0 == 2  # one launch per pass for the whole batch
    got = got.cpu().numpy()
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), (SIZES[i], int(np.abs(g.astype(int) - w.astype(int)).max()))
    assert np.array_equal(got, _stack_resized(imgs, S).cpu().numpy())


def test_resize_list_limit(cuda_device):
    """A side of CA_RESIZE_MAX_SIDE is resized (test above); one pixel more is refused by the wrapper and by the C entry
    point, before anything is launched."""
    from cognitive_aim_depth_estimation_b200 import _lib, ops
    ok = torch.zeros(2, 8, 3, dtype=torch.uint8, device=cuda_device)
    for shape in ((4, MAX_SIDE + 1, 3), (MAX_SIDE + 1, 4, 3)):
        with pytest.raises(ValueError):
            ops.resize_u8_list([ok, torch.zeros(*shape, dtype=torch.uint8, device=cuda_device)], 224, 224)
    lib = _lib.load()
    out = torch.empty(1, 224, 224, 3, dtype=torch.uint8, device=cuda_device)
    ptrs = (ctypes.c_void_p * 1)(ok.data_ptr())
    for h, w in ((4, MAX_SIDE + 1), (MAX_SIDE + 1, 4)):
        hw = (ctypes.c_int * 2)(h, w)
        st = lib.ca_resize_u8_list(ptrs, hw, 1, 224, 224, None, 1 << 30, ctypes.c_void_p(out.data_ptr()),
                                   _lib.stream_ptr())
        assert st == 1 and b"CA_RESIZE_MAX_SIDE" in lib.ca_last_error()


def _list(B, S, seed):
    rng = np.random.default_rng(seed)
    sizes = [(int(rng.integers(40, 900)), int(rng.integers(40, 900))) for _ in range(B)]
    sizes[0] = (S, S)  # one image already at model resolution
    return [torch.from_numpy(a) for a in _photos(sizes, seed)]  # CPU tensors: uploaded like the uniform uint8 path


def _same_call(m, fn, a, b, seed=11):
    """fn(a) and fn(b) from the same generator and ring-buffer state: outputs, generator and ring must agree."""
    ring0 = _ring(m)
    torch.manual_seed(seed)
    want = [t.clone() for t in fn(b)]
    want_state = (m._last_attention_weights.clone() if hasattr(m, "_last_attention_weights") else None,
                  getattr(m, "_last_argmax", torch.zeros(1)).clone(), torch.get_rng_state(), _ring(m))
    _set_ring(m, ring0)
    torch.manual_seed(seed)
    got = fn(a)
    for x, y in zip(got, want):
        assert torch.equal(x, y)
    assert torch.equal(torch.get_rng_state(), want_state[2])
    ring = _ring(m)
    assert torch.equal(ring[0], want_state[3][0]) and torch.equal(ring[1], want_state[3][1])
    if want_state[0] is not None:
        assert torch.equal(m._last_attention_weights, want_state[0])
    assert torch.equal(getattr(m, "_last_argmax", torch.zeros(1)), want_state[1])
    return got


@pytest.mark.parametrize("B,S", [(5, 224), (2, 518)])
def test_forward_with_guidance_list_equals_uniform_u8(model, B, S):
    imgs = _list(B, S, seed=B)
    ref = _stack_resized(imgs, S)
    ex = _exif(B)
    model.input_size = S
    try:
        for ins in ("top-left", ["center", "left", "right", "top", "bottom"][:B]):
            _same_call(model, lambda x: model.forward_with_guidance(x, ex, ins, return_attention=True), imgs, ref)
    finally:
        model.input_size = None


def test_sweep_and_forward_list_equal_uniform_u8(model):
    B, S = 5, 224
    imgs = _list(B, S, seed=21)
    ref = _stack_resized(imgs, S)
    ex = _exif(B)
    model.input_size = S
    try:
        _same_call(model, lambda x: model.forward_with_guidance_sweep(x, ex, list(orc.INSTRUCTIONS),
                                                                      return_attention=True), imgs, ref)
        _same_call(model, lambda x: model.forward(x, ex, return_attention=True) + (model.fusion_features,), imgs, ref)
        _same_call(model, lambda x: (model.get_features(x, ex),), imgs, ref)
        _same_call(model, lambda x: (model.backbone_tokens(x).clone(),), imgs, ref)
        got = model.tokens_from_uint8(imgs).clone()
        assert torch.equal(got, model.tokens_from_uint8(ref).clone())
    finally:
        model.input_size = None


def test_graph_replay_with_other_sizes(model, sd, cuda_device):
    """Three lists of different sizes at one (B, S): eager call, graph capture, graph replay — each equal to the eager
    result of its own list, through the module and through the handle."""
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    B, S = 3, 224
    lists = [_list(B, S, seed=s) for s in (31, 32, 33)]
    ex = _exif(B)
    model.input_size = S
    graphs = model.use_cuda_graphs
    try:
        ring0 = _ring(model)
        model.use_cuda_graphs = False
        want = []
        for imgs in lists:
            _set_ring(model, ring0)
            torch.manual_seed(5)
            want.append([t.clone() for t in model.forward_with_guidance(imgs, ex, "center", return_attention=True)])
        model.use_cuda_graphs = True
        model._ws.pop((B, S), None)
        for imgs, w in zip(lists, want):
            _set_ring(model, ring0)
            torch.manual_seed(5)
            got = model.forward_with_guidance(imgs, ex, "center", return_attention=True)
            assert all(torch.equal(a, b) for a, b in zip(got, w))
        assert len(model._ws[(B, S)]["graphs"]) == 1
    finally:
        model.input_size = None
        model.use_cuda_graphs = graphs

    eager = NativeModel(sd, device=cuda_device, use_graph=False)
    graph = NativeModel(sd, device=cuda_device, use_graph=True)
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        for imgs in lists:
            torch.manual_seed(5)
            want = eager.forward_with_guidance(imgs, ex, "center", S=S)
            with torch.cuda.stream(side):  # the legacy stream cannot be captured
                torch.manual_seed(5)
                got = graph.forward_with_guidance(imgs, ex, "center", S=S)
            side.synchronize()
            assert all(torch.equal(a, b) for a, b in zip(got, want))
    finally:
        eager.close()
        graph.close()


def test_handle_list_equals_stacked_u8(sd, cuda_device):
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    B, S = 5, 224
    imgs = _list(B, S, seed=41)
    ref = _stack_resized(imgs, S)
    ex = _exif(B)
    nm = NativeModel(sd, device=cuda_device, use_graph=False)
    try:
        calls = (lambda x, **k: nm.forward_with_guidance(x, ex, "bottom-right", **k),
                 lambda x, **k: nm.forward_with_guidance_sweep(x, ex, list(orc.INSTRUCTIONS), **k),
                 lambda x, **k: nm.forward(x, ex, runs=2, **k),
                 lambda x, **k: (nm.backbone_tokens(x, **k),))
        for fn in calls:
            torch.manual_seed(3)
            want = [t.clone() for t in fn(ref)]
            torch.manual_seed(3)
            got = fn(imgs, S=S)
            assert all(torch.equal(a, b) for a, b in zip(got, want))
        with pytest.raises(ValueError):
            nm.forward(imgs, ex)  # a list needs S
    finally:
        nm.close()


def _jpeg(arr):
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(arr).save(buf, format="JPEG", quality=90)
    return buf.getvalue()


def test_preprocess_jpeg_unchanged_and_launches_independent_of_sizes(model):
    from cognitive_aim_depth_estimation_b200 import ops
    S = 224
    rng = np.random.default_rng(2)
    mixed = [_jpeg(rng.integers(0, 256, hw + (3,), dtype=np.uint8))
             for hw in ((480, 640), (300, 200), (480, 640), (517, 389), (300, 200))]
    same = [_jpeg(rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)) for _ in range(5)]
    counts = []
    for files in (mixed, same):
        n0 = ops.launch_count()
        got = model.preprocess_jpeg(files, S)
        counts.append(ops.launch_count() - n0)
        imgs = ops.jpeg_decode_batch(files)
        want = torch.cat([model.preprocess(t[None], S) for t in imgs])  # one image at a time
        assert torch.equal(got, want)
    assert counts[0] == counts[1] == 3  # one batched decode, the two resize passes


def test_predict_batch(sd, cuda_device):
    from cognitive_aim_depth_estimation_b200 import ops
    spec = importlib.util.spec_from_file_location(
        "predict_like_demo", os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "predict_like_demo.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    p = mod.Predictor(sd, image_size=224)
    rng = np.random.default_rng(9)
    files = [_jpeg(rng.integers(0, 256, hw + (3,), dtype=np.uint8)) for hw in ((240, 320), (517, 389), (64, 48))]
    ins = ["top-left", "center", "bottom-right"]
    ring0 = _ring(p.model)
    torch.manual_seed(0)
    got = p.predict_batch(files, ins)
    # the same photographs resized one by one, stacked, through the uniform uint8 path in one call
    _set_ring(p.model, ring0)
    torch.manual_seed(0)
    x = torch.cat([ops.resize_u8(t[None].contiguous(), 224, 224) for t in ops.jpeg_decode_batch(files)])
    depth, conf, heat = p.model.forward_with_guidance(x, p.default_exif(3), ins, return_attention=True)
    for i, (d, c, meta) in enumerate(got):
        assert d == float(depth[i]) and c == float(conf[i])
        cell = int(heat[i].argmax())
        assert meta["attention_cell"] == (cell // 16, cell % 16) and meta["instruction"] == ins[i]
    # per-file predict (demo.py's loop): its own per-call projection changes depth, not the attention
    for f, one, (_, _, meta) in zip(files, ins, got):
        assert p.predict(f, one)[2]["attention_cell"] == meta["attention_cell"]


def test_list_argument_errors(model, cuda_device):
    """Bad lists raise ValueError before anything is drawn or launched: generator and ring buffer untouched."""
    ok = [torch.zeros(60, 80, 3, dtype=torch.uint8, device=cuda_device) for _ in range(2)]
    ex = _exif(2)
    bad = [
        (None, ok, "center"),                                                                  # no input_size
        (224, [ok[0], torch.zeros(60, 80, 3, device=cuda_device)], "center"),                  # float element
        (224, [ok[0], torch.zeros(60, 80, 4, dtype=torch.uint8, device=cuda_device)], "center"),  # 4 channels
        (224, [], "center"),                                                                   # empty list
        (224, ok, ["center", "left", "right"]),                                                # 3 instructions, 2 images
        (224, [ok[0], torch.zeros(4, MAX_SIDE + 1, 3, dtype=torch.uint8)], "center"),          # beyond the limit
    ]
    ring0 = _ring(model)
    for S, imgs, ins in bad:
        model.input_size = S
        try:
            torch.manual_seed(1)
            state = torch.get_rng_state()
            with pytest.raises(ValueError):
                model.forward_with_guidance(imgs, ex, ins)
            assert torch.equal(torch.get_rng_state(), state)
            ring = _ring(model)
            assert torch.equal(ring[0], ring0[0]) and torch.equal(ring[1], ring0[1])
        finally:
            model.input_size = None
    model.input_size = 224
    try:
        with pytest.raises(ValueError):
            model.forward_with_guidance(ok, _exif(3), "center")  # EXIF for three images
    finally:
        model.input_size = None
