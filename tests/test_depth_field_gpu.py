"""Depth fields (`model.depth_field(scene)`): cell (y, x) is the guided call with `tables.focus_mask(y, x, g)` from the
same draws, within |d| <= 1e-5 + 1e-4 |guide| for depth and confidence; one field draws and mutates what one guide
call does; eager, captured and replayed fields agree bit for bit; the kernels (`ops.token_project`,
`ops.depth_field_cells`) agree with a float64 restatement that takes the softmax over all N cells."""
import pytest
import torch

from cognitive_aim_depth_estimation_b200 import ops, tables
from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu

CFG = {"model": {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}}
CFG_GUIDED = dict(CFG, curiosity_guided_attention={"enabled": True})
ATOL, RTOL = 1e-5, 1e-4
OFF_CENTRE = [i for i in orc.INSTRUCTIONS if i != "center"]


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


def _assert_close(got, want, what):
    d = (got - want).abs()
    bad = d > ATOL + RTOL * want.abs()
    assert not bad.any(), f"{what}: {int(bad.sum())} cells outside tolerance, max |d| {d.max().item():.3e}"


def _field(m, scene, ring, seed):
    _set_ring(m, ring)
    torch.manual_seed(seed)
    d, c = m.depth_field(scene)
    return d.flatten(1), c.flatten(1)


def _guide_cells(m, scene, ring, seed, cells):
    """guide(scene, focus_mask(c)) for each cell c, each from the same ring and seed: depth, conf [B, len(cells)]."""
    g = scene.S // 14
    ds, cs = [], []
    for c in cells:
        _set_ring(m, ring)
        torch.manual_seed(seed)
        d, cf = m.guide(scene, tables.focus_mask(c // g, c % g, g))
        ds.append(d[:, 0])
        cs.append(cf[:, 0])
    return torch.stack(ds, 1), torch.stack(cs, 1)


def _cell_sample(g, n, seed):
    """n seeded cells plus the corners, the border midpoints and the eight instruction cells."""
    must = {(0, 0), (0, g - 1), (g - 1, 0), (g - 1, g - 1), (0, g // 2), (g // 2, 0), (g - 1, g // 2), (g // 2, g - 1)}
    must |= {tables.focus_cell(i, g) for i in OFF_CENTRE}
    cells = {y * g + x for y, x in must}
    perm = torch.randperm(g * g, generator=torch.Generator().manual_seed(seed)).tolist()
    for c in perm:
        if len(cells) >= n + len(must):
            break
        cells.add(c)
    return sorted(cells)


@pytest.mark.parametrize("S,B,sample", [(224, 1, None), (518, 1, None), (224, 4, None), (518, 32, 256), (1036, 1, 256)])
def test_field_equals_guide_cell_by_cell(model, S, B, sample):
    g = S // 14
    x, ex = orc.synthetic_images(B, S, seed=S + B).cuda(), _exif(orc.synthetic_exif(B, seed=B))
    scene = model.encode(x, ex)
    ring = _ring(model)
    depth, conf = _field(model, scene, ring, 17)
    cells = list(range(g * g)) if sample is None else _cell_sample(g, sample, S)
    want_d, want_c = _guide_cells(model, scene, ring, 17, cells)
    _assert_close(depth[:, cells], want_d, "depth")
    _assert_close(conf[:, cells], want_c, "confidence")


@pytest.mark.parametrize("S", [224, 518, 1036])
def test_instruction_cells_are_the_instruction_predictions(model, S):
    B, g = 2, S // 14
    x, ex = orc.synthetic_images(B, S, seed=3).cuda(), _exif(orc.synthetic_exif(B, seed=4))
    scene = model.encode(x, ex)
    ring = _ring(model)
    depth, conf = _field(model, scene, ring, 23)
    depth, conf = depth.view(B, g, g), conf.view(B, g, g)
    for name in OFF_CENTRE:
        y, xx = tables.focus_cell(name, g)
        assert torch.equal(tables.focus_mask(y, xx, g), tables.instruction_mask(name, g))
        _set_ring(model, ring)
        torch.manual_seed(23)
        d, c = model.guide(scene, name)
        _assert_close(depth[:, y, xx], d[:, 0], f"{name} depth")
        _assert_close(conf[:, y, xx], c[:, 0], f"{name} confidence")


def test_state_after_a_field_is_the_state_after_one_guide(model):
    B = 3
    x, ex = orc.synthetic_images(B, 224, seed=30).cuda(), _exif(orc.synthetic_exif(B, seed=31))
    scene = model.encode(x, ex)
    model.curiosity_module.history_pointer.fill_(1000 - 2)  # the field's B entries wrap around the ring
    ring = _ring(model)
    torch.manual_seed(8)
    model.guide(scene, "bottom-left")
    torch.cuda.synchronize()
    want = (torch.get_rng_state(), _ring(model), model._last_curiosity.clone())
    model.guide(scene, "top")  # leaves _last_attention_weights / _last_argmax that the field must not touch
    last_att, last_arg = model._last_attention_weights.clone(), model._last_argmax.clone()
    _set_ring(model, ring)
    torch.manual_seed(8)
    model.depth_field(scene)
    torch.cuda.synchronize()
    assert torch.equal(torch.get_rng_state(), want[0]), "generator state"
    assert torch.equal(model.curiosity_module.exploration_history, want[1][0]), "ring buffer"
    assert torch.equal(model.curiosity_module.history_pointer, want[1][1]), "ring pointer"
    assert torch.equal(model._last_curiosity, want[2]), "_last_curiosity"
    assert torch.equal(model._last_attention_weights, last_att) and torch.equal(model._last_argmax, last_arg)


def test_eager_capture_and_replay_are_bit_identical(model):
    """The first field of a scene runs eagerly, the second captures a graph, later ones replay it; other forwards on
    the same (B, S) workspace in between change nothing."""
    B, S = 2, 518
    x, ex = orc.synthetic_images(B, S, seed=40).cuda(), _exif(orc.synthetic_exif(B, seed=41))
    y, ey = orc.synthetic_images(B, S, seed=42).cuda(), _exif(orc.synthetic_exif(B, seed=43))
    scene = model.encode(x, ex)
    ring = _ring(model)
    runs = []
    for i in range(4):
        if i >= 2:
            model.forward(y, ey)
            model.forward_with_guidance(y, ey, "right")
            other = model.encode(y, ey)
            model.guide(other, "left")
            model.guide(scene, "top")
        runs.append([t.clone() for t in _field(model, scene, ring, 5)])
    torch.cuda.synchronize()
    assert not model.use_cuda_graphs or any(k[0] == "field" for k in scene._graphs)
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
    assert not torch.isnan(runs[0][0]).any()


def test_curiosity_guided_configuration(cuda_device):
    """Each call's focal attention depends on its own curiosity score: the field reruns the focal iterations once."""
    m = _model(cuda_device, CFG_GUIDED, orc.build_state_dict(0, curiosity_guided=True))
    B, g = 2, 16
    x, ex = orc.synthetic_images(B, 224).cuda(), _exif(orc.synthetic_exif(B))
    scene = m.encode(x, ex)
    assert scene.base is None
    ring = _ring(m)
    depth, conf = _field(m, scene, ring, 13)
    cells = _cell_sample(g, 24, 1)
    want_d, want_c = _guide_cells(m, scene, ring, 13, cells)
    _assert_close(depth[:, cells], want_d, "depth")
    _assert_close(conf[:, cells], want_c, "confidence")


def test_field_matches_the_oracle(model, sd):
    """8 cells (corners included) against the oracle's guided call with the cell's focus mask, from the same seed
    (README bar: depth abs-rel 1e-2, confidence max-abs 1e-2)."""
    B, S, g = 2, 224, 16
    x, ex = orc.synthetic_images(B, S, seed=21), orc.synthetic_exif(B, seed=22)
    tokens = orc.dinov2_tokens(sd, x)
    scene = model.encode(x.cuda(), _exif(ex))
    torch.manual_seed(11)
    depth, conf = (t.cpu().flatten(1) for t in model.depth_field(scene))
    for c in (0, g - 1, g * (g - 1), g * g - 1, 5 * g + 7, 9 * g + 2, 12 * g + 12, 3 * g + 14):
        torch.manual_seed(11)
        ref = orc.forward_with_guidance(sd, None, ex, tables.focus_mask(c // g, c % g, g), tokens=tokens,
                                        update_history=False)
        assert ((depth[:, c] - ref["depth"][:, 0]).abs() / ref["depth"][:, 0].abs()).max().item() <= 1e-2, c
        assert (conf[:, c] - ref["confidence"][:, 0]).abs().max().item() <= 1e-2, c


def _focus_masks(g):
    """[N, N] float64: row c is tables.focus_mask at cell c."""
    yy, xx = torch.meshgrid(torch.arange(g), torch.arange(g), indexing="ij")
    yy, xx = yy.flatten(), xx.flatten()
    d2 = (yy[:, None] - yy[None, :]) ** 2 + (xx[:, None] - xx[None, :]) ** 2
    r = max(1, g // 6)
    m = torch.ones(g * g, g * g, dtype=torch.float64)
    m[d2 <= 4 * r * r] = 2.0
    m[d2 <= r * r] = 5.0
    return m


@pytest.mark.parametrize("g", [5, 16, 37, 74])
def test_kernels_against_a_full_softmax_restatement(model, sd, g):
    """ops.token_project and ops.depth_field_cells against float64 torch with the softmax over all N cells (no
    truncation), NaN-filled scratch and outputs, and a base with one cell near 1."""
    dev = torch.device("cuda")
    B, N = 2, g * g
    gen = torch.Generator().manual_seed(g)
    tokens = torch.randn(B, N + 1, 768, generator=gen)
    tmp_w = torch.randn(64, 768, generator=gen) / 768 ** 0.5
    tmp_b = torch.randn(64, generator=gen) * 0.1
    base = torch.rand(B, N, generator=gen)
    base = base / base.sum(1, keepdim=True)
    base[1] = 1e-6
    base[1, N // 3] = 1.0 - 1e-6 * (N - 1)  # one cell near 1
    ex = orc.synthetic_exif(B, seed=g)
    exif = torch.stack([ex["focal_length"], ex["aperture"], ex["iso"]], 1).float()
    cam = ex["camera_idx"].long().reshape(-1)
    nan = lambda *s: torch.full(s, float("nan"), device=dev)  # noqa: E731
    P, cst, depth, conf = nan(B, N, 64), nan(B, 192), nan(B, N), nan(B, N)
    tok, w, b = tokens.to(dev), tmp_w.to(dev), tmp_b.to(dev)
    pk = model._pack()
    ops.token_project(tok, (N + 1) * 768, 1, w, P, B, N)
    ops.depth_field_cells(pk["heads"], base=base.to(dev), P=P, cst=cst, depth=depth, conf=conf, tokens=tok, tmp_b=b,
                          B=B, g=g, exif=exif.to(dev), camera_idx=cam.to(dev), num_cameras=71,
                          fault_ptr=model._fault_word().data_ptr())
    torch.cuda.synchronize()

    t64 = tokens.double().to(dev)
    P64 = t64[:, 1:] @ tmp_w.double().to(dev).T
    assert torch.allclose(P.double(), P64, rtol=1e-4, atol=1e-5), (P.double() - P64).abs().max()
    sd64 = {k: (v.double().to(dev) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    ex64 = {k: (v.double().to(dev) if v.is_floating_point() else v.to(dev)) for k, v in ex.items()}
    amb = orc.ambient_stream(sd64, t64[:, 0])
    ep = orc.exif_prior(sd64, ex64)
    masks = _focus_masks(g).to(dev)
    for c in (0, N - 1, N // 2):
        assert torch.equal(masks[c].float().cpu(), tables.focus_mask(c // g, c % g, g))
    for i in range(B):
        wts = torch.softmax((0.7 * masks + 0.3 * base[i].double().to(dev)) / 0.05, dim=-1)  # [cells, N]
        feat = wts @ P64[i] + tmp_b.double().to(dev)
        cat = torch.cat([amb[i].expand(N, -1), feat, ep[i].expand(N, -1)], 1)
        d64, c64, _ = orc.heads(sd64, cat)
        _assert_close(depth[i].double(), d64[:, 0], f"depth, image {i}")
        _assert_close(conf[i].double(), c64[:, 0], f"confidence, image {i}")


def test_native_field_and_refusals(cuda_device, sd, model):
    import ctypes as C
    from cognitive_aim_depth_estimation_b200._lib import CogAimError
    from cognitive_aim_depth_estimation_b200.native import NativeModel, NativeScene
    nat = NativeModel(sd, device=cuda_device, fold_layernorm=model._ln_folded())
    B, S = 2, 518
    x, ex = orc.synthetic_images(B, S, seed=60).cuda(), _exif(orc.synthetic_exif(B, seed=61))
    scene = nat.encode(x, ex)
    runs = []
    for _ in range(3):  # eager, captured, replayed
        torch.manual_seed(3)
        runs.append([t.clone() for t in nat.depth_field(scene)])
    torch.cuda.synchronize()
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
    # the handle builds its focal tables on the host (C++ sinf / expf): the model agrees to that rounding
    torch.manual_seed(3)
    want = model.depth_field(model.encode(x, ex))
    for a, b in zip(runs[0], want):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6), (a - b).abs().max()
    stale = NativeScene(nat.lib, C.c_void_p(scene.ptr.value), scene.B, scene.S, scene.device)
    scene.close()
    try:
        with pytest.raises(CogAimError):
            nat.depth_field(stale)
    finally:
        stale.ptr = None
    other = nat.encode(x, ex)
    h = nat._h
    nat.close()
    nat._h = h  # the destroyed handle's address: its scenes are refused, not dereferenced
    with pytest.raises(CogAimError):
        nat.depth_field(other)
    nat._h = None
    other.close()  # a scene outlives its handle and is still released


def test_bad_device_camera_index_is_reported_by_the_next_call(cuda_device, sd):
    m = _model(cuda_device, CFG, sd)
    x, ex = orc.synthetic_images(1, 224).cuda(), _exif(orc.synthetic_exif(1))
    ex["camera_idx"] = torch.full_like(ex["camera_idx"], 500)
    scene = m.encode(x, ex)
    m.depth_field(scene)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="camera_idx"):
        m.depth_field(scene)


def test_stale_scene_is_refused_before_any_draw(cuda_device, sd):
    m = _model(cuda_device, CFG, sd)
    x, ex = orc.synthetic_images(1, 224).cuda(), _exif(orc.synthetic_exif(1))
    scene = m.encode(x, ex)
    m.depth_field(scene)
    other = _model(cuda_device, CFG, sd)  # create_model draws its random init: before the state is taken
    foreign = m.encode(x, ex)
    m.load_state_dict(sd)
    state = torch.get_rng_state()
    with pytest.raises(ValueError, match="stale"):
        m.depth_field(scene)
    assert torch.equal(torch.get_rng_state(), state)
    with pytest.raises(ValueError, match="another model"):
        other.depth_field(foreign)
    assert torch.equal(torch.get_rng_state(), state)


def test_example_saves_the_field(cuda_device, tmp_path):
    import subprocess
    import sys

    import numpy as np
    from PIL import Image
    path = tmp_path / "photo.jpg"
    Image.fromarray(np.random.default_rng(7).integers(0, 256, (240, 320, 3), dtype=np.uint8)).save(path, format="JPEG")
    out = tmp_path / "field.npz"
    root = __file__.rsplit("/tests/", 1)[0]
    env = dict(__import__("os").environ, PYTHONNOUSERSITE="1")
    res = subprocess.run([sys.executable, f"{root}/examples/predict_like_demo.py", str(path), "--depth-field", str(out)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stderr
    f = np.load(out)
    assert f["depth"].shape == (16, 16) and f["confidence"].shape == (16, 16)
    assert np.isfinite(f["depth"]).all() and np.isfinite(f["confidence"]).all()
