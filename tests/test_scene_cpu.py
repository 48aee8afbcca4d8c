"""Host side of scenes (`encode` / `guide` / `guide_sweep`) without a device: what each call draws from the global
generator, and the argument checks, which all happen before anything is drawn or launched."""
import pytest
import torch
import torch.nn as nn

from cognitive_aim_depth_estimation_b200.model import Scene, create_model

CFG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}


class _Stop(Exception):
    pass


def _stop(*a, **k):
    raise _Stop()


@pytest.fixture()
def model():
    return create_model(CFG, {"num_cameras": 71})


def _exif(B):
    return {"focal_length": torch.full((B,), 50.0), "aperture": torch.full((B,), 2.8), "iso": torch.full((B,), 100.0),
            "camera_idx": torch.zeros(B, dtype=torch.long)}


def _scene(model, B=2, S=224):
    """A scene as encode builds it, on the model's (CPU) device: enough for the host-side checks."""
    g = S // 14
    return Scene(model, B, S, torch.zeros(B, g * g + 1, 768), torch.zeros(B, g * g), torch.zeros(B, 3),
                 torch.zeros(B, dtype=torch.long))


def _stub_device_work(model, monkeypatch, stop_at):
    """Stand-ins for the packing and mask tables (device work), and a stop right after the random draws."""
    monkeypatch.setattr(model, "_pack", lambda: {"heads": None})
    monkeypatch.setattr(model, "_mask", lambda gd, g: torch.zeros(g * g))
    monkeypatch.setattr(model, stop_at, _stop)


def test_encode_draws_nothing(model, monkeypatch):
    _stub_device_work(model, monkeypatch, "_workspace")
    torch.manual_seed(5)
    state = torch.get_rng_state()
    with pytest.raises(_Stop):
        model.encode(torch.zeros(2, 3, 224, 224), _exif(2))
    assert torch.equal(torch.get_rng_state(), state)


@pytest.mark.parametrize("B", [1, 3])
def test_guide_draws_what_forward_with_guidance_draws(model, monkeypatch, B):
    """randn(B, 192), randn(B, 768), then nn.Linear(768, 64) — the draws of one forward_with_guidance, in its order."""
    torch.manual_seed(7)
    eps, noise = torch.randn(B, 192), torch.randn(B, 768)
    tmp = nn.Linear(768, 64)
    want = torch.get_rng_state()

    _stub_device_work(model, monkeypatch, "_workspace")
    torch.manual_seed(7)
    with pytest.raises(_Stop):
        model.forward_with_guidance(torch.zeros(B, 3, 224, 224), _exif(B), "center")
    assert torch.equal(torch.get_rng_state(), want)

    monkeypatch.setattr(model, "_scene_ws", _stop)
    torch.manual_seed(7)
    with pytest.raises(_Stop):
        model.guide(_scene(model, B), "center")
    assert torch.equal(torch.get_rng_state(), want)
    assert eps.shape == (B, 192) and noise.shape == (B, 768) and tmp.weight.shape == (64, 768)


def test_guide_sweep_draws_what_the_sweep_draws(model, monkeypatch):
    monkeypatch.setattr(model, "_pack", lambda: {"heads": None})
    monkeypatch.setattr(model, "_mask", lambda gd, g: torch.zeros(g * g))
    monkeypatch.setattr(model, "_scene_ws", lambda scene: ({}, {}))
    monkeypatch.setattr(model, "_sweep_buffers", _stop)
    torch.manual_seed(9)
    model._sweep_draws(2, 3)
    want = torch.get_rng_state()
    torch.manual_seed(9)
    with pytest.raises(_Stop):
        model.guide_sweep(_scene(model, 2), ["center", "left", "top"])
    assert torch.equal(torch.get_rng_state(), want)


def _assert_no_draw(fn):
    torch.manual_seed(1)
    state = torch.get_rng_state()
    with pytest.raises(ValueError):
        fn()
    assert torch.equal(torch.get_rng_state(), state)


def test_argument_errors_come_before_any_draw(model):
    scene = _scene(model, 2)
    x = torch.zeros(2, 3, 224, 224)
    _assert_no_draw(lambda: model.encode(x, None))                      # no EXIF
    _assert_no_draw(lambda: model.guide(scene, None))                   # None guidance
    _assert_no_draw(lambda: model.guide(scene, ["center"]))             # per-image list of the wrong length
    _assert_no_draw(lambda: model.guide("not a scene", "center"))
    _assert_no_draw(lambda: model.guide_sweep(scene, ["center", None]))
    _assert_no_draw(lambda: model.guide_sweep(scene, []))
    _assert_no_draw(lambda: model.guide_sweep(scene, [["center"] * 3]))
    _assert_no_draw(lambda: model.encode(x, {"focal_length": torch.zeros(3), "aperture": torch.zeros(3),
                                             "iso": torch.zeros(3), "camera_idx": torch.zeros(3, dtype=torch.long)}))


def test_model_without_exif_prior_refuses_to_encode():
    m = create_model({"cognitive_modules": ["ambient_stream", "iterative_focal_stream"]}, {"num_cameras": 71})
    _assert_no_draw(lambda: m.encode(torch.zeros(1, 3, 224, 224), _exif(1)))


def test_scene_of_another_model_or_stale_weights_is_refused(model):
    other = create_model(CFG, {"num_cameras": 71})
    _assert_no_draw(lambda: other.guide(_scene(model), "center"))
    scene = _scene(model)
    model.load_state_dict(model.state_dict())
    _assert_no_draw(lambda: model.guide(scene, "center"))
    _assert_no_draw(lambda: model.guide_sweep(scene, ["center"]))


def test_scene_on_another_device_is_refused(model):
    scene = _scene(model)
    scene.device = torch.device("cuda", 0)
    _assert_no_draw(lambda: model.guide(scene, "center"))
