"""Lists of differently sized photographs without a device: every bad list is refused with ValueError before the weights
are packed for a device and before anything is drawn from the global generator."""
import pytest
import torch

from cognitive_aim_depth_estimation_b200.model import create_model

CFG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}
OK = [torch.zeros(60, 80, 3, dtype=torch.uint8), torch.zeros(90, 50, 3, dtype=torch.uint8)]


@pytest.fixture(scope="module")
def model():
    return create_model(CFG, {"num_cameras": 71})


def _exif(B):
    return {"focal_length": torch.full((B,), 50.0), "aperture": torch.full((B,), 2.8), "iso": torch.full((B,), 100.0),
            "camera_idx": torch.zeros(B, dtype=torch.long)}


BAD = [
    ("no input_size", None, OK, "center", 2),
    ("float element", 224, [OK[0], torch.zeros(60, 80, 3)], "center", 2),
    ("4 channels", 224, [OK[0], torch.zeros(60, 80, 4, dtype=torch.uint8)], "center", 2),
    ("CHW element", 224, [OK[0], torch.zeros(3, 60, 80, dtype=torch.uint8)], "center", 2),
    ("empty list", 224, [], "center", 0),
    ("instructions", 224, OK, ["center", "left", "right"], 2),
    ("exif length", 224, OK, "center", 3),
    ("beyond the limit", 224, [OK[0], torch.zeros(4, 16385, 3, dtype=torch.uint8)], "center", 2),
    ("side not a multiple of 14", 230, OK, "center", 2),
]


@pytest.mark.parametrize("what,S,imgs,ins,n_exif", BAD, ids=[b[0] for b in BAD])
def test_list_errors_before_packing_or_drawing(model, what, S, imgs, ins, n_exif):
    model.input_size = S
    try:
        torch.manual_seed(5)
        state = torch.get_rng_state()
        calls = [lambda: model.forward_with_guidance(imgs, _exif(n_exif), ins),
                 lambda: model.forward_with_guidance_sweep(imgs, _exif(n_exif), [ins, "left"])]
        if what not in ("instructions", "exif length"):  # the un-guided entry points take no instruction, read no EXIF count
            calls += [lambda: model.forward(imgs, None), lambda: model.get_features(imgs),
                      lambda: model.backbone_tokens(imgs), lambda: model.tokens_from_uint8(imgs)]
        for call in calls:
            with pytest.raises(ValueError):
                call()
            assert model._packed is None
            assert torch.equal(torch.get_rng_state(), state)
    finally:
        model.input_size = None


def test_valid_list_reaches_the_device_check(model):
    """A well-formed list passes the checks and is then refused for want of a device (there is no CPU fallback)."""
    model.input_size = 224
    try:
        with pytest.raises(RuntimeError):
            model.forward_with_guidance(OK, _exif(2), "center")
    finally:
        model.input_size = None
