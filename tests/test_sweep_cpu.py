"""Host side of the instruction sweep (`forward_with_guidance_sweep`) without a device: the random draws of K guided
calls and the argument checks, which all happen before anything is launched."""
import pytest
import torch
import torch.nn as nn

from cognitive_aim_depth_estimation_b200.model import create_model

CFG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}


@pytest.fixture(scope="module")
def model():
    return create_model(CFG, {"num_cameras": 71})


def _exif(B):
    return {"focal_length": torch.full((B,), 50.0), "aperture": torch.full((B,), 2.8), "iso": torch.full((B,), 100.0),
            "camera_idx": torch.zeros(B, dtype=torch.long)}


@pytest.mark.parametrize("B,K", [(1, 9), (3, 1), (2, 16)])
def test_sweep_draws_equal_successive_calls(model, B, K):
    """The draws of a K-sweep are those of K successive guided calls (src/model.py:609, 744, then the nn.Linear(768, 64)
    of :1421, per call, as oracle/cogaim_oracle.py forward_with_guidance makes them), and the generator ends where
    those K calls leave it."""
    torch.manual_seed(11)
    want = []
    for _ in range(K):
        eps, noise = torch.randn(B, 192), torch.randn(B, 768)
        tmp = nn.Linear(768, 64)
        want.append((eps, noise, tmp.weight.detach(), tmp.bias.detach()))
    state = torch.get_rng_state()
    torch.manual_seed(11)
    got = model._sweep_draws(B, K)
    assert torch.equal(torch.get_rng_state(), state)
    assert len(got) == K
    for w, g in zip(want, got):
        for a, b in zip(w, g):
            assert torch.equal(a, b)


def test_sweep_draws_follow_the_sharded_replay(model):
    """With `rng_replay_batch` set (a shard of a larger batch) each call draws at the global batch size and keeps this
    shard's rows, as `forward_with_guidance` does."""
    torch.manual_seed(3)
    full = model._sweep_draws(8, 3)
    state = torch.get_rng_state()
    model.rng_replay_batch, model.rng_replay_offset = 8, 5
    try:
        torch.manual_seed(3)
        part = model._sweep_draws(3, 3)
    finally:
        model.rng_replay_batch, model.rng_replay_offset = None, 0
    assert torch.equal(torch.get_rng_state(), state)
    for f, p in zip(full, part):
        assert torch.equal(f[0][5:8], p[0]) and torch.equal(f[1][5:8], p[1])
        assert torch.equal(f[2], p[2]) and torch.equal(f[3], p[3])


@pytest.mark.parametrize("guidances,exif", [
    ([], True),                                       # K = 0
    (["center"] * 17, True),                          # K above the cap of 16
    (["center", None], True),                         # None: the un-guided focal path, not a sweep
    (["center"], False),                              # no EXIF: the reference falls back to forward()
    ("center", True),                                 # not a list
])
def test_sweep_rejects_bad_arguments_before_drawing(model, guidances, exif):
    x = torch.zeros(2, 3, 56, 56)
    torch.manual_seed(5)
    state = torch.get_rng_state()
    with pytest.raises(ValueError):
        model.forward_with_guidance_sweep(x, _exif(2) if exif else None, guidances)
    assert torch.equal(torch.get_rng_state(), state)


def test_sweep_needs_the_exif_prior():
    m = create_model({"cognitive_modules": ["ambient_stream", "iterative_focal_stream"]}, {"num_cameras": 71})
    with pytest.raises(ValueError):
        m.forward_with_guidance_sweep(torch.zeros(1, 3, 56, 56), _exif(1), ["center"])


def test_sweep_has_no_cpu_fallback(model):
    with pytest.raises(RuntimeError):
        model.forward_with_guidance_sweep(torch.zeros(1, 3, 56, 56), _exif(1), ["center", "left"])
