"""Host side of depth fields without a device: the focus-mask family the field is defined by, what `depth_field` draws
from the global generator, its refusals (all before any draw), and the exported entry points."""
import ctypes

import pytest
import torch
import torch.nn as nn

from cognitive_aim_depth_estimation_b200 import _lib, tables
from cognitive_aim_depth_estimation_b200.model import Scene, create_model

CFG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}
OFF_CENTRE = ("left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right")


class _Stop(Exception):
    pass


def _stop(*a, **k):
    raise _Stop()


@pytest.fixture()
def model():
    return create_model(CFG, {"num_cameras": 71})


def _scene(model, B=2, S=224, device="cpu"):
    g = S // 14
    z = dict(device=device)
    return Scene(model, B, S, torch.zeros(B, g * g + 1, 768, **z), torch.zeros(B, g * g, **z), torch.zeros(B, 3, **z),
                 torch.zeros(B, dtype=torch.long, **z))


@pytest.mark.parametrize("g", range(4, 91))
def test_focus_mask_is_the_instruction_mask_at_the_instruction_cells(g):
    for name in OFF_CENTRE:
        y, x = tables.focus_cell(name, g)
        assert torch.equal(tables.focus_mask(y, x, g), tables.instruction_mask(name, g)), (g, name)
    assert tables.focus_cell("center", g) is None


@pytest.mark.parametrize("g", [5, 16, 37, 74, 90])
def test_focus_mask_is_the_integer_disk(g):
    """The table's fp64 sqrt(dy^2 + dx^2) <= r is exactly the integer test dy^2 + dx^2 <= r^2 the kernel uses."""
    r = max(1, g // 6)
    yy, xx = torch.meshgrid(torch.arange(g), torch.arange(g), indexing="ij")
    for y, x in [(0, 0), (g - 1, g // 3), (g // 2, g // 2), (g // 4, g - 1)]:
        d2 = (yy - y) ** 2 + (xx - x) ** 2
        want = torch.where(d2 <= r * r, 5.0, torch.where(d2 <= 4 * r * r, 2.0, 1.0)).flatten()
        assert torch.equal(tables.focus_mask(y, x, g), want)
    with pytest.raises(ValueError):
        tables.focus_mask(g, 0, g)


@pytest.mark.parametrize("B", [1, 3])
def test_depth_field_draws_what_guide_draws(model, monkeypatch, B):
    """randn(B, 192), randn(B, 768), then nn.Linear(768, 64): one guide call's draws, in its order."""
    torch.manual_seed(7)
    torch.randn(B, 192), torch.randn(B, 768)
    nn.Linear(768, 64)
    want = torch.get_rng_state()
    monkeypatch.setattr(model, "_pack", lambda: {"heads": None})
    monkeypatch.setattr(model, "_mask", lambda gd, g: torch.zeros(g * g))
    monkeypatch.setattr(model, "_scene_ws", _stop)
    torch.manual_seed(7)
    with pytest.raises(_Stop):
        model.guide(_scene(model, B), "left")
    assert torch.equal(torch.get_rng_state(), want)
    torch.manual_seed(7)
    with pytest.raises(_Stop):
        model.depth_field(_scene(model, B))
    assert torch.equal(torch.get_rng_state(), want)


def test_refusals_happen_before_any_draw(model, monkeypatch):
    monkeypatch.setattr(model, "_pack", lambda: {"heads": None})
    monkeypatch.setattr(model, "_scene_ws", _stop)
    other = create_model(CFG, {"num_cameras": 71})
    stale = _scene(model)
    model._weights_version += 1
    torch.manual_seed(3)
    state = torch.get_rng_state()
    for scene, match in ((stale, "stale"), (_scene(other), "another model"), (_scene(model, device="meta"), "lives on"),
                         ("not a scene", "Scene")):
        with pytest.raises(ValueError, match=match):
            model.depth_field(scene)
        assert torch.equal(torch.get_rng_state(), state), match


def test_library_exports_the_field_entry_points():
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in ("ca_depth_field", "ca_token_project", "ca_depth_field_cells"):
        assert hasattr(lib, name), name
        assert name in _lib.exported_symbols()
