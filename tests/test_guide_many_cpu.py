"""Host side of `guide_many` without a device: the exported symbols, the caps shared by the header and the binding, what
one call draws from the global generator, and the argument checks, which all happen before anything is drawn."""
import re
from pathlib import Path

import pytest
import torch
import torch.nn as nn

from cognitive_aim_depth_estimation_b200 import _lib
from cognitive_aim_depth_estimation_b200.model import Scene, create_model

CFG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"]}
HEADER = Path(__file__).resolve().parent.parent / "include" / "cogaim_b200.h"


class _Stop(Exception):
    pass


def _stop(*a, **k):
    raise _Stop()


@pytest.fixture()
def model():
    return create_model(CFG, {"num_cameras": 71})


def _scene(model, B=2, S=224):
    g = S // 14
    return Scene(model, B, S, torch.zeros(B, g * g + 1, 768), torch.zeros(B, g * g), torch.zeros(B, 3),
                 torch.zeros(B, dtype=torch.long))


def test_exported_symbols():
    for name in ("ca_gather_rows", "ca_weighted_pool_rows"):
        assert name in _lib.exported_symbols()
        assert re.search(rf"\bint {name}\(", HEADER.read_text())


def test_header_and_binding_caps_agree():
    text = HEADER.read_text()
    for name, value in (("CA_GUIDE_MANY_MAX_CALLS", _lib.GUIDE_MANY_MAX_CALLS),
                        ("CA_GUIDE_MANY_MAX_ROWS", _lib.GUIDE_MANY_MAX_ROWS)):
        m = re.search(rf"#define {name} (\d+)", text)
        assert m and int(m.group(1)) == value, name
    # ca_guide_many_row: four pointers and a long long, no padding
    body = re.search(r"typedef struct ca_guide_many_row \{(.*?)\} ca_guide_many_row;", text, re.S).group(1)
    assert len(re.findall(r";", body)) == _lib.GUIDE_MANY_ROW_WORDS
    assert [f[0] for f in _lib.HeadsInputs._fields_][-1] == "call_of_row"


def test_draws_are_the_guide_loop_draws(model, monkeypatch):
    """For each call in order: randn(B_j, 192), randn(B_j, 768), then nn.Linear(768, 64)."""
    sizes = (1, 3, 2)
    torch.manual_seed(7)
    for B in sizes:
        torch.randn(B, 192), torch.randn(B, 768)
        nn.Linear(768, 64)
    want = torch.get_rng_state()
    monkeypatch.setattr(model, "_pack", lambda: {"heads": None})
    monkeypatch.setattr(model, "_mask", lambda gd, g: torch.zeros(g * g))
    monkeypatch.setattr(model, "_many_buffers", _stop)
    torch.manual_seed(7)
    with pytest.raises(_Stop):
        model.guide_many([_scene(model, B) for B in sizes], ["center", "left", "top"])
    assert torch.equal(torch.get_rng_state(), want)


def _assert_no_draw(fn, match):
    torch.manual_seed(1)
    state = torch.get_rng_state()
    with pytest.raises(ValueError, match=match):
        fn()
    assert torch.equal(torch.get_rng_state(), state)


def test_refusals_come_before_any_draw(model):
    a, b = _scene(model, 2), _scene(model, 1)
    other = create_model(CFG, {"num_cameras": 71})
    foreign = _scene(other, 1)
    wide = _scene(model, 1, 518)
    away = _scene(model, 1)
    away.device = torch.device("cuda", 0)
    stale = _scene(model, 1)
    many = _lib.GUIDE_MANY_MAX_CALLS + 1
    big = _scene(model, _lib.GUIDE_MANY_MAX_ROWS // 2 + 1)
    g = model.guide_many
    _assert_no_draw(lambda: g(a, ["left"]), "list")
    _assert_no_draw(lambda: g([a], "left"), "list")
    _assert_no_draw(lambda: g([], []), "m >= 1")
    _assert_no_draw(lambda: g([a, b], ["left"]), "one guidance")
    _assert_no_draw(lambda: g([a, b], ["left", None]), "None")
    _assert_no_draw(lambda: g([a, "scene"], ["left", "top"]), "Scene")
    _assert_no_draw(lambda: g([a, foreign], ["left", "top"]), "another model")
    _assert_no_draw(lambda: g([a, away], ["left", "top"]), "lives on")
    _assert_no_draw(lambda: g([a, wide], ["left", "top"]), "share the image side")
    _assert_no_draw(lambda: g([a, b], [["left"], "top"]), "per-image")
    _assert_no_draw(lambda: g([a, b], ["left", "sideways"]), "unknown instruction")
    _assert_no_draw(lambda: g([a, b], [["left", "up"], "top"]), "unknown instruction")
    _assert_no_draw(lambda: g([b] * many, ["left"] * many), "at most")
    _assert_no_draw(lambda: g([big, big], ["left", "top"]), "at most")
    model.load_state_dict(model.state_dict())
    _assert_no_draw(lambda: g([a, stale], ["left", "top"]), "stale")
