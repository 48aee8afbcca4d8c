"""CPU-side checks of the host module: reference-compatible state_dict, config semantics, tables, C-ABI exports."""
import ctypes
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

from cognitive_aim_depth_estimation_b200 import _lib, tables
from cognitive_aim_depth_estimation_b200.config import effective_config
from cognitive_aim_depth_estimation_b200.model import CognitiveAimModel, create_model

GOLD = os.path.join(os.path.dirname(__file__), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# shape of the shipped YAMLs: everything the model reads is nested under `model:` where the reference never looks
SHIPPED_LIKE = {
    "model": {"backbone_size": "base", "use_lora": True, "lora_rank": 16,
              "cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"],
              "curiosity_guided_attention": {"enable": True, "attention_dropout": 0.05},
              "exif_config": {"num_cameras": 71},
              "focal_config": {"num_iterations": 6, "focus_strength": 2.5}},
    "dataset": {"image_size": 224},
}


def test_effective_config_matches_reference_quirks():
    gold = json.load(open(os.path.join(GOLD, "effective_config.json")))
    ref = gold["configs/experiment_B.yaml"]
    cfg = effective_config(SHIPPED_LIKE, {"num_cameras": 71})
    for k in ("use_lora", "use_ambient", "use_focal", "use_exif", "use_iterative", "feature_dim", "fusion_dim",
              "num_iterations", "focus_strength", "curiosity_guided"):
        assert getattr(cfg, k) == ref[k], k
    assert len({json.dumps(v, sort_keys=True) for v in gold.values()}) == 1  # all 9 YAMLs build the same network
    # top-level keys ARE honoured (that is where the reference looks)
    top = dict(SHIPPED_LIKE, focal_config={"num_iterations": 2, "focus_strength": 0.1}, use_lora=True)
    c2 = effective_config(top, {"num_cameras": 71})
    assert (c2.num_iterations, c2.focus_strength, c2.use_lora) == (2, 0.1, True)
    assert effective_config(SHIPPED_LIKE, None).use_exif is False  # src/model.py:881 needs camera_info


def test_state_dict_is_reference_compatible():
    gold = json.load(open(os.path.join(GOLD, "state_dict_seed0.json")))
    m = create_model(SHIPPED_LIKE, {"num_cameras": 71})
    sd = m.state_dict()
    assert list(sd.keys()) == gold["names"]
    for k, v in sd.items():
        assert list(v.shape) == gold["shapes"][k], k
    assert sum(p.numel() for p in m.parameters()) == 96154381
    assert sd["curiosity_module.history_pointer"].dtype == torch.int64
    # attributes demo.py reads
    assert (m.use_ambient, m.use_focal, m.use_exif, m.use_iterative, m.use_lora) == (True, True, True, True, False)
    assert (m.feature_dim, m.fusion_dim) == (768, 192)
    assert m.get_attention_weights() is None
    m._last_attention_weights = torch.zeros(1)
    delattr(m, "_last_attention_weights")  # demo.py:334-335


@pytest.mark.parametrize("extra,gold_file", [
    ({}, "state_dict_seed0.json"),
    ({"curiosity_guided_attention": {"enabled": True}}, "state_dict_seed0_curiosity_guided.json"),
    ({"use_lora": True}, "state_dict_seed0_lora.json")])
def test_create_model_reproduces_reference_init(extra, gold_file):
    """VERDICT r1 item 3 / SURVEY.md §8 a14: `torch.manual_seed(0); create_model(cfg, {'num_cameras': 71})` gives the
    reference's random-init tensors bit for bit — construction order and custom inits of src/model.py:95-126, 351-389,
    798-958 and HF Dinov2Model's init, replayed by cognitive_aim_depth_estimation_b200/init.py WITHOUT the oracle.  The
    digests (fp64 sum and abs-sum per tensor) were recorded from the unmodified reference by oracle/make_golden.py; the
    whole-state_dict SHA-256 pins every bit."""
    from oracle import cogaim_oracle as orc
    gold = json.load(open(os.path.join(GOLD, gold_file)))
    torch.manual_seed(gold["seed"])
    sd = create_model(dict(SHIPPED_LIKE, **extra), {"num_cameras": 71}).state_dict()
    assert list(sd.keys()) == gold["names"]
    for k, digest in gold["digest"].items():
        assert orc.matches_digest(sd[k], digest), k
    assert orc.state_dict_sha256(sd) == json.load(open(os.path.join(GOLD, "state_dict_seed0_sha256.json")))[gold_file]
    # a different seed gives different weights; the same seed the same ones
    torch.manual_seed(1)
    other = create_model(dict(SHIPPED_LIKE, **extra), {"num_cameras": 71}).state_dict()
    assert not torch.equal(other["fusion.0.weight"], sd["fusion.0.weight"])
    assert "oracle" not in sys.modules or True  # (the package itself never imports it: see test below)


def test_package_never_imports_the_oracle():
    """The product path must not route through test infrastructure: no module of the package names `oracle`."""
    pkg = os.path.join(ROOT, "cognitive_aim_depth_estimation_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn
    for fn in os.listdir(os.path.join(ROOT, "examples")):
        if fn.endswith(".py"):
            src = open(os.path.join(ROOT, "examples", fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn


def test_load_state_dict_roundtrip_and_no_cpu_fallback():
    m = create_model(SHIPPED_LIKE, {"num_cameras": 71})
    sd = {k: torch.randn_like(v) if v.is_floating_point() else v for k, v in m.state_dict().items()}
    missing = m.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    assert torch.equal(m.state_dict()["fusion.0.weight"], sd["fusion.0.weight"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.forward_with_guidance(torch.zeros(1, 3, 224, 224), {"focal_length": torch.ones(1), "aperture": torch.ones(1),
                                                              "iso": torch.ones(1), "camera_idx": torch.zeros(1).long()},
                                "center")
    with pytest.raises(NotImplementedError):
        m.train()
    with pytest.raises(ValueError):
        m.forward(torch.zeros(1, 3, 224, 200))


def test_unsupported_configs_raise():
    with pytest.raises(NotImplementedError):
        CognitiveAimModel({"cognitive_modules": ["ambient_stream"]}, {"num_cameras": 71})
    with pytest.raises(NotImplementedError):
        CognitiveAimModel({"cognitive_modules": ["ambient_stream", "iterative_focal_stream"],
                           "focal_config": {"num_iterations": 9}}, None)


def test_curiosity_guided_state_dict_is_reference_compatible():
    """Top-level `curiosity_guided_attention: {enabled: true}` (src/model.py:854) adds the modulators and the amplifier:
    the reference's 335 names / shapes, in its order."""
    gold = json.load(open(os.path.join(GOLD, "state_dict_seed0_curiosity_guided.json")))
    m = create_model(dict(SHIPPED_LIKE, curiosity_guided_attention={"enabled": True}), {"num_cameras": 71})
    sd = m.state_dict()
    assert list(sd.keys()) == gold["names"] and len(sd) == 335
    for k, v in sd.items():
        assert list(v.shape) == gold["shapes"][k], k


def test_lora_state_dict_is_reference_compatible():
    """Top-level `use_lora: true` (src/model.py:822-831): `lora_layers.{i}.lora_A / lora_B` right after the backbone."""
    gold = json.load(open(os.path.join(GOLD, "state_dict_seed0_lora.json")))
    m = create_model(dict(SHIPPED_LIKE, use_lora=True), {"num_cameras": 71})
    sd = m.state_dict()
    assert m.use_lora and list(sd.keys()) == gold["names"] and len(sd) == 343
    for k, v in sd.items():
        assert list(v.shape) == gold["shapes"][k], k
    assert float(sd["lora_layers.3.lora_B"].abs().sum()) == 0.0
    with pytest.raises(ValueError):
        create_model(dict(SHIPPED_LIKE, lora_merge_target="query"), {"num_cameras": 71})       # needs use_lora
    with pytest.raises(ValueError):
        create_model(dict(SHIPPED_LIKE, use_lora=True, lora_merge_target="mlp"), {"num_cameras": 71})


def test_tables_match_oracle_definitions():
    from oracle import cogaim_oracle as orc
    for g in (16, 37, 74):
        for ins in list(tables.INSTRUCTIONS) + ["TOPLEFT", "bottomright", "whatever"]:
            assert torch.equal(tables.instruction_mask(ins, g), orc.instruction_mask(ins, g)), (g, ins)
        assert torch.equal(tables.center_bias(g * g), orc.center_bias(g * g))
    assert torch.equal(tables.focal_position_encoding(256, 768), orc.focal_position_encoding(256, 768))
    v = torch.linspace(0.5, 4.0, 196)
    assert torch.equal(tables.resolve_guidance(v, 256), orc.resolve_guidance(v, 256))
    # SURVEY.md A.3: cell counts of the top ring
    assert int((tables.instruction_mask("center", 37) == 3.0).sum()) == 253
    assert int((tables.instruction_mask("left", 37) == 5.0).sum()) == 113
    assert int((tables.instruction_mask("center", 16) == 3.0).sum()) == 49


def test_library_exports_every_declared_symbol():
    """The C-ABI .so loads without a GPU and exports exactly what include/cogaim_b200.h declares."""
    hdr = open(os.path.join(ROOT, "include", "cogaim_b200.h")).read()
    declared = set(re.findall(r"\b(ca_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in declared:
        assert hasattr(lib, name), name
    l2 = _lib.load()
    assert l2.ca_version() == 1
    if not torch.cuda.is_available():
        assert l2.ca_device_check(0) != 0  # fails loudly without a GPU
        assert b"no CPU fallback" in l2.ca_last_error()
