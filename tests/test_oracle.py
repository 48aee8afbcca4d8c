"""Pin the CPU oracle (oracle/cogaim_oracle.py) against outputs of the UNMODIFIED reference.

The fixtures in tests/golden/ were produced by oracle/make_golden.py, which imports /root/reference in the build
container.  These tests run on CPU (`-m "not gpu"`) and never touch /root/reference.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import cogaim_oracle as orc

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _assert_reference_init(sd, gold_file):
    """Digests recorded from the reference (up to fp64 summation order) and the state_dict's SHA-256 (every bit)."""
    gold = json.load(open(os.path.join(GOLD, gold_file)))
    assert list(sd.keys()) == gold["names"]
    for k, v in sd.items():
        assert list(v.shape) == gold["shapes"][k], k
        assert orc.matches_digest(v, gold["digest"][k]), k
    assert orc.state_dict_sha256(sd) == json.load(open(os.path.join(GOLD, "state_dict_seed0_sha256.json")))[gold_file]


@pytest.fixture(scope="module")
def sd():
    return orc.build_state_dict(0)


@pytest.fixture(scope="module")
def tokens224(sd):
    return orc.dinov2_tokens(sd, orc.synthetic_images(2, 224))


def test_state_dict_matches_reference_init(sd):
    """Same seed + same construction order => the reference's 319 tensors, bit for bit."""
    assert len(sd) == 319
    _assert_reference_init(sd, "state_dict_seed0.json")


def test_backbone_restated_vs_hf(sd, tokens224):
    gold = np.load(os.path.join(GOLD, "backbone.npz"))
    t = tokens224
    np.testing.assert_allclose(t[:, :8, :32].numpy(), gold["S224_B2_tokens_head"], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(t[:, -4:, -32:].numpy(), gold["S224_B2_tokens_tail"], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(t.norm(dim=-1).numpy(), gold["S224_B2_token_norms"], rtol=1e-5)


@pytest.mark.parametrize("instruction", orc.INSTRUCTIONS + ["TopLeft", "CENTER", "nonsense"])
def test_guided_224(sd, tokens224, instruction):
    gold = np.load(os.path.join(GOLD, "guided.npz"))
    torch.manual_seed(11)
    out = orc.forward_with_guidance(sd, None, orc.synthetic_exif(2), instruction, tokens=tokens224,
                                    update_history=False)
    key = f"S224_B2_{instruction}"
    np.testing.assert_allclose(out["depth"].numpy(), gold[key + "_depth"], rtol=2e-5)
    np.testing.assert_allclose(out["confidence"].numpy(), gold[key + "_conf"], rtol=1e-6)
    np.testing.assert_allclose(out["heatmap"].numpy(), gold[key + "_heat"], rtol=2e-3, atol=1e-9)
    assert (out["heatmap"].argmax(-1).numpy() == gold[key + "_heat"].argmax(-1)).all()


def test_guided_tensor_guidance_is_resized(sd, tokens224):
    gold = np.load(os.path.join(GOLD, "guided.npz"))
    torch.manual_seed(11)
    out = orc.forward_with_guidance(sd, None, orc.synthetic_exif(2), torch.linspace(0.5, 4.0, 196), tokens=tokens224,
                                    update_history=False)
    np.testing.assert_allclose(out["heatmap"].numpy(), gold["S224_B2_tensor196_heat"], rtol=2e-3, atol=1e-9)
    np.testing.assert_allclose(out["depth"].numpy(), gold["S224_B2_tensor196_depth"], rtol=2e-5)


def test_guided_518_center_and_corner(sd):
    gold = np.load(os.path.join(GOLD, "guided.npz"))
    tokens = orc.dinov2_tokens(sd, orc.synthetic_images(1, 518))
    bg = np.load(os.path.join(GOLD, "backbone.npz"))
    np.testing.assert_allclose(tokens.norm(dim=-1).numpy(), bg["S518_B1_token_norms"], rtol=1e-5)
    for ins in ("center", "top-left", "bottom-right"):
        torch.manual_seed(11)
        out = orc.forward_with_guidance(sd, None, orc.synthetic_exif(1), ins, tokens=tokens, update_history=False)
        key = f"S518_B1_{ins}"
        np.testing.assert_allclose(out["depth"].numpy(), gold[key + "_depth"], rtol=2e-5)
        np.testing.assert_allclose(out["heatmap"].numpy(), gold[key + "_heat"], rtol=2e-3, atol=1e-9)
        assert (out["heatmap"].argmax(-1).numpy() == gold[key + "_heat"].argmax(-1)).all()


@pytest.mark.parametrize("tag", ["exif", "noexif"])
def test_unguided_224(sd, tokens224, tag):
    gold = np.load(os.path.join(GOLD, "unguided.npz"))
    torch.manual_seed(11)
    ex = orc.synthetic_exif(2) if tag == "exif" else None
    out = orc.forward_unguided(sd, None, ex, tokens=tokens224, update_history=False)
    key = f"S224_B2_{tag}"
    np.testing.assert_allclose(out["depth"].numpy(), gold[key + "_depth"], rtol=2e-5)
    np.testing.assert_allclose(out["confidence"].numpy(), gold[key + "_conf"], rtol=1e-6)
    np.testing.assert_allclose(out["heatmap"].numpy(), gold[key + "_heat"], rtol=2e-3, atol=1e-9)
    np.testing.assert_allclose(out["fusion_features"].numpy(), gold[key + "_fusion"], rtol=1e-4, atol=1e-6)


def test_confidence_degenerate_constant():
    """SURVEY.md §4 degeneracy guard: at seed-0 init every confidence is sigmoid(2.0)."""
    gold = np.load(os.path.join(GOLD, "guided.npz"))
    assert np.allclose(gold["S224_B2_center_conf"], 0.8807970285, atol=1e-7)


def test_pillow_resize_restatement_is_bit_exact():
    """oracle.pil_resize_bilinear (restated from Pillow's Resample.c) against PIL.Image.resize itself — the third-party
    arithmetic behind demo.py:162-163 `Resize((S, S))` (Pillow 12.2.0 here)."""
    import numpy as np
    from PIL import Image
    from oracle import cogaim_oracle as orc
    rng = np.random.default_rng(0)
    for H, W, oh, ow in [(480, 640, 518, 518), (480, 640, 224, 224), (100, 77, 224, 224), (224, 224, 518, 518),
                         (300, 518, 518, 518), (518, 300, 518, 518), (37, 41, 14, 70), (64, 64, 64, 64)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        want = np.asarray(Image.fromarray(img).resize((ow, oh), Image.BILINEAR))
        assert np.array_equal(orc.pil_resize_bilinear(img, oh, ow), want), (H, W, oh, ow)


def test_demo_preprocess_restatement_matches_torchvision():
    import numpy as np
    from PIL import Image
    from torchvision import transforms
    from oracle import cogaim_oracle as orc
    img = np.random.default_rng(3).integers(0, 256, (120, 200, 3), dtype=np.uint8)
    tf = transforms.Compose([transforms.Resize((56, 56)), transforms.ToTensor(),
                             transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    assert torch.equal(orc.demo_preprocess(img, 56), tf(Image.fromarray(img)))


def test_focus_map_restatement_shapes_and_range():
    from oracle import cogaim_oracle as orc
    heat = torch.softmax(torch.randn(2, 256, generator=torch.Generator().manual_seed(0)), -1)
    fm = orc.focus_map(heat, 100, 150)
    assert fm.shape == (2, 100, 150) and float(fm.min()) >= 0.0 and float(fm.max()) <= 1.0
    grid = orc.focus_map(heat, 16, 16)  # identity zoom = the min-max normalised grid itself
    assert abs(float(grid.max()) - 1.0) < 1e-4 and float(grid.min()) == 0.0  # (max - min) / (max - min + 1e-8)
    # 70 % of the cubed cells sit at or below the percentile threshold and were scaled by 0.3
    assert 0.6 < float((grid < grid.flatten(1).quantile(0.7, dim=1).view(2, 1, 1) + 1e-9).float().mean()) < 0.8


# --- CuriosityModule side effects and the curiosity-guided configuration (tests/golden/curiosity*.npz) -------------------

def _curiosity_sequence(sd, tokens, gold, check_outputs):
    """Replays oracle/make_golden.py `run_sequence` on the oracle; compares rewards, ring buffer and pointer per step."""
    ex = orc.synthetic_exif(2)
    p = "curiosity_module."
    sd[p + "exploration_history"] = torch.zeros(1000)
    sd[p + "history_pointer"] = torch.tensor(0)

    def check(step, rewards):
        np.testing.assert_allclose(torch.stack(rewards).numpy(), gold[f"seq{step}_rewards"], rtol=2e-5)
        np.testing.assert_allclose(sd[p + "exploration_history"][:32].numpy(), gold[f"seq{step}_history"], rtol=2e-5)
        np.testing.assert_allclose(sd[p + "exploration_history"][-4:].numpy(), gold[f"seq{step}_history_tail"], rtol=2e-5)
        assert int(sd[p + "history_pointer"]) == int(gold[f"seq{step}_pointer"])

    rewards = []
    real = orc.curiosity_module

    def spy(*a, **k):
        r = real(*a, **k)
        rewards.append(r.clone())
        return r

    orc.curiosity_module = spy
    try:
        torch.manual_seed(11)
        o = orc.forward_with_guidance(sd, None, ex, "center", tokens=tokens)
        check(1, rewards)
        if check_outputs:
            np.testing.assert_allclose(o["depth"].numpy(), gold["seq1_depth"], rtol=2e-5)
            np.testing.assert_allclose(o["heatmap"].numpy(), gold["seq1_heat"], rtol=2e-3, atol=1e-9)
        rewards.clear()
        torch.manual_seed(11)
        o = orc.forward_unguided(sd, None, ex, tokens=tokens, has_last_attention=True)
        check(2, rewards)
        if check_outputs:
            np.testing.assert_allclose(o["depth"].numpy(), gold["seq2_depth"], rtol=2e-5)
            np.testing.assert_allclose(o["heatmap"].numpy(), gold["seq2_heat"], rtol=2e-3, atol=1e-9)
            np.testing.assert_allclose(o["fusion_features"].numpy(), gold["seq2_fusion"], rtol=1e-4, atol=1e-6)
        rewards.clear()
        torch.manual_seed(11)
        o = orc.forward_unguided(sd, None, None, tokens=tokens, has_last_attention=False)
        check(3, rewards)
        if check_outputs:
            np.testing.assert_allclose(o["depth"].numpy(), gold["seq3_depth"], rtol=2e-5)
            np.testing.assert_allclose(o["heatmap"].numpy(), gold["seq3_heat"], rtol=2e-3, atol=1e-9)
        rewards.clear()
        torch.manual_seed(11)
        orc.forward_unguided(sd, None, ex, tokens=tokens, has_last_attention=True, return_attention=False)
        check(4, rewards)
    finally:
        orc.curiosity_module = real


def test_curiosity_rewards_and_ring_buffer(sd, tokens224):
    gold = np.load(os.path.join(GOLD, "curiosity.npz"))
    _curiosity_sequence(dict(sd), tokens224, gold, check_outputs=False)
    # ring-buffer wrap-around: pointer 999 + 2 rewards -> slots 999, 0; pointer 1   (src/model.py:770-773)
    s2 = dict(sd)
    s2["curiosity_module.exploration_history"] = torch.zeros(1000)
    s2["curiosity_module.history_pointer"] = torch.tensor(999)
    torch.manual_seed(11)
    orc.forward_with_guidance(s2, None, orc.synthetic_exif(2), "top", tokens=tokens224)
    assert int(s2["curiosity_module.history_pointer"]) == int(gold["seq6_pointer"]) == 1
    np.testing.assert_allclose(s2["curiosity_module.exploration_history"][-1].item(), gold["seq6_history_tail"][-1], rtol=2e-5)
    np.testing.assert_allclose(s2["curiosity_module.exploration_history"][0].item(), gold["seq6_history"][0], rtol=2e-5)


def test_curiosity_guided_state_dict_and_forward():
    """Top-level `curiosity_guided_attention: {enabled: true}` (src/model.py:854): 335 tensors, modulated attention."""
    sd = orc.build_state_dict(0, curiosity_guided=True)
    assert len(sd) == 335
    _assert_reference_init(sd, "state_dict_seed0_curiosity_guided.json")
    tokens = orc.dinov2_tokens(sd, orc.synthetic_images(2, 224))
    gold = np.load(os.path.join(GOLD, "curiosity_guided.npz"))
    _curiosity_sequence(dict(sd), tokens, gold, check_outputs=True)
    for ins in ("top-left", "right"):
        torch.manual_seed(11)
        o = orc.forward_with_guidance(dict(sd), None, orc.synthetic_exif(2), ins, tokens=tokens)
        np.testing.assert_allclose(o["depth"].numpy(), gold[f"guided_{ins}_depth"], rtol=2e-5)
        np.testing.assert_allclose(o["heatmap"].numpy(), gold[f"guided_{ins}_heat"], rtol=2e-3, atol=1e-9)
        assert (o["heatmap"].argmax(-1).numpy() == gold[f"guided_{ins}_heat"].argmax(-1)).all()


def test_lora_is_built_saved_and_ignored_by_the_reference():
    """Top-level `use_lora: true` (src/model.py:822-831): 24 more tensors, bit-identical init, and a forward that never
    reads them — the fixture was recorded with non-zero lora_B; the oracle, which has no LoRA code at all, reproduces it."""
    sd = orc.build_state_dict(0, use_lora=True)
    assert len(sd) == 343
    _assert_reference_init(sd, "state_dict_seed0_lora.json")
    assert float(sd["lora_layers.0.lora_B"].abs().sum()) == 0.0
    gold = np.load(os.path.join(GOLD, "lora.npz"))
    torch.manual_seed(11)
    out = orc.forward_with_guidance(sd, orc.synthetic_images(2, 224), orc.synthetic_exif(2), "center", update_history=False)
    np.testing.assert_allclose(out["depth"].numpy(), gold["depth"], rtol=2e-5)
    np.testing.assert_allclose(out["heatmap"].numpy(), gold["heat"], rtol=2e-3, atol=1e-9)
