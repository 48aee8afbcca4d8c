"""CPU ORACLE — test infrastructure, NOT product code.

A plain PyTorch fp32 restatement of the reference's forward path, written against a flat `state_dict`
(name -> tensor) so it can travel to the GPU box where `/root/reference` does not exist.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg may import this module;
the product package `cognitive_aim_depth_estimation_b200` never does.

What is restated (reference file:line given at each function):
  * HF transformers 5.5.0 `Dinov2Model` forward (third-party dependency of the reference, unpinned in
    its requirements.txt:12; arithmetic lives in transformers/models/dinov2/modeling_dinov2.py),
  * reference src/model.py: AmbientStream, FocalStream, IterativeFocalStream, EXIFPriorDatabase,
    CuriosityModule (for its RNG draws and ring buffer), fusion + heads, `forward_with_guidance`,
    `_guided_focal_stream`, `forward`, and the construction order / custom inits of `create_model`
    (so that `build_state_dict(seed)` reproduces the reference's random-init weights bit-for-bit),
  * reference demo.py:162-166 preprocessing: Pillow's antialiased bilinear resample (third-party, `Pillow>=8.3.0`
    unpinned in requirements.txt:8; 12.2.0 here) restated from its Resample.c, ToTensor, Normalize
    (`pil_resize_bilinear`, `demo_preprocess`) — pinned bit-exactly against PIL / torchvision in tests/test_oracle.py,
  * reference demo.py:530-563 heat-map post-processing (`focus_map`), with the numpy / scipy calls the reference makes.

Pinning: the reference ships no golden vectors or tests (SURVEY.md §4).  This oracle is pinned against
outputs of the reference itself, imported unmodified in the build container by `oracle/make_golden.py`;
those outputs are committed under `tests/golden/` and checked by `tests/test_oracle.py`.
"""
from __future__ import annotations

import hashlib
import math
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

SD = Dict[str, torch.Tensor]

INSTRUCTIONS = ["center", "left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right"]

# --------------------------------------------------------------------------------------------------
# Weights: same seed + same construction order as reference src/model.py:798-958  ->  same tensors
# --------------------------------------------------------------------------------------------------


def _xavier_u(lin: nn.Linear, gain: float):
    nn.init.xavier_uniform_(lin.weight, gain=gain)
    nn.init.constant_(lin.bias, 0.0)


class _FocalInit(nn.Module):
    """Parameter container with the construction + init order of FocalStream (src/model.py:58-126).
    curiosity_guided=False is the effective config (SURVEY.md §0 quirk 1); True adds the modulator (:73-79)."""

    def __init__(self, d=768, h=256, curiosity_guided=False):
        super().__init__()
        self.query_proj = nn.Linear(d, d)
        self.key_proj = nn.Linear(d, d)
        self.value_proj = nn.Linear(d, d)
        if curiosity_guided:
            self.curiosity_modulator = nn.Sequential(nn.Linear(1, h // 8), nn.ReLU(), nn.Linear(h // 8, 8), nn.Sigmoid())
        self.projection = nn.Sequential(nn.Linear(d, h), nn.ReLU(), nn.Dropout(0.1), nn.Linear(h, h // 4))
        self.adaptive_weight = nn.Parameter(torch.tensor(0.5))
        for m in self.projection:  # :98-103
            if isinstance(m, nn.Linear):
                _xavier_u(m, 0.8)
        if curiosity_guided:  # :106-111
            for m in self.curiosity_modulator:
                if isinstance(m, nn.Linear):
                    _xavier_u(m, 0.8)
        with torch.no_grad():  # :114-126
            nn.init.xavier_normal_(self.query_proj.weight, gain=2.0)
            nn.init.xavier_normal_(self.key_proj.weight, gain=2.0)
            nn.init.xavier_normal_(self.value_proj.weight, gain=1.0)
            nn.init.uniform_(self.query_proj.bias, -0.05, 0.05)
            nn.init.uniform_(self.key_proj.bias, -0.05, 0.05)
            nn.init.constant_(self.value_proj.bias, 0.0)


class _IterFocalInit(nn.Module):
    """IterativeFocalStream construction (src/model.py:318-389)."""

    def __init__(self, d=768, h=256, iters=3, curiosity_guided=False):
        super().__init__()
        self.focal_streams = nn.ModuleList([_FocalInit(d, h, curiosity_guided) for _ in range(iters)])
        self.initial_focus = nn.Parameter(torch.randn(1, d))
        if curiosity_guided:  # :333-339
            self.curiosity_amplifier = nn.Sequential(nn.Linear(1, 32), nn.ReLU(), nn.Linear(32, iters),
                                                     nn.Softmax(dim=-1))
        self.fusion = nn.Sequential(nn.Linear(h // 4 * iters, h // 2), nn.ReLU(), nn.Linear(h // 2, h // 4))
        for m in self.fusion:  # :354-358
            if isinstance(m, nn.Linear):
                _xavier_u(m, 0.8)
        if curiosity_guided:  # :361-366
            for m in self.curiosity_amplifier:
                if isinstance(m, nn.Linear):
                    _xavier_u(m, 0.8)
        nn.init.normal_(self.initial_focus, mean=0.0, std=0.02)  # :369
        for i, fs in enumerate(self.focal_streams):  # :372-389
            with torch.no_grad():
                f = 1.0 + 0.1 * i
                nn.init.xavier_normal_(fs.query_proj.weight, gain=1.2 * f)
                nn.init.xavier_normal_(fs.key_proj.weight, gain=1.2 * f)
                nn.init.xavier_normal_(fs.value_proj.weight, gain=1.0 * f)
                nn.init.uniform_(fs.query_proj.bias, -0.01 * f, 0.01 * f)
                nn.init.uniform_(fs.key_proj.bias, -0.01 * f, 0.01 * f)
                nn.init.constant_(fs.value_proj.bias, 0.0)


class _AlignerInit(nn.Module):  # DimensionAligner, src/model.py:1467-1476
    def __init__(self, target, source):
        super().__init__()
        self.projection = nn.Linear(source, target)


class _CuriosityInit(nn.Module):  # CuriosityModule.__init__, src/model.py:524-584
    def __init__(self, d=768, h=256):
        super().__init__()
        lat = d // 4

        def mlp(a, b, c):
            return nn.Sequential(nn.Linear(a, b), nn.ReLU(), nn.Dropout(0.1), nn.Linear(b, c))

        self.encoder_mean = mlp(d, d // 2, lat)
        self.encoder_logvar = mlp(d, d // 2, lat)
        self.decoder = mlp(lat, d // 2, lat)
        self.uncertainty_head = nn.Sequential(nn.Linear(d, d // 4), nn.ReLU(), nn.Linear(d // 4, 1), nn.Softplus())
        self.geometric_curiosity = nn.Sequential(nn.Linear(d + 4, h), nn.ReLU(), nn.Linear(h, 1), nn.Sigmoid())
        self.local_curiosity = nn.Sequential(nn.Linear(d, h // 2), nn.ReLU(), nn.Linear(h // 2, 1), nn.Sigmoid())
        self.curiosity_weights = nn.Parameter(torch.tensor([0.4, 0.3, 0.3]))
        self.register_buffer("exploration_history", torch.zeros(1000))
        self.register_buffer("history_pointer", torch.tensor(0))


class _ModelInit(nn.Module):
    """Construction order of CognitiveAimModel.__init__ (src/model.py:798-958) under the effective config."""

    def __init__(self, num_cameras=71, curiosity_guided=False, use_lora=False, lora_rank=16):
        super().__init__()
        from transformers import Dinov2Config, Dinov2Model  # the reference's own backbone dependency
        self.backbone = Dinov2Model(Dinov2Config(image_size=518, patch_size=14))  # :814 (offline: random init)
        if use_lora:  # :822-831, LoRALayer.__init__ :15-24 (built and saved, never applied: quirk 4)
            self.lora_layers = nn.ModuleList()
            for _ in range(12):
                lo = nn.Module()
                lo.lora_A = nn.Parameter(torch.randn(lora_rank, 768) * 0.01)
                lo.lora_B = nn.Parameter(torch.zeros(768, lora_rank))
                self.lora_layers.append(lo)
        self.ambient_stream = nn.Module()
        self.ambient_stream.mlp = nn.Sequential(nn.Linear(768, 256), nn.ReLU(), nn.Dropout(0.1), nn.Linear(256, 128),
                                                nn.ReLU(), nn.Linear(128, 64))  # :37-44
        self.focal_stream = _IterFocalInit(768, 256, 3, curiosity_guided)  # :857-864
        ex = nn.Module()  # EXIFPriorDatabase :460-480
        ex.camera_embedding = nn.Embedding(num_cameras, 64)
        ex.exif_encoder = nn.Sequential(nn.Linear(3, 64), nn.ReLU(), nn.Linear(64, 64))
        ex.fusion = nn.Sequential(nn.Linear(128, 256), nn.ReLU(), nn.Dropout(0.1), nn.Linear(256, 64))
        self.exif_prior = ex
        self.fusion = nn.Sequential(nn.Linear(192, 192), nn.ReLU(), nn.Dropout(0.1))  # :908-912
        self.ambient_dim_aligner = _AlignerInit(768, 64)  # :920-922
        self.focal_dim_aligner = _AlignerInit(768, 64)
        self.exif_dim_aligner = _AlignerInit(768, 64)
        self.decision_head = nn.Sequential(nn.Linear(192, 1), nn.Softplus())  # :925-933
        with torch.no_grad():
            nn.init.xavier_uniform_(self.decision_head[0].weight, gain=1.0)
            nn.init.constant_(self.decision_head[0].bias, 1.0)
        self.confidence_head = nn.Sequential(nn.Linear(192, 1), nn.ReLU(), nn.Linear(1, 1), nn.Sigmoid())  # :936-945
        with torch.no_grad():
            self.confidence_head[2].bias.fill_(2.0)
        self.curiosity_module = _CuriosityInit(768, 256)  # :948-952
        self.global_aligner = _AlignerInit(768, 768 * 3)  # :958


def build_state_dict(seed: int = 0, num_cameras: int = 71, curiosity_guided: bool = False,
                     use_lora: bool = False) -> SD:
    """`torch.manual_seed(seed); create_model(cfg, {'num_cameras': 71}).state_dict()` of the reference
    (SURVEY.md §8c seed protocol), without the reference.  curiosity_guided=True is what a config with the top-level
    key `curiosity_guided_attention: {enabled: true}` builds (src/model.py:854): 16 more tensors; use_lora=True is
    top-level `use_lora: true` (:822): 24 more tensors that no forward path reads."""
    torch.manual_seed(seed)
    m = _ModelInit(num_cameras, curiosity_guided, use_lora).eval()
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def state_dict_digest(sd: SD) -> Dict[str, float]:
    """Cheap fingerprint used by the golden fixtures: per-tensor fp64 sum and abs-sum."""
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items()}


def matches_digest(v: torch.Tensor, digest) -> bool:
    """`v` against its `state_dict_digest` entry (sum, abs-sum), up to the order of the fp64 additions: torch splits a
    CPU sum across its threads, so the order depends on the host's core count, and two orders of n additions differ by
    at most 2 n 2^-53 sum|x|.  Bit-exactness is `state_dict_sha256`'s job."""
    s, a = digest
    v = v.double()
    tol = 2 * v.numel() * 2.0 ** -53 * a
    return abs(float(v.sum()) - s) <= tol and abs(float(v.abs().sum()) - a) <= tol


def state_dict_sha256(sd: SD) -> str:
    """Bit-exact fingerprint of a whole state_dict: names, dtypes, shapes and bytes, in order."""
    h = hashlib.sha256()
    for k, v in sd.items():
        v = v.detach().cpu().contiguous()
        h.update(f"{k}:{v.dtype}:{tuple(v.shape)};".encode())
        h.update(v.numpy().tobytes())
    return h.hexdigest()


# --------------------------------------------------------------------------------------------------
# DINOv2 ViT-B/14 (HF transformers 5.5.0 modeling_dinov2.py)
# --------------------------------------------------------------------------------------------------


def dinov2_pos_embed(sd: SD, g: int, prefix: str = "backbone.") -> torch.Tensor:
    """[1+g*g, D] position embedding for a g x g patch grid (modeling_dinov2.py:57-95: identity at the native
    37 x 37 grid, otherwise bicubic, align_corners=False, computed in fp32)."""
    pos = sd[prefix + "embeddings.position_embeddings"][0]
    n0 = pos.shape[0] - 1
    if g * g == n0:
        return pos
    g0 = int(round(n0 ** 0.5))
    grid = pos[1:].reshape(1, g0, g0, -1).permute(0, 3, 1, 2).float()
    grid = F.interpolate(grid, size=(g, g), mode="bicubic", align_corners=False)
    return torch.cat([pos[:1], grid.permute(0, 2, 3, 1).reshape(g * g, -1)], dim=0)


def dinov2_tokens(sd: SD, images: torch.Tensor, prefix: str = "backbone.", n_layers: int = 12, heads: int = 12,
                  eps: float = 1e-6) -> torch.Tensor:
    """`Dinov2Model(images).last_hidden_state` [B, 1+N, 768] (modeling_dinov2.py:97-116, 367-386, 473-478)."""
    B, _, H, W = images.shape
    p = prefix
    w = sd[p + "embeddings.patch_embeddings.projection.weight"]
    x = F.conv2d(images, w, sd[p + "embeddings.patch_embeddings.projection.bias"], stride=w.shape[-1])
    g = x.shape[-1]
    x = x.flatten(2).transpose(1, 2)
    x = torch.cat([sd[p + "embeddings.cls_token"].expand(B, -1, -1), x], dim=1)
    x = x + dinov2_pos_embed(sd, g, p).unsqueeze(0)
    D = x.shape[-1]
    dh = D // heads
    for i in range(n_layers):
        q = f"{p}encoder.layer.{i}."
        h = F.layer_norm(x, (D,), sd[q + "norm1.weight"], sd[q + "norm1.bias"], eps)
        a = q + "attention.attention."

        def split(t):
            return t.view(B, -1, heads, dh).transpose(1, 2)

        qq = split(F.linear(h, sd[a + "query.weight"], sd[a + "query.bias"]))
        kk = split(F.linear(h, sd[a + "key.weight"], sd[a + "key.bias"]))
        vv = split(F.linear(h, sd[a + "value.weight"], sd[a + "value.bias"]))
        att = torch.softmax(qq @ kk.transpose(-1, -2) * dh ** -0.5, dim=-1) @ vv
        att = att.transpose(1, 2).reshape(B, -1, D)
        o = F.linear(att, sd[q + "attention.output.dense.weight"], sd[q + "attention.output.dense.bias"])
        x = x + o * sd[q + "layer_scale1.lambda1"]
        h = F.layer_norm(x, (D,), sd[q + "norm2.weight"], sd[q + "norm2.bias"], eps)
        h = F.gelu(F.linear(h, sd[q + "mlp.fc1.weight"], sd[q + "mlp.fc1.bias"]))
        h = F.linear(h, sd[q + "mlp.fc2.weight"], sd[q + "mlp.fc2.bias"])
        x = x + h * sd[q + "layer_scale2.lambda1"]
    return F.layer_norm(x, (D,), sd[p + "layernorm.weight"], sd[p + "layernorm.bias"], eps)


# --------------------------------------------------------------------------------------------------
# Cognitive streams (reference src/model.py)
# --------------------------------------------------------------------------------------------------


def focal_position_encoding(n: int, d: int) -> torch.Tensor:
    """2-D sinusoidal table of FocalStream.forward (src/model.py:140-177), vectorised."""
    pe = torch.zeros(n, d)
    g = int(n ** 0.5)
    if g * g == n:
        half = d // 2
        div = torch.exp(torch.arange(0, half, 2, dtype=torch.float) * -(math.log(10000.0) / half))
        idx = torch.arange(n)
        row = (idx // g).float().unsqueeze(1)
        col = (idx % g).float().unsqueeze(1)
        pe[:, 0:half:2] = torch.sin(row * div)
        pe[:, 1:half:2] = torch.cos(row * div)
        pe[:, half::2] = torch.sin(col * div)
        pe[:, half + 1::2] = torch.cos(col * div)
    else:
        pos = torch.arange(0, n, dtype=torch.float).unsqueeze(1)
        div = torch.exp(torch.arange(0, d, 2, dtype=torch.float) * -(math.log(10000.0) / d))
        pe[:, 0::2] = torch.sin(pos * div)
        pe[:, 1::2] = torch.cos(pos * div)
    return pe


def center_bias(n: int, strength: float = 0.3) -> torch.Tensor:
    """create_center_bias_mask (src/model.py:208-231)."""
    g = int(n ** 0.5)
    if g * g != n:
        d = (torch.arange(n, dtype=torch.float) - n // 2).abs()
        return torch.exp(-d ** 2 / (2 * (n / 12) ** 2)) * strength
    c = g // 2
    y, x = torch.meshgrid(torch.arange(g), torch.arange(g), indexing="ij")
    dist = torch.sqrt((x - c).float() ** 2 + (y - c).float() ** 2)
    return torch.exp(-dist ** 2 / (2 * (g / 6) ** 2)).flatten() * strength


def _mlp(sd: SD, x, names, relu_last=False):
    for i, n in enumerate(names):
        x = F.linear(x, sd[n + ".weight"], sd[n + ".bias"])
        if i < len(names) - 1 or relu_last:
            x = F.relu(x)
    return x


def focal_stream(sd: SD, prefix: str, tokens: torch.Tensor, need_features: bool = True, curiosity_score=None):
    """One FocalStream.forward (src/model.py:128-313).  `curiosity_score` [B] is used only when the state dict holds a
    curiosity_modulator (curiosity_guided=True, :264-276).  Returns (features [B,64] or None, attention [B,N])."""
    B, N, D = tokens.shape
    x = tokens + focal_position_encoding(N, D).unsqueeze(0)  # :184
    q = F.linear(x, sd[prefix + "query_proj.weight"], sd[prefix + "query_proj.bias"])
    k = F.linear(x, sd[prefix + "key_proj.weight"], sd[prefix + "key_proj.bias"])
    A = torch.softmax(q @ k.transpose(-2, -1) / math.sqrt(D // 8), dim=-1)  # :69,197-200
    cb = center_bias(N).unsqueeze(0)
    pa = A.mean(dim=1) + cb  # :234-239
    if pa.var() < 1e-6:  # :242-257 (batch-wide variance; never fires for g >= 4)
        pa = torch.diagonal(A, dim1=-2, dim2=-1) + cb
    if pa.var() < 1e-6:
        pa = A.max(dim=-1).values + cb
    if pa.var() < 1e-6:
        norms = x.norm(dim=-1)
        pa = norms + torch.randn_like(norms) * 0.1 * norms.std()
    pa = pa / (pa.sum(dim=-1, keepdim=True) + 1e-8)  # :261
    if prefix + "curiosity_modulator.0.weight" in sd and curiosity_score is not None:  # :264-276
        mod = torch.sigmoid(_mlp(sd, curiosity_score.unsqueeze(-1),
                                 [prefix + "curiosity_modulator.0", prefix + "curiosity_modulator.2"]))
        cw = mod.mean(dim=-1, keepdim=True)
        aw = sd[prefix + "adaptive_weight"]
        pa = aw * (pa * (1.0 + cw)) + (1 - aw) * pa
    pa = pa.clamp(min=1e-8)  # :281-282
    pa = pa / (pa.sum(dim=-1, keepdim=True) + 1e-8)
    feats = None
    if need_features:
        v = F.linear(x, sd[prefix + "value_proj.weight"], sd[prefix + "value_proj.bias"])
        weighted = ((A @ v) * pa.unsqueeze(-1)).sum(dim=1)  # :204,308
        feats = _mlp(sd, weighted, [prefix + "projection.0", prefix + "projection.3"])  # :311
    return feats, pa


def iterative_focal_stream(sd: SD, tokens: torch.Tensor, need_features: bool = True, iters: int = 3,
                           focus_strength: float = 1.5, prefix: str = "focal_stream.", curiosity_score=None):
    """IterativeFocalStream.forward (src/model.py:391-455). Returns (fused [B,64] or None, last attention [B,N])."""
    cur = tokens
    feats = []
    att = None
    iter_w = None
    if prefix + "curiosity_amplifier.0.weight" in sd and curiosity_score is not None:  # :406-409
        iter_w = torch.softmax(_mlp(sd, curiosity_score.unsqueeze(-1),
                                    [prefix + "curiosity_amplifier.0", prefix + "curiosity_amplifier.2"]), dim=-1)
    for i in range(iters):
        sc = curiosity_score * iter_w[:, i] if iter_w is not None else curiosity_score  # :412-417
        f, att = focal_stream(sd, f"{prefix}focal_streams.{i}.", cur, need_features, sc)
        feats.append(f)
        if i < iters - 1:
            cur = cur * (1 + focus_strength * att.unsqueeze(-1))  # :426
    fused = None
    if need_features:
        fused = _mlp(sd, torch.cat(feats, dim=1), [prefix + "fusion.0", prefix + "fusion.2"])  # :430
    return fused, att


_FOCUS = {  # (y, x) as functions of g ; src/model.py:1282-1376
    "left": lambda g: (g // 2, g // 4), "right": lambda g: (g // 2, g * 3 // 4),
    "top": lambda g: (g // 4, g // 2), "bottom": lambda g: (g * 3 // 4, g // 2),
    "top-left": lambda g: (g // 4, g // 4), "top-right": lambda g: (g // 4, g * 3 // 4),
    "bottom-left": lambda g: (g * 3 // 4, g // 4), "bottom-right": lambda g: (g * 3 // 4, g * 3 // 4),
}
_ALIASES = {"topleft": "top-left", "topright": "top-right", "bottomleft": "bottom-left", "bottomright": "bottom-right"}


def instruction_mask(instruction: str, g: int) -> torch.Tensor:
    """String -> flattened g x g guidance mask (src/model.py:1262-1379). Unknown strings give all-ones."""
    name = instruction.lower()
    name = _ALIASES.get(name, name)
    mask = torch.ones(g, g)
    if name == "center":
        fy, fx, r, hi, lo = g // 2, g // 2, max(1, g // 4), 3.0, 1.5
    elif name in _FOCUS:
        (fy, fx), r, hi, lo = _FOCUS[name](g), max(1, g // 6), 5.0, 2.0
    else:
        return mask.flatten()
    for y in range(g):
        for x in range(g):
            d = math.sqrt((y - fy) ** 2 + (x - fx) ** 2)
            if d <= r:
                mask[y, x] = hi
            elif d <= r * 2:
                mask[y, x] = lo
    return mask.flatten()


def resolve_guidance(guidance, n: int) -> torch.Tensor:
    """attention_guidance (str or tensor of any square length) -> [N] (src/model.py:1262-1398)."""
    g = int(math.sqrt(n))
    if isinstance(guidance, str):
        guidance = instruction_mask(guidance, g)
    if guidance.size(0) != n:
        gs = int(math.sqrt(guidance.size(0)))
        guidance = F.interpolate(guidance.view(1, 1, gs, gs), size=(g, g), mode="bilinear",
                                 align_corners=False).squeeze().flatten()
    return guidance


def exif_prior(sd: SD, exif: dict, prefix: str = "exif_prior.") -> torch.Tensor:
    """EXIFPriorDatabase.forward (src/model.py:482-519)."""
    def flat(t):
        return t.squeeze(1) if t.dim() > 1 else t
    cam = F.embedding(flat(exif["camera_idx"]), sd[prefix + "camera_embedding.weight"])
    cont = torch.stack([flat(exif["focal_length"]), flat(exif["aperture"]), torch.log(flat(exif["iso"]) + 1)], dim=1)
    e = _mlp(sd, cont, [prefix + "exif_encoder.0", prefix + "exif_encoder.2"])
    return _mlp(sd, torch.cat([cam, e], dim=1), [prefix + "fusion.0", prefix + "fusion.3"])


def ambient_stream(sd: SD, cls: torch.Tensor) -> torch.Tensor:
    """AmbientStream.forward (src/model.py:46-53)."""
    return _mlp(sd, cls, ["ambient_stream.mlp.0", "ambient_stream.mlp.3", "ambient_stream.mlp.5"])


def _randn_rows(like: torch.Tensor, rng_rows):
    """`torch.randn_like(like)`, or — when `like` holds only the rows `rows` of a batch of `Bg` images — the same rows
    of the draw the reference would make for the whole batch (identical generator consumption)."""
    if rng_rows is None:
        return torch.randn_like(like)
    Bg, rows = rng_rows
    return torch.randn(Bg, like.size(1))[list(rows)]


def curiosity_module(sd: SD, cls: torch.Tensor, update_history: bool = True, prefix: str = "curiosity_module.",
                     rng_rows=None):
    """CuriosityModule.forward (src/model.py:586-688) with exif_data=None, loss_type='robust'.
    Output-dead under the effective config, but it draws randn(B,192) then randn(B,768) from the global
    CPU generator (:609, :744) and writes the exploration ring buffer (:760-773).
    `rng_rows=(Bg, rows)`: `cls` holds rows `rows` of a batch of `Bg` images (tests of images picked out of a large
    batch): the noise is drawn at the full batch size, so the generator ends where the reference's would."""
    p = prefix
    mu = _mlp(sd, cls, [p + "encoder_mean.0", p + "encoder_mean.3"])
    logvar = _mlp(sd, cls, [p + "encoder_logvar.0", p + "encoder_logvar.3"])
    std = torch.exp(0.5 * logvar)
    z = mu + _randn_rows(std, rng_rows) * std
    rec = _mlp(sd, z, [p + "decoder.0", p + "decoder.3"])
    diff = rec - cls[:, :rec.size(1)]
    err = torch.sqrt((diff ** 2).sum(dim=1) + 1e-8)
    err = err / (1.0 + err)
    kl = -0.5 * torch.sum(1 + logvar - mu.pow(2) - logvar.exp(), dim=1)
    unc = F.softplus(_mlp(sd, cls, [p + "uncertainty_head.0", p + "uncertainty_head.2"])).squeeze(-1)
    basic = err.clamp(min=0) + 0.1 * kl.clamp(min=0) + 0.1 * unc.clamp(0.0, 10.0)
    geo = torch.full((cls.size(0),), 0.5)  # exif_data is None at every call site (:690-700)
    base = torch.sigmoid(_mlp(sd, cls, [p + "local_curiosity.0", p + "local_curiosity.2"])).squeeze(-1)
    noisy = cls + _randn_rows(cls, rng_rows) * 0.01
    nz = torch.sigmoid(_mlp(sd, noisy, [p + "local_curiosity.0", p + "local_curiosity.2"])).squeeze(-1)
    local = (base + (base - nz).abs() * 0.2).clamp(0.0, 1.0)
    w = torch.softmax(sd[p + "curiosity_weights"], dim=0)
    reward = w[0] * geo + w[1] * local + w[2] * basic
    if update_history:
        hist = sd[p + "exploration_history"]
        ptr = int(sd[p + "history_pointer"])
        for r in reward:
            hist[ptr % hist.size(0)] = r.item()
            ptr = (ptr + 1) % hist.size(0)
        sd[p + "history_pointer"] = torch.tensor(ptr)
    return reward.clamp(0.0, 100.0)


def heads(sd: SD, feats192: torch.Tensor):
    """fusion + decision_head + confidence_head (src/model.py:908-945, 1223-1230)."""
    f = F.relu(F.linear(feats192, sd["fusion.0.weight"], sd["fusion.0.bias"]))
    depth = F.softplus(F.linear(f, sd["decision_head.0.weight"], sd["decision_head.0.bias"]))
    c = F.relu(F.linear(f, sd["confidence_head.0.weight"], sd["confidence_head.0.bias"]))
    conf = torch.sigmoid(F.linear(c, sd["confidence_head.2.weight"], sd["confidence_head.2.bias"]))
    return depth, conf, f


@torch.no_grad()
def forward_with_guidance(sd: SD, images: torch.Tensor, exif: Optional[dict], guidance, tokens=None,
                          update_history: bool = True, rng_rows=None):
    """CognitiveAimModel.forward_with_guidance(..., return_attention=True) (src/model.py:1157-1240) for
    `guidance` a string or tensor and exif given.  Consumes the global CPU RNG exactly like the reference:
    randn(B,192), randn(B,768) (curiosity), then nn.Linear(768,64) init (:1421).
    Returns dict(depth [B,1], confidence [B,1], heatmap [B,N], base_attention [B,N], pooled [B,768])."""
    if tokens is None:
        tokens = dinov2_tokens(sd, images)
    cls, patches = tokens[:, 0], tokens[:, 1:]
    score = curiosity_module(sd, cls, update_history, rng_rows=rng_rows)  # :1185 (only consumed when curiosity_guided=True)
    amb = ambient_stream(sd, cls)  # :1196
    _, base = iterative_focal_stream(sd, patches, need_features=False,
                                     curiosity_score=score)  # :1257 (features discarded at :1424)
    g = resolve_guidance(guidance, patches.size(1))
    guided = torch.softmax((0.7 * g.unsqueeze(0) + 0.3 * base) / 0.05, dim=-1)  # :1404-1409
    pooled = (patches * guided.unsqueeze(-1)).sum(dim=1)  # :1412-1414
    temp = nn.Linear(768, 64)  # :1421 fresh random projection on every call
    focal = temp(pooled)
    ex = exif_prior(sd, exif)  # :1216
    depth, conf, _ = heads(sd, torch.cat([amb, focal, ex], dim=1))
    return {"depth": depth, "confidence": conf, "heatmap": guided, "base_attention": base, "pooled": pooled,
            "tokens": tokens, "curiosity": score}


@torch.no_grad()
def forward_unguided(sd: SD, images: torch.Tensor, exif: Optional[dict], tokens=None, update_history: bool = True,
                     has_last_attention: bool = False, return_attention: bool = True):
    """CognitiveAimModel.forward(images, exif, return_attention) (src/model.py:1064-1155): identical repeated backbone
    passes of the reference are computed once (they are bit-identical in eval).  The CuriosityModule runs once in
    get_features_aligned (:992), once more when the model holds no `_last_attention_weights` (:1093-1104,
    `has_last_attention=False`) and once more for return_attention (:1138) — each run draws fresh noise and appends B
    rewards to the exploration ring buffer.  With curiosity_guided=True the features use the first score un-clamped and
    the returned attention the last score clamped to [0.5, 1] (:1107, :1141)."""
    if tokens is None:
        tokens = dinov2_tokens(sd, images)
    cls, patches = tokens[:, 0], tokens[:, 1:]
    score = curiosity_module(sd, cls, update_history)
    amb = ambient_stream(sd, cls)
    fused, att = iterative_focal_stream(sd, patches, need_features=True, curiosity_score=score)
    guided_cfg = "focal_stream.curiosity_amplifier.0.weight" in sd
    for extra in ([] if has_last_attention else ["last"]) + (["ret"] if return_attention else []):
        sc = curiosity_module(sd, cls, update_history).clamp(0.5, 1.0)
        if guided_cfg and extra == "ret":
            _, att = iterative_focal_stream(sd, patches, need_features=False, curiosity_score=sc)
    parts = [amb, fused]
    if exif is not None:
        parts.append(exif_prior(sd, exif))
    x = torch.cat(parts, dim=1)
    if x.size(1) < 192:  # :1035-1039 zero-pad the missing EXIF slot
        x = torch.cat([x, torch.zeros(x.size(0), 192 - x.size(1))], dim=1)
    depth, conf, f = heads(sd, x)
    return {"depth": depth, "confidence": conf, "heatmap": att, "fusion_features": f, "tokens": tokens}


# --------------------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md §8d)
# --------------------------------------------------------------------------------------------------


def focus_map(attention: torch.Tensor, height: int, width: int):
    """demo.py:530-563, per image: cube, 70th-percentile threshold (x0.3 at or below), min-max, g x g, scipy zoom order 1
    to the image size — with the very numpy / scipy calls the reference makes.  attention [B, N] -> float32 [B, h, w]."""
    import numpy as np
    from scipy.ndimage import zoom
    outs = []
    for row in attention.detach().cpu().numpy().astype(np.float32):
        attn_map = np.power(row, 3)                                                   # :533
        threshold = np.percentile(attn_map, 70)                                       # :536
        attn_map = np.where(attn_map > threshold, attn_map, attn_map * 0.3)           # :537
        attn_map = (attn_map - attn_map.min()) / (attn_map.max() - attn_map.min() + 1e-8)  # :540
        g = int(np.sqrt(len(attn_map)))                                               # :543-546
        assert g * g == len(attn_map)
        m = attn_map.reshape(g, g)
        outs.append(zoom(m, (height / g, width / g), order=1))                        # :558-563
    return torch.from_numpy(np.stack(outs).astype(np.float32))


def synthetic_images(B: int, S: int, seed: int = 1234) -> torch.Tensor:
    return torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(seed))


def synthetic_exif(B: int, seed: int = 1236) -> dict:
    g = torch.Generator().manual_seed(seed)
    return {
        "focal_length": torch.rand(B, generator=g) * 190 + 10,
        "aperture": torch.rand(B, generator=g) * 21 + 1,
        "iso": torch.rand(B, generator=g) * 6350 + 50,
        "camera_idx": torch.randint(0, 71, (B,), generator=g),
    }


# ------------------------------------------------------------------------------------------------------
# demo.py:162-166 preprocessing: torchvision Resize((S,S)) on a PIL image = Pillow's antialiased bilinear resample.
# Pillow is a third-party dependency of the reference (requirements.txt:8 `Pillow>=8.3.0`, unpinned; 12.2.0 here).
# Restated from Pillow's published algorithm (src/libImaging/Resample.c: precompute_coeffs, normalize_coeffs_8bpc,
# ImagingResampleHorizontal_8bpc / Vertical_8bpc, two passes with a uint8 intermediate); tests/test_oracle.py pins it
# bit-exactly against PIL.Image.resize itself.
# ------------------------------------------------------------------------------------------------------
_PIL_PRECISION_BITS = 32 - 8 - 2


def pil_bilinear_coeffs(in_size: int, out_size: int):
    """Resample.c precompute_coeffs + normalize_coeffs_8bpc for the triangle filter (support 1.0), box = whole axis.
    Returns (xmin[out], count[out], kk[out, ksize] int32)."""
    import math
    import numpy as np
    scale = in_size / out_size
    filterscale = max(scale, 1.0)
    support = 1.0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    xmin = np.zeros(out_size, np.int32)
    cnt = np.zeros(out_size, np.int32)
    kk = np.zeros((out_size, ksize), np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        lo = int(center - support + 0.5)  # C (int) cast: truncation toward zero
        lo = max(lo, 0)
        hi = int(center + support + 0.5)
        hi = min(hi, in_size)
        n = hi - lo
        w = np.zeros(ksize, np.float64)
        for x in range(n):
            t = abs((x + lo - center + 0.5) * ss)
            w[x] = 1.0 - t if t < 1.0 else 0.0
        ww = w[:n].sum() if n else 0.0
        # Pillow accumulates ww sequentially in double; np.sum of <= ksize doubles may pair differently, so redo it
        ww = 0.0
        for x in range(n):
            ww += w[x]
        if ww != 0.0:
            w[:n] /= ww
        for x in range(n):
            kk[xx, x] = int(-0.5 + w[x] * (1 << _PIL_PRECISION_BITS)) if w[x] < 0 else int(0.5 + w[x] * (1 << _PIL_PRECISION_BITS))
        xmin[xx], cnt[xx] = lo, n
    return xmin, cnt, kk


def pil_resize_bilinear(img_u8, out_h: int, out_w: int):
    """uint8 [H, W, C] -> uint8 [out_h, out_w, C] exactly as PIL.Image.resize((out_w, out_h), BILINEAR) (what
    torchvision Resize((S, S)) calls for a PIL image, demo.py:162-163): horizontal pass, uint8 rounding, vertical pass."""
    import numpy as np
    img = np.asarray(img_u8)
    H, W, _ = img.shape
    if (H, W) == (out_h, out_w):
        return img.copy()

    def one_pass(src, out_size, axis):
        xmin, cnt, kk = pil_bilinear_coeffs(src.shape[axis], out_size)
        src = np.moveaxis(src, axis, 0).astype(np.int64)
        acc = np.full((out_size,) + src.shape[1:], 1 << (_PIL_PRECISION_BITS - 1), np.int64)
        for j in range(kk.shape[1]):
            idx = np.minimum(xmin + j, src.shape[0] - 1)
            coef = np.where(j < cnt, kk[:, j], 0).astype(np.int64)
            acc += src[idx] * coef.reshape((-1,) + (1,) * (src.ndim - 1))
        out = np.clip(acc >> _PIL_PRECISION_BITS, 0, 255).astype(np.uint8)
        return np.moveaxis(out, 0, axis)

    need_h, need_v = W != out_w, H != out_h
    if need_h and need_v:
        # Resample.c runs the horizontal pass only on the source rows the vertical pass will read
        ymin, ycnt, _ = pil_bilinear_coeffs(H, out_h)
        first, last = int(ymin[0]), int(ymin[-1] + ycnt[-1])
        tmp = one_pass(img[first:last], out_w, 1)
        xmin, cnt, kk = pil_bilinear_coeffs(H, out_h)
        src = tmp.astype(np.int64)
        acc = np.full((out_h,) + src.shape[1:], 1 << (_PIL_PRECISION_BITS - 1), np.int64)
        for j in range(kk.shape[1]):
            idx = np.minimum(xmin - first + j, src.shape[0] - 1)
            coef = np.where(j < cnt, kk[:, j], 0).astype(np.int64)
            acc += src[idx] * coef.reshape(-1, 1, 1)
        return np.clip(acc >> _PIL_PRECISION_BITS, 0, 255).astype(np.uint8)
    if need_h:
        return one_pass(img, out_w, 1)
    return one_pass(img, out_h, 0)


def demo_preprocess(img_u8, S: int, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)) -> torch.Tensor:
    """demo.py:162-166: Resize((S,S)) -> ToTensor -> Normalize, uint8 [H, W, 3] -> float32 [3, S, S]."""
    import numpy as np
    r = pil_resize_bilinear(img_u8, S, S)
    x = torch.from_numpy(r.astype(np.float32) / np.float32(255.0)).permute(2, 0, 1)
    return (x - torch.tensor(mean).view(3, 1, 1)) / torch.tensor(std).view(3, 1, 1)
