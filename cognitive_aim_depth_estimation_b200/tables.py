"""Input-independent tables of the focal / guidance path, built once per grid size on the host and cached.

The reference rebuilds these with Python loops on every forward (src/model.py:149-166 costs 0.12 s per call on CPU);
here they are vectorised, computed once in fp32 with the same elementary operations, and kept resident on the GPU.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

INSTRUCTIONS = ("center", "left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right")
_ALIASES = {"topleft": "top-left", "topright": "top-right", "bottomleft": "bottom-left",
            "bottomright": "bottom-right"}  # src/model.py:1330,1342,1354,1366


def canonical_instruction(s: str) -> str:
    s = s.lower()  # src/model.py:1270 `.lower()`
    return _ALIASES.get(s, s)


def focus_cell(name: str, g: int):
    """(y, x) of an off-centre instruction's focus cell (src/model.py:1282-1376), or None for "center" and unknown
    strings."""
    q, h, t = g // 4, g // 2, g * 3 // 4
    return {"left": (h, q), "right": (h, t), "top": (q, h), "bottom": (t, h), "top-left": (q, q), "top-right": (q, t),
            "bottom-left": (t, q), "bottom-right": (t, t)}.get(name)


def _disk_mask(fy: int, fx: int, g: int, r: int, hi: float, lo: float) -> torch.Tensor:
    """hi where the distance to (fy, fx) is <= r, lo where it is <= 2r, 1 elsewhere."""
    mask = torch.ones(g, g, dtype=torch.float32)
    y, x = torch.meshgrid(torch.arange(g), torch.arange(g), indexing="ij")
    dist = torch.sqrt(((y - fy) ** 2 + (x - fx) ** 2).double())  # math.sqrt on Python ints == exact fp64
    mask[dist <= 2 * r] = lo
    mask[dist <= r] = hi
    return mask.flatten()


def focus_mask(y: int, x: int, g: int) -> torch.Tensor:
    """Flattened g x g mask of the off-centre instructions with the focus moved to cell (y, x): 5.0 where
    dy^2 + dx^2 <= r^2, 2.0 where dy^2 + dx^2 <= 4 r^2, 1.0 elsewhere, r = max(1, g // 6) (src/model.py:1282-1376).
    Each of the eight off-centre instructions is this mask at its `focus_cell`; "center" is not (it has its own radius
    and weights).  Cell (y, x) of `CognitiveAimModel.depth_field` is the guided call with this mask."""
    if not (0 <= y < g and 0 <= x < g):
        raise ValueError(f"focus cell ({y}, {x}) lies outside the {g} x {g} grid")
    return _disk_mask(y, x, g, max(1, g // 6), 5.0, 2.0)


def instruction_mask(instruction: str, g: int) -> torch.Tensor:
    """Flattened g x g spatial mask of a textual instruction; unknown strings give all ones (reference behaviour)."""
    name = canonical_instruction(instruction)
    if name == "center":
        h = g // 2
        return _disk_mask(h, h, g, max(1, g // 4), 3.0, 1.5)
    cell = focus_cell(name, g)
    if cell is None:
        return torch.ones(g * g, dtype=torch.float32)
    return focus_mask(*cell, g)


def resolve_guidance(guidance, n: int) -> torch.Tensor:
    """str | Tensor[N'] -> fp32 CPU tensor [N] (bilinear resize when N' != N, src/model.py:1386-1398)."""
    g = int(math.sqrt(n))
    if isinstance(guidance, str):
        return instruction_mask(guidance, g)
    if not torch.is_tensor(guidance) or guidance.dim() != 1:
        raise ValueError("attention_guidance must be an instruction string or a 1-D tensor")
    v = guidance.detach().to("cpu", torch.float32)
    if v.numel() != n:
        gs = int(math.sqrt(v.numel()))
        if gs * gs != v.numel():
            raise ValueError(f"guidance of length {v.numel()} is not a square grid")
        v = F.interpolate(v.view(1, 1, gs, gs), size=(g, g), mode="bilinear", align_corners=False).reshape(-1)
    return v.contiguous()


def focal_position_encoding(n: int, d: int) -> torch.Tensor:
    """[N, D] 2-D sinusoidal table added to the patch tokens in every FocalStream (src/model.py:140-177)."""
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
    """[N] Gaussian centre prior, sigma = g/6 (src/model.py:208-231)."""
    g = int(n ** 0.5)
    if g * g != n:
        d = (torch.arange(n, dtype=torch.float) - n // 2).abs()
        return torch.exp(-d ** 2 / (2 * (n / 12) ** 2)) * strength
    c = g // 2
    y, x = torch.meshgrid(torch.arange(g), torch.arange(g), indexing="ij")
    dist = torch.sqrt((x - c).float() ** 2 + (y - c).float() ** 2)
    return torch.exp(-dist ** 2 / (2 * (g / 6) ** 2)).flatten() * strength


def interpolate_pos_embed(pos: torch.Tensor, g: int) -> torch.Tensor:
    """[1+g*g, D] DINOv2 position embedding for a g x g grid: identity at the native grid, bicubic otherwise
    (HF modeling_dinov2.py:57-95).  `pos` is [1, 1+N0, D]; computed on CPU fp32 once per resolution."""
    p = pos.detach().to("cpu", torch.float32)[0]
    n0 = p.shape[0] - 1
    if g * g == n0:
        return p.contiguous()
    g0 = int(round(n0 ** 0.5))
    grid = p[1:].reshape(1, g0, g0, -1).permute(0, 3, 1, 2)
    grid = F.interpolate(grid, size=(g, g), mode="bicubic", align_corners=False)
    return torch.cat([p[:1], grid.permute(0, 2, 3, 1).reshape(g * g, -1)], dim=0).contiguous()
