"""Host-side mirror of the reference's model surface (reference src/model.py), driving the sm_100a kernels.

`create_model(config, camera_info, device)` returns a `CognitiveAimModel` whose `forward` /
`forward_with_guidance` / `get_attention_weights` / `get_features` signatures, return shapes, side effects
(`_last_attention_weights`, `fusion_features`) and `state_dict()` names match the reference (src/model.py:1064,
1157, 1058, 1428, 1534; SURVEY.md §8b), so `demo.py` can switch imports and keep working.

Differences that are deliberate (DESIGN.md):
  * the forward runs ONLY on a CUDA sm_100 device through libcogaim_b200.so; there is no CPU fallback and errors
    are raised, never swallowed (the reference prints and falls back, src/model.py:1050-1056,1237-1240);
  * the reference's redundant passes (backbone x3, focal stream x4 in `forward`) are computed once;
  * output-dead work of the effective configuration (value path / projections in guided mode, DimensionAligners,
    LoRA) is not executed;
  * the CuriosityModule (src/model.py:586-688) runs on the GPU as often as the reference runs it (once per guided call,
    one to three times per `forward`), for its observable state — the `exploration_history` ring buffer and
    `history_pointer` — and, with `curiosity_guided_attention.enabled`, for the attention modulation.  Its two
    `randn_like` draws per run come from the global CPU generator, where a CPU reference takes them, so that the
    per-call random projection (src/model.py:1421) matches the reference under a shared `torch.manual_seed`.
"""
from __future__ import annotations

import contextlib
import functools
import math
import os
import weakref
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import ops, tables
from ._lib import RESIZE_MAX_SIDE as _RESIZE_MAX_SIDE  # largest photograph side the resize stages in shared memory
from ._lib import GUIDE_TAIL_MAX_B as _GUIDE_TAIL_MAX_B  # single guided calls of larger batches run the three-kernel tail
from ._lib import SWEEP_MAX_K as _SWEEP_MAX_K  # instructions per sweep: the sweep pool keeps one accumulator each
from ._lib import GUIDE_MANY_MAX_CALLS as _GUIDE_MANY_MAX_CALLS, GUIDE_MANY_MAX_ROWS as _GUIDE_MANY_MAX_ROWS
from ._lib import GUIDE_MANY_ROW_WORDS as _GUIDE_MANY_ROW_WORDS
from .config import DEFAULT_COGNITIVE_MODULES, EffectiveConfig, effective_config
from .init import reference_init_

_D = 768
_HEADS = 12
_LAYERS = 12
_MLP = 3072
_POOL_SPLITS = 32  # 1024 CTAs at B = 32: the 8-way split (256 CTAs) reached 39 % of the HBM rate (profiles/r01e_bw_kernels.md)
_LORA_PAD = 64  # fused LoRA: the rank is padded to one 64-wide K block of the tcgen05 GEMM (K = 768 + 64 = 13 blocks)
_MAX_SIDE = 1260  # 90 x 90 patch tokens: the focal vector stages keep an image's N <= 8192 columns in one CTA (csrc/focal.cu)


def _poison(tensors):
    """Test aid (CA_POISON_WS): fresh floating-point buffers start as NaN, so a kernel that reads a slot nobody wrote
    (e.g. an unwritten partial-sum column) produces NaN instead of plausible stale data."""
    if os.environ.get("CA_POISON_WS", "0") not in ("", "0"):
        for t in tensors:
            if torch.is_tensor(t) and t.is_floating_point():
                t.fill_(float("nan"))


# ------------------------------------------------------------------------------------------------------
# Parameter tree with the reference's state_dict names
# ------------------------------------------------------------------------------------------------------

def _param_specs(cfg: EffectiveConfig):
    """(name, shape, kind) in reference state_dict order; kind in {w, b, ones, zeros, const:<v>, buf...}."""
    s = []
    e = "backbone.embeddings."
    s += [(e + "cls_token", (1, 1, _D), "w"), (e + "mask_token", (1, _D), "zeros"),
          (e + "position_embeddings", (1, 1370, _D), "w"),
          (e + "patch_embeddings.projection.weight", (_D, 3, 14, 14), "w"),
          (e + "patch_embeddings.projection.bias", (_D,), "zeros")]
    for i in range(_LAYERS):
        p = f"backbone.encoder.layer.{i}."
        s += [(p + "norm1.weight", (_D,), "ones"), (p + "norm1.bias", (_D,), "zeros")]
        for n in ("query", "key", "value"):
            s += [(p + f"attention.attention.{n}.weight", (_D, _D), "w"),
                  (p + f"attention.attention.{n}.bias", (_D,), "zeros")]
        s += [(p + "attention.output.dense.weight", (_D, _D), "w"), (p + "attention.output.dense.bias", (_D,), "zeros"),
              (p + "layer_scale1.lambda1", (_D,), "ones"),
              (p + "norm2.weight", (_D,), "ones"), (p + "norm2.bias", (_D,), "zeros"),
              (p + "mlp.fc1.weight", (_MLP, _D), "w"), (p + "mlp.fc1.bias", (_MLP,), "zeros"),
              (p + "mlp.fc2.weight", (_D, _MLP), "w"), (p + "mlp.fc2.bias", (_D,), "zeros"),
              (p + "layer_scale2.lambda1", (_D,), "ones")]
    s += [("backbone.layernorm.weight", (_D,), "ones"), ("backbone.layernorm.bias", (_D,), "zeros")]
    if cfg.use_lora:  # src/model.py:822-831: one LoRALayer(768, 768, rank) per encoder layer, lora_B zero-initialised
        for i in range(_LAYERS):
            s += [(f"lora_layers.{i}.lora_A", (cfg.lora_rank, _D), "w"), (f"lora_layers.{i}.lora_B", (_D, cfg.lora_rank), "zeros")]

    def lin(name, o, i):
        return [(name + ".weight", (o, i), "w"), (name + ".bias", (o,), "zeros")]

    s += lin("ambient_stream.mlp.0", 256, _D) + lin("ambient_stream.mlp.3", 128, 256) + lin("ambient_stream.mlp.5", 64, 128)
    h = cfg.focal_hidden_dim
    s += [("focal_stream.initial_focus", (1, _D), "w")]
    for i in range(cfg.num_iterations):
        p = f"focal_stream.focal_streams.{i}."
        s += [(p + "adaptive_weight", (), "const:0.5")]
        s += lin(p + "query_proj", _D, _D) + lin(p + "key_proj", _D, _D) + lin(p + "value_proj", _D, _D)
        if cfg.curiosity_guided:  # src/model.py:73-79
            s += lin(p + "curiosity_modulator.0", h // 8, 1) + lin(p + "curiosity_modulator.2", 8, h // 8)
        s += lin(p + "projection.0", h, _D) + lin(p + "projection.3", h // 4, h)
    if cfg.curiosity_guided:  # src/model.py:333-339
        s += lin("focal_stream.curiosity_amplifier.0", 32, 1)
        s += lin("focal_stream.curiosity_amplifier.2", cfg.num_iterations, 32)
    s += lin("focal_stream.fusion.0", h // 2, h // 4 * cfg.num_iterations) + lin("focal_stream.fusion.2", h // 4, h // 2)
    if cfg.use_exif:
        s += [("exif_prior.camera_embedding.weight", (cfg.num_cameras, 64), "w")]
        s += lin("exif_prior.exif_encoder.0", 64, 3) + lin("exif_prior.exif_encoder.2", 64, 64)
        s += lin("exif_prior.fusion.0", 256, 128) + lin("exif_prior.fusion.3", 64, 256)
    s += lin("fusion.0", 192, 192)
    for n in ("ambient", "focal", "exif"):
        s += lin(f"{n}_dim_aligner.projection", _D, 64)
    s += [("decision_head.0.weight", (1, 192), "w"), ("decision_head.0.bias", (1,), "const:1.0")]
    s += lin("confidence_head.0", 1, 192)
    s += [("confidence_head.2.weight", (1, 1), "const:0.5"), ("confidence_head.2.bias", (1,), "const:2.0")]
    c = "curiosity_module."
    s += [(c + "curiosity_weights", (3,), "curw"), (c + "exploration_history", (1000,), "buf_zeros"),
          (c + "history_pointer", (), "buf_long")]
    s += lin(c + "encoder_mean.0", 384, _D) + lin(c + "encoder_mean.3", 192, 384)
    s += lin(c + "encoder_logvar.0", 384, _D) + lin(c + "encoder_logvar.3", 192, 384)
    s += lin(c + "decoder.0", 384, 192) + lin(c + "decoder.3", 192, 384)
    s += lin(c + "uncertainty_head.0", 192, _D) + lin(c + "uncertainty_head.2", 1, 192)
    if cfg.enable_hierarchical_curiosity:
        s += lin(c + "geometric_curiosity.0", 256, _D + 4) + lin(c + "geometric_curiosity.2", 1, 256)
        s += lin(c + "local_curiosity.0", 128, _D) + lin(c + "local_curiosity.2", 1, 128)
    s += lin("global_aligner.projection", _D, 3 * _D)
    return s


_NVTX = os.environ.get("CA_NVTX", "0") not in ("", "0")


@contextlib.contextmanager
def _nvtx(name: str):
    """Named NVTX range around a stage of the forward (CA_NVTX=1; visible in eager launches and at graph capture, e.g.
    under `nsys` / `ncu --nvtx`).  The reference has no tracing hooks at all (SURVEY.md §5)."""
    if not _NVTX:
        yield
        return
    torch.cuda.nvtx.range_push(name)
    try:
        yield
    finally:
        torch.cuda.nvtx.range_pop()


def _on_own_device(fn):
    """Run a public entry point with the model's GPU as the current CUDA device: every ca_* launch goes to the CURRENT
    device and torch.cuda.current_stream() is per device, so a model living on cuda:1 must not launch on cuda:0 just
    because the caller never called torch.cuda.set_device(1)."""
    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        dev = self._device()
        if dev.type != "cuda":
            return fn(self, *a, **k)  # argument checks first; _pack() then refuses: there is no CPU fallback
        with torch.cuda.device(dev):
            return fn(self, *a, **k)
    return wrapped


def _register(root: nn.Module, dotted: str, tensor: torch.Tensor, buffer: bool):
    mod = root
    parts = dotted.split(".")
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    if buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


class Scene:
    """The instruction-independent part of a guided call over one batch, kept for any number of later instructions
    (`CognitiveAimModel.encode` -> `guide` / `guide_sweep`).  Owns its buffers: the backbone tokens [B, T, 768] fp32
    (not the workspace the next forward overwrites), the last focal iteration's attention [B, N] (None with
    curiosity-guided attention, where every call's focal pass depends on its own curiosity score), the EXIF and camera
    indices on the device, and the CUDA graphs captured on these buffers.  Everything is released with the scene.
    Valid for the model and weights it was encoded with: re-packed weights (`load_state_dict`, `.to()`,
    `set_lora_adapters`) make it stale."""

    def __init__(self, model, B: int, S: int, tokens, base, exif, cam):
        self._model = weakref.ref(model)
        self._stamp = model._weights_version
        self.B, self.S, self.device = B, S, tokens.device
        self.tokens, self.base, self.exif, self.camera_idx = tokens, base, exif, cam
        self._graphs: Dict = {}
        self._guided = 0


class CognitiveAimModel(nn.Module):
    """Drop-in for the reference `CognitiveAimModel` (inference only)."""

    def __init__(self, config: dict, camera_info: Optional[dict] = None):
        super().__init__()
        self.config = config
        cfg = effective_config(config, camera_info)
        self.cfg = cfg
        if cfg.backbone_size != "base":
            raise NotImplementedError("only the DINOv2 ViT-B/14 backbone (backbone_size='base') is built")
        if not (cfg.use_ambient and cfg.use_iterative):
            raise NotImplementedError(
                "the B200 path is built for the configuration every shipped YAML resolves to "
                "(ambient_stream + iterative_focal_stream [+ exif_prior_database]); got cognitive_modules without them")
        if not 1 <= cfg.num_iterations <= 4:
            raise NotImplementedError("1..4 focal iterations are built (focal_value / focal_fusion kernels, csrc/heads.cu)")
        if cfg.focal_hidden_dim != 256:
            raise NotImplementedError("focal_hidden_dim must be 256 (the 768 -> 256 -> 64 focal projection is what the "
                                      "kernels instantiate; every shipped YAML resolves to it)")
        # attributes demo.py reads (demo.py:71-73,380-382)
        self.backbone_size = cfg.backbone_size
        self.feature_dim = cfg.feature_dim
        self.fusion_dim = cfg.fusion_dim
        # LoRA is dead code in the reference (quirk 4): `lora_layers` are built and saved, never applied.  Same here,
        # unless the NON-reference key `lora_merge_target` asks for the adapters to be merged into a weight (_lora_delta).
        self.use_lora = cfg.use_lora
        if cfg.lora_merge_target not in (None, "query", "key", "value", "attention_output"):
            raise ValueError("lora_merge_target must be one of query / key / value / attention_output")
        if cfg.lora_merge_target and not cfg.use_lora:
            raise ValueError("lora_merge_target needs use_lora: true")
        if cfg.lora_mode not in ("merge", "fused"):
            raise ValueError("lora_mode must be 'merge' or 'fused'")
        if cfg.lora_mode == "fused" and not cfg.lora_merge_target:
            raise ValueError("lora_mode: fused needs lora_merge_target (which projection the adapters apply to)")
        if cfg.lora_mode == "fused" and cfg.lora_rank > _LORA_PAD:
            raise ValueError(f"lora_mode: fused supports ranks up to {_LORA_PAD}")
        self.use_ambient, self.use_focal = cfg.use_ambient, cfg.use_focal
        self.use_iterative, self.use_exif = cfg.use_iterative, cfg.use_exif
        self.target_fusion_dim = 768
        # Parameter tree by reference name; values come from reference_init_, which consumes the global CPU generator
        # exactly like the reference's constructor: torch.manual_seed(s) + create_model(...) == the reference's weights.
        for name, shape, kind in _param_specs(cfg):
            t = torch.tensor(0) if kind == "buf_long" else torch.zeros(shape)
            _register(self, name, t, buffer=kind.startswith("buf"))
        reference_init_(dict(self.state_dict(keep_vars=True)), cfg)
        self._weights_version = 0  # bumped whenever the packed weights change: a Scene records it
        self._packed = None       # device-side packed weights (bf16 GEMM operands etc.)
        self._packed_key = None
        self._tables: Dict = {}   # per-grid tables (pos-embed, PE, centre bias, masks)
        self._ws: Dict = {}       # workspaces keyed by (B, S)
        self._many: Dict = {}     # guide_many buffers keyed by (S, R, m)
        self.input_size = None        # side uint8 [B, H, W, 3] inputs are resized to (demo.py's dataset.image_size); None = as given
        self.validate_inputs = True   # camera_idx range faults (checked on the device) are raised at the next call
        self._fault = None            # pinned int32 the heads kernel flags input faults in
        self.rng_replay_batch = None  # sharded runs: replay the reference's RNG draws at the GLOBAL batch size
        self.rng_replay_offset = 0    # ... and take this shard's rows of them
        # The ~110 launches of one forward are captured once per (batch, resolution, path) into a CUDA graph and
        # replayed: the launch gaps between dependent kernels (~0.4 ms of a 14 ms step) and the host-side launch work
        # disappear.  Per-call inputs (mask, per-call projection, EXIF) are copied into fixed buffers the graph reads.
        self.use_cuda_graphs = os.environ.get("CA_NO_GRAPHS", "0") in ("", "0")
        self.eval()

    # -- nn.Module protocol -----------------------------------------------------------------------------
    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("inference-only implementation: training mode is not built")
        return super().train(False)

    def _apply(self, fn, *a, **k):
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        self._invalidate()
        return super().load_state_dict(state_dict, strict=strict, assign=assign)

    def _invalidate(self):
        self._weights_version = getattr(self, "_weights_version", 0) + 1  # scenes encoded before are stale
        self._packed = None
        self._tables = {}
        self._ws = {}
        self._many = {}

    def _sd(self) -> Dict[str, torch.Tensor]:
        return dict(self.state_dict(keep_vars=True))

    # -- weight packing ---------------------------------------------------------------------------------
    def _lora_delta(self, sd, layer: int, target: str):
        """(alpha / rank) * lora_B @ lora_A of encoder layer `layer` when `lora_merge_target == target`, else None.

        The reference constructs one LoRALayer(768, 768, rank, alpha=16) per encoder layer (src/model.py:15-24, 822-831) and
        never applies it (its forward calls a non-existent `lora_projection`, :30), so the reference-faithful behaviour —
        the default here — is that LoRA parameters travel in the state_dict and change nothing.  For a deployment that
        does want y = W x + (alpha/rank) B A x on one of the 768 -> 768 projections, the adapters are MERGED into that
        projection's weight when the bf16 operands are packed: on an inference path with one adapter set this is
        exactly the LoRA output at zero extra HBM traffic, FLOPs or launches, which no epilogue-fused rank-16 MMA step
        can beat (that form only pays when adapters change per request, which the reference cannot express)."""
        if not self.cfg.use_lora or self.cfg.lora_merge_target != target or self.cfg.lora_mode != "merge":
            return None
        A = sd[f"lora_layers.{layer}.lora_A"].float()
        Bm = sd[f"lora_layers.{layer}.lora_B"].float()
        return (16.0 / self.cfg.lora_rank) * (Bm @ A)  # alpha defaults to 16 (:15), scaling = alpha / rank (:19)

    def _lora_fused(self) -> bool:
        return self.cfg.use_lora and self.cfg.lora_mode == "fused"

    def _ln_folded(self) -> bool:
        """CA_LN_FOLD=1 (read when the operands are packed): norm1 / norm2 folded into the GEMMs either side of them
        (ops.fold_layernorm, csrc/gemm.cuh EPI_LN_*) — no LayerNorm pass over HBM inside the encoder.  Opt-in: measured
        at B = 32 x 518^2 it moves 0.88 ms / step out of `layernorm` and 0.78 ms into the residual GEMMs (DESIGN.md §7),
        i.e. no faster than the separate kernels.  Never with fused LoRA adapters on q/k/v (their t = LN(x) A^T GEMM
        wants the normalised rows)."""
        if os.environ.get("CA_LN_FOLD", "0") in ("0", ""):
            return False
        return not (self._lora_fused() and self.cfg.lora_merge_target != "attention_output")

    def _write_lora(self, L, A, Bm):
        """Adapter (A [r, 768], B [768, r]) -> the packed operands of one layer: rows of `lora_a`, and the extra K columns
        of the target projection's weight, (alpha / r) * B in the rows of the adapted projection (zero elsewhere)."""
        r = self.cfg.lora_rank
        tgt = self.cfg.lora_merge_target
        dev = L["lora_a"].device
        L["lora_a"].zero_()
        L["lora_a"][:r] = A.detach().to(dev, torch.bfloat16)
        key = "wo_ext" if tgt == "attention_output" else "wqkv_ext"
        row0 = {"query": 0, "key": _D, "value": 2 * _D, "attention_output": 0}[tgt]
        L[key][:, _D:] = 0
        L[key][row0:row0 + _D, _D:_D + r] = ((16.0 / r) * Bm.detach().float()).to(dev, torch.bfloat16)

    def set_lora_adapters(self, adapters):
        """lora_mode: fused only — swap the adapters of some or all encoder layers WITHOUT re-packing the base weights:
        `adapters` maps layer index -> (lora_A [r, 768], lora_B [768, r]).  Takes effect at the next forward (the CUDA
        graphs read the operands through fixed addresses)."""
        if not self._lora_fused():
            raise ValueError("set_lora_adapters needs use_lora: true and lora_mode: fused")
        pk = self._pack()
        for i, (A, Bm) in adapters.items():
            self._write_lora(pk["layers"][i], A, Bm)
        self._weights_version += 1

    def _device(self) -> torch.device:
        return self.backbone.layernorm.weight.device

    def _pack(self):
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError(
                "CognitiveAimModel runs only on a CUDA sm_100 device (call .to('cuda')); there is no CPU fallback")
        if self._packed is not None:
            return self._packed
        ops._lib.check(ops._lib.load().ca_device_check(dev.index or 0), "ca_device_check")
        sd = {k: v.detach() for k, v in self._sd().items()}
        f32 = lambda t: t.to(dev, torch.float32).contiguous()  # noqa: E731
        b16 = lambda t: t.to(dev, torch.bfloat16).contiguous()  # noqa: E731
        pk = {}
        e = "backbone.embeddings."
        wpe = torch.zeros(_D, ops.PATCH_ROW_STRIDE, device=dev, dtype=torch.bfloat16)
        wpe[:, :588] = b16(sd[e + "patch_embeddings.projection.weight"].reshape(_D, 588))
        pk["patch_w"], pk["patch_b"] = wpe, f32(sd[e + "patch_embeddings.projection.bias"])
        pk["cls"] = f32(sd[e + "cls_token"].reshape(_D))
        layers = []
        for i in range(_LAYERS):
            p = f"backbone.encoder.layer.{i}."
            a = p + "attention.attention."
            def merged(w, target):
                d = self._lora_delta(sd, i, target)
                return w if d is None else w.float() + d.to(w.device)

            L = {
                "n1w": f32(sd[p + "norm1.weight"]), "n1b": f32(sd[p + "norm1.bias"]),
                "wqkv": b16(torch.cat([merged(sd[a + "query.weight"], "query"), merged(sd[a + "key.weight"], "key"),
                                       merged(sd[a + "value.weight"], "value")], 0)),
                "bqkv": f32(torch.cat([sd[a + "query.bias"], sd[a + "key.bias"], sd[a + "value.bias"]], 0)),
                "wo": b16(merged(sd[p + "attention.output.dense.weight"], "attention_output")),
                "bo": f32(sd[p + "attention.output.dense.bias"]),
                "ls1": f32(sd[p + "layer_scale1.lambda1"]),
                "n2w": f32(sd[p + "norm2.weight"]), "n2b": f32(sd[p + "norm2.bias"]),
                "w1": b16(sd[p + "mlp.fc1.weight"]), "b1": f32(sd[p + "mlp.fc1.bias"]),
                "w2": b16(sd[p + "mlp.fc2.weight"]), "b2": f32(sd[p + "mlp.fc2.bias"]),
                "ls2": f32(sd[p + "layer_scale2.lambda1"]),
            }
            if self._lora_fused():
                # lora_mode: fused — y = [h | t] [W | s B]^T with t = h A^T: the adapter is ONE extra 64-wide K block of the
                # projection's tcgen05 GEMM (rank padded with zeros), t written behind each row of the activation by a
                # small GEMM.  W itself is never touched: `set_lora_adapters` swaps adapters between calls by rewriting
                # A and the 64 extra columns only.
                tgt = self.cfg.lora_merge_target
                key = "wo" if tgt == "attention_output" else "wqkv"
                base = L[key]
                ext = torch.zeros(base.shape[0], _D + _LORA_PAD, device=dev, dtype=torch.bfloat16)
                ext[:, :_D] = base
                L[key + "_ext"] = ext
                L["lora_a"] = torch.zeros(_LORA_PAD, _D, device=dev, dtype=torch.bfloat16)
                del L[key]
                self._write_lora(L, sd[f"lora_layers.{i}.lora_A"], sd[f"lora_layers.{i}.lora_B"])
            if self._ln_folded():
                wq = torch.cat([merged(sd[a + "query.weight"], "query"), merged(sd[a + "key.weight"], "key"),
                                merged(sd[a + "value.weight"], "value")], 0).to(dev)
                L["wqkv"], L["bqkv"] = ops.fold_layernorm(wq, L["bqkv"], L["n1w"], L["n1b"])
                L["w1"], L["b1"] = ops.fold_layernorm(sd[p + "mlp.fc1.weight"].to(dev), L["b1"], L["n2w"], L["n2b"])
            layers.append(L)
        pk["layers"] = layers
        pk["zero64"] = torch.zeros(_LORA_PAD, device=dev)
        pk["lnw"], pk["lnb"] = f32(sd["backbone.layernorm.weight"]), f32(sd["backbone.layernorm.bias"])
        focal = []
        for i in range(self.cfg.num_iterations):
            p = f"focal_stream.focal_streams.{i}."
            focal.append({
                "wqk": b16(torch.cat([sd[p + "query_proj.weight"], sd[p + "key_proj.weight"]], 0)),
                "bqk": f32(torch.cat([sd[p + "query_proj.bias"], sd[p + "key_proj.bias"]], 0)),
                "wv": f32(sd[p + "value_proj.weight"]), "bv": f32(sd[p + "value_proj.bias"]),
                "pw0": f32(sd[p + "projection.0.weight"]), "pb0": f32(sd[p + "projection.0.bias"]),
                "pw1": f32(sd[p + "projection.3.weight"]), "pb1": f32(sd[p + "projection.3.bias"]),
            })
        pk["focal"] = focal
        pk["ffw0"], pk["ffb0"] = f32(sd["focal_stream.fusion.0.weight"]), f32(sd["focal_stream.fusion.0.bias"])
        pk["ffw1"], pk["ffb1"] = f32(sd["focal_stream.fusion.2.weight"]), f32(sd["focal_stream.fusion.2.bias"])
        z = lambda *s: torch.zeros(*s, device=dev)  # noqa: E731
        if self.use_exif:
            ex = {"cam_emb": f32(sd["exif_prior.camera_embedding.weight"]),
                  "exif_w0": f32(sd["exif_prior.exif_encoder.0.weight"]), "exif_b0": f32(sd["exif_prior.exif_encoder.0.bias"]),
                  "exif_w1": f32(sd["exif_prior.exif_encoder.2.weight"]), "exif_b1": f32(sd["exif_prior.exif_encoder.2.bias"]),
                  "exif_f0": f32(sd["exif_prior.fusion.0.weight"]), "exif_fb0": f32(sd["exif_prior.fusion.0.bias"]),
                  "exif_f1": f32(sd["exif_prior.fusion.3.weight"]), "exif_fb1": f32(sd["exif_prior.fusion.3.bias"])}
        else:
            ex = {"cam_emb": z(1, 64), "exif_w0": z(64, 3), "exif_b0": z(64), "exif_w1": z(64, 64), "exif_b1": z(64),
                  "exif_f0": z(256, 128), "exif_fb0": z(256), "exif_f1": z(64, 256), "exif_fb1": z(64)}
        hw = {
            "amb_w0": f32(sd["ambient_stream.mlp.0.weight"]), "amb_b0": f32(sd["ambient_stream.mlp.0.bias"]),
            "amb_w1": f32(sd["ambient_stream.mlp.3.weight"]), "amb_b1": f32(sd["ambient_stream.mlp.3.bias"]),
            "amb_w2": f32(sd["ambient_stream.mlp.5.weight"]), "amb_b2": f32(sd["ambient_stream.mlp.5.bias"]),
            **ex,
            "fus_w": f32(sd["fusion.0.weight"]), "fus_b": f32(sd["fusion.0.bias"]),
            "dec_w": f32(sd["decision_head.0.weight"]), "dec_b": f32(sd["decision_head.0.bias"]),
            "conf_w0": f32(sd["confidence_head.0.weight"]), "conf_b0": f32(sd["confidence_head.0.bias"]),
            "conf_w2": f32(sd["confidence_head.2.weight"]), "conf_b2": f32(sd["confidence_head.2.bias"]),
        }
        pk["heads_tensors"] = hw
        pk["heads"] = ops.make_heads_weights(hw)
        c = "curiosity_module."
        cw = {}
        for short, name in (("em", "encoder_mean"), ("el", "encoder_logvar"), ("dec", "decoder")):
            cw[short + "_w0"], cw[short + "_b0"] = f32(sd[c + name + ".0.weight"]), f32(sd[c + name + ".0.bias"])
            cw[short + "_w1"], cw[short + "_b1"] = f32(sd[c + name + ".3.weight"]), f32(sd[c + name + ".3.bias"])
        cw["unc_w0"], cw["unc_b0"] = f32(sd[c + "uncertainty_head.0.weight"]), f32(sd[c + "uncertainty_head.0.bias"])
        cw["unc_w1"], cw["unc_b1"] = f32(sd[c + "uncertainty_head.2.weight"]), f32(sd[c + "uncertainty_head.2.bias"])
        if self.cfg.enable_hierarchical_curiosity:
            cw["loc_w0"], cw["loc_b0"] = f32(sd[c + "local_curiosity.0.weight"]), f32(sd[c + "local_curiosity.0.bias"])
            cw["loc_w1"], cw["loc_b1"] = f32(sd[c + "local_curiosity.2.weight"]), f32(sd[c + "local_curiosity.2.bias"])
        cw["cur_w"] = f32(sd[c + "curiosity_weights"])
        pk["curiosity_tensors"] = cw
        pk["curiosity"] = ops.make_curiosity_weights(cw)
        pk["curiosity_mod"] = None
        if self.cfg.curiosity_guided:
            fsp = "focal_stream."
            amp = tuple(f32(sd[fsp + n]) for n in ("curiosity_amplifier.0.weight", "curiosity_amplifier.0.bias",
                                                   "curiosity_amplifier.2.weight", "curiosity_amplifier.2.bias"))
            mods = []
            for i in range(self.cfg.num_iterations):
                q = f"{fsp}focal_streams.{i}.curiosity_modulator."
                mods.append(tuple(f32(sd[q + n]) for n in ("0.weight", "0.bias", "2.weight", "2.bias")))
            pk["curiosity_mod_tensors"] = (amp, mods)
            pk["curiosity_mod"] = ops.make_curiosity_mod_weights(amp, mods)
            pk["adaptive_weight"] = [float(sd[f"{fsp}focal_streams.{i}.adaptive_weight"])
                                     for i in range(self.cfg.num_iterations)]
        pk["pos_param"] = sd[e + "position_embeddings"]
        self._packed = pk
        return pk

    def _grid_tables(self, g: int):
        dev = self._device()
        t = self._tables.get(g)
        if t is None:
            if g < 4:
                raise ValueError("patch grids smaller than 4 x 4 are not supported (the reference's degenerate-variance "
                                 "fallbacks, src/model.py:242-257, are not built)")
            n = g * g
            pk = self._pack()
            t = {"pos": tables.interpolate_pos_embed(pk["pos_param"], g).to(dev),
                 "pe": tables.focal_position_encoding(n, _D).to(dev),
                 "cbias": tables.center_bias(n).to(dev), "masks": {}}
            self._tables[g] = t
        return t

    def _mask(self, guidance, g: int) -> torch.Tensor:
        """[N] mask of one instruction / guidance tensor, or [B, N] for a list of per-image instructions (a superset of
        the reference, which broadcasts one instruction per call, src/model.py:1401)."""
        if isinstance(guidance, (list, tuple)):
            return torch.stack([self._mask(one, g) for one in guidance], dim=0)
        t = self._grid_tables(g)
        if isinstance(guidance, str):
            key = tables.canonical_instruction(guidance)
            m = t["masks"].get(key)
            if m is None:
                m = tables.resolve_guidance(guidance, g * g).to(self._device())
                t["masks"][key] = m
            return m
        return tables.resolve_guidance(guidance, g * g).to(self._device())

    def _workspace(self, B: int, S: int):
        key = (B, S)
        ws = self._ws.get(key)
        if ws is None:
            dev = self._device()
            g = S // 14
            N, T = g * g, g * g + 1
            P = ops.stats_partials(N)
            bf = dict(device=dev, dtype=torch.bfloat16)
            fl = dict(device=dev, dtype=torch.float32)
            ws = {
                "patches": torch.empty(B * N, ops.PATCH_ROW_STRIDE, **bf),
                "x": torch.empty(B * T, _D, **fl),
                # with lora_mode: fused the rows of the adapted projection's input carry 64 extra columns (t = h A^T)
                "h_ext": torch.empty(B * T, _D + (_LORA_PAD if self._lora_fused() and self.cfg.lora_merge_target != "attention_output" else 0), **bf),
                "att_ext": torch.empty(B * T, _D + (_LORA_PAD if self._lora_fused() and self.cfg.lora_merge_target == "attention_output" else 0), **bf),
                "qkv": torch.empty(B * T, 3 * _D, **bf),
                "mlp": torch.empty(B * T, _MLP, **bf), "tokens": torch.empty(B, T, _D, **fl),
                "xin": torch.empty(B * N, _D, **bf), "qk": torch.empty(B * N, 2 * _D, **bf),
                "pm": torch.empty(B, P, N, **fl), "ps": torch.empty(B, P, N, **fl), "pc": torch.empty(B, P, N, **fl),
                "rmax": torch.empty(B, N, **fl), "rinv": torch.empty(B, N, **fl),
                # span-relative exponentials of the focal scores (fp16) + the per-(row, span) factors that turn them into
                # softmax probabilities: the column sums are a bandwidth pass over E instead of a second Q K^T
                "E": torch.empty(B, N, 64 * ((N + 63) // 64), device=dev, dtype=torch.float16),
                "wtab": torch.empty(B, P, N, **fl),
                "attn": torch.empty(self.cfg.num_iterations, B, N, **fl), "cvec": torch.empty(B, N, **fl),
                "rowscale": torch.empty(2, B, N, **fl),
                # LayerNorm folding: per (row, 128-column span) (sum, M2) of the residual row; `h` then holds the raw rows
                "ln_stats": torch.empty(B * T, _D // 128, 2, **fl),
                "pool": torch.empty(B, _POOL_SPLITS, _D, **fl), "pool_pe": torch.empty(B, _POOL_SPLITS, _D, **fl),
                "feats": torch.empty(B, self.cfg.num_iterations, 64, **fl),
                "focal_feat": torch.empty(B, 64, **fl), "fused": torch.empty(B, 192, **fl),
                # per-call inputs, at fixed addresses so that captured graphs can be replayed
                "exif_in": torch.zeros(B, 3, **fl), "cam_in": torch.zeros(B, device=dev, dtype=torch.int64),
                "graphs": {},
                # the per-call buffers, one set per number of CuriosityModule runs (_sweep_buffers)
                "sweeps": {},
            }
            ws["h"], ws["att"] = ws["h_ext"][:, :_D], ws["att_ext"][:, :_D]
            _poison(t for k, t in ws.items() if k != "exif_in")
            if len(self._ws) >= 4:  # keep the cache bounded
                self._ws.pop(next(iter(self._ws)))
            self._ws[key] = ws
        return ws

    # -- stages -----------------------------------------------------------------------------------------
    def _pinned_slot(self):
        """Next buffer of a 4-deep ring of pinned host staging areas for the per-call projection and the curiosity
        draws; waits (normally not at all: the copy is four calls old) until the previous async copy out of it has
        completed."""
        ring = getattr(self, "_pinned_ring", None)
        if ring is None:
            ring = {"slots": [{"draws": {}, "event": torch.cuda.Event()} for _ in range(4)], "next": 0}
            self._pinned_ring = ring
        slot = ring["slots"][ring["next"]]
        ring["next"] = (ring["next"] + 1) % len(ring["slots"])
        slot["event"].synchronize()
        return slot

    def _stage_runs(self, cs, draws):
        """The host draws of R CuriosityModule runs, made before any buffer is looked up — R tuples (eps [B,192],
        noise [B,768]) of an un-guided forward, or `_sweep_draws`' (eps, noise, projection weight, bias) of R guided calls
        — through the pinned staging of one ring slot into the sweep buffers' cur_eps, cur_noise (and tmpw, tmpb)."""
        R, B = len(draws), draws[0][0].shape[0]

        def fill(bufs):
            for k, d in enumerate(draws):
                for buf, t in zip(bufs, d):
                    buf[k].copy_(t)
            return [(cs[dst], buf) for dst, buf in zip(("cur_eps", "cur_noise", "tmpw", "tmpb")[:len(draws[0])], bufs)]

        self._stage_pinned((B, R), ((R, B, 192), (R, B, _D), (R, 64, _D), (R, 64)), fill)

    def _stage_pinned(self, key, shapes, fill):
        """Per-call host inputs through the pinned staging of one ring slot: `fill` writes the slot's fp32 buffers of
        `shapes` (kept per `key`) and returns the (device destination, pinned source) pairs to read, in order."""
        slot = self._pinned_slot()
        # pinned buffers per key, kept for the life of the model: a kernel reads them asynchronously, so they must
        # never go back to the host allocator while a read may be in flight (the slot's event guards their REUSE)
        bufs = slot["draws"].get(key)
        if bufs is None:
            bufs = slot["draws"][key] = tuple(torch.empty(*s).pin_memory() for s in shapes)
        pairs = fill(bufs)
        # SM-side reads of the pinned staging area (ops.fetch_pinned), not cudaMemcpyAsync: these few hundred KB must not
        # wait on the H2D copy engine behind the application's upload of the next image batch
        for dst, buf in pairs:
            ops.fetch_pinned(dst, buf)
        slot["event"].record()

    @staticmethod
    def _check_side(S):
        if S < 56 or S % 14 != 0 or S > _MAX_SIDE:
            raise ValueError(f"image side must be a multiple of 14 in [56, {_MAX_SIDE}] (got {S})")

    def _check_list(self, images, S):
        """B of a list of photographs of individual sizes (uint8 [H_i, W_i, 3], CPU or CUDA) resized to S x S."""
        if len(images) == 0:
            raise ValueError("empty list of images")
        for i, t in enumerate(images):
            if not torch.is_tensor(t) or t.dtype != torch.uint8 or t.dim() != 3 or t.shape[-1] != 3:
                raise ValueError(f"image {i} of the list must be a uint8 [H, W, 3] tensor")
            if not 0 < min(t.shape[0], t.shape[1]) <= max(t.shape[0], t.shape[1]) <= _RESIZE_MAX_SIDE:
                raise ValueError(f"image {i} of the list is {t.shape[0]} x {t.shape[1]}: sides must be in "
                                 f"[1, {_RESIZE_MAX_SIDE}]")
        if S is None:
            raise ValueError("a list of images is resized to model.input_size: set it (demo.py's dataset.image_size)")
        self._check_side(S)
        return len(images)

    def _check_images(self, images):
        """(B, S) of a forward input: float [B, 3, S, S] already normalised (what the reference's forward takes), or —
        an extension for the demo-shaped flow — uint8 [B, H, W, 3] straight from the decoder (demo.py:312-319 on the
        GPU: Resize((input_size, input_size)) when the size differs, ToTensor, Normalize, fused with the patchify), or a
        list of uint8 [H_i, W_i, 3] photographs of individual sizes, all resized to input_size (demo.py:406-432
        `predict_batch` over a folder)."""
        if isinstance(images, (list, tuple)):
            return self._check_list(images, self.input_size), self.input_size
        if torch.is_tensor(images) and images.dtype == torch.uint8:
            if images.dim() != 4 or images.shape[-1] != 3:
                raise ValueError("uint8 images must be [B, H, W, 3]")
            B, H, W, _ = images.shape
            S = self.input_size if self.input_size is not None else H
            if self.input_size is None and H != W:
                raise ValueError("uint8 images must be square, or set model.input_size to resize like demo.py")
            self._check_side(S)
            return B, S
        if not torch.is_tensor(images) or images.dim() != 4 or images.shape[1] != 3:
            raise ValueError("images must be a [B, 3, S, S] tensor")
        B, _, H, W = images.shape
        if H != W or H < 56 or H > _MAX_SIDE:
            raise ValueError(f"images must be square with side in [56, {_MAX_SIDE}] (got {H} x {W})")
        if not images.is_floating_point():
            raise ValueError("images must be floating point (already normalised) or uint8 [B, H, W, 3]")
        return B, H

    def _patch_rows(self, images, ws, S: int):
        """im2col rows (bf16 [B*N, 592]) of the batch into ws['patches']; returns (patches, tensors to keep alive).
        Runs eagerly in front of the (possibly replayed) graph, so lists of other sizes replay the same graph."""
        dev = self._device()
        if isinstance(images, (list, tuple)):
            src = [t.to(dev).contiguous() for t in images]
            u8 = ops.resize_u8_list(src, S, S)  # demo.py:162-163 per image, the whole batch in one launch per pass
            return ops.preprocess_u8(u8, ws["patches"]), (src, u8)
        if images.dtype == torch.uint8:
            u8 = images.to(dev).contiguous()
            if tuple(u8.shape[1:3]) != (S, S):
                u8 = ops.resize_u8(u8, S, S)  # demo.py:162-163: Pillow's antialiased bilinear resample, bit-exact
            return ops.preprocess_u8(u8, ws["patches"]), u8
        x = images.to(dev, torch.float32).contiguous()
        return ops.patchify_f32(x, ws["patches"]), x

    @_on_own_device
    def backbone_tokens(self, images: torch.Tensor, *, patches: Optional[torch.Tensor] = None, B=None, S=None):
        """DINOv2 ViT-B/14 `last_hidden_state` [B, 1+N, 768] fp32 (HF modeling_dinov2.py:459-485).
        `patches` (bf16 [B*N, 592] from `preprocess_u8`) may be given instead of images.
        The result is a BORROWED view of the (B, S) workspace: the next call at the same shape overwrites it — clone it to
        keep it (the forward passes return fresh tensors)."""
        if patches is None:
            B, S = self._check_images(images)
        pk = self._pack()
        dev = self._device()
        g = S // 14
        N, T = g * g, g * g + 1
        ws = self._workspace(B, S)
        tb = self._grid_tables(g)
        if patches is None:
            patches, images = self._patch_rows(images, ws, S)
        self._run(ws, ("backbone", patches.data_ptr()), lambda: self._backbone_layers(ws, patches, B, S))
        return ws["tokens"]

    def _backbone_layers(self, ws, patches, B: int, S: int):
        """Embedding GEMM + 12 encoder layers + final LayerNorm on patch rows already in `patches` (graph-capturable:
        fixed addresses, no host synchronisation, no allocation)."""
        pk = self._packed
        g = S // 14
        N, T = g * g, g * g + 1
        tb = self._tables[g]
        x, h = ws["x"], ws["h"]
        with _nvtx("cogaim.embeddings"):
            ops.cls_rows(x, pk["cls"], tb["pos"], B, T, _D)
            ops.gemm(patches, pk["patch_w"], ops.EPI_PATCH_F32, x, bias=pk["patch_b"], pos=tb["pos"], patches_per_img=N)
        fused = self._lora_fused()
        on_out = fused and self.cfg.lora_merge_target == "attention_output"
        fold = self._ln_folded()
        st = ws["ln_stats"]
        if fold:
            ops.ln_shadow(x, h, st)  # the residual epilogues keep (h, st) current from here on
        for li, L in enumerate(pk["layers"]):
          with _nvtx(f"cogaim.layer{li}"):
            last = li == len(pk["layers"]) - 1
            if fold:
                ops.gemm_ln(h, L["wqkv"], ops.EPI_LN_BIAS_BF16, ws["qkv"], bias=L["bqkv"], stats=st)
            else:
                ops.layernorm(x, L["n1w"], L["n1b"], h)
                if fused and not on_out:
                    ops.gemm(h, L["lora_a"], ops.EPI_BIAS_BF16, ws["h_ext"][:, _D:], bias=pk["zero64"])  # t = h A^T
                    ops.gemm(ws["h_ext"], L["wqkv_ext"], ops.EPI_BIAS_BF16, ws["qkv"], bias=L["bqkv"])
                else:
                    ops.gemm(h, L["wqkv"], ops.EPI_BIAS_BF16, ws["qkv"], bias=L["bqkv"])
            ops.attention(ws["qkv"], ws["att"], B, T, _HEADS)
            a_out, w_out = (ws["att_ext"], L["wo_ext"]) if on_out else (ws["att"], L["wo"])
            if on_out:
                ops.gemm(ws["att"], L["lora_a"], ops.EPI_BIAS_BF16, ws["att_ext"][:, _D:], bias=pk["zero64"])
            if fold:
                ops.gemm_ln(a_out, w_out, ops.EPI_RESID_LN_F32, x, bias=L["bo"], ls=L["ls1"], stats=st, shadow=h)
                ops.gemm_ln(h, L["w1"], ops.EPI_LN_GELU_BF16, ws["mlp"], bias=L["b1"], stats=st)
            else:
                ops.gemm(a_out, w_out, ops.EPI_RESID_F32, x, bias=L["bo"], ls=L["ls1"])
                ops.layernorm(x, L["n2w"], L["n2b"], h)
                ops.gemm(h, L["w1"], ops.EPI_GELU_BF16, ws["mlp"], bias=L["b1"])
            if fold and not last:
                ops.gemm_ln(ws["mlp"], L["w2"], ops.EPI_RESID_LN_F32, x, bias=L["b2"], ls=L["ls2"], stats=st, shadow=h)
            else:  # the final LayerNorm reads the fp32 rows itself
                ops.gemm(ws["mlp"], L["w2"], ops.EPI_RESID_F32, x, bias=L["b2"], ls=L["ls2"])
        with _nvtx("cogaim.final_norm"):
            ops.layernorm(x, pk["lnw"], pk["lnb"], ws["tokens"].view(B * T, _D))
        return ws["tokens"]

    def _run(self, ws, key, fn, graphs=None):
        """Run `fn` (a fixed sequence of launches on fixed buffers): eagerly, or — with `use_cuda_graphs` — captured
        once per key and replayed.  The first call runs eagerly as well: it performs the library's one-time
        allocations and attribute settings, which are illegal during capture.  `graphs`: the store of the graphs
        (default: the workspace's)."""
        if not self.use_cuda_graphs or ops.tracing_events():
            fn()
            return
        if graphs is None:
            graphs = ws["graphs"]
        graph = graphs.get(key)
        if graph is None:
            fn()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                n0 = ops.launch_count()
                fn()
                launches = ops.launch_count() - n0
            # a graph kept outside the workspace (a Scene's) keeps the workspace buffers it reads alive
            graphs[key] = (graph, launches) if graphs is ws["graphs"] else (graph, launches, ws)
            if len(graphs) > 8:
                graphs.pop(next(iter(graphs)))
            return  # the eager run above produced this call's results
        graph[0].replay()
        ops.count_launches(graph[1])

    def _focal_iterations(self, ws, B: int, g: int, want_features: bool, cur_weight=None, tokens=None):
        """IterativeFocalStream (src/model.py:391-455) on `tokens` [B, 1+N, 768] (default: the workspace's; a scene's
        for a guide call): per iteration Q|K projection, one tensor-core pass over Q K^T (row statistics + stored exponentials), the column sums
        as a bandwidth pass, and the vector epilogue.  `cur_weight` [n_iters, B]: curiosity modulation (only with
        curiosity_guided_attention.enabled, :264-276).  Returns the last iteration's attention [B, N]; fills
        ws['focal_feat'] when `want_features`."""
        pk = self._pack()
        tb = self._grid_tables(g)
        N = g * g
        scale_log2 = ops.LOG2E / math.sqrt(_D // 8)  # src/model.py:69 (single head, sqrt(768 // 8))
        iters = self.cfg.num_iterations
        tokens = ws["tokens"] if tokens is None else tokens
        qk = ws["qk"]
        q, k = qk[:, :_D], qk[:, _D:]
        rs = None
        for i in range(iters):
          with _nvtx(f"cogaim.focal{i}"):
            F_ = pk["focal"][i]
            ops.focal_input(tokens, tb["pe"], rs, ws["xin"], B, N, _D)
            ops.gemm(ws["xin"], F_["wqk"], ops.EPI_BIAS_BF16, qk, bias=F_["bqk"])
            common = dict(M=N, N=N, K=_D, lda=2 * _D, ldw=2 * _D, batch=B, a_batch_stride=N * 2 * _D,
                          w_batch_stride=N * 2 * _D, scale_log2=scale_log2)
            E = ws["E"]
            ops.gemm(q, k, ops.EPI_ROWSTATS, E, part_a=ws["pm"], part_b=ws["ps"], ldo=E.stride(1),
                     out_batch_stride=E.stride(0), **common)
            ops.rowstats_merge(ws["pm"], ws["ps"], None, None, None, ws["wtab"])
            ops.colsum_e(E, ws["wtab"], ws["pc"], B, N)
            last = i == iters - 1
            rs_out = None if last else ws["rowscale"][i % 2]
            ops.focal_finalize(ws["pc"], tb["cbias"], ws["attn"][i], rs, rs_out, B, N, self.cfg.focus_strength, 0,
                               cur_weight=None if cur_weight is None else cur_weight[i],
                               adaptive_weight=pk["adaptive_weight"][i] if cur_weight is not None else 0.5)
            if want_features:
                # value path re-associated: sum_i a_i (A V)_i = ((a^T A) x~) Wv^T + bv   (src/model.py:204,308)
                ops.rowstats_merge(ws["pm"], ws["ps"], ws["attn"][i], None, None, ws["wtab"])
                ops.colsum_e(E, ws["wtab"], ws["pc"], B, N)
                ops.focal_finalize(ws["pc"], None, ws["cvec"], None, None, B, N, 0.0, 1)
                T = N + 1
                ops.weighted_pool(tokens, T * _D, 1, ws["cvec"], rs, ws["pool"], B, N, _D, _POOL_SPLITS)
                ops.weighted_pool(tb["pe"], 0, 0, ws["cvec"], None, ws["pool_pe"], B, N, _D, _POOL_SPLITS)
                ops.focal_value(tok_partial=ws["pool"], pe_partial=ws["pool_pe"], splits=_POOL_SPLITS, wv=F_["wv"],
                                bv=F_["bv"], proj_w0=F_["pw0"], proj_b0=F_["pb0"], proj_w1=F_["pw1"], proj_b1=F_["pb1"],
                                feat_out=ws["feats"], it=i, n_iters=iters, B=B)
            rs = rs_out
        if want_features:
            ops.focal_fusion(ws["feats"], iters, pk["ffw0"], pk["ffb0"], pk["ffw1"], pk["ffb1"], ws["focal_feat"], B)
        return ws["attn"][iters - 1]

    @staticmethod
    def _check_per_image(guidance, B: int):
        if isinstance(guidance, (list, tuple)) and len(guidance) != B:
            raise ValueError(f"{len(guidance)} per-image instructions for a batch of {B}")

    def _check_exif(self, exif_data, B: int):
        """The EXIF entry counts against the batch, before anything is drawn or launched (_exif_tensors converts)."""
        if exif_data is None or not self.use_exif:
            return
        for key in ("focal_length", "aperture", "iso", "camera_idx"):
            if key not in exif_data:
                raise ValueError(f"exif_data is missing '{key}'")
            n = exif_data[key].numel() if torch.is_tensor(exif_data[key]) else torch.as_tensor(exif_data[key]).numel()
            if n != B:
                raise ValueError(f"exif_data['{key}'] has {n} entries for a batch of {B}")

    def _exif_tensors(self, exif_data, B: int):
        if exif_data is None or not self.use_exif:
            return None, None
        dev = self._device()

        def flat(key, dtype):
            if key not in exif_data:
                raise ValueError(f"exif_data is missing '{key}'")
            t = exif_data[key]
            if not torch.is_tensor(t):
                t = torch.as_tensor(t)
            t = t.reshape(-1).to(dev, dtype)
            if t.numel() != B:
                raise ValueError(f"exif_data['{key}'] has {t.numel()} entries for a batch of {B}")
            return t

        cont = torch.stack([flat("focal_length", torch.float32), flat("aperture", torch.float32),
                            flat("iso", torch.float32)], dim=1).contiguous()
        cam_in = exif_data["camera_idx"] if "camera_idx" in exif_data else None
        if self.validate_inputs and cam_in is not None and not (torch.is_tensor(cam_in) and cam_in.is_cuda):
            # host-resident indices: checking them costs no synchronisation, so fail at once like nn.Embedding would
            c = torch.as_tensor(cam_in).reshape(-1)
            if c.numel() and (int(c.min()) < 0 or int(c.max()) >= self.cfg.num_cameras):
                raise ValueError("camera_idx out of range")
        cam = flat("camera_idx", torch.int64).contiguous()
        # device-resident indices are range-checked inside the heads kernel (no device-to-host sync): _raise_on_fault
        return cont, cam

    def _fault_word(self) -> torch.Tensor:
        if self._fault is None:
            self._fault = torch.zeros(1, dtype=torch.int32).pin_memory()
        return self._fault

    def _raise_on_fault(self, sync: bool = False):
        """Input faults found by the kernels of EARLIER calls (a camera_idx outside the embedding table: clamped on the
        device, flagged in a pinned word the host can read without synchronising).  Called at the start of every
        forward; `check_inputs(sync=True)` waits for the device first, i.e. also covers the call just made."""
        if self._fault is None:
            return
        if sync:
            torch.cuda.synchronize(self._device())
        if self.validate_inputs and int(self._fault[0]) != 0:
            self._fault.zero_()
            raise ValueError("camera_idx out of range (reported by the device for an earlier forward call; the lookup "
                             "was clamped into the table)")

    def check_inputs(self, sync: bool = True):
        """Raise ValueError if any forward so far was given an out-of-range camera_idx (reference: nn.Embedding raises
        IndexError at src/model.py:491)."""
        self._raise_on_fault(sync=sync)

    def _curiosity_draw(self, B: int):
        """One CuriosityModule run draws randn(B,192) then randn(B,768) on the global CPU generator in eval
        (src/model.py:609,744), before the per-call projection is initialised (:1421).  A batch-sharded run sets
        `rng_replay_batch` / `rng_replay_offset` to the global batch / this shard's first image so every shard sees the
        draws (and hence the projection) of the un-sharded call.  Returns this shard's (eps [B,192], noise [B,768])."""
        Bg = self.rng_replay_batch or B
        lo = self.rng_replay_offset if self.rng_replay_batch else 0
        eps = torch.randn(Bg, 192)
        noise = torch.randn(Bg, 768)
        return eps[lo:lo + B], noise[lo:lo + B]

    def _curiosity_runs(self, cs, tokens, B: int, T: int, roles):
        """Device side of the CuriosityModule runs of one call on `tokens`, in the reference's order: rewards, ring-buffer
        update, and (curiosity-guided configuration only) the attention modulation weights of each run, in the sweep
        buffers `cs`.  The score of the un-guided attention runs is clamped to [0.5, 1] (src/model.py:1107, :1141); the others
        are not."""
        pk = self._packed
        cm = self.curiosity_module
        # Output-dead under the shipped configurations and latency-bound (one CTA per image through ten small dense
        # layers): it runs on a side stream, forked here and joined by `_curiosity_join`, under the focal stream's GEMMs.
        # The fork / join are stream dependencies, so they are captured into the CUDA graph as a parallel branch.
        side = None
        if not self.cfg.curiosity_guided and not ops.tracing_events():
            side = getattr(self, "_side_stream", None)
            if side is None or side.device != self._device():
                side = self._side_stream = torch.cuda.Stream(device=self._device())
            side.wait_stream(torch.cuda.current_stream())
        self._curiosity_side = side
        with torch.cuda.stream(side) if side is not None else contextlib.nullcontext():
            self._curiosity_launches(cs, tokens, B, T, roles, pk, cm)

    def _curiosity_join(self):
        side, self._curiosity_side = getattr(self, "_curiosity_side", None), None
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)

    def _curiosity_launches(self, cs, tokens, B, T, roles, pk, cm):
        for j, role in enumerate(roles):
            ops.curiosity(pk["curiosity"], tokens=tokens, tokens_per_img=T, eps=cs["cur_eps"][j],
                          noise=cs["cur_noise"][j], reward_raw=cs["cur_raw"][j], reward=cs["cur_reward"][j],
                          history=cm.exploration_history, history_pointer=cm.history_pointer, B=B)
            if self.cfg.curiosity_guided:
                lo, hi = (0.5, 1.0) if role in ("last", "ret") else (1.0, 0.0)
                ops.curiosity_modulation(pk["curiosity_mod"], cs["cur_reward"][j], lo, hi, cs["cur_weight"][j], B,
                                         self.cfg.num_iterations, self.cfg.focal_hidden_dim // 8)

    def _curiosity_key(self):
        cm = self.curiosity_module
        return (cm.exploration_history.data_ptr(), cm.history_pointer.data_ptr())

    # -- public forward passes --------------------------------------------------------------------------
    @torch.no_grad()
    @_on_own_device
    def forward_with_guidance(self, images, exif_data=None, attention_guidance=None, return_attention=False):
        """reference src/model.py:1157-1240.  Returns (depth [B,1], confidence [B,1][, attention [B,N]]).  With EXIF and a
        guidance this is the sweep of one instruction, `forward_with_guidance_sweep(images, exif_data, [guidance])`."""
        self._raise_on_fault()
        if attention_guidance is None and exif_data is not None and self.use_exif:
            # guidance None -> plain focal-stream features and attention (:1206-1212)
            return self._forward_impl(images, exif_data, return_attention, mode="guided_none")
        if exif_data is None or not self.use_exif:
            # reference: the 128-wide concat fails inside `fusion`, the except branch falls back to forward()
            # (:1237-1240) AFTER the guided attention was stored at :1212 — reproduce exactly that end state.
            return self._forward_impl(images, exif_data, return_attention, mode="guided_fallback",
                                      guidance=attention_guidance)
        depth, conf, _ = self.forward_with_guidance_sweep(images, exif_data, [attention_guidance], return_attention=True)
        heat = self._last_attention_weights  # :1212
        return (depth[0], conf[0], heat) if return_attention else (depth[0], conf[0])

    def _sweep_draws(self, B: int, K: int):
        """The host-side random draws of K successive guided calls, in the reference's order per call: the
        CuriosityModule's randn(B,192), randn(B,768) (src/model.py:609,744), then the fresh nn.Linear(768, 64) (:1421).
        Returns K tuples (eps [B,192], noise [B,768], projection weight [64,768], projection bias [64])."""
        out = []
        for _ in range(K):
            eps, noise = self._curiosity_draw(B)
            tmp = nn.Linear(_D, 64)
            out.append((eps, noise, tmp.weight.detach(), tmp.bias.detach()))
        return out

    def _sweep_buffers(self, ws, B: int, S: int, R: int):
        """The per-call buffers ("sweep" buffers) of a call with R CuriosityModule runs (rows r * B + b), kept with the
        (B, S) workspace whose backbone, focal and value-path buffers every call shares.  R guided calls of a sweep (R = 1: a single
        guided call or a depth field) use every row; an un-guided forward's heads write rows 0..B-1 of depth / conf and
        its `guided_fallback` softmax uses row 0 of mask_in / heat / argmax.  An un-guided forward of one run and a single
        guided call share a set: both write it before they read it, on one stream."""
        cs = ws["sweeps"].get(R)
        if cs is None:
            dev = self._device()
            N = (S // 14) ** 2
            fl = dict(device=dev, dtype=torch.float32)
            cs = {
                # the host draws (_stage_runs): a Gaussian pair per run, and the fresh projection of each guided call
                "cur_eps": torch.zeros(R, B, 192, **fl), "cur_noise": torch.zeros(R, B, _D, **fl),
                "tmpw": torch.empty(R, 64, _D, **fl), "tmpb": torch.empty(R, 64, **fl),
                # rewards per run; modulation weights per (run, iteration)
                "cur_raw": torch.empty(R, B, **fl), "cur_reward": torch.empty(R, B, **fl),
                "cur_weight": torch.empty(R, self.cfg.num_iterations, B, **fl),
                # curiosity-guided attention: each run's focal attention, modulated by its own score
                "base": torch.empty(R, B, N, **fl) if self.cfg.curiosity_guided and R > 1 else None,
                "mask_in": torch.empty(R, B, N, **fl), "heat": torch.empty(R, B, N, **fl),
                "argmax": torch.empty(R, B, device=dev, dtype=torch.int32),
                "tail_pool": torch.empty(R * B, _POOL_SPLITS, _D, **fl),
                # per-image tickets of ops.guide_tail: zero here, and every launch leaves them at zero
                "tail_ticket": torch.zeros(B, device=dev, dtype=torch.int32),
                "depth": torch.empty(R, B, **fl), "conf": torch.empty(R, B, **fl),
            }
            # a function is handed the workspace and the sweep buffers separately: no name may mean two buffers
            assert ws.keys().isdisjoint(cs), sorted(ws.keys() & cs.keys())
            _poison(cs.values())
            ws["sweeps"][R] = cs
        return cs

    @staticmethod
    def _check_guidances(guidances):
        """K of an instruction sweep's guidance list (checked before anything is drawn or launched)."""
        if not isinstance(guidances, (list, tuple)):
            raise ValueError("guidances must be a list of K instructions / guidance tensors / per-image lists")
        K = len(guidances)
        if not 1 <= K <= _SWEEP_MAX_K:
            raise ValueError(f"an instruction sweep takes 1..{_SWEEP_MAX_K} guidances, got {K}")
        if any(gd is None for gd in guidances):
            raise ValueError("a None guidance runs the un-guided focal path (src/model.py:1206-1212): use "
                             "forward_with_guidance for it")
        return K

    def _sweep_masks(self, guidances, B: int, g: int):
        """The K [B, N] masks of a sweep (views: strings and [N] guidance broadcast over the batch)."""
        N = g * g
        masks = []
        for gd in guidances:
            m = self._mask(gd, g)
            if m.dim() == 2 and m.shape[0] != B:
                raise ValueError(f"{m.shape[0]} per-image instructions for a batch of {B}")
            masks.append(m.expand(B, N))
        return masks

    def _guided_device(self, ws, cs, tokens, B: int, g: int, K: int, base, exif, cam):
        """Device side of K guided calls after the backbone, on `tokens` (the workspace's, or a Scene's for `guide_sweep`):
        the K CuriosityModule runs, the focal pass (`base` [B, N] when it is shared; with curiosity-guided attention one
        pass per call), then the tail: for one call of at most _GUIDE_TAIL_MAX_B images ops.guide_tail (one launch), else
        the softmax, pool and heads of the K * B rows.  Shared by every guided entry point."""
        pk = self._packed
        N, T = g * g, g * g + 1
        self._curiosity_runs(cs, tokens, B, T, ("guided",) * K)
        base_k_stride = 0
        if self.cfg.curiosity_guided and K == 1:
            base = self._focal_iterations(ws, B, g, want_features=False, cur_weight=cs["cur_weight"][0], tokens=tokens)
        elif self.cfg.curiosity_guided:
            # each call's focal attention is modulated by its own curiosity score (src/model.py:264-276)
            for k in range(K):
                cs["base"][k].copy_(self._focal_iterations(ws, B, g, want_features=False, cur_weight=cs["cur_weight"][k],
                                                           tokens=tokens))
            base, base_k_stride = cs["base"], B * N
        elif base is None:
            base = self._focal_iterations(ws, B, g, want_features=False, tokens=tokens)
        heads_in = dict(exif=exif, camera_idx=cam, num_cameras=self.cfg.num_cameras,
                        fault_ptr=self._fault_word().data_ptr())
        if K == 1 and B <= _GUIDE_TAIL_MAX_B:  # one launch (include/cogaim_b200.h CA_GUIDE_TAIL_MAX_B)
            ops.guide_tail(pk["heads"], base=base, mask=cs["mask_in"][0], heat=cs["heat"][0], argmax=cs["argmax"][0],
                           ticket=cs["tail_ticket"], tokens=tokens, depth=cs["depth"][0], conf=cs["conf"][0], B=B,
                           N=N, pool_partial=cs["tail_pool"], tmp_w=cs["tmpw"][0], tmp_b=cs["tmpb"][0], **heads_in)
        else:
            ops.guided_softmax_sweep(base, base_k_stride, cs["mask_in"], cs["heat"], cs["argmax"], K, B, N)
            ops.weighted_pool_sweep(tokens, T * _D, 1, cs["heat"], cs["tail_pool"], K, B, N, _D, _POOL_SPLITS)
            ops.heads(pk["heads"], tokens=tokens, tokens_per_img=T, depth=cs["depth"], conf=cs["conf"], B=K * B,
                      pool_partial=cs["tail_pool"], pool_splits=_POOL_SPLITS, tmp_w=cs["tmpw"], tmp_b=cs["tmpb"],
                      sweep_images=B, **heads_in)
        self._curiosity_join()

    def _sweep_results(self, cs, K: int, return_attention: bool):
        heat = cs["heat"].clone()
        # what the last of the K calls leaves behind
        self._last_attention_weights = heat[K - 1]
        self._last_argmax = cs["argmax"][K - 1].clone()
        self._last_curiosity = cs["cur_reward"][K - 1]
        depth, conf = cs["depth"].clone().unsqueeze(-1), cs["conf"].clone().unsqueeze(-1)
        return (depth, conf, heat) if return_attention else (depth, conf)

    @torch.no_grad()
    @_on_own_device
    def forward_with_guidance_sweep(self, images, exif_data, guidances, return_attention=False):
        """K = len(guidances) guided calls over one batch in one pass: bit-identical to
        `[forward_with_guidance(images, exif_data, g) for g in guidances]` from the same global-RNG state — outputs,
        generator state, CuriosityModule ring buffer and `_last_*` state — with the backbone and (unless curiosity-guided
        attention is enabled) the focal iterations run once instead of K times.  Each entry is what `attention_guidance`
        accepts: an instruction string or alias, a guidance tensor [N'], or a list of B per-image instructions.
        Returns depth [K, B, 1], confidence [K, B, 1] (and the heat maps [K, B, N] with `return_attention`)."""
        self._raise_on_fault()
        K = self._check_guidances(guidances)
        if exif_data is None or not self.use_exif:
            raise ValueError("an instruction sweep needs EXIF data and a model with the EXIF prior (otherwise the "
                             "reference falls back to forward(): use forward_with_guidance)")
        B, S = self._check_images(images)
        for gd in guidances:
            self._check_per_image(gd, B)
        self._check_exif(exif_data, B)
        self._pack()
        g = S // 14
        mask = self._sweep_masks(guidances, B, g)
        exif, cam = self._exif_tensors(exif_data, B)
        draws = self._sweep_draws(B, K)
        ws = self._workspace(B, S)
        cs = self._sweep_buffers(ws, B, S, K)
        self._stage_runs(cs, draws)
        torch.stack(mask, out=cs["mask_in"])
        ws["exif_in"].copy_(exif, non_blocking=True)
        ws["cam_in"].copy_(cam, non_blocking=True)
        self._grid_tables(g)
        patches, images = self._patch_rows(images, ws, S)

        def device_pass():
            self._backbone_layers(ws, patches, B, S)
            self._guided_device(ws, cs, ws["tokens"], B, g, K, None, ws["exif_in"], ws["cam_in"])

        self._run(ws, ("sweep", K, self._curiosity_key()), device_pass)
        self._keepalive = (exif, cam, mask, images)
        return self._sweep_results(cs, K, return_attention)

    # -- scenes: encode a batch once, guide it any number of times ---------------------------------------
    @torch.no_grad()
    @_on_own_device
    def encode(self, images, exif_data) -> Scene:
        """The instruction-independent part of `forward_with_guidance` — the backbone and (unless curiosity-guided
        attention is enabled) the focal iterations — run once and kept in a `Scene` for `guide` / `guide_sweep`.
        Takes the images `forward_with_guidance` takes.  Draws nothing from the global generator and leaves the
        CuriosityModule state and every `_last_*` attribute as they are."""
        self._raise_on_fault()
        if exif_data is None or not self.use_exif:
            raise ValueError("a scene needs EXIF data and a model with the EXIF prior (otherwise the reference falls "
                             "back to forward(): use forward_with_guidance)")
        B, S = self._check_images(images)
        self._check_exif(exif_data, B)
        self._pack()
        dev = self._device()
        g = S // 14
        N, T = g * g, g * g + 1
        exif, cam = self._exif_tensors(exif_data, B)
        ws = self._workspace(B, S)
        self._grid_tables(g)
        patches, images = self._patch_rows(images, ws, S)
        cg = self.cfg.curiosity_guided

        def device_pass():
            self._backbone_layers(ws, patches, B, S)
            if not cg:
                self._focal_iterations(ws, B, g, want_features=False)

        self._run(ws, ("encode", patches.data_ptr(), cg), device_pass)
        tokens = torch.empty(B, T, _D, device=dev, dtype=torch.float32)
        base = None if cg else torch.empty(B, N, device=dev, dtype=torch.float32)
        _poison((tokens, base))
        tokens.copy_(ws["tokens"])
        if base is not None:
            base.copy_(ws["attn"][self.cfg.num_iterations - 1])
        # cloned: the scene owns its EXIF even when the caller's tensors were already contiguous device tensors
        scene = Scene(self, B, S, tokens, base, exif.clone(), cam.clone())
        self._keepalive = (exif, cam, images)  # until the next call, like the forwards (the copies are enqueued)
        return scene

    def _check_scene(self, scene):
        if not isinstance(scene, Scene):
            raise ValueError("expected a Scene from model.encode")
        if scene._model() is not self:
            raise ValueError("the scene was encoded by another model")
        if scene.device != self._device():
            raise ValueError(f"the scene lives on {scene.device}, the model on {self._device()}")
        if scene._stamp != self._weights_version:
            scene._graphs.clear()  # their workspace is no longer the model's: do not keep it alive
            raise ValueError("stale scene: the model's weights changed after it was encoded (encode the images again)")

    def _scene_ws(self, scene):
        """The (B, S) workspace whose scratch buffers a guide call on `scene` uses; the scene's tokens are passed on
        separately (nothing is copied)."""
        self._pack()
        self._grid_tables(scene.S // 14)
        return self._workspace(scene.B, scene.S)

    def _run_scene(self, scene, ws, key, fn):
        """Eager at a scene's first guide call; from the second on captured (once, on the scene's own buffers and this
        workspace) and replayed.  The graphs go with the scene."""
        first = scene._guided == 0
        scene._guided += 1
        if first:
            fn()
        else:
            for k in [k for k, v in scene._graphs.items() if v[2] is not ws]:
                del scene._graphs[k]  # captured on a workspace the model has since replaced: release it
            self._run(ws, key + (id(ws), self._curiosity_key()), fn, graphs=scene._graphs)

    def guide(self, scene: Scene, attention_guidance, return_attention=False):
        """`forward_with_guidance(images, exif_data, attention_guidance, return_attention)` for the images and EXIF of
        `scene`, bit for bit — outputs, global generator draws, CuriosityModule ring buffer and pointer, `_last_*` —
        without re-running the backbone (nor, unless curiosity-guided attention is enabled, the focal iterations):
        `guide_sweep(scene, [attention_guidance])`."""
        depth, conf, _ = self.guide_sweep(scene, [attention_guidance], return_attention=True)
        heat = self._last_attention_weights  # :1212
        return (depth[0], conf[0], heat) if return_attention else (depth[0], conf[0])

    @torch.no_grad()
    @_on_own_device
    def guide_sweep(self, scene: Scene, guidances, return_attention=False):
        """`forward_with_guidance_sweep(images, exif_data, guidances, return_attention)` for the images and EXIF of
        `scene`, bit for bit, without re-running the backbone (nor, unless curiosity-guided attention is enabled, the
        focal iterations)."""
        self._raise_on_fault()
        self._check_scene(scene)
        K = self._check_guidances(guidances)
        B, S = scene.B, scene.S
        for gd in guidances:
            self._check_per_image(gd, B)
        self._pack()
        g = S // 14
        mask = self._sweep_masks(guidances, B, g)
        draws = self._sweep_draws(B, K)
        ws = self._scene_ws(scene)
        cs = self._sweep_buffers(ws, B, S, K)
        self._stage_runs(cs, draws)
        torch.stack(mask, out=cs["mask_in"])

        def device_pass():
            self._guided_device(ws, cs, scene.tokens, B, g, K, scene.base, scene.exif, scene.camera_idx)

        self._run_scene(scene, ws, ("sweep", K), device_pass)
        self._keepalive = (mask,)
        return self._sweep_results(cs, K, return_attention)

    # -- many scenes: one guide call on each of m scenes, answered together -----------------------------------
    def _check_many(self, scenes, guidances):
        """(S, R) of a guide_many call, R = the images of all its scenes; checked before anything is drawn or launched."""
        if not isinstance(scenes, (list, tuple)) or not isinstance(guidances, (list, tuple)):
            raise ValueError("guide_many takes a list of scenes and a list of guidances")
        m = len(scenes)
        if m == 0 or len(guidances) != m:
            raise ValueError(f"guide_many takes m >= 1 scenes and one guidance per scene (got {m} scenes and "
                             f"{len(guidances)} guidances)")
        if m > _GUIDE_MANY_MAX_CALLS:
            raise ValueError(f"guide_many takes at most {_GUIDE_MANY_MAX_CALLS} scenes, got {m}")
        if any(gd is None for gd in guidances):
            raise ValueError("a None guidance runs the un-guided focal path (src/model.py:1206-1212): use "
                             "forward_with_guidance for it")
        for scene in scenes:
            self._check_scene(scene)
        S = scenes[0].S
        if any(scene.S != S for scene in scenes):
            raise ValueError(f"the scenes of one guide_many call must share the image side (got "
                             f"{sorted({scene.S for scene in scenes})})")
        for scene, gd in zip(scenes, guidances):
            self._check_per_image(gd, scene.B)
            for one in (gd if isinstance(gd, (list, tuple)) else [gd]):
                if isinstance(one, str) and tables.canonical_instruction(one) not in tables.INSTRUCTIONS:
                    raise ValueError(f"unknown instruction {one!r} (one of {', '.join(tables.INSTRUCTIONS)} or an alias)")
        R = sum(scene.B for scene in scenes)
        if R > _GUIDE_MANY_MAX_ROWS:
            raise ValueError(f"guide_many takes at most {_GUIDE_MANY_MAX_ROWS} images over all scenes, got {R}")
        return S, R

    def _many_buffers(self, S: int):
        """The buffers of guide_many calls at side S, sized at the caps (CA_GUIDE_MANY_MAX_ROWS rows,
        CA_GUIDE_MANY_MAX_CALLS calls): a call of R rows and m calls uses the first R rows / m projections of each, and
        its graph is kept per (R, m).  Nothing here is per (B, S): no backbone workspace is needed."""
        cs = self._many.get(S)
        if cs is None:
            dev = self._device()
            N = (S // 14) ** 2
            R, m = _GUIDE_MANY_MAX_ROWS, _GUIDE_MANY_MAX_CALLS
            fl = dict(device=dev, dtype=torch.float32)
            cs = {
                # ca_guide_many_row [R] as fp32 words, staged with the draws (ops.fetch_pinned reads fp32)
                "rows": torch.empty(R, 2 * _GUIDE_MANY_ROW_WORDS, **fl),
                "cls": torch.empty(R, _D, **fl), "base": torch.empty(R, N, **fl), "exif": torch.empty(R, 3, **fl),
                "cam": torch.empty(R, device=dev, dtype=torch.int64),
                "call": torch.empty(R, device=dev, dtype=torch.int32),
                # one CuriosityModule run over the R rows: the ring receives them in call order
                "cur_eps": torch.zeros(1, R, 192, **fl), "cur_noise": torch.zeros(1, R, _D, **fl),
                "cur_raw": torch.empty(1, R, **fl), "cur_reward": torch.empty(1, R, **fl),
                "tmpw": torch.empty(m, 64, _D, **fl), "tmpb": torch.empty(m, 64, **fl),
                "mask_in": torch.empty(R, N, **fl), "heat": torch.empty(R, N, **fl),
                "argmax": torch.empty(R, device=dev, dtype=torch.int32),
                "tail_pool": torch.empty(R, _POOL_SPLITS, _D, **fl),
                "depth": torch.empty(R, **fl), "conf": torch.empty(R, **fl),
                "graphs": {}, "calls": {},
            }
            _poison(cs.values())
            if len(self._many) >= 4:  # keep the cache bounded
                self._many.pop(next(iter(self._many)))
            self._many[S] = cs
        return cs

    @staticmethod
    def _many_rows(cs, R: int, m: int):
        """The views of the first R rows / m calls of a guide_many buffer set (leading slices: contiguous)."""
        per_call = ("tmpw", "tmpb")
        rows = {k: (v[:m] if k in per_call else v[:, :R] if k.startswith("cur_") else v[:R])
                for k, v in cs.items() if torch.is_tensor(v)}
        rows["graphs"] = cs["graphs"]
        return rows

    @staticmethod
    def _row_table(scenes, N: int, fault: int):
        """ca_guide_many_row [R] as int64 words: per image of each scene in call order, the addresses of its tokens,
        focal attention, EXIF and camera index in the scene, the fault word a bad camera index is reported in, and its
        call index."""
        words = []
        for j, scene in enumerate(scenes):
            tok, base, exif, cam = (t.data_ptr() for t in (scene.tokens, scene.base, scene.exif, scene.camera_idx))
            for b in range(scene.B):
                words += [tok + b * (N + 1) * _D * 4, base + b * N * 4, exif + b * 12, cam + b * 8, fault, j]
        return torch.tensor(words, dtype=torch.int64)

    @torch.no_grad()
    @_on_own_device
    def guide_many(self, scenes, guidances, return_attention=False):
        """One guide call on each of m scenes, answered together: returns the list of m tuples
        `[guide(scenes[j], guidances[j], return_attention) for j in range(m)]`, bit for bit, and leaves the global
        generator, the CuriosityModule ring buffer and pointer and `_last_*` (from call m) as that loop would.  The
        scenes may differ in batch size and repeat; they share the model, the device and the image side S.  A guidance
        is what `guide` takes, except that an unknown instruction string is refused.  At most
        CA_GUIDE_MANY_MAX_CALLS scenes of CA_GUIDE_MANY_MAX_ROWS images in all (include/cogaim_b200.h).
        The R images of all calls run as one batch: the CLS tokens, focal attention rows and EXIF are gathered through
        a row table (the patch tokens are read where the scenes keep them), then one CuriosityModule run, one guided
        softmax, pool and heads pass.  With curiosity-guided attention every call needs its own focal pass, and the m
        calls run one after another."""
        self._raise_on_fault()
        S, R = self._check_many(scenes, guidances)
        self._pack()
        g = S // 14
        N = g * g
        masks = [self._sweep_masks([gd], scene.B, g)[0] for scene, gd in zip(scenes, guidances)]
        if self.cfg.curiosity_guided:
            return [self.guide(scene, gd, return_attention) for scene, gd in zip(scenes, guidances)]
        m = len(scenes)
        draws = [self._sweep_draws(scene.B, 1)[0] for scene in scenes]  # call order: :609, :744, :1421 per call
        full = self._many_buffers(S)
        cs = self._many_rows(full, R, m)
        table = self._row_table(scenes, N, self._fault_word().data_ptr())
        caps = (_GUIDE_MANY_MAX_ROWS, _GUIDE_MANY_MAX_CALLS)

        def fill(bufs):
            eps, noise, tmpw, tmpb, rows = bufs
            r = 0
            for j, (scene, d) in enumerate(zip(scenes, draws)):
                eps[r:r + scene.B].copy_(d[0])
                noise[r:r + scene.B].copy_(d[1])
                tmpw[j].copy_(d[2])
                tmpb[j].copy_(d[3])
                r += scene.B
            rows[:R].view(torch.int64).copy_(table.view(R, _GUIDE_MANY_ROW_WORDS))
            return [(cs["cur_eps"][0], eps[:R]), (cs["cur_noise"][0], noise[:R]), (cs["tmpw"], tmpw[:m]),
                    (cs["tmpb"], tmpb[:m]), (cs["rows"], rows[:R])]

        # one pinned set per ring slot, at the caps: the staging memory does not grow with the (R, m) seen
        self._stage_pinned("many", ((caps[0], 192), (caps[0], _D), (caps[1], 64, _D), (caps[1], 64),
                                    (caps[0], 2 * _GUIDE_MANY_ROW_WORDS)), fill)
        torch.cat(masks, out=cs["mask_in"])
        pk = self._packed

        def device_pass():
            ops.gather_rows(cs["rows"], R, N, cs["cls"], cs["base"], cs["exif"], cs["cam"], cs["call"],
                            num_cameras=self.cfg.num_cameras)  # reports a bad camera index in the row's fault word
            self._curiosity_runs(cs, cs["cls"], R, 1, ("guided",))
            ops.guided_softmax(cs["base"], cs["mask_in"], cs["heat"], cs["argmax"], R, N)
            ops.weighted_pool_rows(cs["rows"], cs["heat"], cs["tail_pool"], R, N, _D, _POOL_SPLITS)
            ops.heads(pk["heads"], tokens=cs["cls"], tokens_per_img=1, depth=cs["depth"], conf=cs["conf"], B=R,
                      pool_partial=cs["tail_pool"], pool_splits=_POOL_SPLITS, tmp_w=cs["tmpw"], tmp_b=cs["tmpb"],
                      exif=cs["exif"], camera_idx=cs["cam"], num_cameras=self.cfg.num_cameras, call_of_row=cs["call"])
            self._curiosity_join()

        # eager at the first call of this (R, m), captured at the second, replayed after — with any scenes: the row
        # table is data
        calls = full["calls"][(R, m)] = full["calls"].get((R, m), 0) + 1
        if calls == 1:
            device_pass()
        else:
            self._run(cs, ("many", R, m, self._curiosity_key()), device_pass)
        self._keepalive = (tuple(scenes), masks)
        heat = cs["heat"].clone()
        depth, conf = cs["depth"].clone().unsqueeze(-1), cs["conf"].clone().unsqueeze(-1)
        out, r = [], 0
        for scene in scenes:
            rows = slice(r, r + scene.B)
            out.append((depth[rows], conf[rows], heat[rows]) if return_attention else (depth[rows], conf[rows]))
            r += scene.B
        last = slice(R - scenes[-1].B, R)  # what call m leaves behind
        self._last_attention_weights = heat[last]
        self._last_argmax = cs["argmax"][last].clone()
        self._last_curiosity = cs["cur_reward"][0, last].clone()
        return out

    def _field_buffers(self, ws, B: int, N: int):
        """The depth-field buffers of a (B, S) workspace, added at its first field: the projected tokens [B, N, 64], the
        per-image fusion constant [B, 192] and the field itself."""
        if "field_P" not in ws:
            fl = dict(device=self._device(), dtype=torch.float32)
            ws.update(field_P=torch.empty(B, N, 64, **fl), field_cst=torch.empty(B, 192, **fl),
                      field_depth=torch.empty(B, N, **fl), field_conf=torch.empty(B, N, **fl))
            _poison(ws[k] for k in ("field_P", "field_cst", "field_depth", "field_conf"))
        return ws

    @torch.no_grad()
    @_on_own_device
    def depth_field(self, scene: Scene):
        """The guided depth and confidence with the focus on every cell of the g x g patch grid (g = S / 14): returns
        depth, confidence [B, g, g] fp32.  Cell (y, x) of image b is what `guide(scene, tables.focus_mask(y, x, g))` gives
        for image b with the same draws, within fp32 rounding (the field projects the tokens before pooling them and sums
        each cell's softmax over its focus disk, where all but < N e^-36 of the weight lies).  So cell (g//4, g//4) is the
        "top-left" prediction, and likewise for the other off-centre instructions; "center" has its own mask, and cell
        (g//2, g//2) is not its prediction.
        One call draws what one `guide` call draws, in its order (the CuriosityModule's randn(B, 192), randn(B, 768),
        then nn.Linear(768, 64)); every cell uses that one projection, and the CuriosityModule runs once (B ring
        entries).  `_last_curiosity` is set as `guide` sets it; `_last_attention_weights` and `_last_argmax` are left as
        they are (there is no single heat map)."""
        self._raise_on_fault()
        self._check_scene(scene)
        B, S = scene.B, scene.S
        pk = self._pack()
        g = S // 14
        N, T = g * g, g * g + 1
        draws = self._sweep_draws(B, 1)  # :1185, :1421
        ws = self._scene_ws(scene)
        self._field_buffers(ws, B, N)
        cs = self._sweep_buffers(ws, B, S, 1)
        self._stage_runs(cs, draws)
        cg = self.cfg.curiosity_guided

        def device_pass():
            self._curiosity_runs(cs, scene.tokens, B, T, ("guided",))
            base = (self._focal_iterations(ws, B, g, want_features=False, cur_weight=cs["cur_weight"][0],
                                           tokens=scene.tokens) if cg else scene.base)
            ops.token_project(scene.tokens, T * _D, 1, cs["tmpw"][0], ws["field_P"], B, N)
            ops.depth_field_cells(pk["heads"], base=base, P=ws["field_P"], cst=ws["field_cst"], depth=ws["field_depth"],
                                  conf=ws["field_conf"], tokens=scene.tokens, tmp_b=cs["tmpb"][0], B=B, g=g,
                                  exif=scene.exif, camera_idx=scene.camera_idx, num_cameras=self.cfg.num_cameras,
                                  fault_ptr=self._fault_word().data_ptr())
            self._curiosity_join()

        self._run_scene(scene, ws, ("field",), device_pass)
        self._last_curiosity = cs["cur_reward"][0]
        return ws["field_depth"].clone().view(B, g, g), ws["field_conf"].clone().view(B, g, g)

    @torch.no_grad()
    @_on_own_device
    def forward(self, images, exif_data=None, return_attention=False):
        """reference src/model.py:1064-1155 (un-guided).  One backbone + one focal pass instead of 3 + 4."""
        return self._forward_impl(images, exif_data, return_attention, mode="forward")

    def _forward_impl(self, images, exif_data, return_attention, mode, guidance=None):
        """The un-guided paths.  `mode` selects which of the reference's entry points is being mirrored — they differ in
        how often the CuriosityModule runs (RNG draws, ring-buffer entries) and in what `_last_attention_weights` ends as:
          forward          get_features_aligned (:992) [+ :1104 when no `_last_attention_weights` is stored] [+ :1138 for
                           return_attention]
          features         get_features_aligned alone (:960-1048)
          guided_none      forward_with_guidance(guidance=None) (:1185, :1206-1212): one run, attention always stored
          guided_fallback  forward_with_guidance without EXIF: the guided attempt (:1185 [+ :1421 projection draws]) fails in
                           `fusion` and falls back to forward() (:1237-1240) with the guided attention already stored."""
        self._raise_on_fault()
        B, S = self._check_images(images)
        self._check_per_image(guidance, B)
        self._check_exif(exif_data, B)
        pk = self._pack()
        g = S // 14
        N, T = g * g, g * g + 1
        exif, cam = self._exif_tensors(exif_data, B)
        has_last = hasattr(self, "_last_attention_weights")
        if mode == "forward":
            roles = ["features"] + ([] if has_last else ["last"]) + (["ret"] if return_attention else [])
        elif mode in ("features", "guided_none"):
            roles = ["features"]
        elif mode == "guided_fallback":
            roles = ["guided", "features"] + (["ret"] if return_attention else [])
        else:
            raise AssertionError(mode)
        mask = None
        draws = []
        for j, role in enumerate(roles):
            draws.append(self._curiosity_draw(B))
            if role == "guided" and guidance is not None:
                mask = self._mask(guidance, g)
                nn.Linear(_D, 64)  # :1421 is reached (and draws) before the 128-wide concat fails in `fusion`
        ws = self._workspace(B, S)
        cs = self._sweep_buffers(ws, B, S, len(roles))
        self._stage_runs(cs, draws)
        has_exif = exif is not None
        if has_exif:
            ws["exif_in"].copy_(exif, non_blocking=True)
            ws["cam_in"].copy_(cam, non_blocking=True)
        if mask is not None:
            cs["mask_in"][0].copy_(mask, non_blocking=True)
        self._grid_tables(g)
        patches, images = self._patch_rows(images, ws, S)
        cg = self.cfg.curiosity_guided
        jf = roles.index("features")

        def device_pass():
            self._backbone_layers(ws, patches, B, S)
            tokens = ws["tokens"]
            self._curiosity_runs(cs, tokens, B, T, roles)
            if cg:
                # the attention-only calls of the reference see their own run's (clamped) score: separate passes
                for j, role in enumerate(roles):
                    if role != "features":
                        att_j = self._focal_iterations(ws, B, g, want_features=False, cur_weight=cs["cur_weight"][j])
                        cs["base"][j].copy_(att_j)
            att_f = self._focal_iterations(ws, B, g, want_features=True, cur_weight=cs["cur_weight"][jf] if cg else None)
            if mask is not None:
                base = cs["base"][roles.index("guided")] if cg else att_f
                ops.guided_softmax(base, cs["mask_in"][0], cs["heat"][0], cs["argmax"][0], B, N)
            ops.heads(pk["heads"], tokens=tokens, tokens_per_img=T, depth=cs["depth"][0], conf=cs["conf"][0], B=B,
                      focal_feat=ws["focal_feat"], exif=ws["exif_in"] if has_exif else None,
                      camera_idx=ws["cam_in"] if has_exif else None, fused_out=ws["fused"],
                      num_cameras=self.cfg.num_cameras, fault_ptr=self._fault_word().data_ptr())
            self._curiosity_join()

        self._run(ws, ("unguided", has_exif, tuple(roles), mask is not None, self._curiosity_key()), device_pass)
        self._keepalive = (exif, cam, images, mask)
        att_feat = ws["attn"][self.cfg.num_iterations - 1]

        def att_of(role):
            return (cs["base"][roles.index(role)] if cg and role != "features" else att_feat).clone()

        self.fusion_features = ws["fused"].clone()  # :1089
        self._last_curiosity = cs["cur_reward"][jf]
        if mode == "forward":
            if not has_last:  # :1093-1113 only set when absent
                self._last_attention_weights = att_of("last")
        elif mode == "guided_none":
            self._last_attention_weights = att_of("features")  # :1212 always stores
        elif mode == "guided_fallback":
            self._last_attention_weights = cs["heat"][0].clone() if mask is not None else att_of("guided")  # :1212
        depth, conf = cs["depth"][0].clone().unsqueeze(1), cs["conf"][0].clone().unsqueeze(1)
        if not return_attention:
            return depth, conf
        return depth, conf, att_of("ret" if "ret" in roles else "features")

    # -- accessors ----------------------------------------------------------------------------------------
    def get_attention_weights(self):
        """reference src/model.py:1058-1062."""
        return getattr(self, "_last_attention_weights", None)

    @torch.no_grad()
    @_on_own_device
    def get_features_aligned(self, images, exif_data=None):
        """[B, 192] fused features (reference src/model.py:960-1048)."""
        self._forward_impl(images, exif_data, False, mode="features")
        return self.fusion_features

    def get_features(self, images, exif_data=None):
        """reference src/model.py:1428-1430."""
        return self.get_features_aligned(images, exif_data)

    @torch.no_grad()
    @_on_own_device
    def focal_attention(self, tokens: torch.Tensor, want_features: bool = False):
        """IterativeFocalStream on given backbone tokens [B, 1+N, 768] fp32 (test / analysis hook): returns the
        last-iteration attention [B, N] (and the fused 64-d focal features when `want_features`)."""
        if tokens.dim() != 3 or tokens.shape[-1] != _D:
            raise ValueError("tokens must be [B, 1+N, 768]")
        B, T, _ = tokens.shape
        g = int(math.isqrt(T - 1))
        if g * g != T - 1:
            raise ValueError("token count - 1 must be a square grid")
        self._pack()
        ws = self._workspace(B, g * 14)
        ws["tokens"].copy_(tokens.to(self._device(), torch.float32))
        att = self._focal_iterations(ws, B, g, want_features).clone()
        return (att, ws["focal_feat"].clone()) if want_features else att

    @torch.no_grad()
    @_on_own_device
    def focus_map(self, size, attention: Optional[torch.Tensor] = None):
        """The overlay heat map `demo.py:_save_prediction_image` renders (demo.py:530-563): cube, 70th-percentile
        threshold, min-max normalisation, g x g grid, order-1 zoom to `size` = (height, width) of the image it is laid
        over — computed on the GPU from the attention of the last forward (or `attention` [B, N]) instead of numpy /
        scipy on a D2H copy.  Returns float32 [B, height, width] in [0, 1]."""
        att = self.get_attention_weights() if attention is None else attention
        if att is None:
            raise ValueError("no attention weights: run a forward pass first or pass `attention`")
        att = att.to(self._device(), torch.float32).reshape(att.shape[0], -1).contiguous()
        B, N = att.shape
        g = int(math.isqrt(N))
        if g * g != N:
            raise ValueError("attention length must be a square grid")
        h, w = int(size[0]), int(size[1])
        norm = torch.empty(B, N, device=att.device, dtype=torch.float32)
        out = torch.empty(B, h, w, device=att.device, dtype=torch.float32)
        ops.focus_map(att, g, h, w, norm, out)
        return out

    # -- demo-style preprocessing ---------------------------------------------------------------------------
    @torch.no_grad()
    @_on_own_device
    def preprocess(self, images_hwc_u8: torch.Tensor, size: int, mean=ops.IMAGENET_MEAN, std=ops.IMAGENET_STD):
        """demo.py:162-166 for a batch of same-sized uint8 [B, H, W, 3] images, on the GPU: Resize((size, size)) (Pillow's
        antialiased bilinear resample, bit-exact) -> ToTensor -> Normalize.  Returns float32 [B, 3, size, size], the
        tensor `forward` / `forward_with_guidance` take."""
        if images_hwc_u8.dtype != torch.uint8 or images_hwc_u8.dim() != 4 or images_hwc_u8.shape[-1] != 3:
            raise ValueError("expected uint8 [B, H, W, 3]")
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("preprocess runs only on a CUDA sm_100 device; there is no CPU fallback")
        return self._normalise(ops.resize_u8(images_hwc_u8.to(dev).contiguous(), size, size), mean, std)

    @staticmethod
    def _normalise(r, mean, std):
        """uint8 [B, S, S, 3] -> ToTensor -> Normalize: float32 [B, 3, S, S] (demo.py:164-166)."""
        dev = r.device
        # ToTensor: a true division (a tensor divisor; dividing by a Python scalar multiplies by the reciprocal on CUDA)
        x = r.permute(0, 3, 1, 2).to(torch.float32) / torch.full((1,), 255.0, device=dev)
        m = torch.tensor(mean, device=dev).view(1, 3, 1, 1)
        s = torch.tensor(std, device=dev).view(1, 3, 1, 1)
        return x.sub_(m).div_(s).contiguous()                          # Normalize

    @torch.no_grad()
    @_on_own_device
    def preprocess_jpeg(self, jpeg_files, size: int, mean=ops.IMAGENET_MEAN, std=ops.IMAGENET_STD):
        """demo.py:312-319 for a list of JPEG files given as bytes: decode (nvJPEG) -> Resize((size, size)) (exact Pillow
        arithmetic) -> ToTensor -> Normalize, all on the GPU.  Images may differ in size (each is resized on its own, as
        `predict_batch` does, demo.py:406-432, in one resize for the whole list).  Returns float32 [B, 3, size, size]."""
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("preprocess_jpeg runs only on a CUDA sm_100 device; there is no CPU fallback")
        if len(jpeg_files) == 0:
            raise ValueError("empty list of JPEG files")
        # one batched nvJPEG decode for all files, one ragged resize, one normalisation: the launch count does not depend on
        # the number of distinct source sizes
        imgs = ops.jpeg_decode_batch(list(jpeg_files), dev)
        return self._normalise(ops.resize_u8_list(imgs, size, size), mean, std)

    @torch.no_grad()
    @_on_own_device
    def tokens_from_uint8(self, images_hwc_u8, size: Optional[int] = None):
        """uint8 [B, H, W, 3] -> backbone tokens: demo.py:162-166 on the GPU — Resize((size, size)) exactly as Pillow does
        it (skipped when the images already have that size or `size` is None), then ToTensor + Normalize + patchify
        fused in one kernel.  A list of uint8 [H_i, W_i, 3] photographs of individual sizes is resized to `size` (or,
        when it is None, model.input_size)."""
        if isinstance(images_hwc_u8, (list, tuple)):
            S = size if size is not None else self.input_size
            B = self._check_list(images_hwc_u8, S)
            self._pack()
            ws = self._workspace(B, S)
            patches, self._keepalive = self._patch_rows(images_hwc_u8, ws, S)
            return self.backbone_tokens(None, patches=patches, B=B, S=S)
        if images_hwc_u8.dtype != torch.uint8 or images_hwc_u8.dim() != 4 or images_hwc_u8.shape[-1] != 3:
            raise ValueError("expected uint8 [B, H, W, 3]")
        if size is not None and tuple(images_hwc_u8.shape[1:3]) != (size, size):
            # demo.py:162-163 Resize((S, S)): Pillow's antialiased bilinear resample, bit-exact, on the GPU
            images_hwc_u8 = ops.resize_u8(images_hwc_u8.to(self._device()).contiguous(), size, size)
        B, S = images_hwc_u8.shape[0], images_hwc_u8.shape[1]
        if images_hwc_u8.shape[2] != S:
            raise ValueError("expected square images (or pass size=S to resize like demo.py)")
        ws = self._workspace(B, S)
        patches = ops.preprocess_u8(images_hwc_u8.to(self._device()).contiguous(), ws["patches"])
        return self.backbone_tokens(None, patches=patches, B=B, S=S)


def create_model(config: dict, camera_info: Optional[dict] = None, device=None) -> CognitiveAimModel:
    """Factory with the reference's signature (src/model.py:1534).  `config` is the whole YAML dict."""
    cfg = dict(config)
    if "cognitive_modules" not in cfg and "cognitive_modules" not in (cfg.get("model") or {}):
        cfg["cognitive_modules"] = list(DEFAULT_COGNITIVE_MODULES)
    model = CognitiveAimModel(cfg, camera_info)
    if device is not None:
        model = model.to(device)
    ckpt = config.get("load_checkpoint")  # :1549 (top-level key; absent in every shipped YAML)
    if ckpt:
        state = torch.load(ckpt, map_location="cpu")
        skip = ("decision_head.", "confidence_head.", "curiosity_module.", "global_aligner.", "ambient_stream.",
                "focal_stream.", "exif_prior.", "fusion.")  # :1556-1559
        model.load_state_dict({k: v for k, v in state.items() if not k.startswith(skip)}, strict=False)
    return model
