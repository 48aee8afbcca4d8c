"""Thin ctypes driver of the handle-level C-ABI (`ca_create / ca_forward_guided / ca_forward / ca_backbone / ca_destroy`,
include/cogaim_b200.h): ONE native call per forward; tables, workspaces, staging, the launch sequence and the CUDA graphs
all live in libcogaim_b200.so (csrc/launcher.cu).  This module does not use model.py: it is what a non-Python host would
write — pack the reference's state_dict into device operands, fill `ca_model_weights`, call.

Random numbers stay with the caller, as in the reference: the two Gaussian draws of each CuriosityModule run
(src/model.py:609, 744) and the per-call projection `nn.Linear(768, 64)` (:1421) are drawn HERE from torch's global CPU
generator, in the reference's order, and handed to the library as host arrays.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib

_D, _LAYERS = 768, 12


def _fold(weight, bias, gamma, beta):
    """LayerNorm (gamma, beta) folded into the Linear after it (include/cogaim_b200.h, ca_layer_weights.cqkv / c1):
    W' = bf16(rows of W diag(gamma), centred), b' = b + W beta."""
    w32 = weight.float()
    wg = w32 * gamma.float()[None, :]
    return (wg - wg.mean(dim=1, keepdim=True)).to(torch.bfloat16), bias.float() + w32 @ beta.float()


def _pack(sd: Dict[str, torch.Tensor], dev: torch.device, num_cameras: int, fold_layernorm: bool = False):
    """reference state_dict -> (ca_model_weights, tensors to keep alive)."""
    keep = []

    def f32(t):
        t = t.detach().to(dev, torch.float32).contiguous()
        keep.append(t)
        return t.data_ptr()

    def b16(t):
        t = t.detach().to(dev, torch.bfloat16).contiguous()
        keep.append(t)
        return t.data_ptr()

    w = _lib.ModelWeights()
    e = "backbone.embeddings."
    pw = torch.zeros(_D, 592, dtype=torch.bfloat16)
    pw[:, :588] = sd[e + "patch_embeddings.projection.weight"].detach().reshape(_D, 588).to(torch.bfloat16)
    w.patch_w, w.patch_b = b16(pw), f32(sd[e + "patch_embeddings.projection.bias"])
    w.cls_token = f32(sd[e + "cls_token"].reshape(_D))
    pos = sd[e + "position_embeddings"].detach().to("cpu", torch.float32).reshape(-1, _D).contiguous()  # HOST
    if pos.shape[0] != 1 + 37 * 37:
        raise ValueError("position_embeddings must be the native 37 x 37 grid (+ CLS)")
    keep.append(pos)
    w.pos_embed = pos.data_ptr()
    for i in range(_LAYERS):
        p, L = f"backbone.encoder.layer.{i}.", w.layer[i]
        a = p + "attention.attention."
        L.n1w, L.n1b = f32(sd[p + "norm1.weight"]), f32(sd[p + "norm1.bias"])
        L.wqkv = b16(torch.cat([sd[a + "query.weight"], sd[a + "key.weight"], sd[a + "value.weight"]], 0))
        L.bqkv = f32(torch.cat([sd[a + "query.bias"], sd[a + "key.bias"], sd[a + "value.bias"]], 0))
        L.wo, L.bo = b16(sd[p + "attention.output.dense.weight"]), f32(sd[p + "attention.output.dense.bias"])
        L.ls1 = f32(sd[p + "layer_scale1.lambda1"])
        L.n2w, L.n2b = f32(sd[p + "norm2.weight"]), f32(sd[p + "norm2.bias"])
        L.w1, L.b1 = b16(sd[p + "mlp.fc1.weight"]), f32(sd[p + "mlp.fc1.bias"])
        L.w2, L.b2 = b16(sd[p + "mlp.fc2.weight"]), f32(sd[p + "mlp.fc2.bias"])
        L.ls2 = f32(sd[p + "layer_scale2.lambda1"])
        if fold_layernorm:
            # norm1 -> (wqkv, bqkv), norm2 -> (w1, b1): the library then runs the encoder without LayerNorm passes
            wq = torch.cat([sd[a + "query.weight"], sd[a + "key.weight"], sd[a + "value.weight"]], 0).detach().to(dev)
            bq = torch.cat([sd[a + "query.bias"], sd[a + "key.bias"], sd[a + "value.bias"]], 0).detach().to(dev)
            g1, be1 = sd[p + "norm1.weight"].detach().to(dev), sd[p + "norm1.bias"].detach().to(dev)
            g2, be2 = sd[p + "norm2.weight"].detach().to(dev), sd[p + "norm2.bias"].detach().to(dev)
            wp, bp = _fold(wq, bq, g1, be1)
            L.wqkv, L.bqkv = b16(wp), f32(bp)
            wp, bp = _fold(sd[p + "mlp.fc1.weight"].detach().to(dev), sd[p + "mlp.fc1.bias"].detach().to(dev), g2, be2)
            L.w1, L.b1 = b16(wp), f32(bp)
    w.lnw, w.lnb = f32(sd["backbone.layernorm.weight"]), f32(sd["backbone.layernorm.bias"])
    n_focal = 0
    while f"focal_stream.focal_streams.{n_focal}.query_proj.weight" in sd:
        n_focal += 1
    if not 1 <= n_focal <= 4:
        raise ValueError("1..4 focal iterations are built")
    w.n_focal, w.focus_strength = n_focal, 1.5  # every shipped YAML resolves to 3 iterations, focus 1.5 (SURVEY.md §0)
    for i in range(n_focal):
        p, F = f"focal_stream.focal_streams.{i}.", w.focal[i]
        F.wqk = b16(torch.cat([sd[p + "query_proj.weight"], sd[p + "key_proj.weight"]], 0))
        F.bqk = f32(torch.cat([sd[p + "query_proj.bias"], sd[p + "key_proj.bias"]], 0))
        F.wv, F.bv = f32(sd[p + "value_proj.weight"]), f32(sd[p + "value_proj.bias"])
        F.pw0, F.pb0 = f32(sd[p + "projection.0.weight"]), f32(sd[p + "projection.0.bias"])
        F.pw1, F.pb1 = f32(sd[p + "projection.3.weight"]), f32(sd[p + "projection.3.bias"])
    w.ffw0, w.ffb0 = f32(sd["focal_stream.fusion.0.weight"]), f32(sd["focal_stream.fusion.0.bias"])
    w.ffw1, w.ffb1 = f32(sd["focal_stream.fusion.2.weight"]), f32(sd["focal_stream.fusion.2.bias"])
    H = w.heads
    for field, name in (("amb_w0", "ambient_stream.mlp.0.weight"), ("amb_b0", "ambient_stream.mlp.0.bias"),
                        ("amb_w1", "ambient_stream.mlp.3.weight"), ("amb_b1", "ambient_stream.mlp.3.bias"),
                        ("amb_w2", "ambient_stream.mlp.5.weight"), ("amb_b2", "ambient_stream.mlp.5.bias"),
                        ("cam_emb", "exif_prior.camera_embedding.weight"),
                        ("exif_w0", "exif_prior.exif_encoder.0.weight"), ("exif_b0", "exif_prior.exif_encoder.0.bias"),
                        ("exif_w1", "exif_prior.exif_encoder.2.weight"), ("exif_b1", "exif_prior.exif_encoder.2.bias"),
                        ("exif_f0", "exif_prior.fusion.0.weight"), ("exif_fb0", "exif_prior.fusion.0.bias"),
                        ("exif_f1", "exif_prior.fusion.3.weight"), ("exif_fb1", "exif_prior.fusion.3.bias"),
                        ("fus_w", "fusion.0.weight"), ("fus_b", "fusion.0.bias"),
                        ("dec_w", "decision_head.0.weight"), ("dec_b", "decision_head.0.bias"),
                        ("conf_w0", "confidence_head.0.weight"), ("conf_b0", "confidence_head.0.bias"),
                        ("conf_w2", "confidence_head.2.weight"), ("conf_b2", "confidence_head.2.bias")):
        if name not in sd:
            raise ValueError(f"state_dict has no {name} (the handle API is built for ambient + iterative focal + EXIF)")
        setattr(H, field, f32(sd[name]))
    c, Cw = "curiosity_module.", w.curiosity
    for short, name in (("em", "encoder_mean"), ("el", "encoder_logvar"), ("dec", "decoder")):
        setattr(Cw, short + "_w0", f32(sd[c + name + ".0.weight"]))
        setattr(Cw, short + "_b0", f32(sd[c + name + ".0.bias"]))
        setattr(Cw, short + "_w1", f32(sd[c + name + ".3.weight"]))
        setattr(Cw, short + "_b1", f32(sd[c + name + ".3.bias"]))
    Cw.unc_w0, Cw.unc_b0 = f32(sd[c + "uncertainty_head.0.weight"]), f32(sd[c + "uncertainty_head.0.bias"])
    Cw.unc_w1, Cw.unc_b1 = f32(sd[c + "uncertainty_head.2.weight"]), f32(sd[c + "uncertainty_head.2.bias"])
    if c + "local_curiosity.0.weight" in sd:
        Cw.loc_w0, Cw.loc_b0 = f32(sd[c + "local_curiosity.0.weight"]), f32(sd[c + "local_curiosity.0.bias"])
        Cw.loc_w1, Cw.loc_b1 = f32(sd[c + "local_curiosity.2.weight"]), f32(sd[c + "local_curiosity.2.bias"])
    Cw.cur_w = f32(sd[c + "curiosity_weights"])
    hist = sd[c + "exploration_history"].detach().to(dev, torch.float32).contiguous().clone()
    ptr = sd[c + "history_pointer"].detach().to(dev, torch.int64).reshape(1).contiguous().clone()
    w.exploration_history, w.history_len, w.history_pointer = hist.data_ptr(), hist.numel(), ptr.data_ptr()
    w.num_cameras = num_cameras
    w.layernorm_folded = 1 if fold_layernorm else 0
    return w, keep, hist, ptr


class NativeModel:
    """`forward_with_guidance` / `forward` / backbone tokens through the handle-level C-ABI."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device="cuda:0", num_cameras: int = 71,
                 use_graph: bool = True, fold_layernorm: bool = False):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("the Cognitive-Aim B200 path runs only on a CUDA sm_100 device; there is no CPU fallback")
        self.lib = _lib.load()
        self.use_graph = use_graph
        w, self._keep, self.exploration_history, self.history_pointer = _pack(state_dict, self.device, num_cameras,
                                                                              fold_layernorm)
        h = C.c_void_p()
        _lib.check(self.lib.ca_create(C.byref(h), C.byref(w), self.device.index or 0), "ca_create")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ca_destroy(self._h)
            self._h = None

    __del__ = close

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _image_list(self, images, S):
        """A list of uint8 [H_i, W_i, 3] photographs -> (device tensors, HOST pointer array, HOST (H, W) array)."""
        if S is None:
            raise ValueError("a list of images needs S, the side they are resized to")
        if len(images) == 0 or any(t.dtype != torch.uint8 or t.dim() != 3 or t.shape[-1] != 3 for t in images):
            raise ValueError("expected a non-empty list of uint8 [H, W, 3] tensors")
        imgs = [t.to(self.device).contiguous() for t in images]
        ptrs, hw = _lib.image_arrays(imgs)
        return imgs, C.cast(ptrs, C.POINTER(C.c_void_p)), C.cast(hw, C.POINTER(C.c_int)), [imgs, ptrs, hw]

    def _call(self, images, exif, S=None) -> _lib.ForwardCall:
        c = _lib.ForwardCall()
        if isinstance(images, (list, tuple)):
            imgs, c.image_list, c.image_hw, held = self._image_list(images, S)
            B = len(imgs)
            c.B, c.S = B, S
        elif images.dtype == torch.uint8:
            B, S = images.shape[0], images.shape[1]
            c.images_u8 = 1
        else:
            B, S = images.shape[0], images.shape[-1]
            images = images.to(self.device, torch.float32)
        if not isinstance(images, (list, tuple)):
            images = images.to(self.device).contiguous()
            c.images, c.B, c.S = images.data_ptr(), B, S
            held = [images]
        if exif is not None:
            cont = torch.stack([exif["focal_length"].reshape(-1), exif["aperture"].reshape(-1),
                                exif["iso"].reshape(-1)], dim=1).to(self.device, torch.float32).contiguous()
            cam = exif["camera_idx"].reshape(-1).to(self.device, torch.int64).contiguous()
            c.exif, c.camera_idx = cont.data_ptr(), cam.data_ptr()
            held += [cont, cam]
        c.use_graph = int(self.use_graph)
        return c, held, B, S

    @staticmethod
    def _draws(c, B: int, R: int, held, projections: bool = True):
        """The HOST draws of R CuriosityModule runs, in the reference's order per run: randn(B, 192), randn(B, 768)
        (:609, :744), then for a guided call nn.Linear(768, 64) (:1421: same constructor => same generator draws);
        stacked over the runs and set in the call struct `c`."""
        draws = []
        for _ in range(R):
            eps, noise = torch.randn(B, 192), torch.randn(B, _D)
            tmp = nn.Linear(_D, 64) if projections else None
            draws.append((eps, noise) + ((tmp.weight.detach(), tmp.bias.detach()) if projections else ()))
        stacked = [torch.stack(t).contiguous() for t in zip(*draws)]
        held += stacked
        for field, t in zip(("eps", "noise", "tmp_w", "tmp_b"), stacked):
            setattr(c, field, t.data_ptr())

    def _outputs(self, c, K: int, B: int, N: int):
        """The outputs of K guided calls — depth, confidence [K, B], heat maps [K, B, N], arg-max cells [K, B] — with
        their pointers set in the call struct `c`."""
        out = {"depth": torch.empty(K, B, device=self.device), "conf": torch.empty(K, B, device=self.device),
               "heat": torch.empty(K, B, N, device=self.device),
               "argmax": torch.empty(K, B, device=self.device, dtype=torch.int32)}
        c.depth, c.conf, c.attention, c.argmax = (out[k].data_ptr() for k in ("depth", "conf", "heat", "argmax"))
        return out

    def _guidance(self, c, guidance, N: int, held):
        """One call's instruction string, or guidance tensor [N] / [B, N], into the call struct `c`."""
        if isinstance(guidance, str):
            c.instruction = guidance.encode()
        else:
            m = guidance.to(self.device, torch.float32).contiguous()
            held.append(m)
            c.mask, c.mask_batch_stride = m.data_ptr(), (N if m.dim() == 2 else 0)

    def _guidances(self, s, guidances, N: int, held):
        """A sweep's K instruction strings, or K guidance tensors [N], into the sweep struct `s`."""
        K = len(guidances)
        if not 1 <= K <= _lib.SWEEP_MAX_K:
            raise ValueError(f"an instruction sweep takes 1..{_lib.SWEEP_MAX_K} guidances, got {K}")
        s.K = K
        if all(isinstance(g, str) for g in guidances):
            names = (C.c_char_p * K)(*[g.encode() for g in guidances])
            held.append(names)
            s.instructions = C.cast(names, C.POINTER(C.c_char_p))
        elif all(torch.is_tensor(g) and g.dim() == 1 and g.numel() == N for g in guidances):
            m = torch.stack([g.to(self.device, torch.float32) for g in guidances]).contiguous()
            held.append(m)
            s.masks = m.data_ptr()
        else:
            raise ValueError(f"guidances must be K instruction strings or K guidance tensors of length {N}")
        return K

    @torch.no_grad()
    def forward_with_guidance(self, images, exif, guidance, S=None):
        """-> depth [B,1], confidence [B,1], heat map [B,N], arg-max cell [B] (reference src/model.py:1157-1240).
        `images` may be a list of uint8 [H_i, W_i, 3] photographs of individual sizes: the library resizes them to S."""
        c, held, B, S = self._call(images, exif, S)
        N = (S // 14) ** 2
        self._draws(c, B, 1, held)
        c.curiosity_runs = 1
        self._guidance(c, guidance, N, held)
        out = self._outputs(c, 1, B, N)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_forward_guided(self._h, C.byref(c), self._stream()), "ca_forward_guided")
        self._held = held  # inputs stay referenced until the next call (their reads are enqueued, not finished)
        return out["depth"][0].unsqueeze(1), out["conf"][0].unsqueeze(1), out["heat"][0], out["argmax"][0]

    @torch.no_grad()
    def forward_with_guidance_sweep(self, images, exif, guidances, S=None):
        """K = len(guidances) `forward_with_guidance` calls in one native call (ca_forward_guided_sweep): the backbone and
        the focal pass run once.  `guidances`: K instruction strings, or K guidance tensors [N].  Draws the K calls'
        random numbers in the reference's order per call.  -> depth [K,B,1], confidence [K,B,1], heat maps [K,B,N],
        arg-max cells [K,B]."""
        c, held, B, S = self._call(images, exif, S)
        N = (S // 14) ** 2
        s = _lib.SweepCall()
        K = self._guidances(s, guidances, N, held)
        self._draws(s, B, K, held)
        out = self._outputs(s, K, B, N)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_forward_guided_sweep(self._h, C.byref(c), C.byref(s), self._stream()),
                       "ca_forward_guided_sweep")
        self._held = held
        return out["depth"].unsqueeze(-1), out["conf"].unsqueeze(-1), out["heat"], out["argmax"]

    @torch.no_grad()
    def forward(self, images, exif: Optional[dict] = None, runs: int = 1, S=None):
        """-> depth [B,1], confidence [B,1], focal attention [B,N], fusion features [B,192] (src/model.py:1064-1155).
        `runs`: how often the reference would run its CuriosityModule in this call (1..3, :992, :1104, :1138)."""
        c, held, B, S = self._call(images, exif, S)
        N = (S // 14) ** 2
        self._draws(c, B, runs, held, projections=False)
        c.curiosity_runs = runs
        out = {"depth": torch.empty(B, device=self.device), "conf": torch.empty(B, device=self.device),
               "att": torch.empty(B, N, device=self.device), "fused": torch.empty(B, 192, device=self.device)}
        c.depth, c.conf, c.attention, c.fused = (out[k].data_ptr() for k in ("depth", "conf", "att", "fused"))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_forward(self._h, C.byref(c), self._stream()), "ca_forward")
        self._held = held
        return out["depth"].unsqueeze(1), out["conf"].unsqueeze(1), out["att"], out["fused"]

    @torch.no_grad()
    def backbone_tokens(self, images, S=None):
        if isinstance(images, (list, tuple)):
            imgs, ptrs, hw, held = self._image_list(images, S)
            B, g = len(imgs), S // 14
            tokens = torch.empty(B, g * g + 1, _D, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.ca_backbone_list(self._h, ptrs, hw, B, S, tokens.data_ptr(), self._stream()),
                           "ca_backbone_list")
            self._held = held
            return tokens
        u8 = images.dtype == torch.uint8
        B, S = (images.shape[0], images.shape[1]) if u8 else (images.shape[0], images.shape[-1])
        images = (images if u8 else images.to(torch.float32)).to(self.device).contiguous()
        g = S // 14
        tokens = torch.empty(B, g * g + 1, _D, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_backbone(self._h, images.data_ptr(), int(u8), B, S, tokens.data_ptr(), self._stream()),
                       "ca_backbone")
        self._held = [images]
        return tokens

    @torch.no_grad()
    def encode(self, images, exif, S=None, fault=None) -> "NativeScene":
        """ca_encode: the backbone and the focal pass of the batch, once, kept in a scene for `guide` / `guide_sweep`.
        Draws nothing from the global generator.  `fault`: an optional pinned int32 tensor in which the scene's guide
        calls report a camera index outside the embedding table (bit 0)."""
        if exif is None:
            raise ValueError("a scene needs EXIF data (without it the reference falls back to forward())")
        c, held, B, S = self._call(images, exif, S)
        if fault is not None:
            c.fault = fault.data_ptr()
            held.append(fault)
        out = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_encode(self._h, C.byref(c), C.byref(out), self._stream()), "ca_encode")
        self._held = held
        return NativeScene(self.lib, out, B, S, self.device)

    @torch.no_grad()
    def guide(self, scene: "NativeScene", guidance):
        """ca_guide: `forward_with_guidance` on the encoded images (same draws, same results, same order of draws)."""
        if guidance is None:
            raise ValueError("guide needs an instruction or a guidance tensor")
        B, N = scene.B, (scene.S // 14) ** 2
        c = _lib.GuideCall()
        held = []
        self._guidance(c, guidance, N, held)
        self._draws(c, B, 1, held)
        out = self._outputs(c, 1, B, N)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_guide(self._h, scene.ptr, C.byref(c), self._stream()), "ca_guide")
        self._held = held
        return out["depth"][0].unsqueeze(1), out["conf"][0].unsqueeze(1), out["heat"][0], out["argmax"][0]

    @torch.no_grad()
    def guide_sweep(self, scene: "NativeScene", guidances):
        """ca_guide_sweep: `forward_with_guidance_sweep` on the encoded images."""
        B, N = scene.B, (scene.S // 14) ** 2
        s = _lib.SweepCall()
        held = []
        K = self._guidances(s, guidances, N, held)
        self._draws(s, B, K, held)
        out = self._outputs(s, K, B, N)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_guide_sweep(self._h, scene.ptr, C.byref(s), self._stream()), "ca_guide_sweep")
        self._held = held
        return out["depth"].unsqueeze(-1), out["conf"].unsqueeze(-1), out["heat"], out["argmax"]

    @torch.no_grad()
    def guide_many(self, scenes, guidances):
        """ca_guide_many: one `guide` call on each of m scenes of one side S in one native call, bit for bit what the m
        `guide` calls return, with their draws made in the same order.  `guidances`: m instruction strings, or m guidance
        tensors ([N] or [B_j, N]).  -> a list of m (depth [B_j,1], confidence [B_j,1], heat map [B_j,N], arg-max
        cell [B_j])."""
        m = len(scenes)
        if m == 0 or len(guidances) != m:
            raise ValueError("guide_many takes m >= 1 scenes and one guidance per scene")
        S = scenes[0].S
        N = (S // 14) ** 2
        R = sum(sc.B for sc in scenes)
        c = _lib.GuideManyCall()
        c.m = m
        ptrs = (C.c_void_p * m)(*[sc.ptr.value if sc.ptr is not None else None for sc in scenes])
        c.scenes = C.cast(ptrs, C.POINTER(C.c_void_p))
        held = [ptrs]
        if all(isinstance(g, str) for g in guidances):
            names = (C.c_char_p * m)(*[g.encode() for g in guidances])
            held.append(names)
            c.instructions = C.cast(names, C.POINTER(C.c_char_p))
        elif all(torch.is_tensor(g) for g in guidances):
            rows = [g.to(self.device, torch.float32).reshape(-1, N).expand(sc.B, N) for sc, g in zip(scenes, guidances)]
            masks = torch.cat(rows).contiguous()
            held.append(masks)
            c.masks = masks.data_ptr()
        else:
            raise ValueError("guidances must be m instruction strings or m guidance tensors")
        draws = []
        for sc in scenes:  # per call in order: randn(B_j, 192), randn(B_j, 768), nn.Linear(768, 64)
            eps, noise = torch.randn(sc.B, 192), torch.randn(sc.B, _D)
            tmp = nn.Linear(_D, 64)
            draws.append((eps, noise, tmp.weight.detach(), tmp.bias.detach()))
        eps, noise = torch.cat([d[0] for d in draws]), torch.cat([d[1] for d in draws])
        tmp_w, tmp_b = torch.stack([d[2] for d in draws]).contiguous(), torch.stack([d[3] for d in draws]).contiguous()
        held += [eps, noise, tmp_w, tmp_b]
        c.eps, c.noise, c.tmp_w, c.tmp_b = eps.data_ptr(), noise.data_ptr(), tmp_w.data_ptr(), tmp_b.data_ptr()
        out = self._outputs(c, 1, R, N)
        c.use_graph = int(self.use_graph)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_guide_many(self._h, C.byref(c), self._stream()), "ca_guide_many")
        self._held = held
        res, r = [], 0
        for sc in scenes:
            rows = slice(r, r + sc.B)
            res.append((out["depth"][0, rows].unsqueeze(1), out["conf"][0, rows].unsqueeze(1), out["heat"][0, rows],
                        out["argmax"][0, rows]))
            r += sc.B
        return res

    @torch.no_grad()
    def depth_field(self, scene: "NativeScene"):
        """ca_depth_field: `CognitiveAimModel.depth_field` on the encoded images (the draws of one guide call, in its
        order).  Returns depth, confidence [B, g, g]."""
        B, g = scene.B, scene.S // 14
        c = _lib.DepthFieldCall()
        held = []
        self._draws(c, B, 1, held)
        depth, conf = torch.empty(B, g, g, device=self.device), torch.empty(B, g, g, device=self.device)
        c.depth, c.conf = depth.data_ptr(), conf.data_ptr()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ca_depth_field(self._h, scene.ptr, C.byref(c), self._stream()), "ca_depth_field")
        self._held = held
        return depth, conf

    def launch_count(self) -> int:
        return int(self.lib.ca_last_launch_count(self._h))


class NativeScene:
    """A ca_scene: released by `close()` or when dropped."""

    def __init__(self, lib, ptr, B: int, S: int, device):
        self.lib, self.ptr, self.B, self.S, self.device = lib, ptr, B, S, device

    def close(self):
        if self.ptr is not None and self.ptr.value:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.ca_scene_destroy(self.ptr), "ca_scene_destroy")
        self.ptr = None

    __del__ = close
