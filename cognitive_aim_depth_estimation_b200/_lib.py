"""ctypes binding of libcogaim_b200.so (C-ABI declared in include/cogaim_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing or a call fails, a
RuntimeError carrying `ca_last_error()` is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / "libcogaim_b200.so"

_lib = None

c_f32p = C.c_void_p  # device pointers travel as integers
c_ptr = C.c_void_p


class CogAimError(RuntimeError):
    pass




class HeadsWeights(C.Structure):
    """ca_heads_weights (include/cogaim_b200.h)."""
    _names = ["amb_w0", "amb_b0", "amb_w1", "amb_b1", "amb_w2", "amb_b2", "cam_emb", "exif_w0", "exif_b0", "exif_w1",
              "exif_b1", "exif_f0", "exif_fb0", "exif_f1", "exif_fb1", "fus_w", "fus_b", "dec_w", "dec_b", "conf_w0",
              "conf_b0", "conf_w2", "conf_b2"]
    _fields_ = [(n, C.c_void_p) for n in _names]


class HeadsInputs(C.Structure):
    """ca_heads_inputs (include/cogaim_b200.h)."""
    _fields_ = [("tokens", C.c_void_p), ("tokens_per_img", C.c_int), ("focal_feat", C.c_void_p),
                ("pool_partial", C.c_void_p), ("pool_splits", C.c_int), ("tmp_w", C.c_void_p), ("tmp_b", C.c_void_p),
                ("pooled_out", C.c_void_p), ("exif", C.c_void_p), ("camera_idx", C.c_void_p),
                ("num_cameras", C.c_int), ("fault", C.c_void_p), ("sweep_images", C.c_int)]


class FocalValueArgs(C.Structure):
    """ca_focal_value_args (include/cogaim_b200.h)."""
    _fields_ = [("tok_partial", C.c_void_p), ("pe_partial", C.c_void_p), ("splits", C.c_int), ("wv", C.c_void_p),
                ("bv", C.c_void_p), ("proj_w0", C.c_void_p), ("proj_b0", C.c_void_p), ("proj_w1", C.c_void_p),
                ("proj_b1", C.c_void_p), ("feat_out", C.c_void_p), ("iter", C.c_int), ("n_iters", C.c_int)]


class CuriosityWeights(C.Structure):
    """ca_curiosity_weights (include/cogaim_b200.h)."""
    _names = ["em_w0", "em_b0", "em_w1", "em_b1", "el_w0", "el_b0", "el_w1", "el_b1", "dec_w0", "dec_b0", "dec_w1",
              "dec_b1", "unc_w0", "unc_b0", "unc_w1", "unc_b1", "loc_w0", "loc_b0", "loc_w1", "loc_b1", "cur_w"]
    _fields_ = [(n, C.c_void_p) for n in _names]


class CuriosityModWeights(C.Structure):
    """ca_curiosity_mod_weights (include/cogaim_b200.h)."""
    _fields_ = [("amp_w0", C.c_void_p), ("amp_b0", C.c_void_p), ("amp_w1", C.c_void_p), ("amp_b1", C.c_void_p),
                ("mod_w0", C.c_void_p * 8), ("mod_b0", C.c_void_p * 8), ("mod_w1", C.c_void_p * 8),
                ("mod_b1", C.c_void_p * 8)]


class LayerWeights(C.Structure):
    """ca_layer_weights (include/cogaim_b200.h)."""
    _names = ["n1w", "n1b", "wqkv", "bqkv", "wo", "bo", "ls1", "n2w", "n2b", "w1", "b1", "w2", "b2", "ls2"]
    _fields_ = [(n, C.c_void_p) for n in _names]


class FocalWeights(C.Structure):
    """ca_focal_weights (include/cogaim_b200.h)."""
    _names = ["wqk", "bqk", "wv", "bv", "pw0", "pb0", "pw1", "pb1"]
    _fields_ = [(n, C.c_void_p) for n in _names]


class ModelWeights(C.Structure):
    """ca_model_weights (include/cogaim_b200.h)."""
    _fields_ = [("patch_w", C.c_void_p), ("patch_b", C.c_void_p), ("cls_token", C.c_void_p), ("pos_embed", C.c_void_p),
                ("layer", LayerWeights * 12), ("lnw", C.c_void_p), ("lnb", C.c_void_p), ("n_focal", C.c_int),
                ("focus_strength", C.c_float), ("focal", FocalWeights * 4), ("ffw0", C.c_void_p), ("ffb0", C.c_void_p),
                ("ffw1", C.c_void_p), ("ffb1", C.c_void_p), ("heads", HeadsWeights), ("curiosity", CuriosityWeights),
                ("exploration_history", C.c_void_p), ("history_len", C.c_int), ("history_pointer", C.c_void_p),
                ("num_cameras", C.c_int), ("layernorm_folded", C.c_int)]


class ForwardCall(C.Structure):
    """ca_forward_call (include/cogaim_b200.h)."""
    _fields_ = [("images", C.c_void_p), ("images_u8", C.c_int), ("B", C.c_int), ("S", C.c_int), ("exif", C.c_void_p),
                ("camera_idx", C.c_void_p), ("instruction", C.c_char_p), ("mask", C.c_void_p),
                ("mask_batch_stride", C.c_longlong), ("tmp_w", C.c_void_p), ("tmp_b", C.c_void_p), ("eps", C.c_void_p),
                ("noise", C.c_void_p), ("curiosity_runs", C.c_int), ("depth", C.c_void_p), ("conf", C.c_void_p),
                ("attention", C.c_void_p), ("argmax", C.c_void_p), ("fused", C.c_void_p), ("fault", C.c_void_p),
                ("use_graph", C.c_int), ("image_list", C.POINTER(C.c_void_p)), ("image_hw", C.POINTER(C.c_int))]


SWEEP_MAX_K = 16  # CA_SWEEP_MAX_K (include/cogaim_b200.h)
GUIDE_TAIL_MAX_B = 1  # CA_GUIDE_TAIL_MAX_B: guide calls of larger batches run the three-kernel chain
RESIZE_MAX_SIDE = 16384  # CA_RESIZE_MAX_SIDE
RESIZE_LIST_CHUNK = 128  # CA_RESIZE_LIST_CHUNK


class SweepCall(C.Structure):
    """ca_sweep_call (include/cogaim_b200.h)."""
    _fields_ = [("K", C.c_int), ("instructions", C.POINTER(C.c_char_p)), ("masks", C.c_void_p), ("tmp_w", C.c_void_p),
                ("tmp_b", C.c_void_p), ("eps", C.c_void_p), ("noise", C.c_void_p), ("depth", C.c_void_p),
                ("conf", C.c_void_p), ("attention", C.c_void_p), ("argmax", C.c_void_p)]


class GuideCall(C.Structure):
    """ca_guide_call (include/cogaim_b200.h)."""
    _fields_ = [("instruction", C.c_char_p), ("mask", C.c_void_p), ("mask_batch_stride", C.c_longlong),
                ("tmp_w", C.c_void_p), ("tmp_b", C.c_void_p), ("eps", C.c_void_p), ("noise", C.c_void_p),
                ("depth", C.c_void_p), ("conf", C.c_void_p), ("attention", C.c_void_p), ("argmax", C.c_void_p)]


# name -> (argtypes); every function returns int status except where noted in _RESTYPES
_SIGNATURES = {
    "ca_version": [],
    "ca_device_check": [C.c_int],
    "ca_gemm_bf16": [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong,
                     C.c_longlong, C.c_int, c_ptr, C.c_int, C.c_longlong, c_ptr, c_ptr, c_ptr, C.c_int, C.c_float,
                     c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    "ca_gemm_bf16_ln": [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr,
                        c_ptr, C.c_int, C.c_float, c_ptr, C.c_int, c_ptr],
    "ca_ln_shadow": [c_ptr, c_ptr, C.c_int, c_ptr, C.c_int, C.c_int, c_ptr],
    "ca_attention_bf16": [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_attention_bf16_ld": [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_patchify_f32": [c_ptr, c_ptr, C.c_int, C.c_int, c_ptr],
    "ca_preprocess_u8": [c_ptr, c_ptr, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), c_ptr],
    "ca_cls_rows": [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_layernorm": [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_float, c_ptr],
    "ca_layernorm_ld": [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, c_ptr],
    "ca_focal_input": [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_fetch_pinned_f32": [c_ptr, c_ptr, C.c_size_t, c_ptr],
    "ca_rowstats_merge": [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_colsum_e": [c_ptr, C.c_int, C.c_longlong, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_focal_finalize": [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, c_ptr,
                          C.c_float, c_ptr],
    "ca_curiosity": [C.POINTER(CuriosityWeights), c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr,
                     C.c_int, c_ptr],
    "ca_curiosity_modulation": [C.POINTER(CuriosityModWeights), c_ptr, C.c_float, C.c_float, c_ptr, C.c_int, C.c_int,
                                C.c_int, c_ptr],
    "ca_resize_u8": [c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr],
    "ca_resize_u8_list_tmp_bytes": [C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int],
    "ca_resize_u8_list": [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr,
                          c_ptr],
    "ca_jpeg_info": [C.c_char_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "ca_jpeg_decode": [C.c_char_p, C.c_size_t, c_ptr, C.c_int, C.c_int, c_ptr],
    "ca_jpeg_decode_batch": [C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), C.c_int, C.POINTER(C.c_void_p),
                             C.POINTER(C.c_int), C.POINTER(C.c_int), c_ptr],
    "ca_focus_map": [c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr],
    "ca_guided_softmax": [c_ptr, c_ptr, C.c_longlong, c_ptr, c_ptr, C.c_int, C.c_int, C.c_float, C.c_float, c_ptr],
    "ca_weighted_pool": [c_ptr, C.c_longlong, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr],
    "ca_guided_softmax_sweep": [c_ptr, C.c_longlong, c_ptr, C.c_longlong, C.c_longlong, c_ptr, c_ptr, C.c_int, C.c_int,
                                C.c_int, C.c_float, C.c_float, c_ptr],
    "ca_weighted_pool_sweep": [c_ptr, C.c_longlong, C.c_int, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               c_ptr],
    "ca_heads": [C.POINTER(HeadsWeights), C.POINTER(HeadsInputs), c_ptr, c_ptr, c_ptr, C.c_int, c_ptr],
    "ca_guide_tail": [C.POINTER(HeadsWeights), C.POINTER(HeadsInputs), c_ptr, c_ptr, C.c_longlong, c_ptr, c_ptr, c_ptr,
                      c_ptr, c_ptr, C.c_int, C.c_int, C.c_float, C.c_float, c_ptr],
    "ca_focal_value": [C.POINTER(FocalValueArgs), C.c_int, c_ptr],
    "ca_focal_fusion": [c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr],
    "ca_create": [C.POINTER(C.c_void_p), C.POINTER(ModelWeights), C.c_int],
    "ca_destroy": [c_ptr],
    "ca_forward_guided": [c_ptr, C.POINTER(ForwardCall), c_ptr],
    "ca_forward_guided_sweep": [c_ptr, C.POINTER(ForwardCall), C.POINTER(SweepCall), c_ptr],
    "ca_forward": [c_ptr, C.POINTER(ForwardCall), c_ptr],
    "ca_backbone": [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr],
    "ca_backbone_list": [c_ptr, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int, C.c_int, c_ptr, c_ptr],
    "ca_last_launch_count": [c_ptr],
    "ca_encode": [c_ptr, C.POINTER(ForwardCall), C.POINTER(C.c_void_p), c_ptr],
    "ca_guide": [c_ptr, c_ptr, C.POINTER(GuideCall), c_ptr],
    "ca_guide_sweep": [c_ptr, c_ptr, C.POINTER(SweepCall), c_ptr],
    "ca_scene_destroy": [c_ptr],
}


_RESTYPES = {"ca_resize_u8_list_tmp_bytes": C.c_size_t}


def exported_symbols():
    """Every symbol include/cogaim_b200.h declares (used by the CPU-side ABI test)."""
    return ["ca_last_error", *_SIGNATURES.keys()]


def load():
    """Load the library once; raise loudly if it has not been built (`__graft_entry__.build()`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CogAimError(
            f"{LIB_PATH} is missing: build it with `python -m cognitive_aim_depth_estimation_b200.build` "
            "(there is no CPU / PyTorch fallback for the Cognitive-Aim forward path)")
    lib = C.CDLL(str(LIB_PATH))
    lib.ca_last_error.restype = C.c_char_p
    lib.ca_last_error.argtypes = []
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = _RESTYPES.get(name, C.c_int)
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(status: int, what: str):
    if status != 0:
        msg = load().ca_last_error()
        raise CogAimError(f"{what} failed with status {status}: {msg.decode() if msg else '?'}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def image_arrays(images):
    """HOST arrays (device pointers [B], (H, W) pairs [B, 2]) of a list of uint8 [H_i, W_i, 3] CUDA tensors, as the
    list entry points (ca_resize_u8_list, ca_forward_call.image_list) take them."""
    ptrs = (C.c_void_p * len(images))(*[t.data_ptr() for t in images])
    hw = (C.c_int * (2 * len(images)))(*[int(d) for t in images for d in t.shape[:2]])
    return ptrs, hw


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
