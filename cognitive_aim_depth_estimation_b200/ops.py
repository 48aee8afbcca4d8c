"""Thin Python wrappers over the C-ABI entry points (one wrapper per entry point, no arithmetic here).

Tensors are torch CUDA tensors used purely as device-memory handles; every wrapper validates dtype /
contiguity, forwards raw pointers and raises `CogAimError` on a non-zero status.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

EPI_BIAS_BF16 = 0
EPI_GELU_BF16 = 1
EPI_RESID_F32 = 2
EPI_PATCH_F32 = 3
EPI_ROWSTATS = 4
EPI_COLSUM = 5
EPI_F32 = 6
EPI_LN_BIAS_BF16, EPI_LN_GELU_BF16, EPI_RESID_LN_F32 = 7, 8, 9


class _Trace:
    """Launch accounting: `launches` counts kernels enqueued by this module; when `events` is a list every call is
    bracketed by CUDA events on the launching stream (bench.py reads per-kernel device time from them)."""
    launches = 0
    events = None


def trace_start(with_events: bool):
    _Trace.launches = 0
    _Trace.events = [] if with_events else None


def trace_stop():
    ev, n = _Trace.events, _Trace.launches
    _Trace.events = None
    return n, ev


def tracing_events() -> bool:
    """True while per-launch CUDA events are being recorded (graph replay would hide the launches from them)."""
    return _Trace.events is not None


def launch_count() -> int:
    return _Trace.launches


def count_launches(n: int):
    """Account for `n` kernels launched by replaying a captured graph."""
    _Trace.launches += n


def _begin():
    if _Trace.events is None:
        return None
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def _end(e0, name, n_kernels, work=0.0):
    _Trace.launches += n_kernels
    if e0 is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        _Trace.events.append((name, work, e0, e1))


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (no CPU fallback)")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")


def stats_partials(n: int) -> int:
    """P: per-row partial slots of the statistics epilogues = one per 64-column span of the 256-wide tiles."""
    return 4 * ((n + 255) // 256)


def gemm(A, W, epilogue, out=None, *, M=None, N=None, K=None, lda=None, ldw=None, batch=1, a_batch_stride=0,
         w_batch_stride=0, ldo=None, out_batch_stride=0, bias=None, ls=None, pos=None, patches_per_img=0,
         scale_log2=0.0, part_a=None, part_b=None, col_max=None, col_rinv=None):
    """C = epilogue(A @ W^T) on tcgen05 tensor cores (csrc/gemm.cu). A:[M,K] bf16, W:[N,K] bf16."""
    lib = _lib.load()
    _req(A, torch.bfloat16, "A")
    _req(W, torch.bfloat16, "W")
    M = A.shape[-2] if M is None else M
    K = A.shape[-1] if K is None else K
    N = W.shape[-2] if N is None else N
    lda = A.stride(-2) if lda is None else lda
    ldw = W.stride(-2) if ldw is None else ldw
    if out is not None and ldo is None:
        ldo = out.stride(-2)
    for t, n in ((bias, "bias"), (ls, "ls"), (pos, "pos"), (part_a, "part_a"), (part_b, "part_b"),
                 (col_max, "col_max"), (col_rinv, "col_rinv")):
        _req(t, torch.float32, n)
    e0 = _begin()
    st = lib.ca_gemm_bf16(ptr(A), ptr(W), M, N, K, lda, ldw, batch, a_batch_stride, w_batch_stride, epilogue,
                          ptr(out), ldo or 0, out_batch_stride, ptr(bias), ptr(ls), ptr(pos), patches_per_img,
                          float(scale_log2), ptr(part_a), ptr(part_b), ptr(col_max), ptr(col_rinv), stream_ptr())
    check(st, "ca_gemm_bf16")
    _end(e0, "gemm_stats" if epilogue in (EPI_ROWSTATS, EPI_COLSUM) else "gemm", 1, 2.0 * M * N * K * batch)
    return out


def gemm_ln(A, W, epilogue, out, *, bias, stats, ls=None, shadow=None, eps=1e-6):
    """The LayerNorm-folded forms of `gemm` (csrc/gemm.cuh EPI_LN_* / EPI_RESID_LN_F32; include/cogaim_b200.h
    ca_gemm_bf16_ln).  stats: fp32 [M, slots, 2]."""
    lib = _lib.load()
    _req(A, torch.bfloat16, "A")
    _req(W, torch.bfloat16, "W")
    for t, n in ((bias, "bias"), (ls, "ls"), (stats, "stats")):
        _req(t, torch.float32, n)
    _req(shadow, torch.bfloat16, "shadow")
    M, K, N = A.shape[-2], A.shape[-1], W.shape[-2]
    e0 = _begin()
    st = lib.ca_gemm_bf16_ln(ptr(A), ptr(W), M, N, K, A.stride(-2), W.stride(-2), epilogue, ptr(out), out.stride(-2),
                             ptr(bias), ptr(ls), ptr(stats), stats.shape[-2], float(eps), ptr(shadow),
                             shadow.stride(-2) if shadow is not None else 0, stream_ptr())
    check(st, "ca_gemm_bf16_ln")
    _end(e0, "gemm", 1, 2.0 * M * N * K)
    return out


def fold_layernorm(weight, bias, gamma, beta):
    """Operands of an EPI_LN_* GEMM from a Linear (weight [N, K], bias [N]) and the LayerNorm (gamma, beta [K]) in front of
    it:  LN(x) W^T + b = rstd * (x W'^T) + b'  with  W' = bf16(rows of W diag(gamma), centred)  and  b' = b + W beta.
    Centring the rows (sum_k W'[n,k] = 0) makes x W'^T = (x - mean(x)) W'^T: the GEMM on the RAW rows already carries the
    mean subtraction, and the epilogue is left with the row's 1/std."""
    w32 = weight.float()
    wg = w32 * gamma.float()[None, :]
    wp = (wg - wg.mean(dim=1, keepdim=True)).to(torch.bfloat16).contiguous()
    bp = (bias.float() + w32 @ beta.float()).contiguous()
    return wp, bp


def ln_shadow(x, shadow, stats):
    """bf16 copy of the fp32 rows + the per-128-column (sum, M2) row statistics: entry of the LayerNorm-folded chain."""
    _req(x, torch.float32, "x")
    _req(shadow, torch.bfloat16, "shadow")
    _req(stats, torch.float32, "stats")
    rows, D = x.shape[-2], x.shape[-1]
    e0 = _begin()
    check(_lib.load().ca_ln_shadow(ptr(x), ptr(shadow), shadow.stride(-2), ptr(stats), rows, D, stream_ptr()),
          "ca_ln_shadow")
    _end(e0, "layernorm", 1, 0.0)
    return shadow


LOG2E = math.log2(math.e)

PATCH_ROW_STRIDE = 592
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def attention(qkv, out, B, T, H):
    """out[B*T, H*64] = softmax(QK^T/8)V per (image, head) (csrc/attention.cu)."""
    _req(qkv, torch.bfloat16, "qkv")
    _req(out, torch.bfloat16, "out")
    e0 = _begin()
    if out.stride(-2) != H * 64:  # a strided view: the rows carry LoRA columns behind the H*64 outputs
        check(_lib.load().ca_attention_bf16_ld(ptr(qkv), ptr(out), out.stride(-2), B, T, H, stream_ptr()),
              "ca_attention_bf16_ld")
    else:
        check(_lib.load().ca_attention_bf16(ptr(qkv), ptr(out), B, T, H, stream_ptr()), "ca_attention_bf16")
    _end(e0, "attention", 1, 4.0 * B * H * T * T * 64)
    return out


def patchify_f32(images, patches):
    _req(images, torch.float32, "images")
    _req(patches, torch.bfloat16, "patches")
    B, _, S, _ = images.shape
    e0 = _begin()
    check(_lib.load().ca_patchify_f32(ptr(images), ptr(patches), B, S, stream_ptr()), "ca_patchify_f32")
    _end(e0, "patchify", 1, float(images.numel() * 4 + patches.numel() * 2))
    return patches


def preprocess_u8(images_hwc, patches, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    import ctypes as C
    _req(images_hwc, torch.uint8, "images")
    _req(patches, torch.bfloat16, "patches")
    B, S = images_hwc.shape[0], images_hwc.shape[1]
    m = (C.c_float * 3)(*mean)
    s = (C.c_float * 3)(*std)
    e0 = _begin()
    check(_lib.load().ca_preprocess_u8(ptr(images_hwc), ptr(patches), B, S, m, s, stream_ptr()), "ca_preprocess_u8")
    _end(e0, "preprocess_u8", 1, float(images_hwc.numel() + patches.numel() * 2))
    return patches


def cls_rows(x, cls, pos, B, T, D):
    e0 = _begin()
    check(_lib.load().ca_cls_rows(ptr(x), ptr(cls), ptr(pos), B, T, D, stream_ptr()), "ca_cls_rows")
    _end(e0, "small", 1)


def layernorm(x, gamma, beta, out, eps=1e-6):
    _req(x, torch.float32, "x")
    rows, D = x.numel() // x.shape[-1], x.shape[-1]
    e0 = _begin()
    if out.dim() >= 2 and out.stride(-2) != D:  # strided rows (LoRA columns behind each row)
        check(_lib.load().ca_layernorm_ld(ptr(x), ptr(gamma), ptr(beta), ptr(out), int(out.dtype == torch.bfloat16),
                                          out.stride(-2), rows, D, eps, stream_ptr()), "ca_layernorm_ld")
    else:
        check(_lib.load().ca_layernorm(ptr(x), ptr(gamma), ptr(beta), ptr(out), int(out.dtype == torch.bfloat16), rows,
                                       D, eps, stream_ptr()), "ca_layernorm")
    _end(e0, "layernorm", 1, float(rows * D * (4 + out.element_size())))
    return out


def focal_input(tokens, pe, rowscale, xin, B, N, D):
    e0 = _begin()
    check(_lib.load().ca_focal_input(ptr(tokens), ptr(pe), ptr(rowscale), ptr(xin), B, N, D, stream_ptr()),
          "ca_focal_input")
    _end(e0, "focal_input", 1, float(B * N * D * 6))
    return xin


def fetch_pinned(dst, src_pinned):
    """dst (CUDA fp32) <- src_pinned (pinned CPU fp32, contiguous, same numel) through an SM-side read of host memory:
    never queues behind a bulk upload on the H2D copy engine (csrc/rowops.cu)."""
    import ctypes as C
    _req(dst, torch.float32, "dst")
    if src_pinned.is_cuda or not src_pinned.is_pinned() or src_pinned.dtype != torch.float32:
        raise ValueError("fetch_pinned expects a pinned fp32 CPU tensor")
    if not (dst.is_contiguous() and src_pinned.is_contiguous()) or dst.numel() != src_pinned.numel():
        raise ValueError("fetch_pinned expects contiguous tensors of equal size")
    e0 = _begin()
    check(_lib.load().ca_fetch_pinned_f32(ptr(dst), C.c_void_p(src_pinned.data_ptr()), dst.numel(), stream_ptr()),
          "ca_fetch_pinned_f32")
    _end(e0, "small", 1)


def rowstats_merge(pm, ps, weight, rmax, rinv, wtab=None):
    """pm, ps (and wtab): span-major [B, P, N] partials of the CA_EPI_ROWSTATS epilogue."""
    P, n = pm.shape[-2], pm.shape[-1]
    rows = pm.numel() // P
    e0 = _begin()
    check(_lib.load().ca_rowstats_merge(ptr(pm), ptr(ps), ptr(weight), ptr(rmax), ptr(rinv), ptr(wtab), rows, n, P,
                                        stream_ptr()), "ca_rowstats_merge")
    _end(e0, "small", 1)


def colsum_e(E, wtab, pc, B, N):
    """pc[B, P, N] (span-major) column-sum partials of the (weighted) row softmax from the stored fp16 exponentials
    E [B, N, lde]."""
    _req(E, torch.float16, "E")
    _req(wtab, torch.float32, "wtab")
    _req(pc, torch.float32, "pc")
    P = pc.shape[-2]
    if pc.shape[-1] != N or wtab.shape[-2] != P or wtab.shape[-1] != N:
        raise ValueError("colsum_e: pc and wtab must be span-major [B, P, N]")
    e0 = _begin()
    check(_lib.load().ca_colsum_e(ptr(E), E.stride(-2), E.stride(0), ptr(wtab), ptr(pc), B, N, P, stream_ptr()),
          "ca_colsum_e")
    _end(e0, "colsum_e", 1, float(E.numel() * 2))


def focal_finalize(pc, cbias, attn, rs_in, rs_out, B, N, focus_strength=1.5, mode=0, cur_weight=None,
                   adaptive_weight=0.5):
    """pc [B, P, N] span-major partials; cur_weight [B] (optional) + adaptive_weight: the curiosity modulation of
    src/model.py:264-276."""
    P = pc.shape[-2]
    _req(cur_weight, torch.float32, "cur_weight")
    e0 = _begin()
    check(_lib.load().ca_focal_finalize(ptr(pc), ptr(cbias), ptr(attn), ptr(rs_in), ptr(rs_out), B, N, P,
                                        float(focus_strength), mode, ptr(cur_weight), float(adaptive_weight),
                                        stream_ptr()), "ca_focal_finalize")
    _end(e0, "small", 1)


def guided_softmax(base, mask, heat, argmax, B, N, alpha=0.7, temperature=0.05):
    """mask: [N] (one instruction for the batch) or [B, N] (one per image)."""
    _req(base, torch.float32, "base")
    _req(mask, torch.float32, "mask")
    _req(argmax, torch.int32, "argmax")
    if mask.dim() == 2 and mask.shape[0] != B:
        raise ValueError(f"per-image mask has {mask.shape[0]} rows for a batch of {B}")
    stride = mask.stride(0) if mask.dim() == 2 else 0
    e0 = _begin()
    check(_lib.load().ca_guided_softmax(ptr(base), ptr(mask), stride, ptr(heat), ptr(argmax), B, N, alpha, temperature,
                                        stream_ptr()), "ca_guided_softmax")
    _end(e0, "small", 1)


def weighted_pool(src, src_batch_stride, row_offset, w, w2, partial, B, N, D, splits):
    e0 = _begin()
    check(_lib.load().ca_weighted_pool(ptr(src), src_batch_stride, row_offset, ptr(w), ptr(w2), ptr(partial), B, N, D,
                                       splits, stream_ptr()), "ca_weighted_pool")
    _end(e0, "pool", 1, float(B * N * D * 4))


def guided_softmax_sweep(base, base_k_stride, mask, heat, argmax, K, B, N, alpha=0.7, temperature=0.05):
    """K * B rows of `guided_softmax` (instruction sweep): mask [K, B, N], heat [K, B, N], argmax [K, B]; row k * B + b
    reads base + k * base_k_stride + b * N (base_k_stride 0: one base attention [B, N] shared by every instruction)."""
    _req(base, torch.float32, "base")
    _req(mask, torch.float32, "mask")
    _req(heat, torch.float32, "heat")
    _req(argmax, torch.int32, "argmax")
    if mask.shape != (K, B, N) or not mask.is_contiguous():
        raise ValueError(f"sweep mask must be a contiguous [K, B, N] = [{K}, {B}, {N}] tensor, got {tuple(mask.shape)}")
    e0 = _begin()
    check(_lib.load().ca_guided_softmax_sweep(ptr(base), base_k_stride, ptr(mask), B * N, N, ptr(heat), ptr(argmax), K, B,
                                              N, alpha, temperature, stream_ptr()), "ca_guided_softmax_sweep")
    _end(e0, "small", 1)


def weighted_pool_sweep(src, src_batch_stride, row_offset, w, partial, K, B, N, D, splits):
    """`weighted_pool` for K weight vectors w [K, B, N] at once: partial [K * B, splits, D], the tokens read once."""
    e0 = _begin()
    check(_lib.load().ca_weighted_pool_sweep(ptr(src), src_batch_stride, row_offset, ptr(w), ptr(partial), K, B, N, D,
                                             splits, stream_ptr()), "ca_weighted_pool_sweep")
    _end(e0, "pool", 1, float(B * N * D * 4))


def _row_table(rows, R):
    """A device row table (`ca_guide_many_row` [R]) held as int64 [R, GUIDE_MANY_ROW_WORDS] or fp32 [R, 2 * words]."""
    if not rows.is_cuda or rows.dtype not in (torch.int64, torch.float32) or not rows.is_contiguous():
        raise ValueError("rows must be a contiguous CUDA tensor (int64 or fp32 words of ca_guide_many_row)")
    if rows.numel() * rows.element_size() != R * _lib.GUIDE_MANY_ROW_WORDS * 8:
        raise ValueError(f"rows must hold {R} ca_guide_many_row entries")


def gather_rows(rows, R, N, cls, base, exif, camera_idx, call_of_row, num_cameras=0):
    """Through the row table `rows` (ca_guide_many_row [R]): cls [R, 768], base [R, N], exif [R, 3], camera_idx [R]
    (int64) and call_of_row [R] (int32), one launch (csrc/focal.cu).  A camera index outside [0, num_cameras) sets bit 0
    of the row's fault word."""
    _row_table(rows, R)
    for t, n in ((cls, "cls"), (base, "base"), (exif, "exif")):
        _req(t, torch.float32, n)
    _req(camera_idx, torch.int64, "camera_idx")
    _req(call_of_row, torch.int32, "call_of_row")
    if cls.numel() < R * 768 or base.numel() < R * N or exif.numel() < R * 3 or camera_idx.numel() < R \
            or call_of_row.numel() < R:
        raise ValueError("gather_rows: the outputs are smaller than R rows")
    e0 = _begin()
    check(_lib.load().ca_gather_rows(ptr(rows), R, N, int(num_cameras), ptr(cls), ptr(base), ptr(exif), ptr(camera_idx),
                                     ptr(call_of_row), stream_ptr()), "ca_gather_rows")
    _end(e0, "small", 1)


def weighted_pool_rows(rows, w, partial, R, N, D, splits):
    """`weighted_pool` over R rows of several scenes: row r pools w [R, N] against the tokens the row table points to
    (rows 1..N of that image); partial [R, splits, D]."""
    _row_table(rows, R)
    _req(w, torch.float32, "w")
    _req(partial, torch.float32, "partial")
    if w.numel() < R * N or partial.numel() < R * splits * D:
        raise ValueError("weighted_pool_rows: w needs R * N and partial R * splits * D floats")
    e0 = _begin()
    check(_lib.load().ca_weighted_pool_rows(ptr(rows), ptr(w), ptr(partial), R, N, D, splits, stream_ptr()),
          "ca_weighted_pool_rows")
    _end(e0, "pool", 1, float(R * N * D * 4))


def resize_u8(src, out_h, out_w):
    """uint8 [B, H0, W0, 3] -> uint8 [B, out_h, out_w, 3], bit-exact PIL.Image.resize(..., BILINEAR) (csrc/resize.cu)."""
    _req(src, torch.uint8, "src")
    if src.dim() != 4 or src.shape[-1] != 3 or not src.is_contiguous():
        raise ValueError("resize_u8 expects a contiguous uint8 [B, H, W, 3] tensor")
    B, H0, W0, _ = src.shape
    out = torch.empty(B, out_h, out_w, 3, device=src.device, dtype=torch.uint8)
    tmp = torch.empty(B, H0, out_w, 3, device=src.device, dtype=torch.uint8) if (H0 != out_h and W0 != out_w) else None
    e0 = _begin()
    check(_lib.load().ca_resize_u8(ptr(src), B, H0, W0, out_h, out_w, ptr(tmp), ptr(out), stream_ptr()), "ca_resize_u8")
    _end(e0, "resize", 2 if tmp is not None else 1, float(src.numel() + out.numel()))
    return out


def resize_u8_list(images, out_h, out_w):
    """list of B uint8 [H_i, W_i, 3] CUDA tensors (individual sizes) -> uint8 [B, out_h, out_w, 3], each image bit-exact
    PIL.Image.resize(..., BILINEAR); two launches for the whole batch whatever its mix of sizes (csrc/resize.cu)."""
    import ctypes as C
    if not isinstance(images, (list, tuple)) or len(images) == 0:
        raise ValueError("resize_u8_list expects a non-empty list of images")
    for t in images:
        _req(t, torch.uint8, "images")
        if t.dim() != 3 or t.shape[-1] != 3 or not t.is_contiguous():
            raise ValueError("resize_u8_list expects contiguous uint8 [H, W, 3] tensors")
        if not 0 < min(t.shape[0], t.shape[1]) <= max(t.shape[0], t.shape[1]) <= _lib.RESIZE_MAX_SIDE:
            raise ValueError(f"image sides must be in [1, {_lib.RESIZE_MAX_SIDE}], got {tuple(t.shape[:2])}")
    B = len(images)
    dev = images[0].device
    if any(t.device != dev for t in images):
        raise ValueError("resize_u8_list expects every image on one device")
    lib = _lib.load()
    ptrs, hw = _lib.image_arrays(images)
    tmp_bytes = int(lib.ca_resize_u8_list_tmp_bytes(hw, B, out_h, out_w))
    out = torch.empty(B, out_h, out_w, 3, device=dev, dtype=torch.uint8)
    tmp = torch.empty(tmp_bytes, device=dev, dtype=torch.uint8) if tmp_bytes else None
    # kernels per chunk of images: one per pass that some image of the chunk needs (an image of the target size is copied)
    n = 0
    for c0 in range(0, B, _lib.RESIZE_LIST_CHUNK):
        chunk = images[c0:c0 + _lib.RESIZE_LIST_CHUNK]
        n += any(t.shape[1] != out_w for t in chunk) + any(t.shape[0] != out_h for t in chunk)
    e0 = _begin()
    with torch.cuda.device(dev):
        check(lib.ca_resize_u8_list(ptrs, hw, B, out_h, out_w, ptr(tmp), tmp_bytes, ptr(out), stream_ptr()),
              "ca_resize_u8_list")
    _end(e0, "resize", n, float(sum(t.numel() for t in images) + out.numel()))
    return out


def jpeg_decode(data: bytes, device=None):
    """One JPEG file's bytes -> uint8 [H, W, 3] RGB CUDA tensor, decoded by nvJPEG on the current stream
    (csrc/jpeg.cu; reference demo.py:312 `Image.open(path).convert('RGB')`)."""
    import ctypes as C
    if not isinstance(data, (bytes, bytearray, memoryview)):
        raise ValueError("jpeg_decode expects the file's bytes")
    data = bytes(data)
    lib = _lib.load()
    w, h = C.c_int(0), C.c_int(0)
    check(lib.ca_jpeg_info(data, len(data), C.byref(w), C.byref(h)), "ca_jpeg_info")
    out = torch.empty(h.value, w.value, 3, device=device or "cuda", dtype=torch.uint8)
    e0 = _begin()
    with torch.cuda.device(out.device):
        check(lib.ca_jpeg_decode(data, len(data), ptr(out), w.value, h.value, stream_ptr()), "ca_jpeg_decode")
    _end(e0, "jpeg", 1, float(out.numel()))
    return out


def jpeg_decode_batch(files, device=None, return_groups=False):
    """List of JPEG files (bytes) -> list of uint8 [H_i, W_i, 3] RGB CUDA tensors, decoded in ONE nvjpegDecodeBatched call
    (reference demo.py:406-432 `predict_batch` opens and decodes its files one at a time).  Images of equal size share
    one contiguous [k, H, W, 3] allocation (the returned tensors are its slices); `return_groups=True` also returns
    [(block [k, H, W, 3], indices into the list)].  `resize_u8_list` takes the returned list whatever its sizes."""
    import ctypes as C
    if len(files) == 0:
        raise ValueError("empty list of JPEG files")
    datas = []
    for f in files:
        if not isinstance(f, (bytes, bytearray, memoryview)):
            raise ValueError("jpeg_decode_batch expects each file's bytes")
        datas.append(bytes(f))
    lib = _lib.load()
    n = len(datas)
    ws, hs = (C.c_int * n)(), (C.c_int * n)()
    for i, d in enumerate(datas):
        w, h = C.c_int(0), C.c_int(0)
        check(lib.ca_jpeg_info(d, len(d), C.byref(w), C.byref(h)), "ca_jpeg_info")
        ws[i], hs[i] = w.value, h.value
    dev = torch.device(device or "cuda")
    groups = {}
    for i in range(n):
        groups.setdefault((hs[i], ws[i]), []).append(i)
    outs = [None] * n
    blocks = []
    for (h, w), idx in groups.items():
        block = torch.empty(len(idx), h, w, 3, device=dev, dtype=torch.uint8)
        blocks.append((block, idx))
        for j, i in enumerate(idx):
            outs[i] = block[j]
    data_arr = (C.c_char_p * n)(*datas)
    len_arr = (C.c_size_t * n)(*[len(d) for d in datas])
    out_arr = (C.c_void_p * n)(*[o.data_ptr() for o in outs])
    e0 = _begin()
    with torch.cuda.device(dev):
        check(lib.ca_jpeg_decode_batch(data_arr, len_arr, n, out_arr, ws, hs, stream_ptr()), "ca_jpeg_decode_batch")
    _end(e0, "jpeg", 1, float(sum(o.numel() for o in outs)))
    return (outs, blocks) if return_groups else outs


def focus_map(heat, g, out_h, out_w, norm, out):
    """norm [B, g*g], out [B, out_h, out_w] (or None): heat-map post-processing of demo.py:530-563 (csrc/visual.cu)."""
    _req(heat, torch.float32, "heat")
    _req(norm, torch.float32, "norm")
    _req(out, torch.float32, "out")
    B = heat.shape[0]
    e0 = _begin()
    check(_lib.load().ca_focus_map(ptr(heat), B, g, out_h, out_w, ptr(norm), ptr(out), stream_ptr()), "ca_focus_map")
    _end(e0, "focus_map", 1 if out is None else 2, float(B * (2 * g * g + out_h * out_w) * 4))
    return out if out is not None else norm


def _dp(t):
    return None if t is None else t.data_ptr()


def make_heads_weights(named):
    """named: dict field -> fp32 CUDA tensor (kept alive by the caller)."""
    w = _lib.HeadsWeights()
    for n in _lib.HeadsWeights._names:
        t = named[n]
        _req(t, torch.float32, n)
        setattr(w, n, t.data_ptr())
    return w


def heads(weights, *, tokens, tokens_per_img, depth, conf, B, focal_feat=None, pool_partial=None, pool_splits=0,
          tmp_w=None, tmp_b=None, pooled_out=None, exif=None, camera_idx=None, fused_out=None, num_cameras=0,
          fault_ptr=None, sweep_images=0, call_of_row=None):
    """`fault_ptr`: address of a device-visible int32 (pinned host memory) that receives bit 0 when a camera index lies
    outside [0, num_cameras) — the range check of the embedding lookup, done on the device so the call never syncs.
    `sweep_images` > 0: an instruction sweep of B / sweep_images calls over `sweep_images` images (rows k * images + b,
    tmp_w [K, 64, 768], tmp_b [K, 64]; include/cogaim_b200.h ca_heads_inputs).  `call_of_row` (int32 [B]): row r uses
    projection call_of_row[r] of tmp_w [m, 64, 768] / tmp_b [m, 64] (the rows of several guide calls)."""
    import ctypes as C
    _req(call_of_row, torch.int32, "call_of_row")
    inp = _lib.HeadsInputs(_dp(tokens), tokens_per_img, _dp(focal_feat), _dp(pool_partial), pool_splits, _dp(tmp_w),
                           _dp(tmp_b), _dp(pooled_out), _dp(exif), _dp(camera_idx), int(num_cameras), fault_ptr,
                           int(sweep_images), _dp(call_of_row))
    e0 = _begin()
    check(_lib.load().ca_heads(C.byref(weights), C.byref(inp), ptr(depth), ptr(conf), ptr(fused_out), B, stream_ptr()),
          "ca_heads")
    _end(e0, "heads", 1)


def guide_tail(weights, *, base, mask, heat, argmax, ticket, tokens, depth, conf, B, N, pool_partial, tmp_w, tmp_b,
               exif=None, camera_idx=None, num_cameras=0, fault_ptr=None, pooled_out=None, alpha=0.7, temperature=0.05):
    """`guided_softmax` -> `weighted_pool` (pool_partial [B, splits, 768], rows 1..N of each image's tokens) -> `heads`
    of one guided call in ONE launch, bit for bit.  mask: [N] or [B, N]; ticket: int32 [B], zero before the first call
    (every call leaves it at zero)."""
    import ctypes as C
    _req(base, torch.float32, "base")
    _req(mask, torch.float32, "mask")
    _req(heat, torch.float32, "heat")
    _req(ticket, torch.int32, "ticket")
    _req(pool_partial, torch.float32, "pool_partial")
    _req(tokens, torch.float32, "tokens")
    if tuple(tokens.shape) != (B, N + 1, 768) or not tokens.is_contiguous() or tokens.data_ptr() % 16:
        raise ValueError(f"guide_tail: tokens must be a contiguous, 16-byte aligned [B, N + 1, 768] = [{B}, {N + 1}, 768] "
                         f"tensor, got {tuple(tokens.shape)}")
    if not pool_partial.is_contiguous() or pool_partial.data_ptr() % 16:
        raise ValueError("guide_tail: pool_partial must be contiguous and 16-byte aligned")
    if argmax is not None:
        _req(argmax, torch.int32, "argmax")
    if mask.dim() == 2 and mask.shape[0] != B:
        raise ValueError(f"per-image mask has {mask.shape[0]} rows for a batch of {B}")
    if ticket.numel() < B or pool_partial.dim() != 3 or pool_partial.shape[0] < B or pool_partial.shape[2] != 768:
        raise ValueError("guide_tail: ticket needs B entries and pool_partial must be [B, splits, 768]")
    stride = mask.stride(0) if mask.dim() == 2 else 0
    inp = _lib.HeadsInputs(_dp(tokens), N + 1, None, _dp(pool_partial), pool_partial.shape[1], _dp(tmp_w), _dp(tmp_b),
                           _dp(pooled_out), _dp(exif), _dp(camera_idx), int(num_cameras), fault_ptr, 0)
    e0 = _begin()
    check(_lib.load().ca_guide_tail(C.byref(weights), C.byref(inp), ptr(base), ptr(mask), stride, ptr(heat), ptr(argmax),
                                    ptr(ticket), ptr(depth), ptr(conf), B, N, alpha, temperature, stream_ptr()),
          "ca_guide_tail")
    _end(e0, "tail", 1, float(B * N * 768 * 4))


def token_project(src, src_batch_stride, row_offset, tmp_w, P, B, N):
    """P [B, N, 64] = rows row_offset .. row_offset + N - 1 of each image of `src` (fp32, 768 wide, images
    `src_batch_stride` floats apart) times tmp_w [64, 768] transposed: the per-call projection of every patch token."""
    _req(src, torch.float32, "src")
    _req(tmp_w, torch.float32, "tmp_w")
    _req(P, torch.float32, "P")
    if tuple(tmp_w.shape) != (64, 768) or not tmp_w.is_contiguous():
        raise ValueError("token_project: tmp_w must be a contiguous [64, 768] tensor")
    if P.numel() < B * N * 64 or not P.is_contiguous():
        raise ValueError("token_project: P must be a contiguous tensor of at least B * N * 64 floats")
    if src.numel() < (B - 1) * src_batch_stride + (row_offset + N) * 768:
        raise ValueError("token_project: src is smaller than B images of row_offset + N rows")
    e0 = _begin()
    check(_lib.load().ca_token_project(ptr(src), src_batch_stride, row_offset, ptr(tmp_w), ptr(P), B, N, stream_ptr()),
          "ca_token_project")
    _end(e0, "token_project", 1, float(B * N * 768 * 4))


def depth_field_cells(weights, *, base, P, cst, depth, conf, tokens, tmp_b, B, g, exif=None, camera_idx=None,
                      num_cameras=0, fault_ptr=None, alpha=0.7, temperature=0.05):
    """depth, conf [B, g * g]: for every cell c, the guided call whose mask is `tables.focus_mask` at c, from the
    projected tokens P [B, g * g, 64] (`token_project`), the focal attention `base` [B, g * g], the CLS rows of `tokens`
    [B, g * g + 1, 768], the projection bias tmp_b [64] and the EXIF inputs as `heads` takes them.  cst: [B, 192]
    scratch.  Two launches (the per-image fusion constant, then the cells)."""
    import ctypes as C
    N = g * g
    for t, name in ((base, "base"), (P, "P"), (cst, "cst"), (depth, "depth"), (conf, "conf"), (tokens, "tokens"),
                    (tmp_b, "tmp_b")):
        _req(t, torch.float32, name)
        if not t.is_contiguous():
            raise ValueError(f"depth_field_cells: {name} must be contiguous")
    if tuple(tokens.shape) != (B, N + 1, 768):
        raise ValueError(f"depth_field_cells: tokens must be [B, N + 1, 768] = [{B}, {N + 1}, 768], got "
                         f"{tuple(tokens.shape)}")
    if (base.numel() < B * N or P.numel() < B * N * 64 or cst.numel() < B * 192 or depth.numel() < B * N
            or conf.numel() < B * N or tmp_b.numel() != 64):
        raise ValueError("depth_field_cells: base / depth / conf need B * g * g floats, P B * g * g * 64, cst B * 192 "
                         "and tmp_b 64")
    inp = _lib.HeadsInputs(_dp(tokens), N + 1, None, None, 0, None, _dp(tmp_b), None, _dp(exif), _dp(camera_idx),
                           int(num_cameras), fault_ptr, 0)
    e0 = _begin()
    check(_lib.load().ca_depth_field_cells(C.byref(weights), C.byref(inp), ptr(base), ptr(P), ptr(cst), ptr(depth),
                                           ptr(conf), B, g, alpha, temperature, stream_ptr()), "ca_depth_field_cells")
    _end(e0, "field_cells", 2, float(B * N * 64 * 4))


def make_curiosity_weights(named):
    """named: dict field -> fp32 CUDA tensor or None for the four local_curiosity fields (kept alive by the caller)."""
    w = _lib.CuriosityWeights()
    for n in _lib.CuriosityWeights._names:
        t = named.get(n)
        _req(t, torch.float32, n)
        setattr(w, n, None if t is None else t.data_ptr())
    return w


def make_curiosity_mod_weights(amp, mods):
    """amp: (w0, b0, w1, b1) of curiosity_amplifier; mods: per iteration (w0, b0, w1, b1) of curiosity_modulator."""
    w = _lib.CuriosityModWeights()
    for n, t in zip(("amp_w0", "amp_b0", "amp_w1", "amp_b1"), amp):
        _req(t, torch.float32, n)
        setattr(w, n, t.data_ptr())
    if len(mods) > 8:
        raise ValueError("at most 8 focal iterations")
    for i, four in enumerate(mods):
        for n, t in zip(("mod_w0", "mod_b0", "mod_w1", "mod_b1"), four):
            _req(t, torch.float32, n)
            getattr(w, n)[i] = t.data_ptr()
    return w


def curiosity(weights, *, tokens, tokens_per_img, eps, noise, reward_raw, reward, history, history_pointer, B):
    """CuriosityModule.forward on the CLS rows of `tokens` + the exploration ring-buffer update (csrc/curiosity.cu)."""
    import ctypes as C
    for t, n in ((tokens, "tokens"), (eps, "eps"), (noise, "noise"), (reward_raw, "reward_raw"), (reward, "reward"),
                 (history, "history")):
        _req(t, torch.float32, n)
    _req(history_pointer, torch.int64, "history_pointer")
    if eps.numel() < B * 192 or (noise is not None and noise.numel() < B * 768):
        raise ValueError("eps / noise draws are smaller than the batch")
    e0 = _begin()
    check(_lib.load().ca_curiosity(C.byref(weights), ptr(tokens), tokens_per_img, ptr(eps), ptr(noise), ptr(reward_raw),
                                   ptr(reward), ptr(history), 0 if history is None else history.numel(),
                                   ptr(history_pointer), B, stream_ptr()), "ca_curiosity")
    _end(e0, "curiosity", 1 if history is None else 2)


def curiosity_modulation(weights, reward, lo, hi, cur_weight, B, n_iters, mod_hidden):
    """cur_weight [n_iters, B]: head-mean modulator output per iteration (csrc/curiosity.cu); lo > hi = no clamp."""
    import ctypes as C
    _req(reward, torch.float32, "reward")
    _req(cur_weight, torch.float32, "cur_weight")
    e0 = _begin()
    check(_lib.load().ca_curiosity_modulation(C.byref(weights), ptr(reward), float(lo), float(hi), ptr(cur_weight), B,
                                              n_iters, mod_hidden, stream_ptr()), "ca_curiosity_modulation")
    _end(e0, "curiosity", 1)


def focal_value(*, tok_partial, pe_partial, splits, wv, bv, proj_w0, proj_b0, proj_w1, proj_b1, feat_out, it, n_iters,
                B):
    import ctypes as C
    a = _lib.FocalValueArgs(_dp(tok_partial), _dp(pe_partial), splits, _dp(wv), _dp(bv), _dp(proj_w0), _dp(proj_b0),
                            _dp(proj_w1), _dp(proj_b1), _dp(feat_out), it, n_iters)
    e0 = _begin()
    check(_lib.load().ca_focal_value(C.byref(a), B, stream_ptr()), "ca_focal_value")
    _end(e0, "heads", 1)


def focal_fusion(feats, n_iters, w0, b0, w1, b1, out, B):
    e0 = _begin()
    check(_lib.load().ca_focal_fusion(ptr(feats), n_iters, ptr(w0), ptr(b0), ptr(w1), ptr(b1), ptr(out), B,
                                      stream_ptr()), "ca_focal_fusion")
    _end(e0, "heads", 1)
