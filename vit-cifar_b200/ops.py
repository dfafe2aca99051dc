"""Tensor-level wrappers over the C ABI: torch tensors in, raw device pointers + current stream out.

PyTorch is plumbing here (device memory, streams); every FLOP on this path runs in libvitb200.so.
All functions launch on ``torch.cuda.current_stream()`` and never synchronise, so a sequence of them can be
captured into a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import BF16, F32, GEMM_DY_F32, GEMM_GELU, GEMM_OUT_F32, check

_DT = {torch.float32: F32, torch.bfloat16: BF16}


def dt_of(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"activation dtype must be float32 or bfloat16, got {t.dtype}") from None


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.VitbError("libvitb200 kernels take CUDA tensors only (no CPU fallback)")
    return t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _contig(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_contiguous():
            raise ValueError("libvitb200 ops need contiguous tensors")


def require_device() -> None:
    """Fail loudly when there is no usable B200 / library (the product path has no fallback)."""
    lib = _lib.load()
    if not torch.cuda.is_available():
        raise _lib.VitbError("no CUDA device: the vit-cifar_b200 hot path runs on sm_100a only")
    if not lib.vitb_device_supported():
        raise _lib.VitbError("current CUDA device is not compute capability 10.x (B200)")


def launch_count() -> int:
    """Kernels launched (or captured) by libvitb200 so far in this process."""
    return int(_lib.load().vitb_launch_count())


# ---------------------------------------------------------------------------------------------
# workspace: one growing scratch buffer per device; old buffers stay alive (graph safety)
# ---------------------------------------------------------------------------------------------
_ws: dict = {}
_ws_keep: list = []


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    cur = _ws.get(key)
    if cur is None or cur.numel() < nbytes:
        size = max(int(nbytes), 1 << 20)
        if cur is not None:
            _ws_keep.append(cur)
            size = max(size, 2 * cur.numel())
        cur = torch.empty(size, dtype=torch.uint8, device=device)
        _ws[key] = cur
    return cur


# ---------------------------------------------------------------------------------------------
# ops
# ---------------------------------------------------------------------------------------------
def cast_f32_to_bf16(src: torch.Tensor, dst: torch.Tensor) -> None:
    assert src.dtype == torch.float32 and dst.dtype == torch.bfloat16 and src.numel() == dst.numel()
    _contig(src, dst)
    check(_lib.load().vitb_cast_f32_to_bf16(_ptr(src), _ptr(dst), src.numel(), _stream()), "cast_f32_to_bf16")


def patch_embed_fwd(img, w, w_act, bias, cls, pos, out, words, P: int, has_cls: bool) -> None:
    """w_act / words: bf16 shadow of emb.weight and the (B*P*P, K) patch-matrix buffer (tensor-core path) or None."""
    B, _, S, _ = img.shape
    H = w.shape[0]
    assert img.dtype == torch.float32 and w.dtype == torch.float32
    _contig(img, w, bias, cls, pos, out, words)
    lib = _lib.load()
    dt = dt_of(out)
    nb = lib.vitb_patch_embed_fwd_ws_bytes(B, S, P, H, dt)
    ws = workspace(nb, img.device) if nb else None
    check(lib.vitb_patch_embed_fwd(_ptr(img), _ptr(w), _ptr(w_act), _ptr(bias), _ptr(cls), _ptr(pos), _ptr(out), _ptr(words),
                                   _ptr(ws), ws.numel() if ws is not None else 0, B, S, P, H, int(has_cls), dt, _stream()), "patch_embed_fwd")


def patch_embed_bwd(img, words, dout, dw, dbias, dcls, dpos, P: int, has_cls: bool) -> None:
    B, _, S, _ = img.shape
    H = dw.shape[0]
    lib = _lib.load()
    _contig(img, dout, dw, dbias, dcls, dpos, words)
    nb = lib.vitb_patch_embed_bwd_ws_bytes(B, S, P, H, int(has_cls))
    ws = workspace(nb, img.device)
    check(lib.vitb_patch_embed_bwd(_ptr(img), _ptr(words), _ptr(dout), _ptr(dw), _ptr(dbias), _ptr(dcls), _ptr(dpos), _ptr(ws), ws.numel(),
                                   B, S, P, H, int(has_cls), dt_of(dout), _stream()), "patch_embed_bwd")


def layernorm_fwd(x, x_row_stride: int, gamma, beta, y, mean, rstd, rows: int, H: int, eps: float = 1e-5) -> None:
    check(_lib.load().vitb_layernorm_fwd(_ptr(x), x_row_stride, _ptr(gamma), _ptr(beta), _ptr(y), _ptr(mean), _ptr(rstd),
                                         rows, H, eps, dt_of(y), _stream()), "layernorm_fwd")


def layernorm_bwd(dy, x, x_row_stride: int, gamma, mean, rstd, dres, dx, dx_row_stride: int, dgamma, dbeta, dx_colsum,
                  rows: int, H: int) -> None:
    lib = _lib.load()
    nb = lib.vitb_layernorm_bwd_ws_bytes(rows, H)
    ws = workspace(nb, dy.device)
    check(lib.vitb_layernorm_bwd(_ptr(dy), _ptr(x), x_row_stride, _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dres), _ptr(dx),
                                 dx_row_stride, _ptr(dgamma), _ptr(dbeta), _ptr(dx_colsum), _ptr(ws), ws.numel(), rows, H,
                                 dt_of(dy), _stream()), "layernorm_bwd")


def drop_desc(p: float, seed: int, site: int, step: int = 0, step_dev=None):
    """A vitb_dropout_t for the fused dropout sites (None when p == 0).  Keep the returned object alive across the call."""
    if not p:
        return None
    return _lib.DropoutDesc(float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, int(site), int(step) & 0xFFFFFFFF, _ptr(step_dev))


def _dref(d):
    return C.byref(d) if d is not None else None


def layernorm_bwd_fused(dy, x, x_row_stride: int, gamma, mean, rstd, dres, dx, dx_row_stride: int, dgamma, dbeta, z, dx2, dx2_colsum,
                        rows: int, H: int, drop=None) -> None:
    """layernorm_bwd plus a second output dx2 = dropout(dx) [* gelu'(z)] and its column sums (vitb_layernorm_bwd_fused)."""
    lib = _lib.load()
    nb = lib.vitb_layernorm_bwd_ws_bytes(rows, H)
    ws = workspace(nb, dy.device)
    check(lib.vitb_layernorm_bwd_fused(_ptr(dy), _ptr(x), x_row_stride, _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dres), _ptr(dx),
                                       dx_row_stride, _ptr(dgamma), _ptr(dbeta), _ptr(z), _ptr(dx2), _ptr(dx2_colsum), _dref(drop),
                                       _ptr(ws), ws.numel(), rows, H, dt_of(dy), _stream()), "layernorm_bwd_fused")


def gemm_fwd(a, w_act, bias, residual, out, preact, M: int, N: int, K: int, gelu: bool = False, out_f32: bool = False, drop=None) -> None:
    """out = dropout(act(a w^T + bias)) + residual; `drop`: a drop_desc (mask in the GEMM epilogue) or None."""
    flags = (GEMM_GELU if gelu else 0) | (GEMM_OUT_F32 if out_f32 else 0)
    check(_lib.load().vitb_gemm_bias_act_fwd_drop(_ptr(a), _ptr(w_act), _ptr(bias), _ptr(residual), _ptr(out), _ptr(preact),
                                                  M, N, K, flags, dt_of(a), _dref(drop), _stream()), "gemm_bias_act_fwd")


def gemm_dgrad(dy, w_act, z, dx, M: int, N: int, K: int, dy_f32: bool = False, drop=None) -> None:
    """dx = dropout(dy w * gelu'(z)); `drop`: a drop_desc or None."""
    flags = GEMM_DY_F32 if dy_f32 else 0
    check(_lib.load().vitb_gemm_dgrad_drop(_ptr(dy), _ptr(w_act), _ptr(z), _ptr(dx), M, N, K, flags, dt_of(dx), _dref(drop), _stream()),
          "gemm_dgrad")


def gemm_wgrad(dy, x, dw, dbias, M: int, N: int, K: int, dy_f32: bool = False) -> None:
    lib = _lib.load()
    dt = dt_of(x)
    nb = lib.vitb_gemm_wgrad_ws_bytes(M, N, K, dt)
    ws = workspace(nb, x.device)
    flags = GEMM_DY_F32 if dy_f32 else 0
    check(lib.vitb_gemm_wgrad_dbias(_ptr(dy), _ptr(x), _ptr(dw), _ptr(dbias), _ptr(ws), ws.numel(), M, N, K, flags, dt, _stream()),
          "gemm_wgrad_dbias")


def bwd_fused_ws_bytes(M: int, N: int, K: int, dt: int = BF16) -> int:
    """Workspace of gemm_bwd_fused, 0 when this shape / dtype has no fused kernel (use gemm_dgrad + gemm_wgrad)."""
    return int(_lib.load().vitb_gemm_bwd_fused_ws_bytes(M, N, K, dt))


def gemm_bwd_fused(dy, x, w_act, z, dx, dw, dx_colsum, M: int, N: int, K: int) -> None:
    """Backward of y = x W^T in one pass over dy: dx = dy W (* gelu'(z)), dw = dy^T x, dx_colsum = column sums of dx (optional)."""
    lib = _lib.load()
    dt = dt_of(x)
    nb = lib.vitb_gemm_bwd_fused_ws_bytes(M, N, K, dt)
    ws = workspace(max(int(nb), 256), x.device)
    check(lib.vitb_gemm_bwd_fused(_ptr(dy), _ptr(x), _ptr(w_act), _ptr(z), _ptr(dx), _ptr(dw), _ptr(dx_colsum), _ptr(ws), ws.numel(), M, N, K, dt,
                                  _stream()), "gemm_bwd_fused")


def attn_fwd(qkv, o, lse, attn_map, B: int, T: int, heads: int, d: int, scale: float) -> None:
    check(_lib.load().vitb_attn_fwd(_ptr(qkv), _ptr(o), _ptr(lse), _ptr(attn_map), B, T, heads, d, scale, dt_of(qkv), _stream()), "attn_fwd")


def attn_bwd(qkv, o, d_o, lse, dqkv, B: int, T: int, heads: int, d: int, scale: float) -> None:
    check(_lib.load().vitb_attn_bwd(_ptr(qkv), _ptr(o), _ptr(d_o), _ptr(lse), _ptr(dqkv), B, T, heads, d, scale, dt_of(qkv), _stream()),
          "attn_bwd")


def gelu_bwd_colsum(dy, z, dz, colsum, rows: int, cols: int, drop=None) -> None:
    """dz = dropout(dy) * gelu'(z), colsum = column sums of dz; `drop`: a drop_desc or None."""
    lib = _lib.load()
    ws = workspace(lib.vitb_colsum_ws_bytes(rows, cols), dy.device)
    check(lib.vitb_gelu_bwd_colsum_drop(_ptr(dy), _ptr(z), _ptr(dz), _ptr(colsum), _ptr(ws), ws.numel(), rows, cols, dt_of(dy), _dref(drop),
                                        _stream()), "gelu_bwd_colsum")


def colsum(x, out, rows: int, cols: int) -> None:
    lib = _lib.load()
    ws = workspace(lib.vitb_colsum_ws_bytes(rows, cols), x.device)
    check(lib.vitb_colsum(_ptr(x), _ptr(out), _ptr(ws), ws.numel(), rows, cols, dt_of(x), _stream()), "colsum")


def pool_fwd(x, y, B: int, T: int, H: int, mode: int) -> None:
    check(_lib.load().vitb_pool_fwd(_ptr(x), _ptr(y), B, T, H, mode, dt_of(x), _stream()), "pool_fwd")


def pool_bwd(dy, dx, B: int, T: int, H: int, mode: int) -> None:
    check(_lib.load().vitb_pool_bwd(_ptr(dy), _ptr(dx), B, T, H, mode, dt_of(dx), _stream()), "pool_bwd")


_F3 = C.c_float * 3


def augment(img_u8, dx, dy, flip, mean, std, out, pad: int) -> None:
    """RandomCrop(pad) + RandomHorizontalFlip + ToTensor + Normalize (utils.py:337-355) of a uint8 (B,S,S,3) device batch into
    fp32 (B,3,S,S); dx / dy (int32, device) and flip (uint8, device) are the per-image random draws (None = identity)."""
    B, S = img_u8.shape[0], img_u8.shape[1]
    assert img_u8.dtype == torch.uint8 and img_u8.shape == (B, S, S, 3) and out.dtype == torch.float32 and out.shape == (B, 3, S, S)
    assert (dx is None or dx.dtype == torch.int32) and (dy is None or dy.dtype == torch.int32) and (flip is None or flip.dtype == torch.uint8)
    _contig(img_u8, out, dx, dy, flip)
    m, s_ = _F3(*[float(v) for v in mean]), _F3(*[float(v) for v in std])
    check(_lib.load().vitb_augment_crop_flip_normalize(_ptr(img_u8), _ptr(dx), _ptr(dy), _ptr(flip), C.cast(m, C.c_void_p), C.cast(s_, C.c_void_p),
                                                       _ptr(out), B, S, int(pad), _stream()), "augment_crop_flip_normalize")


def augment_autoaugment(img_u8, dx, dy, flip, code, op_ids, mags, mean, std, out, pad: int) -> None:
    """`augment` with an AutoAugment sub-policy (the reference's autoaugment.py) applied between the flip and ToTensor.  code (int32,
    device): per image, bits 0-7 sub-policy index, 8/9 apply op 1/2, 10/11 negative sign of op 1/2; op_ids / mags: the table, two
    (op code, magnitude) entries per sub-policy (autoaugment.kernel_table)."""
    B, S = img_u8.shape[0], img_u8.shape[1]
    assert img_u8.dtype == torch.uint8 and img_u8.shape == (B, S, S, 3) and out.dtype == torch.float32 and out.shape == (B, 3, S, S)
    assert (dx is None or dx.dtype == torch.int32) and (dy is None or dy.dtype == torch.int32) and (flip is None or flip.dtype == torch.uint8)
    assert code.dtype == torch.int32 and code.shape == (B,) and len(op_ids) == len(mags) and len(op_ids) % 2 == 0
    _contig(img_u8, out, dx, dy, flip, code)
    m, s_ = _F3(*[float(v) for v in mean]), _F3(*[float(v) for v in std])
    n = len(op_ids)
    ids, mg = (C.c_int32 * n)(*[int(v) for v in op_ids]), (C.c_double * n)(*[float(v) for v in mags])
    check(_lib.load().vitb_augment_autoaugment(_ptr(img_u8), _ptr(dx), _ptr(dy), _ptr(flip), _ptr(code), C.cast(ids, C.c_void_p), C.cast(mg, C.c_void_p),
                                               n // 2, C.cast(m, C.c_void_p), C.cast(s_, C.c_void_p), _ptr(out), B, S, int(pad), _stream()),
          "augment_autoaugment")


def _check_gather(data_u8, labels_src, idx, out, labels_dst, dx, dy, flip, policy: bool) -> tuple:
    """Host-side checks of the gather forms: dtype, layout and device of every tensor; returns (N, B, S)."""
    if data_u8.dtype != torch.uint8 or data_u8.dim() != 4 or data_u8.shape[3] != 3 or data_u8.shape[1] != data_u8.shape[2]:
        raise ValueError(f"data_u8 must be uint8 (N, S, S, 3) HWC, got {data_u8.dtype} {tuple(data_u8.shape)}")
    N, S = int(data_u8.shape[0]), int(data_u8.shape[1])
    if N < 1:
        raise ValueError("empty dataset: data_u8 has no images")
    if policy and S > 64:
        raise ValueError(f"the AutoAugment kernel takes images of at most 64 x 64 pixels, got S={S}")
    if idx.dtype != torch.int32 or idx.dim() != 1 or idx.numel() < 1:
        raise ValueError(f"idx must be a non-empty int32 vector, got {idx.dtype} {tuple(idx.shape)}")
    B = int(idx.numel())
    if labels_src.dtype != torch.int64 or tuple(labels_src.shape) != (N,):
        raise ValueError(f"labels_src must be int64 ({N},), got {labels_src.dtype} {tuple(labels_src.shape)}")
    if out.dtype != torch.float32 or tuple(out.shape) != (B, 3, S, S):
        raise ValueError(f"out must be float32 ({B}, 3, {S}, {S}), got {out.dtype} {tuple(out.shape)}")
    if labels_dst.dtype != torch.int64 or tuple(labels_dst.shape) != (B,):
        raise ValueError(f"labels_dst must be int64 ({B},), got {labels_dst.dtype} {tuple(labels_dst.shape)}")
    for name, t, dt in (("dx", dx, torch.int32), ("dy", dy, torch.int32), ("flip", flip, torch.uint8)):
        if t is not None and (t.dtype != dt or tuple(t.shape) != (B,)):
            raise ValueError(f"{name} must be {dt} ({B},), got {t.dtype} {tuple(t.shape)}")
    ts = [t for t in (data_u8, labels_src, idx, out, labels_dst, dx, dy, flip) if t is not None]
    if any(t.device != data_u8.device for t in ts) or not data_u8.is_cuda:
        raise ValueError("every tensor of a gather must be on the same CUDA device: " + ", ".join(str(t.device) for t in ts))
    _contig(*ts)
    return N, B, S


def augment_gather(data_u8, labels_src, idx, dx, dy, flip, mean, std, out, labels_dst, pad: int) -> None:
    """`augment` of the batch data_u8[idx] of a device-resident (N, S, S, 3) dataset, gathered inside the kernel, with
    labels_dst = labels_src[idx] in the same launch.  A row outside [0, N) gives a NaN image and label -1."""
    N, B, S = _check_gather(data_u8, labels_src, idx, out, labels_dst, dx, dy, flip, False)
    m, s_ = _F3(*[float(v) for v in mean]), _F3(*[float(v) for v in std])
    check(_lib.load().vitb_augment_crop_flip_normalize_gather(_ptr(data_u8), _ptr(labels_src), N, _ptr(idx), _ptr(dx), _ptr(dy), _ptr(flip),
                                                              C.cast(m, C.c_void_p), C.cast(s_, C.c_void_p), _ptr(out), _ptr(labels_dst), B, S,
                                                              int(pad), _stream()), "augment_crop_flip_normalize_gather")


def augment_autoaugment_gather(data_u8, labels_src, idx, dx, dy, flip, code, op_ids, mags, mean, std, out, labels_dst, pad: int) -> None:
    """`augment_autoaugment` of the batch data_u8[idx], gathered inside the kernel, as `augment_gather`."""
    N, B, S = _check_gather(data_u8, labels_src, idx, out, labels_dst, dx, dy, flip, True)
    if code.dtype != torch.int32 or tuple(code.shape) != (B,) or code.device != data_u8.device:
        raise ValueError(f"code must be int32 ({B},) on {data_u8.device}, got {code.dtype} {tuple(code.shape)} on {code.device}")
    if len(op_ids) != len(mags) or len(op_ids) % 2 != 0:
        raise ValueError("op_ids and mags: two entries per sub-policy")
    _contig(code)
    m, s_ = _F3(*[float(v) for v in mean]), _F3(*[float(v) for v in std])
    n = len(op_ids)
    ids, mg = (C.c_int32 * n)(*[int(v) for v in op_ids]), (C.c_double * n)(*[float(v) for v in mags])
    check(_lib.load().vitb_augment_autoaugment_gather(_ptr(data_u8), _ptr(labels_src), N, _ptr(idx), _ptr(dx), _ptr(dy), _ptr(flip), _ptr(code),
                                                      C.cast(ids, C.c_void_p), C.cast(mg, C.c_void_p), n // 2, C.cast(m, C.c_void_p),
                                                      C.cast(s_, C.c_void_p), _ptr(out), _ptr(labels_dst), B, S, int(pad), _stream()),
          "augment_autoaugment_gather")


CROP_PASTE_MAX_S = 64  # vitb_random_crop_paste stages an image in 3 * S * S floats of shared memory


def random_crop_paste(img, params, alpha) -> None:
    """da.RandomCropPaste in place on a normalised fp32 (B, 3, S, S) device batch, for given draws: params int32 (B, 8) =
    [fx1, fy1, fw, fh, x1, y1, flip_front, flip_img] per image, alpha float64 (B,) = the blend weight a (vitb_random_crop_paste)."""
    if img.dtype != torch.float32 or img.dim() != 4 or img.shape[1] != 3 or img.shape[2] != img.shape[3] or img.shape[0] < 1:
        raise ValueError(f"img must be a non-empty float32 (B, 3, S, S) batch, got {img.dtype} {tuple(img.shape)}")
    B, S = int(img.shape[0]), int(img.shape[2])
    if S > CROP_PASTE_MAX_S:
        raise ValueError(f"the crop-paste kernel takes images of at most {CROP_PASTE_MAX_S} x {CROP_PASTE_MAX_S} pixels, got S={S}")
    if params.dtype != torch.int32 or tuple(params.shape) != (B, 8):
        raise ValueError(f"params must be int32 ({B}, 8), got {params.dtype} {tuple(params.shape)}")
    if alpha.dtype != torch.float64 or tuple(alpha.shape) != (B,):
        raise ValueError(f"alpha must be float64 ({B},), got {alpha.dtype} {tuple(alpha.shape)}")
    if not img.is_cuda or params.device != img.device or alpha.device != img.device:
        raise ValueError(f"img, params and alpha must be on the same CUDA device: {img.device}, {params.device}, {alpha.device}")
    _contig(img, params, alpha)
    check(_lib.load().vitb_random_crop_paste(_ptr(img), _ptr(params), _ptr(alpha), B, S, _stream()), "random_crop_paste")


def batch_mix(img, perm, out, mode: int, lam: float = 1.0, box=(0, 0, 0, 0)) -> None:
    """CutMix (mode 0: paste rows box[0]:box[1], columns box[2]:box[3] of img[perm[b]] into img[b], da.py:68) or MixUp (mode 1:
    lam * img + (1 - lam) * img[perm], da.py:90) of an fp32 (B, C, S, S) batch into `out`."""
    B, Cn, S, S2 = img.shape
    assert S == S2 and img.dtype == torch.float32 and out.dtype == torch.float32 and out.shape == img.shape and perm.dtype == torch.int32
    _contig(img, perm, out)
    x1, x2, y1, y2 = (int(v) for v in box)
    check(_lib.load().vitb_batch_mix(_ptr(img), _ptr(perm), _ptr(out), B, Cn, S, int(mode), float(lam), x1, x2, y1, y2, _stream()), "batch_mix")


def set_l2_persisting_window(t: Optional[torch.Tensor], carve_out_bytes: int = 0) -> None:
    """Keep reads of tensor `t` (the bf16 weight shadow) in a persisting carve-out of L2 for every kernel launched from now on
    (recorded in captured graph nodes); None clears it."""
    if t is None:
        check(_lib.load().vitb_set_l2_persisting_window(None, 0, 0), "set_l2_persisting_window")
        return
    nbytes = t.numel() * t.element_size()
    check(_lib.load().vitb_set_l2_persisting_window(_ptr(t), nbytes, int(carve_out_bytes) or nbytes), "set_l2_persisting_window")


def dropout(x, residual, out, p: float, seed: int, site: int, step: int = 0, step_dev=None) -> None:
    """out = x * keep / (1 - p) (+ residual), nn.Dropout semantics (layers.py:35, 38, 102).  keep is a pure function of
    (seed, site, step, element index): the backward pass is the same call on the gradient.  `step_dev`: 1-element int32 device
    tensor that overrides `step` (graph replays)."""
    assert x.dtype == out.dtype and x.numel() == out.numel() and (residual is None or residual.dtype == x.dtype)
    _contig(x, out, residual)
    check(_lib.load().vitb_dropout(_ptr(x), _ptr(residual), _ptr(out), x.numel(), float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, int(site),
                                   int(step) & 0xFFFFFFFF, _ptr(step_dev), dt_of(x), _stream()), "dropout")


_ls_ws = {}


def _ls_workspace(device) -> torch.Tensor:
    """Zero-initialised partial-sum / counter buffer of the multi-block loss kernel, one per (device, stream): the kernel leaves the
    counter at zero, so consecutive calls on a stream share it; calls on different streams must not."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _ls_ws.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().vitb_ls_ce_ws_bytes()) // 4, dtype=torch.float32, device=device)
        _ls_ws[key] = ws
    return ws


def ls_ce(logits, labels, loss, dlogits, smoothing: float, grad_scale: float = 1.0, labels_b=None, lam: float = 1.0, lam_dev=None,
          n_valid_dev=None, ws=None) -> None:
    """LS-CE forward + dlogits.  With `labels_b`: the two-target CutMix / MixUp loss lam*L(a) + (1-lam)*L(b) (network.py:149-167);
    `lam_dev` (1-element fp32 device tensor) overrides `lam` so that a captured graph reads a fresh value every step.
    `n_valid_dev` (1-element int32 device tensor): only rows [0, n_valid) are images (partial last batch of an epoch).
    `ws`: zeroed fp32 workspace of vitb_ls_ce_ws_bytes() for the multi-block kernel (default: one per device and stream)."""
    B, Cn = logits.shape
    assert logits.dtype == torch.float32 and labels.dtype == torch.int64
    assert labels_b is None or (labels_b.dtype == torch.int64 and labels_b.shape == labels.shape)
    assert n_valid_dev is None or n_valid_dev.dtype == torch.int32
    _contig(logits, labels, dlogits, labels_b)
    _ptr(logits)  # (CPU tensors: raise before touching the device for a workspace)
    if ws is None:
        ws = _ls_workspace(logits.device)
    check(_lib.load().vitb_ls_ce_blocks_fwd_bwd(_ptr(logits), _ptr(labels), _ptr(labels_b), float(lam), _ptr(lam_dev), _ptr(n_valid_dev), _ptr(loss),
                                                _ptr(dlogits), B, Cn, smoothing, grad_scale, _ptr(ws), ws.numel() * 4, _stream()), "ls_ce_blocks_fwd_bwd")


def ls_ce_single_block(logits, labels, loss, dlogits, smoothing: float, grad_scale: float = 1.0, labels_b=None, lam: float = 1.0,
                       lam_dev=None, n_valid_dev=None) -> None:
    """The workspace-free single-block form of ls_ce (vitb_ls_ce_fwd_bwd / _mix_ / _batch_)."""
    B, Cn = logits.shape
    assert logits.dtype == torch.float32 and labels.dtype == torch.int64
    _contig(logits, labels, dlogits)
    if n_valid_dev is not None:
        assert n_valid_dev.dtype == torch.int32 and (labels_b is None or labels_b.dtype == torch.int64)
        _contig(labels_b)
        check(_lib.load().vitb_ls_ce_batch_fwd_bwd(_ptr(logits), _ptr(labels), _ptr(labels_b), float(lam), _ptr(lam_dev), _ptr(n_valid_dev), _ptr(loss),
                                                   _ptr(dlogits), B, Cn, smoothing, grad_scale, _stream()), "ls_ce_batch_fwd_bwd")
        return
    if labels_b is None:
        check(_lib.load().vitb_ls_ce_fwd_bwd(_ptr(logits), _ptr(labels), _ptr(loss), _ptr(dlogits), B, Cn, smoothing, grad_scale, _stream()),
              "ls_ce_fwd_bwd")
        return
    assert labels_b.dtype == torch.int64 and labels_b.shape == labels.shape
    _contig(labels_b)
    check(_lib.load().vitb_ls_ce_mix_fwd_bwd(_ptr(logits), _ptr(labels), _ptr(labels_b), float(lam), _ptr(lam_dev), _ptr(loss), _ptr(dlogits),
                                             B, Cn, smoothing, grad_scale, _stream()), "ls_ce_mix_fwd_bwd")


def eval_metrics_ws_bytes() -> int:
    return int(_lib.load().vitb_eval_metrics_ws_bytes())


def eval_metrics(logits, labels, totals, ws, smoothing: float, n_valid_dev=None) -> None:
    """Add the batch's [loss_sum, correct, count] to `totals` (3 float64, device): per row the LS-CE loss of `ls_ce` and
    argmax == label, over rows [0, n_valid) (`n_valid_dev`: 1-element int32 device tensor, None = all).  `ws`: a zeroed device
    buffer of eval_metrics_ws_bytes() bytes, reusable by the next call on the same stream."""
    B, Cn = logits.shape
    assert logits.dtype == torch.float32 and labels.dtype == torch.int64 and labels.shape == (B,)
    assert totals.dtype == torch.float64 and totals.numel() == 3 and (n_valid_dev is None or n_valid_dev.dtype == torch.int32)
    _contig(logits, labels, totals, ws)
    check(_lib.load().vitb_eval_metrics(_ptr(logits), _ptr(labels), _ptr(n_valid_dev), B, Cn, float(smoothing), _ptr(totals), _ptr(ws),
                                        ws.numel() * ws.element_size(), _stream()), "eval_metrics")


def defer_begin(arena: torch.Tensor) -> None:
    """From here to defer_flush() the second passes of wgrad / LayerNorm-backward / GELU-backward reductions are postponed: their
    partials go into `arena` (uint8 CUDA tensor that must stay alive and untouched until the flush has executed)."""
    check(_lib.load().vitb_defer_begin(_ptr(arena), arena.numel()), "defer_begin")


def defer_flush() -> None:
    check(_lib.load().vitb_defer_flush(_stream()), "defer_flush")


def defer_flush_partial() -> None:
    """Second passes recorded so far, on the current stream (ordered after the kernels that produced the partials); window stays open."""
    check(_lib.load().vitb_defer_flush_partial(_stream()), "defer_flush_partial")


def defer_used() -> int:
    return int(_lib.load().vitb_defer_used())


def wgrad_ws_bytes(M: int, N: int, K: int, dt: int = BF16) -> int:
    return int(_lib.load().vitb_gemm_wgrad_ws_bytes(M, N, K, dt))


_HyperArr = C.c_float * 16


def adam(p, g, m, v, shadow, hyper_host=None, hyper_dev=None) -> None:
    """hyper_host: sequence of 9 floats (optim.adam_hyper) or None; hyper_dev: 16-float CUDA tensor or None."""
    n = p.numel()
    hh = None
    if hyper_host is not None:
        hh = _HyperArr(*[float(x) for x in hyper_host], *([0.0] * (16 - len(hyper_host))))
    check(_lib.load().vitb_adam_multi(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(shadow), n,
                                      C.cast(hh, C.c_void_p) if hh is not None else None, _ptr(hyper_dev), _stream()), "adam_multi")


def sgd(p, g, buf, shadow, hyper_host=None, hyper_dev=None) -> None:
    """torch.optim.SGD with momentum (network.py:78-84) over flat buffers; hyper as optim.sgd_hyper (Adam's 16-float block layout)."""
    hh = None
    if hyper_host is not None:
        hh = _HyperArr(*[float(x) for x in hyper_host], *([0.0] * (16 - len(hyper_host))))
    check(_lib.load().vitb_sgd_multi(_ptr(p), _ptr(g), _ptr(buf), _ptr(shadow), p.numel(), C.cast(hh, C.c_void_p) if hh is not None else None,
                                     _ptr(hyper_dev), _stream()), "sgd_multi")


# -- data parallel over NVLink peer memory ---------------------------------------------------------
def ipc_export(t: torch.Tensor):
    """(64-byte handle, byte offset) of a CUDA tensor's memory for another process on this node (vitb_ipc_open)."""
    h = C.create_string_buffer(64)
    off = C.c_int64(0)
    check(_lib.load().vitb_ipc_export(_ptr(t), C.cast(h, C.c_void_p), C.cast(C.pointer(off), C.c_void_p)), "ipc_export")
    return bytes(h.raw), int(off.value)


def ipc_open(handle: bytes, offset: int) -> int:
    """Device address, valid in THIS process, of the memory another rank exported."""
    out = C.c_void_p(0)
    buf = C.create_string_buffer(handle, 64)
    check(_lib.load().vitb_ipc_open(C.cast(buf, C.c_void_p), int(offset), C.cast(C.pointer(out), C.c_void_p)), "ipc_open")
    return int(out.value)


class PeerPointers:
    """Host array of `world` device pointers (index = rank) in the form vitb_dp_reduce_adam takes."""

    def __init__(self, ptrs):
        self.ptrs = [int(p) for p in ptrs]
        self.arr = (C.c_void_p * len(self.ptrs))(*self.ptrs)

    def cptr(self):
        return C.cast(self.arr, C.c_void_p)


def dp_reduce_adam(g: PeerPointers, p: PeerPointers, shadow: Optional[PeerPointers], flags: PeerPointers, m, v, sync, n: int, rank: int, world: int,
                   hyper_host=None, hyper_dev=None, optimizer: int = 0) -> None:
    """Barrier, reduce-scatter of the peers' gradients, Adam on the owned slice, all-gather of the new parameters, barrier — one kernel."""
    hh = None
    if hyper_host is not None:
        hh = _HyperArr(*[float(x) for x in hyper_host], *([0.0] * (16 - len(hyper_host))))
    check(_lib.load().vitb_dp_reduce_adam(g.cptr(), p.cptr(), shadow.cptr() if shadow is not None else None, flags.cptr(), _ptr(m), _ptr(v), _ptr(sync),
                                          int(n), int(rank), int(world), int(optimizer), C.cast(hh, C.c_void_p) if hh is not None else None,
                                          _ptr(hyper_dev), _stream()),
          "dp_reduce_adam")


def train_loss_accumulate(loss, acc, B: int, n_valid_dev=None) -> None:
    """acc[0] += loss * n_valid in fp64 (`loss`: the 1-float device result of `ls_ce`; n_valid clamped to [1, B] as there)."""
    assert loss.dtype == torch.float32 and loss.numel() == 1 and acc.dtype == torch.float64 and acc.numel() >= 1
    assert n_valid_dev is None or n_valid_dev.dtype == torch.int32
    check(_lib.load().vitb_train_loss_accumulate(_ptr(loss), _ptr(n_valid_dev), int(B), _ptr(acc), _stream()), "train_loss_accumulate")
