"""``torch.library`` registration of the hot-path operators (SURVEY.md §8b: "registered via torch.library so
DDP/torch.compile see them").

``activezero_b200.ops`` exposes the operators as ``torch.autograd.Function``s -- all the reference's eager
trainer needs.  This module registers the same C-ABI calls as custom ops in the ``az_stereo`` namespace, with
fake (meta) kernels and autograd formulas, so that a traced / compiled program sees opaque, shape-checked
operators instead of Python:

    torch.ops.az_stereo.concat_volume(ref, tgt, num_disp, channels_last) -> vol      (psmnet.py:151-165)
    torch.ops.az_stereo.soft_argmin(cost) -> (disp, lse)                             (psmnet.py:200-217)
    torch.ops.az_stereo.reproj_loss(tgt, src, disp, mask, ps, sign) -> (loss, warped, gpre, stats)
                                                                                    (reprojection.py:81-127)
    torch.ops.az_stereo.gwc_volume(ref, tgt, num_disp, num_groups) -> vol            (SURVEY.md §8a row a3)
    torch.ops.az_stereo.upsample_soft_argmin(lowres, D, H, W) -> (disp, stats)       (psmnet.py:186-217)
    torch.ops.az_stereo.warp(img, disp) -> warped                                    (reprojection.py:13-35)
    torch.ops.az_stereo.scatter_warp(img, disp) -> (out, sign_flags)                 (warp_ops.py:55-95)
    torch.ops.az_stereo.temporal_ir_pattern(frames, ks, threshold) -> pattern        (tools/temporal_ir.py:93-114)
    torch.ops.az_stereo.local_contrast_norm(image, kernel_size, eps) -> (normed, std) (reprojection.py:175-200)

The first six are differentiable (each backward is itself a registered op, so a compiled backward graph stays
opaque too); the last three are the non-differentiable operators of SURVEY.md §8b.  Importing this module also
registers the differentiable first aggregation convolution on the implicit volume (``_volume_conv_library``):

    torch.ops.az_stereo.volume_conv(ref, tgt, weight, num_disp) -> out               (psmnet.py:151-168)

The convenience wrappers below return what the reference-named functions return.  Nothing here computes on the
host: every implementation enqueues the CUDA kernels of ``libaz_stereo.so`` (no CPU fallback).
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import Tensor

from . import _lib, _volume_conv_library
from .ops import (DTYPE16, _cuda_f32, _mask_u8, _ptr, _stream, check_feature_pair, check_reproj_inputs, linspace_table,
                  soft_argmin_backward_into, soft_argmin_forward_into, upsample_soft_argmin_backward_into,
                  upsample_soft_argmin_forward_into)
from .ops import concat_volume_backward as concat_volume_backward_into
from .ops import concat_volume_forward

NS = "az_stereo"
_FLOAT_DTYPES = (torch.float32, *DTYPE16)


def volume_conv(ref: Tensor, tgt: Tensor, weight: Tensor, num_disp: int) -> Tensor:
    """conv3d(concat_volume(ref, tgt, num_disp), weight, padding=1) without the volume, differentiable in all three
    inputs (``torch.ops.az_stereo.volume_conv``)."""
    return _volume_conv_library.volume_conv(ref, tgt, weight, int(num_disp))


# ---------------------------------------------------------------------------------------------
# concat volume
# ---------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NS}::concat_volume", mutates_args=(), device_types="cuda")
def concat_volume(ref: Tensor, tgt: Tensor, num_disp: int, channels_last: bool) -> Tensor:
    # float32 features, or two bfloat16 / two float16 features (the volume has their dtype; ops.build_concat_volume)
    L, R = check_feature_pair(ref, tgt, "az_stereo::concat_volume", allow16=True)
    if num_disp <= 0:
        raise ValueError("az_stereo::concat_volume: num_disp must be positive")
    return concat_volume_forward(L, R, num_disp, channels_last)


@concat_volume.register_fake
def _(ref, tgt, num_disp, channels_last):
    B, C, H, W = ref.shape
    return torch.empty((B, 2 * C, num_disp, H, W), dtype=ref.dtype, device=ref.device,
                       memory_format=torch.channels_last_3d if channels_last else torch.contiguous_format)


@torch.library.custom_op(f"{NS}::concat_volume_backward", mutates_args=(), device_types="cuda")
def concat_volume_backward(gvol: Tensor, C: int) -> Tuple[Tensor, Tensor]:
    # gL, gR have gvol's dtype, which autograd makes the volume's, i.e. the features' dtype
    if gvol.dim() != 5 or gvol.shape[1] != 2 * C or not gvol.is_cuda or gvol.dtype not in _FLOAT_DTYPES:
        raise ValueError("az_stereo::concat_volume_backward: gvol must be a CUDA float32, bfloat16 or float16 "
                         "[B,2C,Dq,H,W] tensor")
    return concat_volume_backward_into(gvol, C)


@concat_volume_backward.register_fake
def _(gvol, C):
    B, _, _, H, W = gvol.shape
    return gvol.new_empty((B, C, H, W)), gvol.new_empty((B, C, H, W))


def _concat_setup(ctx, inputs, output):
    ctx.C = inputs[0].shape[1]


def _concat_backward(ctx, gvol):
    gL, gR = concat_volume_backward(gvol, ctx.C)
    return gL, gR, None, None


concat_volume.register_autograd(_concat_backward, setup_context=_concat_setup)


# ---------------------------------------------------------------------------------------------
# soft-argmin
# ---------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NS}::soft_argmin", mutates_args=(), device_types="cuda")
def soft_argmin_op(cost: Tensor) -> Tuple[Tensor, Tensor]:
    c = _cuda_f32(cost, "cost", allow16=True)
    if c.dim() != 4:
        raise ValueError("az_stereo::soft_argmin: cost must be [B,D,H,W]")
    B, D, H, W = c.shape
    disp = torch.empty((B, 1, H, W), dtype=torch.float32, device=c.device)
    lse = torch.empty((B, 2, H, W), dtype=torch.float32, device=c.device)
    soft_argmin_forward_into(c, disp, lse)
    return disp, lse


@soft_argmin_op.register_fake
def _(cost):
    B, _, H, W = cost.shape  # disp and lse are float32 for 16-bit logits too
    return cost.new_empty((B, 1, H, W), dtype=torch.float32), cost.new_empty((B, 2, H, W), dtype=torch.float32)


@torch.library.custom_op(f"{NS}::soft_argmin_backward", mutates_args=(), device_types="cuda")
def soft_argmin_backward(cost: Tensor, disp: Tensor, lse: Tensor, gdisp: Tensor) -> Tensor:
    c, g = _cuda_f32(cost, "cost", allow16=True), _cuda_f32(gdisp, "grad_disp")
    if c.dim() != 4:
        raise ValueError("az_stereo::soft_argmin_backward: cost must be [B,D,H,W]")
    B, D, H, W = c.shape
    d_, l_ = _cuda_f32(disp, "disp"), _cuda_f32(lse, "lse")
    if tuple(d_.shape) != (B, 1, H, W) or tuple(g.shape) != (B, 1, H, W) or tuple(l_.shape) != (B, 2, H, W) \
            or not (d_.device == l_.device == g.device == c.device):
        raise ValueError("az_stereo::soft_argmin_backward: disp/gdisp [B,1,H,W] and lse [B,2,H,W] on cost's device expected")
    gcost = torch.empty_like(c)
    soft_argmin_backward_into(c, d_, l_, g, gcost)
    return gcost


@soft_argmin_backward.register_fake
def _(cost, disp, lse, gdisp):
    return torch.empty_like(cost)


def _sa_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], output[0], output[1])


def _sa_backward(ctx, gdisp, _glse):
    cost, disp, lse = ctx.saved_tensors
    return soft_argmin_backward(cost, disp, lse, gdisp)


soft_argmin_op.register_autograd(_sa_backward, setup_context=_sa_setup)


def soft_argmin(cost: Tensor) -> Tensor:
    """[B,D,H,W] logits -> [B,1,H,W] expected disparity (softmax + DisparityRegression)."""
    return soft_argmin_op(cost)[0]


# ---------------------------------------------------------------------------------------------
# fused warp + masked-MSE reprojection loss (ps = 1 and patch), with the warped / Fold image
# ---------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NS}::reproj_loss", mutates_args=(), device_types="cuda")
def reproj_loss_op(tgt: Tensor, src: Tensor, disp: Tensor, mask: Tensor, ps: int, sign: float
                   ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    t, s, d = check_reproj_inputs(tgt, src, disp, "az_stereo::reproj_loss")
    m = _mask_u8(mask, t)  # [B,1,H,W] on t's device; non-zero = selected (as ops.reproj_loss)
    if ps < 1 or ps % 2 != 1:
        raise ValueError("az_stereo::reproj_loss: ps must be odd")
    B, C, H, W = t.shape
    dev = t.device
    warped, gpre = torch.empty_like(t), torch.empty_like(d)
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    stats = torch.empty((2,), dtype=torch.float64, device=dev)
    ws = torch.empty((_lib.query("az_reproj_workspace_bytes", B, H),), dtype=torch.uint8, device=dev)
    lx, ly = linspace_table(W, dev), linspace_table(H, dev)
    with torch.cuda.device(dev):
        _lib.call("az_reproj_loss_fwd", _ptr(t), _ptr(s), _ptr(d), float(sign), _ptr(m), _ptr(lx), _ptr(ly), int(ps),
                  _ptr(warped), _ptr(gpre), _ptr(loss), _ptr(stats), _ptr(ws), B, C, H, W, _stream(), batch=B)
    if B == 0:  # F.mse_loss of nothing is NaN
        loss.fill_(float("nan"))
        stats.zero_()
    return loss.reshape(()), warped, gpre, stats


@reproj_loss_op.register_fake
def _(tgt, src, disp, mask, ps, sign):
    return (tgt.new_empty(()), torch.empty_like(tgt), torch.empty_like(disp),
            tgt.new_empty((2,), dtype=torch.float64))


@torch.library.custom_op(f"{NS}::reproj_loss_backward", mutates_args=(), device_types="cuda")
def reproj_loss_backward(gpre: Tensor, stats: Tensor, gloss: Tensor, sign: float, C: int, ps: int) -> Tensor:
    if gpre.dim() != 4 or gpre.shape[1] != 1 or not gpre.is_cuda or gpre.dtype != torch.float32 \
            or stats.numel() != 2 or stats.dtype != torch.float64 or stats.device != gpre.device:
        raise ValueError("az_stereo::reproj_loss_backward: gpre [B,1,H,W] float32 and stats float64[2] on one CUDA device expected")
    gpre = gpre.contiguous()
    B, _, H, W = gpre.shape
    gl = gloss.reshape(1).to(torch.float32).contiguous()
    gdisp = torch.empty_like(gpre)
    with torch.cuda.device(gpre.device):
        _lib.call("az_reproj_loss_bwd", _ptr(gpre), _ptr(stats), _ptr(gl), float(sign), _ptr(gdisp), B, C, H, W, int(ps),
                  _stream(), batch=B)
    return gdisp


@reproj_loss_backward.register_fake
def _(gpre, stats, gloss, sign, C, ps):
    return torch.empty_like(gpre)


def _rl_setup(ctx, inputs, output):
    ctx.save_for_backward(output[2], output[3])
    ctx.meta = (inputs[0].shape[1], int(inputs[4]), float(inputs[5]))


def _rl_backward(ctx, gloss, _gw, _gp, _gs):
    gpre, stats = ctx.saved_tensors
    C, ps, sign = ctx.meta
    return None, None, reproj_loss_backward(gpre, stats, gloss, sign, C, ps), None, None, None


reproj_loss_op.register_autograd(_rl_backward, setup_context=_rl_setup)


def reproj_loss(tgt: Tensor, src: Tensor, disp: Tensor, mask: Tensor, ps: int = 1, sign: float = -1.0):
    """-> (loss, warped): masked MSE between ``tgt`` and ``apply_disparity(unfold(src), sign*disp)`` and the warped
    image (ps = 1) / Fold image (ps > 1); differentiable w.r.t. ``disp``."""
    if tgt.requires_grad or src.requires_grad:
        raise ValueError("az_stereo::reproj_loss is differentiable w.r.t. disp only; use ops.warp() for image gradients")
    loss, warped, _, _ = reproj_loss_op(tgt, src, disp, mask, ps, sign)
    return loss, warped


# ---------------------------------------------------------------------------------------------
# group-wise correlation volume (a3)
# ---------------------------------------------------------------------------------------------
def _gwc_dims(L: Tensor, num_disp: int, num_groups: int, what: str):
    B, C, H, W = L.shape
    if num_disp <= 0 or num_groups <= 0 or C % num_groups != 0:
        raise ValueError(f"{what}: num_disp > 0 and num_groups dividing C={C} expected")
    return B, C, H, W


@torch.library.custom_op(f"{NS}::gwc_volume", mutates_args=(), device_types="cuda")
def gwc_volume(ref: Tensor, tgt: Tensor, num_disp: int, num_groups: int) -> Tensor:
    L, R = check_feature_pair(ref, tgt, "az_stereo::gwc_volume")
    B, C, H, W = _gwc_dims(L, num_disp, num_groups, "az_stereo::gwc_volume")
    vol = torch.empty((B, num_groups, num_disp, H, W), dtype=torch.float32, device=L.device)
    with torch.cuda.device(L.device):
        _lib.call("az_gwc_volume_fwd", _ptr(L), _ptr(R), _ptr(vol), B, C, H, W, num_disp, num_groups, _stream(), batch=B)
    return vol


@gwc_volume.register_fake
def _(ref, tgt, num_disp, num_groups):
    B, _, H, W = ref.shape
    return ref.new_empty((B, num_groups, num_disp, H, W))


@torch.library.custom_op(f"{NS}::gwc_volume_backward", mutates_args=(), device_types="cuda")
def gwc_volume_backward(gvol: Tensor, ref: Tensor, tgt: Tensor) -> Tuple[Tensor, Tensor]:
    L, R = check_feature_pair(ref, tgt, "az_stereo::gwc_volume_backward")
    g = _cuda_f32(gvol, "grad_volume")
    if g.dim() != 5 or g.shape[0] != L.shape[0] or tuple(g.shape[3:]) != tuple(L.shape[2:]) or g.device != L.device:
        raise ValueError("az_stereo::gwc_volume_backward: gvol must be [B,G,Dq,H,W] on the features' device")
    G, Dq = int(g.shape[1]), int(g.shape[2])
    B, C, H, W = _gwc_dims(L, Dq, G, "az_stereo::gwc_volume_backward")
    gL, gR = torch.empty_like(L), torch.empty_like(R)
    with torch.cuda.device(L.device):
        _lib.call("az_gwc_volume_bwd", _ptr(g), _ptr(L), _ptr(R), _ptr(gL), _ptr(gR), B, C, H, W, Dq, G, _stream(), batch=B)
    return gL, gR


@gwc_volume_backward.register_fake
def _(gvol, ref, tgt):
    return torch.empty_like(ref), torch.empty_like(tgt)


def _gwc_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1])


def _gwc_backward(ctx, gvol):
    ref, tgt = ctx.saved_tensors
    gL, gR = gwc_volume_backward(gvol, ref, tgt)
    return gL, gR, None, None


gwc_volume.register_autograd(_gwc_backward, setup_context=_gwc_setup)


# ---------------------------------------------------------------------------------------------
# trilinear upsample + soft-argmin in one kernel (SURVEY.md §8f rank 1)
# ---------------------------------------------------------------------------------------------
def _lowres_dims(lowres: Tensor, what: str):
    c = _cuda_f32(lowres, "lowres", allow16=True)
    if not (c.dim() == 4 or (c.dim() == 5 and c.shape[1] == 1)):
        raise ValueError(f"{what}: expected [B,1,Dq,Hq,Wq] or [B,Dq,Hq,Wq] low-resolution logits")
    return c, (int(c.shape[0]), int(c.shape[-3]), int(c.shape[-2]), int(c.shape[-1]))


@torch.library.custom_op(f"{NS}::upsample_soft_argmin", mutates_args=(), device_types="cuda")
def upsample_soft_argmin_op(lowres: Tensor, D: int, H: int, W: int) -> Tuple[Tensor, Tensor]:
    c, (B, Dq, Hq, Wq) = _lowres_dims(lowres, "az_stereo::upsample_soft_argmin")
    disp = torch.empty((B, 1, H, W), dtype=torch.float32, device=c.device)
    stats = torch.empty((B, 2, H, W), dtype=torch.float32, device=c.device)
    upsample_soft_argmin_forward_into(c, disp, stats, (B, Dq, Hq, Wq, D, H, W))
    return disp, stats


@upsample_soft_argmin_op.register_fake
def _(lowres, D, H, W):
    B = lowres.shape[0]  # disp and stats are float32 for 16-bit logits too
    return lowres.new_empty((B, 1, H, W), dtype=torch.float32), lowres.new_empty((B, 2, H, W), dtype=torch.float32)


@torch.library.custom_op(f"{NS}::upsample_soft_argmin_backward", mutates_args=(), device_types="cuda")
def upsample_soft_argmin_backward(lowres: Tensor, disp: Tensor, stats: Tensor, gdisp: Tensor, D: int) -> Tensor:
    c, (B, Dq, Hq, Wq) = _lowres_dims(lowres, "az_stereo::upsample_soft_argmin_backward")
    d_, s_, g = _cuda_f32(disp, "disp"), _cuda_f32(stats, "stats"), _cuda_f32(gdisp, "grad_disp")
    if d_.dim() != 4 or d_.shape[0] != B or d_.shape[1] != 1 or g.shape != d_.shape \
            or tuple(s_.shape) != (B, 2, d_.shape[2], d_.shape[3]) or not (d_.device == s_.device == g.device == c.device):
        raise ValueError("az_stereo::upsample_soft_argmin_backward: disp/gdisp [B,1,H,W] and stats [B,2,H,W] on the "
                         "logits' device expected")
    H, W = int(d_.shape[2]), int(d_.shape[3])
    glow = torch.empty_like(c)
    upsample_soft_argmin_backward_into(c, d_, s_, g, glow, (B, Dq, Hq, Wq, D, H, W))
    return glow


@upsample_soft_argmin_backward.register_fake
def _(lowres, disp, stats, gdisp, D):
    return torch.empty_like(lowres)


def _usa_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], output[0], output[1])
    ctx.D = int(inputs[1])


def _usa_backward(ctx, gdisp, _gstats):
    lowres, disp, stats = ctx.saved_tensors
    return upsample_soft_argmin_backward(lowres, disp, stats, gdisp, ctx.D), None, None, None


upsample_soft_argmin_op.register_autograd(_usa_backward, setup_context=_usa_setup)


def upsample_soft_argmin(lowres: Tensor, out_size) -> Tensor:
    """[B,1,Dq,Hq,Wq] low-resolution logits -> [B,1,H,W] disparity for ``out_size = (D, H, W)``."""
    D, H, W = (int(v) for v in out_size)
    return upsample_soft_argmin_op(lowres, D, H, W)[0]


# ---------------------------------------------------------------------------------------------
# bilinear disparity warp (a6)
# ---------------------------------------------------------------------------------------------
def _warp_inputs(img: Tensor, disp: Tensor, what: str):
    im, d = _cuda_f32(img, "img"), _cuda_f32(disp, "disp")
    if im.dim() != 4 or tuple(d.shape) != (im.shape[0], 1, im.shape[2], im.shape[3]) or d.device != im.device:
        raise ValueError(f"{what}: img [B,C,H,W] and disp [B,1,H,W] on one device expected, got "
                         f"{tuple(im.shape)} and {tuple(d.shape)}")
    return im, d


@torch.library.custom_op(f"{NS}::warp", mutates_args=(), device_types="cuda")
def warp(img: Tensor, disp: Tensor) -> Tensor:
    im, d = _warp_inputs(img, disp, "az_stereo::warp")
    B, C, H, W = im.shape
    out = torch.empty_like(im)
    lx, ly = linspace_table(W, im.device), linspace_table(H, im.device)
    with torch.cuda.device(im.device):
        _lib.call("az_warp_fwd", _ptr(im), _ptr(d), _ptr(lx), _ptr(ly), _ptr(out), B, C, H, W, _stream(), batch=B)
    return out


@warp.register_fake
def _(img, disp):
    return torch.empty_like(img)


@torch.library.custom_op(f"{NS}::warp_backward", mutates_args=(), device_types="cuda")
def warp_backward(img: Tensor, disp: Tensor, gout: Tensor) -> Tuple[Tensor, Tensor]:
    im, d = _warp_inputs(img, disp, "az_stereo::warp_backward")
    g = _cuda_f32(gout, "grad_out")
    if g.shape != im.shape or g.device != im.device:
        raise ValueError("az_stereo::warp_backward: gout must have img's shape and device")
    B, C, H, W = im.shape
    gimg, gdisp = torch.empty_like(im), torch.empty_like(d)  # both fully written (atomic-free kernels)
    lx, ly = linspace_table(W, im.device), linspace_table(H, im.device)
    with torch.cuda.device(im.device):
        _lib.call("az_warp_bwd", _ptr(im), _ptr(d), _ptr(lx), _ptr(ly), _ptr(g), _ptr(gimg), _ptr(gdisp), B, C, H, W,
                  _stream(), batch=B)
    return gimg, gdisp


@warp_backward.register_fake
def _(img, disp, gout):
    return torch.empty_like(img), torch.empty_like(disp)


def _warp_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1])


def _warp_backward(ctx, gout):
    img, disp = ctx.saved_tensors
    return warp_backward(img, disp, gout)


warp.register_autograd(_warp_backward, setup_context=_warp_setup)


# ---------------------------------------------------------------------------------------------
# non-differentiable operators: scatter warp (a10), temporal IR pattern (a11), LCN (a12)
# ---------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NS}::scatter_warp", mutates_args=(), device_types="cuda")
def scatter_warp_op(img: Tensor, disp: Tensor) -> Tuple[Tensor, Tensor]:
    if not (img.is_cuda and disp.is_cuda) or img.device != disp.device or img.dtype != torch.float32 \
            or disp.dtype != torch.int32 or img.dim() != 4:
        raise ValueError("az_stereo::scatter_warp: img float32 [N,C,H,W] and disp int32 on one CUDA device expected")
    N, C, H, W = img.shape
    if disp.numel() != N * H * W:
        raise ValueError("az_stereo::scatter_warp: disp must be [N,H,W] or [N,1,H,W]")
    im, d = img.contiguous(), disp.contiguous()
    out = torch.empty_like(im)
    flags = torch.zeros((1,), dtype=torch.int32, device=im.device)  # bit 0: a positive, bit 1: a negative disparity
    with torch.cuda.device(im.device):
        _lib.call("az_scatter_warp", _ptr(im), _ptr(d), _ptr(out), _ptr(flags), N, C, H, W, _stream(), batch=N)
    return out, flags


@scatter_warp_op.register_fake
def _(img, disp):
    return torch.empty_like(img), img.new_empty((1,), dtype=torch.int32)


def scatter_warp(img: Tensor, disp: Tensor, check_sign: bool = True) -> Tensor:
    """``apply_disparity_cu`` (utils/warp_ops.py:55-95).  ``check_sign`` reads the 4-byte flag word back, as the
    reference's sign assertion does (warp_ops.py:73-77); pass False inside a compiled region."""
    out, flags = scatter_warp_op(img, disp)
    if check_sign:
        assert int(flags.item()) != 3, "disparities must be all >= 0 or all <= 0"
    return out


@torch.library.custom_op(f"{NS}::temporal_ir_pattern", mutates_args=(), device_types="cuda")
def temporal_ir_pattern(frames: Tensor, ks: int, threshold: float) -> Tensor:
    if not frames.is_cuda or frames.dtype != torch.uint8 or frames.dim() != 4:
        raise ValueError("az_stereo::temporal_ir_pattern: expected a CUDA uint8 [B,T,H,W] tensor")
    f = frames.contiguous()
    B, T, H, W = f.shape
    pat = torch.empty((B, H, W), dtype=torch.float32, device=f.device)
    ws = torch.empty((_lib.query("az_temporal_ir_workspace_bytes", B, H, W),), dtype=torch.uint8, device=f.device)
    with torch.cuda.device(f.device):
        _lib.call("az_temporal_ir", _ptr(f), _ptr(pat), _ptr(ws), B, T, H, W, ks, threshold, _stream(), batch=B)
    return pat


@temporal_ir_pattern.register_fake
def _(frames, ks, threshold):
    B, _, H, W = frames.shape
    return frames.new_empty((B, H, W), dtype=torch.float32)


@torch.library.custom_op(f"{NS}::local_contrast_norm", mutates_args=(), device_types="cuda")
def local_contrast_norm(image: Tensor, kernel_size: int, eps: float) -> Tuple[Tensor, Tensor]:
    if kernel_size < 1 or kernel_size % 2 != 1:
        raise ValueError("az_stereo::local_contrast_norm: kernel size should be odd")
    im = _cuda_f32(image, "image")
    if im.dim() != 4:
        raise ValueError("az_stereo::local_contrast_norm: image must be [B,C,H,W]")
    B, Cin, H, W = im.shape
    normed = torch.empty((B, 1, H, W), dtype=torch.float32, device=im.device)
    std = torch.empty_like(normed)
    with torch.cuda.device(im.device):
        _lib.call("az_local_contrast_norm", _ptr(im), _ptr(normed), _ptr(std), B, Cin, H, W, kernel_size, eps, _stream(), batch=B)
    return normed, std


@local_contrast_norm.register_fake
def _(image, kernel_size, eps):
    B, _, H, W = image.shape
    return image.new_empty((B, 1, H, W)), image.new_empty((B, 1, H, W))
