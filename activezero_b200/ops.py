"""PyTorch-facing operators of the B200 stereo hot path.

One ``torch.autograd.Function`` per differentiable op (the pattern the reference
itself uses for an external CUDA module: ``CorrSampler`` in
``/root/reference/nets/raft/corr.py:18-31``), each a thin marshalling layer over
the C ABI in ``include/az_stereo.h``.  PyTorch provides device memory and the
current stream; all arithmetic happens in ``libaz_stereo.so``.  CUDA float32
tensors only -- there is no CPU path and no eager fallback.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch
from torch.autograd.function import once_differentiable

# Under torch.autocast the operators still compute in fp32 (the reference's PSMNet path does not use AMP;
# the decorators only make the Functions safe to call from an autocast region).
_fwd32 = torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
_bwd = torch.amp.custom_bwd(device_type="cuda")

from . import _lib

_NULL = ctypes.c_void_p(0)


def _ptr(t: Optional[torch.Tensor]):
    return _NULL if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# the 16-bit dtypes of torch.autocast -> the C ABI's dtype codes (AZ_DTYPE_BF16, AZ_DTYPE_F16 in include/az_stereo.h)
DTYPE16 = {torch.bfloat16: 1, torch.float16: 2}


def _cuda_f32(t: torch.Tensor, name: str, allow16: bool = False) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (activezero_b200 has no CPU path)")
    if t.dtype != torch.float32 and not (allow16 and t.dtype in DTYPE16):
        raise ValueError(f"{name}: expected float32{', bfloat16 or float16' if allow16 else ''}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def check_feature_pair(ref_feat, tgt_feat, what: str, allow16: bool = False):
    """Shared by ops and library_ops: both features CUDA float32 [B,C,H,W] of the SAME shape and device
    (``allow16``: or both bfloat16, or both float16)."""
    L = _cuda_f32(ref_feat, "ref_feat", allow16)
    R = _cuda_f32(tgt_feat, "tgt_feat", allow16)
    if L.dim() != 4 or L.shape != R.shape:
        raise ValueError(f"{what}: features must both be [B,C,H,W] with identical shapes, got {tuple(L.shape)} and {tuple(R.shape)}")
    if L.dtype != R.dtype:
        raise ValueError(f"{what}: features of different dtypes ({L.dtype} and {R.dtype})")
    if L.device != R.device:
        raise ValueError(f"{what}: features live on different devices")
    return L, R


def check_reproj_inputs(tgt, src, disp, what: str = "reprojection loss"):
    """tgt, src [B,C,H,W]; disp [B,1,H,W]; all CUDA float32 on one device (rejects before any C-ABI call)."""
    t = _cuda_f32(tgt, "tgt")
    s = _cuda_f32(src, "src")
    d = _cuda_f32(disp, "disp")
    if t.dim() != 4 or t.shape != s.shape or d.dim() != 4 or tuple(d.shape) != (t.shape[0], 1, t.shape[2], t.shape[3]):
        raise ValueError(f"{what}: images [B,C,H,W] of identical shape and disp [B,1,H,W] expected, got "
                         f"{tuple(t.shape)}, {tuple(s.shape)}, {tuple(d.shape)}")
    if not (t.device == s.device == d.device):
        raise ValueError(f"{what}: tensors live on different devices")
    return t, s, d


_LIN_CACHE: dict = {}


def linspace_table(n: int, device: torch.device) -> torch.Tensor:
    """``torch.linspace(0, 1, n)`` evaluated on the CPU in fp32 -- the base grid of
    ``apply_disparity`` (``utils/reprojection.py:18-24``) -- cached on ``device``.
    The table (not a closed form) is what makes the sample position bit-identical
    to the reference's."""
    key = (int(n), str(device))
    tab = _LIN_CACHE.get(key)
    if tab is None:
        tab = torch.linspace(0, 1, int(n), dtype=torch.float32).to(device)
        _LIN_CACHE[key] = tab
    return tab


# ----------------------------------------------------------------------------
# a1/a2 concat volume
# ----------------------------------------------------------------------------
def concat_volume_forward(L, R, num_disp: int, channels_last: bool):
    """Enqueues the concat volume of validated features (float32, or both bfloat16 / both float16: the volume has
    the features' dtype).  Shared by ConcatVolumeFn and library_ops."""
    B, C, H, W = L.shape
    dt = DTYPE16.get(L.dtype)
    # the kernels write channels_last_3d directly when a position's 2C values are whole 16-byte vectors
    ndhwc = bool(channels_last) and C % (4 if dt is None else 8) == 0
    vol = torch.empty((B, 2 * C, num_disp, H, W), dtype=L.dtype, device=L.device,
                      memory_format=torch.channels_last_3d if ndhwc else torch.contiguous_format)
    with torch.cuda.device(L.device):
        if dt is None:
            _lib.call("az_concat_volume_fwd_ndhwc" if ndhwc else "az_concat_volume_fwd", _ptr(L), _ptr(R), _ptr(vol),
                      B, C, H, W, num_disp, _stream(), batch=B)
        else:
            _lib.call("az_concat_volume_fwd_16", _ptr(L), _ptr(R), _ptr(vol), B, C, H, W, num_disp, 1 if ndhwc else 0,
                      _stream(), batch=B)
    if channels_last and not ndhwc:  # C not a multiple of 4 (8 for 16 bits): torch's layout conversion (on the device)
        vol = vol.contiguous(memory_format=torch.channels_last_3d)
    return vol


def concat_volume_backward(gvol, C: int, need_l: bool = True, need_r: bool = True):
    """gL, gR (each None when not needed) of the concat volume for a CUDA gradient [B,2C,Dq,H,W] of dtype float32,
    bfloat16 or float16; the gradients have gvol's dtype.  Shared by ConcatVolumeFn and library_ops."""
    dt = DTYPE16.get(gvol.dtype)
    B, _, Dq, H, W = gvol.shape
    # a gradient that arrives in channels_last_3d (what cuDNN returns for a channels_last_3d input) is consumed
    # in place; anything else is made NCDHW-contiguous
    ndhwc = C % (4 if dt is None else 8) == 0 and Dq * H * W > 1 \
        and gvol.is_contiguous(memory_format=torch.channels_last_3d) and not gvol.is_contiguous()
    g = gvol if ndhwc else _cuda_f32(gvol, "grad_volume", allow16=True)
    gL = torch.empty((B, C, H, W), dtype=g.dtype, device=g.device) if need_l else None
    gR = torch.empty((B, C, H, W), dtype=g.dtype, device=g.device) if need_r else None
    with torch.cuda.device(g.device):
        if dt is None:
            _lib.call("az_concat_volume_bwd_ndhwc" if ndhwc else "az_concat_volume_bwd", _ptr(g), _ptr(gL), _ptr(gR),
                      B, C, H, W, Dq, _stream(), batch=B)
        else:
            _lib.call("az_concat_volume_bwd_16", _ptr(g), _ptr(gL), _ptr(gR), B, C, H, W, Dq, dt, 1 if ndhwc else 0,
                      _stream(), batch=B)
    return gL, gR


class ConcatVolumeFn(torch.autograd.Function):
    """nets/psmnet/psmnet.py:151-165 and its autograd.  Outside torch.autocast, two bfloat16 (or two float16) features
    give a volume of their dtype and gradients of their dtype (RNE of the fp32 sums, DESIGN.md §4.11); inside autocast the
    inputs are cast to float32 as before."""

    @staticmethod
    @_fwd32
    def forward(ctx, ref_feat, tgt_feat, num_disp: int, channels_last: bool = False):
        L, R = check_feature_pair(ref_feat, tgt_feat, "concat volume", allow16=True)
        if int(num_disp) <= 0:
            raise ValueError("concat volume: num_disp must be positive")
        ctx.dims = (L.shape[1], int(num_disp), L.dtype)
        return concat_volume_forward(L, R, int(num_disp), channels_last)

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gvol):
        C, Dq, dtype = ctx.dims
        if not isinstance(gvol, torch.Tensor) or not gvol.is_cuda or gvol.dtype != dtype:
            raise ValueError(f"grad_volume: expected a {dtype} CUDA tensor")
        gL, gR = concat_volume_backward(gvol, C, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return gL, gR, None, None


def build_concat_volume(ref_feat, tgt_feat, num_disp: int, channels_last: bool = False):
    """[B,C,H,W] x2 -> [B,2C,num_disp,H,W] (replaces psmnet.py:151-165).  ``channels_last=True`` returns the
    same tensor in ``torch.channels_last_3d`` memory format (SURVEY.md §8f rank 2): the values and the shape are
    unchanged, only the strides differ, and cuDNN's 3-D convolutions consume it without a layout pass.
    float32 features give a float32 volume; outside torch.autocast, two bfloat16 or two float16 features give a volume
    of their dtype (the same values: a copy), and the backward returns gradients of their dtype."""
    return ConcatVolumeFn.apply(ref_feat, tgt_feat, num_disp, channels_last)


# ----------------------------------------------------------------------------
# §8f rank 2: dres0's first convolution with the concat volume left implicit (tcgen05 TF32 implicit GEMM)
# ----------------------------------------------------------------------------
def pack_volume_conv_weight(weight: torch.Tensor, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """Conv3d weight [32,64,3,3,3] (dres0[0][0].weight, psmnet.py:85-90) -> the per-tap core-matrix order of the
    tensor-core kernel, rounded to TF32; do this once per weight tensor.  ``dtype`` = the dtype of the features it
    will be used with: bfloat16 / float16 round each weight to that dtype first (RNE), as torch.autocast rounds the
    weight of a cuDNN convolution.  A bfloat16 / float16 weight (a converted model) is widened exactly first."""
    w = _cuda_f32(weight.detach(), "weight", allow16=True).float()
    if tuple(w.shape) != (32, 64, 3, 3, 3):
        raise ValueError(f"volume conv: expected a [32,64,3,3,3] Conv3d weight, got {tuple(w.shape)}")
    if dtype != torch.float32 and dtype not in DTYPE16:
        raise ValueError(f"volume conv: dtype must be float32, bfloat16 or float16, got {dtype}")
    packed = torch.empty((27 * 3072,), dtype=torch.float32, device=w.device)  # AZ_VOLUME_CONV0_PACKED_FLOATS
    with torch.cuda.device(w.device):
        if dtype == torch.float32:
            _lib.call("az_volume_conv0_pack", _ptr(w), _ptr(packed), _stream())
        else:
            _lib.call("az_volume_conv0_pack_16", _ptr(w), _ptr(packed), DTYPE16[dtype], _stream())
    return packed


def volume_conv0(ref_feat, tgt_feat, wpacked, num_disp: int, scale=None, shift=None, relu: bool = False):
    """conv3d(concat_volume(ref, tgt, num_disp), weight, padding=1) without the volume (forward only; TF32 operands,
    fp32 accumulation): [B,32,H,W] x2 -> [B,32,num_disp,H,W].  ``scale``/``shift`` [32] fold an eval-mode BatchNorm.
    Two bfloat16 (or float16) features give an output of their dtype, rounded once after the fold and the ReLU;
    ``wpacked`` should then come from ``pack_volume_conv_weight(weight, dtype=<that dtype>)``."""
    L, R = check_feature_pair(ref_feat.detach(), tgt_feat.detach(), "volume conv", allow16=True)
    B, C, H, W = L.shape
    if C != 32:
        raise ValueError("volume conv: PSMNet's 32 feature channels expected")
    wp = _cuda_f32(wpacked, "wpacked")
    if wp.numel() != 27 * 3072 or wp.device != L.device:
        raise ValueError("volume conv: wpacked must come from pack_volume_conv_weight on the features' device")
    if (scale is None) != (shift is None):
        raise ValueError("volume conv: scale and shift go together")
    sc = _cuda_f32(scale.detach().reshape(-1), "scale") if scale is not None else None
    sh = _cuda_f32(shift.detach().reshape(-1), "shift") if shift is not None else None
    if sc is not None and (sc.numel() != 32 or sh.numel() != 32):
        raise ValueError("volume conv: scale / shift must hold 32 values")
    out = torch.empty((B, 32, int(num_disp), H, W), dtype=L.dtype, device=L.device)
    dt = DTYPE16.get(L.dtype)
    with torch.cuda.device(L.device):
        if dt is None:
            _lib.call("az_volume_conv0_fwd", _ptr(L), _ptr(R), _ptr(wp), _ptr(sc), _ptr(sh), _ptr(out), B, C, H, W,
                      int(num_disp), 1 if relu else 0, _stream(), batch=B)
        else:
            _lib.call("az_volume_conv0_fwd_16", _ptr(L), _ptr(R), _ptr(wp), _ptr(sc), _ptr(sh), _ptr(out), B, C, H, W,
                      int(num_disp), 1 if relu else 0, dt, _stream(), batch=B)
    return out


def check_volume_conv_inputs(ref_feat, tgt_feat, weight, num_disp: int, what: str):
    """Shared by ops and library_ops: features CUDA [B,32,H,W], both float32 or both bfloat16 / both float16; weight
    [32,64,3,3,3] on their device, float32 or the features' dtype."""
    L, R = check_feature_pair(ref_feat, tgt_feat, what, allow16=True)
    if L.shape[1] != 32:
        raise ValueError(f"{what}: PSMNet's 32 feature channels expected, got {L.shape[1]}")
    w = _cuda_f32(weight, "weight", allow16=True)
    if w.dtype not in (torch.float32, L.dtype):
        raise ValueError(f"{what}: a {w.dtype} weight with {L.dtype} features (float32 or {L.dtype} expected)")
    if tuple(w.shape) != (32, 64, 3, 3, 3) or w.device != L.device:
        raise ValueError(f"{what}: expected a [32,64,3,3,3] Conv3d weight on the features' device, got {tuple(w.shape)}")
    if int(num_disp) <= 0:
        raise ValueError(f"{what}: num_disp must be positive")
    return L, R, w


def volume_conv_forward(L, R, w, num_disp: int):
    """The raw convolution (no fold, no ReLU) of validated tensors; the output has the features' dtype.  Shared by
    VolumeConv0Fn and library_ops."""
    B, C, H, W = L.shape
    out = torch.empty((B, 32, int(num_disp), H, W), dtype=L.dtype, device=L.device)
    if B > 0:
        dt = DTYPE16.get(L.dtype)
        wp = pack_volume_conv_weight(w, dtype=L.dtype)
        with torch.cuda.device(L.device):
            if dt is None:
                _lib.call("az_volume_conv0_fwd", _ptr(L), _ptr(R), _ptr(wp), _NULL, _NULL, _ptr(out), B, C, H, W,
                          int(num_disp), 0, _stream(), batch=B)
            else:
                _lib.call("az_volume_conv0_fwd_16", _ptr(L), _ptr(R), _ptr(wp), _NULL, _NULL, _ptr(out), B, C, H, W,
                          int(num_disp), 0, dt, _stream(), batch=B)
    return out


def volume_conv_backward_into(gout, L, R, w, gL, gR, gW):
    """Enqueues az_volume_conv0_bwd (float32 features) or az_volume_conv0_bwd_16 (16-bit features) for the validated
    tensors; gL / gR / gW may each be None (skipped).  gout must have the features' dtype."""
    B, C, H, W = L.shape
    if not isinstance(gout, torch.Tensor) or not gout.is_cuda or gout.dtype != L.dtype:
        raise ValueError(f"volume conv backward: grad_out must be a {L.dtype} CUDA tensor, got "
                         f"{getattr(gout, 'dtype', type(gout))}")
    gout = gout.contiguous()
    Dq = gout.shape[2] if gout.dim() == 5 else -1
    if tuple(gout.shape) != (B, 32, Dq, H, W) or gout.device != L.device:
        raise ValueError(f"volume conv backward: grad_out must be [B,32,Dq,H,W] = {(B, 32, Dq, H, W)} on the features' "
                         f"device, got {tuple(gout.shape)}")
    if B == 0:
        if gW is not None:
            gW.zero_()  # a sum over no position
        return
    ws = torch.empty((_lib.query("az_volume_conv0_bwd_workspace_bytes", B, H, W, Dq),), dtype=torch.uint8, device=L.device)
    dt = DTYPE16.get(L.dtype)
    with torch.cuda.device(L.device):
        if dt is None:
            _lib.call("az_volume_conv0_bwd", _ptr(gout), _ptr(L), _ptr(R), _ptr(w), _ptr(gL), _ptr(gR), _ptr(gW),
                      _ptr(ws), B, C, H, W, Dq, _stream(), batch=B)
        else:
            _lib.call("az_volume_conv0_bwd_16", _ptr(gout), _ptr(L), _ptr(R), _ptr(w), _ptr(gL), _ptr(gR), _ptr(gW),
                      _ptr(ws), B, C, H, W, Dq, dt, 0 if w.dtype == torch.float32 else dt, _stream(), batch=B)


class VolumeConv0Fn(torch.autograd.Function):
    """conv3d(concat_volume(ref, tgt, num_disp), weight, padding=1) -- dres0[0][0] on the implicit volume
    (psmnet.py:151-168) -- differentiable in all three inputs.  Forward: the tcgen05 kernel (TF32 operands, fp32
    accumulation).  Backward: the volume-free kernels of csrc/volume_conv_bwd.cu (fp32 arithmetic).  Saves the features
    and the weight only (feature-sized, not volume-sized).  Outside torch.autocast, two bfloat16 (or two float16)
    features with a float32 weight or one of their dtype give an output and feature gradients of their dtype and a
    weight gradient of the weight's dtype, equal to the float32 op on the widened features and the weight rounded to
    their dtype, followed by .to(dtype) (DESIGN.md §4.13); inside autocast the inputs are cast to float32 as before."""

    @staticmethod
    @_fwd32
    def forward(ctx, ref_feat, tgt_feat, weight, num_disp: int):
        L, R, w = check_volume_conv_inputs(ref_feat, tgt_feat, weight, num_disp, "volume conv")
        out = volume_conv_forward(L, R, w, num_disp)
        ctx.save_for_backward(L, R, w)
        return out

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gout):
        L, R, w = ctx.saved_tensors
        g = gout
        gL = torch.empty_like(L) if ctx.needs_input_grad[0] else None
        gR = torch.empty_like(R) if ctx.needs_input_grad[1] else None
        gW = torch.empty_like(w) if ctx.needs_input_grad[2] else None
        volume_conv_backward_into(g, L, R, w, gL, gR, gW)
        return gL, gR, gW, None


def volume_conv(ref_feat, tgt_feat, weight, num_disp: int):
    """[B,32,H,W] x2, Conv3d weight [32,64,3,3,3] -> conv3d(concat_volume(ref, tgt, num_disp), weight, padding=1),
    [B,32,num_disp,H,W], with autograd; the concat volume and its gradient are never materialised.  The raw
    convolution: no BatchNorm fold, no ReLU (``volume_conv0`` is the inference form with both).  Outside
    torch.autocast it also takes two bfloat16 or two float16 features, with a float32 weight or one of their dtype."""
    return VolumeConv0Fn.apply(ref_feat, tgt_feat, weight, num_disp)


# ----------------------------------------------------------------------------
# a3 group-wise correlation volume (no reference counterpart)
# ----------------------------------------------------------------------------
class GwcVolumeFn(torch.autograd.Function):
    @staticmethod
    @_fwd32
    def forward(ctx, ref_feat, tgt_feat, num_disp: int, num_groups: int):
        L, R = check_feature_pair(ref_feat, tgt_feat, "gwc volume")
        B, C, H, W = L.shape
        if int(num_disp) <= 0 or int(num_groups) <= 0 or C % int(num_groups) != 0:
            raise ValueError(f"gwc volume: num_disp > 0 and num_groups dividing C={C} expected")
        vol = torch.empty((B, int(num_groups), int(num_disp), H, W), dtype=torch.float32, device=L.device)
        with torch.cuda.device(L.device):
            _lib.call("az_gwc_volume_fwd", _ptr(L), _ptr(R), _ptr(vol), B, C, H, W, int(num_disp), int(num_groups),
                      _stream(), batch=B)
        ctx.save_for_backward(L, R)
        ctx.dims = (B, C, H, W, int(num_disp), int(num_groups))
        return vol

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gvol):
        L, R = ctx.saved_tensors
        B, C, H, W, Dq, G = ctx.dims
        g = _cuda_f32(gvol, "grad_volume")
        gL = torch.empty_like(L) if ctx.needs_input_grad[0] else None
        gR = torch.empty_like(R) if ctx.needs_input_grad[1] else None
        with torch.cuda.device(g.device):
            _lib.call("az_gwc_volume_bwd", _ptr(g), _ptr(L), _ptr(R), _ptr(gL), _ptr(gR), B, C, H, W, Dq, G, _stream(), batch=B)
        return gL, gR, None, None


def build_gwc_volume(ref_feat, tgt_feat, num_disp: int, num_groups: int):
    return GwcVolumeFn.apply(ref_feat, tgt_feat, num_disp, num_groups)


# ----------------------------------------------------------------------------
# a4/a5 soft-argmin
# ----------------------------------------------------------------------------
# The logits may be float32, bfloat16 or float16; disp, lse / stats and gdisp are always float32 and the logits'
# gradient has the logits' dtype (16 bits: the fp32 gradient rounded once, DESIGN.md §4.12).  Shared by the
# Functions below and library_ops.
def soft_argmin_forward_into(c, disp, lse):
    B, D, H, W = c.shape
    dt = DTYPE16.get(c.dtype)
    with torch.cuda.device(c.device):
        if dt is None:
            _lib.call("az_soft_argmin_fwd", _ptr(c), _ptr(disp), _ptr(lse), B, D, H, W, _stream(), batch=B)
        else:
            _lib.call("az_soft_argmin_fwd_16", _ptr(c), _ptr(disp), _ptr(lse), B, D, H, W, dt, _stream(), batch=B)


def soft_argmin_backward_into(c, disp, lse, g, gcost):
    B, D, H, W = c.shape
    dt = DTYPE16.get(c.dtype)
    with torch.cuda.device(c.device):
        if dt is None:
            _lib.call("az_soft_argmin_bwd", _ptr(c), _ptr(disp), _ptr(lse), _ptr(g), _ptr(gcost), B, D, H, W, _stream(),
                      batch=B)
        else:
            _lib.call("az_soft_argmin_bwd_16", _ptr(c), _ptr(disp), _ptr(lse), _ptr(g), _ptr(gcost), B, D, H, W, dt,
                      _stream(), batch=B)


def upsample_soft_argmin_forward_into(c, disp, stats, dims):
    B, Dq, Hq, Wq, D, H, W = dims
    dt = DTYPE16.get(c.dtype)
    with torch.cuda.device(c.device):
        if dt is None:
            _lib.call("az_upsample_soft_argmin_fwd", _ptr(c), _ptr(disp), _ptr(stats), B, Dq, Hq, Wq, D, H, W, _stream(),
                      batch=B)
        else:
            _lib.call("az_upsample_soft_argmin_fwd_16", _ptr(c), _ptr(disp), _ptr(stats), B, Dq, Hq, Wq, D, H, W, dt,
                      _stream(), batch=B)


def upsample_soft_argmin_backward_into(c, disp, stats, g, glow, dims):
    B, Dq, Hq, Wq, D, H, W = dims
    ws = torch.empty((_lib.query("az_upsample_soft_argmin_workspace_bytes", B, Dq, H, W, Wq),), dtype=torch.uint8,
                     device=c.device)
    dt = DTYPE16.get(c.dtype)
    with torch.cuda.device(c.device):
        if dt is None:
            _lib.call("az_upsample_soft_argmin_bwd", _ptr(c), _ptr(disp), _ptr(stats), _ptr(g), _ptr(glow), _ptr(ws),
                      B, Dq, Hq, Wq, D, H, W, _stream(), batch=B)
        else:
            _lib.call("az_upsample_soft_argmin_bwd_16", _ptr(c), _ptr(disp), _ptr(stats), _ptr(g), _ptr(glow), _ptr(ws),
                      B, Dq, Hq, Wq, D, H, W, dt, _stream(), batch=B)


class SoftArgminFn(torch.autograd.Function):
    """F.softmax(cost, 1) + DisparityRegression (psmnet.py:200-201,
    psmnet_submodule.py:80-89) fused; takes LOGITS.  Outside torch.autocast, bfloat16 / float16 logits are read as
    they are: the disparity is float32 and equal to the float32 operator's on ``cost.float()``, and the gradient has
    the logits' dtype; inside autocast the logits are cast to float32 as before."""

    @staticmethod
    @_fwd32
    def forward(ctx, cost):
        c = _cuda_f32(cost, "cost", allow16=True)
        if c.dim() != 4:
            raise ValueError("soft_argmin: cost must be [B,D,H,W]")
        B, D, H, W = c.shape
        disp = torch.empty((B, 1, H, W), dtype=torch.float32, device=c.device)
        need_bwd = ctx.needs_input_grad[0]
        lse = torch.empty((B, 2, H, W), dtype=torch.float32, device=c.device) if need_bwd else None
        soft_argmin_forward_into(c, disp, lse)
        if need_bwd:
            ctx.save_for_backward(c, disp, lse)
        return disp

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gdisp):
        c, disp, lse = ctx.saved_tensors
        g = _cuda_f32(gdisp, "grad_disp")
        gcost = torch.empty_like(c)
        soft_argmin_backward_into(c, disp, lse, g, gcost)
        return gcost


def soft_argmin(cost):
    """[B,D,H,W] logits (float32, bfloat16 or float16) -> [B,1,H,W] float32 expected disparity."""
    return SoftArgminFn.apply(cost)


class UpsampleSoftArgminFn(torch.autograd.Function):
    """F.interpolate(cost, (D,H,W), 'trilinear', align_corners=False) -> squeeze ->
    softmax -> DisparityRegression (psmnet.py:186-217) in one kernel that reads the
    low-resolution logits only (SURVEY.md §8f rank 1).  bfloat16 / float16 logits outside torch.autocast: as in
    SoftArgminFn, a float32 disparity and a gradient of the logits' dtype."""

    @staticmethod
    @_fwd32
    def forward(ctx, lowres, out_size):
        c = _cuda_f32(lowres, "lowres", allow16=True)
        if c.dim() == 5:
            if c.shape[1] != 1:
                raise ValueError("upsample_soft_argmin: expected [B,1,Dq,Hq,Wq]")
        elif c.dim() != 4:
            raise ValueError("upsample_soft_argmin: expected [B,1,Dq,Hq,Wq] or [B,Dq,Hq,Wq]")
        B, Dq, Hq, Wq = c.shape[0], c.shape[-3], c.shape[-2], c.shape[-1]
        D, H, W = (int(v) for v in out_size)
        disp = torch.empty((B, 1, H, W), dtype=torch.float32, device=c.device)
        need_bwd = ctx.needs_input_grad[0]
        stats = torch.empty((B, 2, H, W), dtype=torch.float32, device=c.device) if need_bwd else None
        ctx.dims = (B, Dq, Hq, Wq, D, H, W)
        upsample_soft_argmin_forward_into(c, disp, stats, ctx.dims)
        if need_bwd:
            ctx.save_for_backward(c, disp, stats)
        return disp

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gdisp):
        c, disp, stats = ctx.saved_tensors
        g = _cuda_f32(gdisp, "grad_disp")
        glow = torch.empty_like(c)
        upsample_soft_argmin_backward_into(c, disp, stats, g, glow, ctx.dims)
        return glow, None


def upsample_soft_argmin(lowres, out_size):
    """[B,1,Dq,Hq,Wq] low-res logits (float32, bfloat16 or float16) -> [B,1,H,W] float32 disparity for
    out_size = (D,H,W)."""
    return UpsampleSoftArgminFn.apply(lowres, tuple(out_size))


# ----------------------------------------------------------------------------
# a6 bilinear disparity warp
# ----------------------------------------------------------------------------
class WarpFn(torch.autograd.Function):
    """apply_disparity (utils/reprojection.py:13-35)."""

    @staticmethod
    @_fwd32
    def forward(ctx, img, disp):
        im = _cuda_f32(img, "img")
        d = _cuda_f32(disp, "disp")
        if im.dim() != 4 or d.dim() != 4 or d.shape[1] != 1 or d.shape[0] != im.shape[0] or d.shape[2:] != im.shape[2:] \
                or d.device != im.device:
            raise ValueError("apply_disparity: img [B,C,H,W], disp [B,1,H,W] on one device expected")
        B, C, H, W = im.shape
        out = torch.empty_like(im)
        lx, ly = linspace_table(W, im.device), linspace_table(H, im.device)
        with torch.cuda.device(im.device):
            _lib.call("az_warp_fwd", _ptr(im), _ptr(d), _ptr(lx), _ptr(ly), _ptr(out), B, C, H, W, _stream(), batch=B)
        ctx.save_for_backward(im, d)
        return out

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gout):
        im, d = ctx.saved_tensors
        B, C, H, W = im.shape
        g = _cuda_f32(gout, "grad_out")
        gimg = torch.empty_like(im) if ctx.needs_input_grad[0] else None  # fully written by the kernel
        gdisp = torch.empty_like(d) if ctx.needs_input_grad[1] else None
        lx, ly = linspace_table(W, im.device), linspace_table(H, im.device)
        with torch.cuda.device(im.device):
            _lib.call("az_warp_bwd", _ptr(im), _ptr(d), _ptr(lx), _ptr(ly), _ptr(g), _ptr(gimg), _ptr(gdisp),
                      B, C, H, W, _stream(), batch=B)
        return gimg, gdisp


def warp(img, disp):
    return WarpFn.apply(img, disp)


# ----------------------------------------------------------------------------
# a7/a8 fused warp + masked MSE
# ----------------------------------------------------------------------------
def _mask_u8(mask: Optional[torch.Tensor], like: torch.Tensor) -> Optional[torch.Tensor]:
    if mask is None:
        return None
    if not isinstance(mask, torch.Tensor) or not mask.is_cuda or mask.device != like.device:
        raise ValueError("mask: expected a CUDA tensor on the images' device")
    B, _, H, W = like.shape
    if mask.dim() != 4 or mask.shape[0] != B or mask.shape[1] != 1 or mask.shape[2] != H or mask.shape[3] != W:
        raise ValueError("mask must be [B,1,H,W]")
    m = mask if mask.dtype == torch.bool else (mask != 0)
    return m.contiguous().view(torch.uint8)


def reproj_image_backward_into(t, s, d, mask_u8, stats, gl, sign: float, ps: int, gtgt, gsrc):
    """Enqueues the image gradients of the reprojection loss of validated inputs (include/az_stereo.h:
    az_reproj_loss_img_bwd): ``gtgt`` / ``gsrc`` (either may be None) are fully written, deterministically."""
    B, C, H, W = t.shape
    lx, ly = linspace_table(W, t.device), linspace_table(H, t.device)
    with torch.cuda.device(t.device):
        _lib.call("az_reproj_loss_img_bwd", _ptr(t), _ptr(s), _ptr(d), float(sign), _ptr(mask_u8), _ptr(lx), _ptr(ly),
                  int(ps), _ptr(stats), _ptr(gl), _ptr(gtgt), _ptr(gsrc), B, C, H, W, _stream(), batch=B)


class ReprojLossFn(torch.autograd.Function):
    """Masked MSE between ``tgt`` and ``apply_disparity(unfold(src), sign*disp)``
    (reprojection.py:81-96 for ps = 1, :99-118 for the patch loss).  Differentiable
    w.r.t. ``disp``, ``tgt`` and ``src`` (the image gradients are recomputed from the
    inputs, without the unfolded planes; DESIGN.md §4.14)."""

    @staticmethod
    @_fwd32
    def forward(ctx, tgt, src, disp, mask_u8, ps: int, sign: float, want_warped: bool):
        t, s, d = check_reproj_inputs(tgt, src, disp)
        if mask_u8 is not None and (mask_u8.dtype != torch.uint8 or tuple(mask_u8.shape) != tuple(d.shape)
                                    or mask_u8.device != t.device or not mask_u8.is_contiguous()):
            raise ValueError("reprojection loss: mask must be a contiguous uint8 [B,1,H,W] tensor on the images' device")
        if int(ps) < 1 or int(ps) % 2 != 1:
            raise ValueError("reprojection loss: ps must be odd")
        B, C, H, W = t.shape
        dev = t.device
        need_bwd = ctx.needs_input_grad[2]
        need_img = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        warped = torch.empty_like(t) if want_warped else None
        gpre = torch.empty_like(d) if need_bwd else None
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        stats = torch.empty((2,), dtype=torch.float64, device=dev)
        ws = torch.empty((_lib.query("az_reproj_workspace_bytes", B, H),), dtype=torch.uint8, device=dev)
        lx, ly = linspace_table(W, dev), linspace_table(H, dev)
        with torch.cuda.device(dev):
            _lib.call("az_reproj_loss_fwd", _ptr(t), _ptr(s), _ptr(d), float(sign), _ptr(mask_u8), _ptr(lx), _ptr(ly),
                      int(ps), _ptr(warped), _ptr(gpre), _ptr(loss), _ptr(stats), _ptr(ws), B, C, H, W, _stream(), batch=B)
        if B == 0:  # F.mse_loss of nothing (reprojection.py:118 on an empty batch) is NaN
            loss.fill_(float("nan"))
            stats.zero_()
        if need_bwd or need_img:
            ctx.save_for_backward(gpre, stats, *((t, s, d, mask_u8) if need_img else (None,) * 4))
        ctx.meta = (B, C, H, W, int(ps), float(sign))
        if warped is not None:
            ctx.mark_non_differentiable(warped)
        return loss.reshape(()), warped

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gloss, _gwarped):
        gpre, stats, t, s, d, mask_u8 = ctx.saved_tensors
        B, C, H, W, ps, sign = ctx.meta
        gl = gloss.reshape(1).to(torch.float32).contiguous()
        gdisp = gtgt = gsrc = None
        if ctx.needs_input_grad[2]:
            gdisp = torch.empty_like(gpre)
            with torch.cuda.device(gpre.device):
                _lib.call("az_reproj_loss_bwd", _ptr(gpre), _ptr(stats), _ptr(gl), sign, _ptr(gdisp), B, C, H, W, ps,
                          _stream(), batch=B)
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            gtgt = torch.empty_like(t) if ctx.needs_input_grad[0] else None  # fully written by the kernels
            gsrc = torch.empty_like(s) if ctx.needs_input_grad[1] else None
            reproj_image_backward_into(t, s, d, mask_u8, stats, gl, sign, ps, gtgt, gsrc)
        return gtgt, gsrc, gdisp, None, None, None, None


def reproj_loss(tgt, src, disp, mask=None, ps: int = 1, sign: float = -1.0, want_warped: bool = False):
    """-> (loss 0-dim, warped [B,C,H,W] or None).  ``warped`` is the warped image for ps == 1 and
    the Fold visualisation image of get_reproj_error_patch for ps > 1 (same pass as the loss).
    Differentiable w.r.t. ``disp``, ``tgt`` and ``src`` (``warped`` is not differentiable).  The image
    gradients are deterministic; with an empty mask they are exactly zero (the loss is NaN)."""
    return ReprojLossFn.apply(tgt, src, disp, _mask_u8(mask, tgt), ps, sign, want_warped)


def patch_fold(src, disp, ps: int, sign: float = -1.0):
    """Fold of the warped unfolded planes, cropped (reprojection.py:120-125); no grad."""
    s = _cuda_f32(src.detach(), "src")
    d = _cuda_f32(disp.detach(), "disp")
    if s.dim() != 4 or d.dim() != 4 or tuple(d.shape) != (s.shape[0], 1, s.shape[2], s.shape[3]) or d.device != s.device:
        raise ValueError(f"patch_fold: src [B,C,H,W] and disp [B,1,H,W] on one device expected, got {tuple(s.shape)}, {tuple(d.shape)}")
    if int(ps) < 1 or int(ps) % 2 != 1:
        raise ValueError("patch_fold: ps must be odd")
    B, C, H, W = s.shape
    vis = torch.empty_like(s)
    lx, ly = linspace_table(W, s.device), linspace_table(H, s.device)
    with torch.cuda.device(s.device):
        _lib.call("az_patch_fold", _ptr(s), _ptr(d), float(sign), _ptr(lx), _ptr(ly), int(ps), _ptr(vis), B, C, H, W,
                  _stream(), batch=B)
    return vis


# ----------------------------------------------------------------------------
# a9: the bilinear rescalings of the multi-scale loss (reprojection.py:153-158), one launch per scale
# ----------------------------------------------------------------------------
class _RescaleDispFn(torch.autograd.Function):
    """disp_rs = F.interpolate(disp, scale_factor=r, mode="bilinear") * r together with the rescaled images and
    mask (non-differentiable outputs); gradient w.r.t. disp through the deterministic adjoint kernel."""

    @staticmethod
    @_fwd32
    def forward(ctx, disp, tgt, src, mask_u8, r: float):
        t, s, d = check_reproj_inputs(tgt, src, disp, "rescale")
        B, C, H, W = t.shape
        Ho, Wo = int(H * r), int(W * r)  # torch: floor(in * scale_factor)
        if Ho < 1 or Wo < 1 or r > 1.0:
            raise ValueError("rescale: 0 < r <= 1 with a non-empty output expected")
        inv = 1.0 / float(r)
        dev = t.device
        t_o = torch.empty((B, C, Ho, Wo), dtype=torch.float32, device=dev)
        s_o = torch.empty_like(t_o)
        d_o = torch.empty((B, 1, Ho, Wo), dtype=torch.float32, device=dev)
        m_o = torch.empty((B, 1, Ho, Wo), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.call("az_bilinear_rescale_fwd", _ptr(t), _ptr(s), _ptr(d), _ptr(mask_u8), _ptr(t_o), _ptr(s_o), _ptr(d_o),
                      _ptr(m_o), B, C, H, W, Ho, Wo, inv, inv, float(r), _stream(), batch=B)
        ctx.meta = (B, H, W, Ho, Wo, inv, float(r))
        ctx.mark_non_differentiable(t_o, s_o, m_o)
        return d_o, t_o, s_o, m_o

    @staticmethod
    @once_differentiable
    @_bwd
    def backward(ctx, gd, _gt, _gs, _gm):
        B, H, W, Ho, Wo, inv, r = ctx.meta
        g = _cuda_f32(gd, "grad_disp_rs")
        gin = torch.empty((B, 1, H, W), dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            _lib.call("az_bilinear_rescale_bwd", _ptr(g), _ptr(gin), B, H, W, Ho, Wo, inv, inv, r, _stream(), batch=B)
        return gin, None, None, None, None


def rescale_for_loss(tgt, src, disp, mask, r: float):
    """-> (tgt_rs, src_rs, disp_rs, mask_rs bool): the four ``F.interpolate(..., scale_factor=r, mode="bilinear")``
    of reprojection.py:153-158 (disp additionally multiplied by r) in one kernel; differentiable w.r.t. disp."""
    if tgt.requires_grad or src.requires_grad:
        raise ValueError("rescale_for_loss is differentiable w.r.t. disp only")
    d_o, t_o, s_o, m_o = _RescaleDispFn.apply(disp, tgt, src, _mask_u8(mask, tgt), float(r))
    return t_o, s_o, d_o, m_o.view(torch.bool)


# ----------------------------------------------------------------------------
# a10 scatter warp, a11 temporal IR, a12 LCN (non-differentiable)
# ----------------------------------------------------------------------------
def scatter_warp(img, disp, check_sign: bool = True):
    """apply_disparity_cu (utils/warp_ops.py:55-95).  ``check_sign`` keeps the
    reference's assertion that the disparities do not mix signs (one 4-byte
    device->host read instead of the reference's two full reductions)."""
    assert img.is_contiguous() and disp.is_contiguous()
    assert img.device.type == disp.device.type == "cuda"
    assert disp.dtype == torch.int
    if img.dtype != torch.float32:
        raise ValueError("apply_disparity_cu: img must be float32")
    if img.dim() != 4 or img.device != disp.device:
        raise ValueError("apply_disparity_cu: img [N,C,H,W] and disp on the same device expected")
    N, C, H, W = img.shape
    if disp.numel() != N * H * W:
        raise ValueError("apply_disparity_cu: disp must be [N,H,W] or [N,1,H,W]")
    out = torch.empty_like(img)
    flags = torch.zeros((1,), dtype=torch.int32, device=img.device) if check_sign else None
    with torch.cuda.device(img.device):
        _lib.call("az_scatter_warp", _ptr(img), _ptr(disp), _ptr(out), _ptr(flags), N, C, H, W, _stream(), batch=N)
    if check_sign:
        assert int(flags.item()) != 3, "disparities must be all >= 0 or all <= 0"
    return out


def scatter_warp_gt(disp_r_2x, max_disp: float, check_sign: bool = True):
    """The trainer's ground-truth chain in one launch (/root/reference/train.py:255-272): nearest x0.5 of the
    double-resolution right-view disparity, ``.type(torch.int)``, ``apply_disparity_cu`` with the disparity as its own
    payload, and the mask ``0 < disp_gt_l < max_disp``.  [N,1,2H,2W] float32 -> (disp_gt_l [N,1,H,W] float32,
    mask [N,1,H,W] bool)."""
    if not isinstance(disp_r_2x, torch.Tensor) or not disp_r_2x.is_cuda or disp_r_2x.dtype != torch.float32:
        raise ValueError("scatter_warp_gt: expected a float32 CUDA tensor")
    if disp_r_2x.dim() != 4 or disp_r_2x.shape[1] != 1 or disp_r_2x.shape[2] < 2 or disp_r_2x.shape[3] < 2:
        raise ValueError("scatter_warp_gt: expected [N,1,2H,2W]")
    d = disp_r_2x.contiguous()
    N, _, H2, W2 = d.shape
    H, W = H2 // 2, W2 // 2
    out = torch.empty((N, 1, H, W), dtype=torch.float32, device=d.device)
    mask = torch.empty((N, 1, H, W), dtype=torch.uint8, device=d.device)
    flags = torch.zeros((1,), dtype=torch.int32, device=d.device) if check_sign else None
    with torch.cuda.device(d.device):
        _lib.call("az_scatter_warp_gt", _ptr(d), _ptr(out), _ptr(mask), _ptr(flags), float(max_disp), N, H2, W2, _stream(), batch=N)
    if check_sign:
        assert int(flags.item()) != 3, "disparities must be all >= 0 or all <= 0"
    return out, mask.view(torch.bool)


def temporal_ir_pattern(frames, ks: int = 11, threshold: float = 0.005):
    """[B,T,H,W] or [T,H,W] uint8 -> [B,H,W] / [H,W] float32 {0,1}
    (tools/temporal_ir.py:93-114)."""
    if not frames.is_cuda or frames.dtype != torch.uint8:
        raise ValueError("temporal_ir_pattern: expected a CUDA uint8 tensor")
    squeeze = frames.dim() == 3
    f = (frames.unsqueeze(0) if squeeze else frames).contiguous()
    if f.dim() != 4:
        raise ValueError("temporal_ir_pattern: [T,H,W] or [B,T,H,W] expected")
    B, T, H, W = f.shape
    pat = torch.empty((B, H, W), dtype=torch.float32, device=f.device)
    ws = torch.empty((_lib.query("az_temporal_ir_workspace_bytes", B, H, W),), dtype=torch.uint8, device=f.device)
    with torch.cuda.device(f.device):
        _lib.call("az_temporal_ir", _ptr(f), _ptr(pat), _ptr(ws), B, T, H, W, int(ks), float(threshold), _stream(), batch=B)
    return pat[0] if squeeze else pat


def local_contrast_norm(image, kernel_size: int = 9, eps: float = 1e-5):
    """utils/reprojection.py:175-200 -> (normed [B,1,H,W], std [B,1,H,W])."""
    assert kernel_size % 2 == 1, "Kernel size should be odd"
    if image.requires_grad:
        # the reference's LCN is ordinary autograd code; this kernel is forward-only (the trainer normalises data)
        raise ValueError("local_contrast_norm: the CUDA operator is not differentiable; detach the image first")
    im = _cuda_f32(image.detach(), "image")
    if im.dim() != 4:
        raise ValueError("local_contrast_norm: image must be [B,C,H,W]")
    B, Cin, H, W = im.shape
    normed = torch.empty((B, 1, H, W), dtype=torch.float32, device=im.device)
    std = torch.empty_like(normed)
    with torch.cuda.device(im.device):
        _lib.call("az_local_contrast_norm", _ptr(im), _ptr(normed), _ptr(std), B, Cin, H, W, int(kernel_size),
                  float(eps), _stream(), batch=B)
    return normed, std


def error_metric_sums(disp_gt, depth_gt, disp_pred, mask, depth_pred=None, focal_length=None, baseline=None):
    """The eight masked sums behind compute_err_metric (utils/cascade_metrics.py:16-57) as ONE
    float64[8] device tensor: n, sum|ddisp|, #>1, #>2, sum clip(|dz*1000|,0,100), #dz>2mm, #>4mm, #>8mm."""
    dg = _cuda_f32(disp_gt.detach(), "disp_gt")
    zg = _cuda_f32(depth_gt.detach(), "depth_gt")
    dp = _cuda_f32(disp_pred.detach(), "disp_pred")
    if dg.dim() != 4 or dg.shape[1] != 1 or zg.shape != dg.shape or dp.shape != dg.shape \
            or not (dg.device == zg.device == dp.device):
        raise ValueError("error metrics: disp_gt, depth_gt, disp_pred must all be [B,1,H,W] on one device")
    B, _, H, W = dg.shape
    m = _mask_u8(mask, dg)
    zp = f = bl = None
    if depth_pred is not None:
        zp = _cuda_f32(depth_pred.detach(), "depth_pred")
        if zp.shape != dg.shape or zp.device != dg.device:
            raise ValueError("error metrics: depth_pred must be [B,1,H,W] like disp_gt, on the same device")
    else:
        f = _cuda_f32(focal_length.detach().reshape(-1), "focal_length")
        bl = _cuda_f32(baseline.detach().reshape(-1), "baseline")
        if f.numel() != B or bl.numel() != B:
            raise ValueError("error metrics: focal_length and baseline must hold one value per sample")
    out = torch.empty((8,), dtype=torch.float64, device=dg.device)
    ws = torch.empty((_lib.query("az_error_metrics_workspace_bytes", B, H, W),), dtype=torch.uint8, device=dg.device)
    with torch.cuda.device(dg.device):
        _lib.call("az_error_metrics", _ptr(dg), _ptr(zg), _ptr(dp), _ptr(zp), _ptr(f), _ptr(bl), _ptr(m), _ptr(out),
                  _ptr(ws), B, H, W, _stream(), batch=B)
    if B == 0:
        out.zero_()  # no pixel selected: compute_err_metric then reports NaN like torch.mean of nothing
    return out


def sim_ir_pattern(img_ir, img_no_ir, ks: int = 11, threshold: float = 0.005):
    """get_smoothed_ir_pattern2 (ks > 0) / get_ir_pattern (ks = 0) of datasets/dataset_utils.py on the
    GPU.  Inputs: CUDA uint8 (raw grey levels) or float64 (already /255) tensors [H,W] or [B,H,W]."""
    if not (img_ir.is_cuda and img_no_ir.is_cuda) or img_ir.shape != img_no_ir.shape or img_ir.dtype != img_no_ir.dtype:
        raise ValueError("sim_ir_pattern: two CUDA tensors of the same shape and dtype expected")
    if img_ir.dtype not in (torch.uint8, torch.float64):
        raise ValueError("sim_ir_pattern: uint8 or float64 images expected (the reference computes in float64)")
    squeeze = img_ir.dim() == 2
    a = (img_ir.unsqueeze(0) if squeeze else img_ir).contiguous()
    b = (img_no_ir.unsqueeze(0) if squeeze else img_no_ir).contiguous()
    if a.dim() != 3:
        raise ValueError("sim_ir_pattern: [H,W] or [B,H,W] expected")
    B, H, W = a.shape
    pat = torch.empty((B, H, W), dtype=torch.float32, device=a.device)
    ws = torch.empty((_lib.query("az_sim_ir_pattern_workspace_bytes", B, H, W, int(ks)),), dtype=torch.uint8,
                     device=a.device)
    with torch.cuda.device(a.device):
        _lib.call("az_sim_ir_pattern", _ptr(a), _ptr(b), 1 if a.dtype == torch.uint8 else 0, _ptr(pat), _ptr(ws),
                  B, H, W, int(ks), float(threshold), _stream(), batch=B)
    return pat[0] if squeeze else pat
