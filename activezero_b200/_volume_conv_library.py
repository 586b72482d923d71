"""``torch.library`` registration of the differentiable implicit-volume convolution (``ops.volume_conv``):

    torch.ops.az_stereo.volume_conv(ref, tgt, weight, num_disp) -> out                     (psmnet.py:151-168)
    torch.ops.az_stereo.volume_conv_backward(gout, ref, tgt, weight) -> (gref, gtgt, gweight)

Both take the dtypes ``ops.volume_conv`` takes (float32, or bfloat16 / float16 features with a float32 weight or one
of their dtype); the fake kernels follow ``ref`` and ``weight`` for the dtypes of the results.

``library_ops`` imports this module, so importing ``library_ops`` registers both operators.  They live in a module of
their own so that the operator set defined in ``library_ops`` itself (pinned by tests/test_library_ops_fake.py) stays
the inference / loss path's.
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import Tensor

from .ops import _cuda_f32, check_volume_conv_inputs, volume_conv_backward_into, volume_conv_forward

NS = "az_stereo"


@torch.library.custom_op(f"{NS}::volume_conv", mutates_args=(), device_types="cuda")
def volume_conv(ref: Tensor, tgt: Tensor, weight: Tensor, num_disp: int) -> Tensor:
    L, R, w = check_volume_conv_inputs(ref, tgt, weight, num_disp, "az_stereo::volume_conv")
    return volume_conv_forward(L, R, w, num_disp)


@volume_conv.register_fake
def _(ref, tgt, weight, num_disp):
    B, _, H, W = ref.shape
    return ref.new_empty((B, 32, num_disp, H, W))


@torch.library.custom_op(f"{NS}::volume_conv_backward", mutates_args=(), device_types="cuda")
def volume_conv_backward(gout: Tensor, ref: Tensor, tgt: Tensor, weight: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    g = _cuda_f32(gout, "grad_out", allow16=True)
    if g.dim() != 5:
        raise ValueError("az_stereo::volume_conv_backward: gout must be [B,32,Dq,H,W]")
    L, R, w = check_volume_conv_inputs(ref, tgt, weight, int(g.shape[2]), "az_stereo::volume_conv_backward")
    gL, gR, gW = torch.empty_like(L), torch.empty_like(R), torch.empty_like(w)
    volume_conv_backward_into(g, L, R, w, gL, gR, gW)
    return gL, gR, gW


@volume_conv_backward.register_fake
def _(gout, ref, tgt, weight):
    return torch.empty_like(ref), torch.empty_like(tgt), torch.empty_like(weight)


def _vc_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1], inputs[2])


def _vc_backward(ctx, gout):
    ref, tgt, weight = ctx.saved_tensors
    gL, gR, gW = volume_conv_backward(gout, ref, tgt, weight)
    return gL, gR, gW, None


volume_conv.register_autograd(_vc_backward, setup_context=_vc_setup)
