"""``torch.library`` registration of the image gradients of the fused reprojection loss (``ops.reproj_loss``):

    torch.ops.az_stereo.reproj_loss_image_backward(tgt, src, disp, mask, stats, gloss, sign, ps) -> (gtgt, gsrc)

``stats`` is the forward's float64[2] output and ``gloss`` the loss gradient; the gradients are recomputed from the
inputs (include/az_stereo.h: az_reproj_loss_img_bwd).  ``library_ops.reproj_loss``'s autograd formula calls it
when ``tgt`` or ``src`` requires grad.

``library_ops`` imports this module, so importing ``library_ops`` registers the operator.  It lives in a module of its
own so that the operator set defined in ``library_ops`` itself (pinned by tests/test_library_ops_fake.py) stays the
inference / loss path's.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from .ops import _mask_u8, check_reproj_inputs, reproj_image_backward_into

NS = "az_stereo"


@torch.library.custom_op(f"{NS}::reproj_loss_image_backward", mutates_args=(), device_types="cuda")
def reproj_loss_image_backward(tgt: Tensor, src: Tensor, disp: Tensor, mask: Optional[Tensor], stats: Tensor,
                               gloss: Tensor, sign: float, ps: int) -> Tuple[Tensor, Tensor]:
    t, s, d = check_reproj_inputs(tgt, src, disp, "az_stereo::reproj_loss_image_backward")
    m = _mask_u8(mask, t)
    if ps < 1 or ps % 2 != 1:
        raise ValueError("az_stereo::reproj_loss_image_backward: ps must be odd")
    if stats.numel() != 2 or stats.dtype != torch.float64 or stats.device != t.device or gloss.numel() != 1 \
            or gloss.device != t.device:
        raise ValueError("az_stereo::reproj_loss_image_backward: stats float64[2] and a one-element gloss on the "
                         "images' device expected")
    gl = gloss.reshape(1).to(torch.float32).contiguous()
    gtgt, gsrc = torch.empty_like(t), torch.empty_like(s)  # fully written by the kernels
    reproj_image_backward_into(t, s, d, m, stats.contiguous(), gl, float(sign), int(ps), gtgt, gsrc)
    return gtgt, gsrc


@reproj_loss_image_backward.register_fake
def _(tgt, src, disp, mask, stats, gloss, sign, ps):
    return torch.empty_like(tgt), torch.empty_like(src)
