"""Drop-in for ``/root/reference/utils/reprojection.py``.

Same function names, argument meaning and return tuples; the bodies route to the
fused CUDA operators of ``activezero_b200.ops`` instead of materialising the
``Unfold`` / ``grid_sample`` / boolean-gather intermediates.  ``utils/losses.py``
of the reference can import this module unchanged.
"""
import torch
import torch.nn.functional as F

from .. import ops
from .warp_ops import apply_disparity_cu

# get_reproj_error_patch returns the Fold of the warped patches for TensorBoard
# only (utils/losses.py / train.py:321-338).  It is computed by default to keep
# the reference's return contract; a training loop that logs images every N
# steps can switch it off in between (the second tuple element is then None).
RETURN_WARPED_PATCH_IMAGE = True


def apply_disparity(img, disp):
    """reprojection.py:13-35: pull ``img`` by ``disp`` (bilinear, zeros padding)."""
    return ops.warp(img, disp)


def _int_mask(mask, like):
    # reprojection.py:91-96, 113-127: mask.repeat(1,C,1,1).type(torch.int), or all ones
    B, C, H, W = like.shape
    if mask is None:
        return torch.ones((B, C, H, W), dtype=torch.int, device=like.device)
    return mask.repeat(1, C, 1, 1).type(torch.int)


def _masked_loss(tgt, src, disp, mask, ps, sign):
    """(loss, warped-or-None).  Fused kernel when only the disparity needs a
    gradient; if an image requires grad (never the case for IR patterns) the
    loss is composed from the differentiable warp kernel instead."""
    if ps == 1 and (tgt.requires_grad or src.requires_grad):
        warped = ops.warp(src, disp if sign > 0 else -disp)
        C = tgt.shape[1]
        sel = (mask.repeat(1, C, 1, 1) if mask is not None else torch.ones_like(warped).type(torch.bool))
        return F.mse_loss(warped[sel], tgt[sel]), warped
    return ops.reproj_loss(tgt, src, disp, mask, ps=ps, sign=sign, want_warped=(ps == 1))


def get_reprojection_error(input_L, input_R, pred_disp_l, pred_disp_r, mask_l=None, mask_r=None):
    """reprojection.py:38-78 (bidirectional)."""
    if mask_l is None:
        # reprojection.py:50-65: occlusion masks from the integer scatter warp
        disp_gt_l = apply_disparity_cu(pred_disp_r.detach().contiguous(), pred_disp_r.detach().type(torch.int).contiguous())
        disp_gt_r = apply_disparity_cu(pred_disp_l.detach().contiguous(), (-pred_disp_l.detach().type(torch.int)).contiguous())
        mask_l = ((disp_gt_l < 192) * (disp_gt_l > 0)).detach()
        mask_r = ((disp_gt_r < 192) * (disp_gt_r > 0)).detach()
    loss_l, warped_l = _masked_loss(input_L, input_R, pred_disp_l, mask_l, 1, -1.0)
    loss_r, warped_r = _masked_loss(input_R, input_L, pred_disp_r, mask_r, 1, +1.0)
    return loss_l, loss_r, warped_l, warped_r, _int_mask(mask_l, input_L), _int_mask(mask_r, input_R)


def get_reprojection_error_old(input_L, input_R, pred_disp_l, mask=None):
    """reprojection.py:81-96."""
    loss, warped = _masked_loss(input_L, input_R, pred_disp_l, mask, 1, -1.0)
    return loss, warped, _int_mask(mask, input_L)


def get_reproj_error_patch(input_L, input_R, pred_disp_l, mask=None, ps=5):
    """reprojection.py:99-127 -- the loss the live trainer uses (ps = 11)."""
    assert ps % 2 == 1
    # An image that requires grad ("feature or image" in the reference's docstring) gets its gradient from the same
    # fused operator.  That call always asks for the Fold image: the x-tiled kernel that computes the loss together
    # with it is the one that stages the widest rows, so a wide input keeps working as it did under the reference's
    # autograd composition.
    img_grad = input_L.requires_grad or input_R.requires_grad
    loss, warped = ops.reproj_loss(input_L, input_R, pred_disp_l, mask, ps=ps, sign=-1.0,
                                   want_warped=RETURN_WARPED_PATCH_IMAGE or img_grad)
    return loss, (warped if RETURN_WARPED_PATCH_IMAGE else None), _int_mask(mask, input_L)


def get_reprojection_error_diff_ratio(input_L, input_R, pred_disp_l, mask=None):
    """reprojection.py:130-173: three scales.  Per scale ONE kernel produces the four bilinear rescalings
    (:153-158) and one fused kernel the warp + masked MSE; an image that requires grad takes torch's
    F.interpolate + the differentiable warp instead."""
    ratio = [0.25, 0.5, 1]
    weight = [0.3, 0.5, 0.2]
    # reprojection.py:142-148: the C mask planes are copies of one [B,1,H,W] plane, so are their rescalings
    output, loss_dict, total_loss = {}, {}, 0
    img_grad = input_L.requires_grad or input_R.requires_grad
    C = input_L.shape[1]
    for i, (r, w) in enumerate(zip(ratio, weight)):
        if img_grad:
            mf = (mask.repeat(1, C, 1, 1) if mask is not None else torch.ones_like(input_L)).type(torch.float32).detach()
            L_rs = F.interpolate(input_L, scale_factor=r, mode="bilinear")
            R_rs = F.interpolate(input_R, scale_factor=r, mode="bilinear")
            d_rs = F.interpolate(pred_disp_l, scale_factor=r, mode="bilinear") * r
            m_rs = F.interpolate(mf, scale_factor=r, mode="bilinear").type(torch.bool)
            warped = ops.warp(R_rs, -d_rs)
            loss = F.mse_loss(warped[m_rs], L_rs[m_rs])
        else:
            L_rs, R_rs, d_rs, m1 = ops.rescale_for_loss(input_L, input_R, pred_disp_l, mask, r)
            loss, warped = ops.reproj_loss(L_rs, R_rs, d_rs, m1, ps=1, sign=-1.0, want_warped=True)
            m_rs = m1.repeat(1, C, 1, 1)
        output[f"stage{i}"] = {"target": L_rs, "warped": warped, "pred_disp": d_rs, "mask": m_rs.type(torch.int)}
        loss_dict[f"stage{i}"] = loss.item()
        total_loss = total_loss + loss * w
    return total_loss, output, loss_dict


def local_contrast_norm(image, kernel_size=9, eps=1e-5):
    """reprojection.py:175-200 -> (normed_image, std), first channel only.  Forward-only kernel (the reference
    runs it on data inside the dataset, datasets/messytable.py:242-250); an image that requires grad takes the
    reference's own Unfold formulation so that the call stays differentiable."""
    if image.requires_grad:
        ks = kernel_size
        assert ks % 2 == 1, "Kernel size should be odd"
        b, _, h, w = image.shape
        img = image[:, :1]
        patches = torch.nn.Unfold(kernel_size=(ks, ks), padding=(ks - 1) // 2)(img).reshape(b, -1, h, w)
        mean, std = patches.mean(1, keepdim=True), patches.std(1, keepdim=True, unbiased=False)
        return (img - mean) / (std + eps), std
    return ops.local_contrast_norm(image, kernel_size=kernel_size, eps=eps)
