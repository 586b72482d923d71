"""CPU: the image gradients of the fused reprojection loss (DESIGN.md §4.14, include/az_stereo.h:
az_reproj_loss_img_bwd) restated in float64 loops -- the gather that gives gtgt and the per-row entry table and
corner splat that give gsrc, with the kernels' border rules -- against torch autograd of the oracle's
reprojection.py:99-127.  The oracle is evaluated at the kernels' fp32 x positions and the model at the oracle's row
positions, so that only the formulas differ.  Also the fake kernel and the registration of ``az_stereo::reproj_loss_image_backward``."""
import numpy as np
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import library_ops as lo  # noqa: F401  (importing registers the ops)
from oracle import stereo_oracle as so


def _positions(d, sign, H, W):
    """fp32 x positions as the kernels form them, the float64 disparity that makes the oracle's
    apply_disparity(., -disp) sample at exactly those positions, and the oracle's own float64 row positions."""
    xs, _ = so.sample_coords(sign * d, H, W, torch.float32)
    _, ys = so.sample_coords(sign * d, H, W, torch.float64)
    lin = torch.linspace(0, 1, W).double().view(1, 1, W)
    pred = -(xs.double() + 0.5 - lin * W)
    return xs.double().numpy(), ys[0, :, 0].numpy(), pred[:, None]


def _axis(pos, size):
    fl = np.floor(pos)
    w = pos - fl
    return int(fl), 1.0 - w, w, 0 <= fl <= size - 1, -1 <= fl <= size - 2


def _model(L, R, xs, ys, m, ps, gl=1.0):
    """float64 restatement of the two kernels' formulas."""
    B, C, H, W = L.shape
    p = (ps - 1) // 2
    K = C * ps * ps
    msum = m.sum()
    gtgt, gsrc = np.zeros_like(L), np.zeros_like(R)
    if msum == 0:
        return gtgt, gsrc
    s = gl * 2.0 / (K * msum)

    def src(b, c, y, x):
        return R[b, c, y, x] if 0 <= y < H and 0 <= x < W else 0.0

    def tgt(b, c, y, x):
        return L[b, c, y, x] if 0 <= y < H and 0 <= x < W else 0.0

    def wu(b, c, i, j, ky, kx):
        y0, ay0, ay1, vy0, vy1 = _axis(ys[i], H)
        x0, bx0, bx1, vx0, vx1 = _axis(xs[b, i, j], W)
        ay0, ay1, bx0, bx1 = ay0 * vy0, ay1 * vy1, bx0 * vx0, bx1 * vx1
        r0, xa = y0 + ky - p, x0 + kx - p
        return (ay0 * (bx0 * src(b, c, r0, xa) + bx1 * src(b, c, r0, xa + 1))
                + ay1 * (bx0 * src(b, c, r0 + 1, xa) + bx1 * src(b, c, r0 + 1, xa + 1)))

    for b in range(B):
        for c in range(C):
            # gtgt: gather over the taps that read tgt[y, x]
            for y in range(H):
                for x in range(W):
                    acc = 0.0
                    for ky in range(ps):
                        for kx in range(ps):
                            i, j = y + p - ky, x + p - kx
                            if 0 <= i < H and 0 <= j < W and m[b, i, j]:
                                acc += wu(b, c, i, j, ky, kx) - L[b, c, y, x]
                    gtgt[b, c, y, x] = -s * acc
            # gsrc: per output row Y the entries (ky, a) -> source row i with y0(i) = Y-a-ky+p, then the splat
            for Y in range(H):
                for ky in range(ps):
                    for a in (0, 1):
                        for i in range(H):
                            y0, ay0, ay1, vy0, vy1 = _axis(ys[i], H)
                            wy = (ay0 * vy0) if a == 0 else (ay1 * vy1)
                            if y0 != Y - a - ky + p or wy == 0:
                                continue
                            for j in range(W):
                                if not m[b, i, j]:
                                    continue
                                x0, bx0, bx1, vx0, vx1 = _axis(xs[b, i, j], W)
                                for kx in range(ps):
                                    r = wu(b, c, i, j, ky, kx) - tgt(b, c, i + ky - p, j + kx - p)
                                    for bb, wx, v in ((0, bx0, vx0), (1, bx1, vx1)):
                                        X = x0 + bb + kx - p
                                        if v and 0 <= X < W:
                                            gsrc[b, c, Y, X] += s * r * wy * wx
    return gtgt, gsrc


@pytest.mark.parametrize("B,C,H,W,ps,field,masked,sign", [
    (1, 1, 6, 9, 3, "random", True, -1.0), (2, 1, 5, 7, 5, "wild", True, -1.0), (1, 2, 7, 6, 3, "wild", False, 1.0),
    (1, 1, 4, 3, 5, "random", True, 1.0), (1, 1, 5, 8, 1, "wild", True, -1.0), (1, 1, 3, 4, 7, "wild", False, -1.0)])
def test_gather_and_splat_formulas_match_oracle_autograd(B, C, H, W, ps, field, masked, sign):
    gen = torch.Generator().manual_seed(B * 100 + H * 10 + W + ps)
    L = torch.rand(B, C, H, W, generator=gen, dtype=torch.float64)
    R = torch.rand(B, C, H, W, generator=gen, dtype=torch.float64)
    scale = W / 3 if field == "random" else 3.0 * W
    off = 0.0 if field == "random" else 0.5
    d = ((torch.rand(B, 1, H, W, generator=gen) - off) * scale).float()
    m = (torch.rand(B, 1, H, W, generator=gen) > 0.3) if masked else torch.ones(B, 1, H, W, dtype=torch.bool)
    xs, ys, pred = _positions(d, sign, H, W)
    Lg, Rg = L.clone().requires_grad_(True), R.clone().requires_grad_(True)
    loss, _, _ = so.reproj_error_patch(Lg, Rg, pred, m if masked else None, ps=ps)
    (0.7 * loss).backward()
    gtgt, gsrc = _model(L.numpy(), R.numpy(), xs, ys, m[:, 0].numpy(), ps, gl=0.7)
    np.testing.assert_allclose(gtgt, Lg.grad.numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(gsrc, Rg.grad.numpy(), rtol=1e-9, atol=1e-12)


def test_empty_mask_gives_zero_image_gradients():
    L = np.random.rand(1, 1, 4, 5)
    xs, ys, _ = _positions(torch.ones(1, 1, 4, 5), -1.0, 4, 5)
    gtgt, gsrc = _model(L, L, xs, ys, np.zeros((1, 4, 5), bool), 3)
    assert not gtgt.any() and not gsrc.any()


def test_image_backward_op_is_registered_with_a_fake_kernel():
    op = torch.ops.az_stereo.reproj_loss_image_backward.default
    assert op._schema.name == "az_stereo::reproj_loss_image_backward" and not op._schema.is_mutable
    with FakeTensorMode():
        t = torch.empty(2, 3, 8, 12, device="cuda")
        d = torch.empty(2, 1, 8, 12, device="cuda")
        stats = torch.empty(2, device="cuda", dtype=torch.float64)
        for mask in (None, torch.empty(2, 1, 8, 12, device="cuda", dtype=torch.bool)):
            gt, gs = torch.ops.az_stereo.reproj_loss_image_backward(t, t, d, mask, stats, torch.empty((), device="cuda"),
                                                                    -1.0, 11)
            assert tuple(gt.shape) == tuple(gs.shape) == (2, 3, 8, 12) and gt.dtype == gs.dtype == torch.float32


def test_reproj_loss_autograd_gives_image_gradients_on_meta():
    """The library op's autograd formula returns gradients of the images' shapes (through the new op's fake
    kernel), also when only one image requires grad."""
    img = torch.empty(2, 3, 8, 12, device="meta", requires_grad=True)
    src = torch.empty(2, 3, 8, 12, device="meta", requires_grad=True)
    disp = torch.empty(2, 1, 8, 12, device="meta", requires_grad=True)
    mask = torch.empty(2, 1, 8, 12, device="meta", dtype=torch.bool)
    loss, _, _, _ = torch.ops.az_stereo.reproj_loss(img, src, disp, mask, 5, -1.0)
    grads = torch.autograd.grad(loss, [img, src, disp])
    assert [tuple(g.shape) for g in grads] == [(2, 3, 8, 12), (2, 3, 8, 12), (2, 1, 8, 12)]
    loss2, _, _, _ = torch.ops.az_stereo.reproj_loss(img.detach(), src, disp, mask, 5, -1.0)
    (gs,) = torch.autograd.grad(loss2, [src])
    assert tuple(gs.shape) == (2, 3, 8, 12)
