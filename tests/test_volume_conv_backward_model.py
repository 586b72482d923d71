"""CPU: the volume-free backward of conv3d(concat_volume(L, R, Dq), W, padding=1) (csrc/volume_conv_bwd.cu), restated
in float64 in the kernels' reduction and index order, against autograd of F.conv3d on the oracle's materialised
volume; and the fake (meta) kernels and autograd wiring of az_stereo::volume_conv / volume_conv_backward."""
import math

import pytest
import torch
import torch.nn.functional as F
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import library_ops  # noqa: F401  (importing registers the ops)
from oracle import stereo_oracle as so


def reduce_planes(g):
    """Kernel 1 (vcb_reduce_kernel): A[kd][kx], Z[kd][kx], each [B,O,H,W]."""
    B, O, Dq, H, W = g.shape
    zero = g.new_zeros(B, O, H)
    A = [[None] * 3 for _ in range(3)]
    Z = [[None] * 3 for _ in range(3)]
    for kd in range(3):
        for kx in range(3):
            A[kd][kx], Z[kd][kx] = g.new_zeros(B, O, H, W), g.new_zeros(B, O, H, W)
    # the shared core diagonal Dg(v), v = -2 .. W+1
    dg = {}
    for v in range(-2, W + 2):
        acc = zero
        for d in range(max(1, -v), min(Dq - 2, W - 2 - v) + 1):
            acc = acc + g[:, :, d, :, v + d]
        dg[v] = acc
    for x in range(W):
        g0 = g[:, :, 0, :, x]
        gl = g[:, :, Dq - 1, :, x] if Dq >= 2 else zero
        M, snap = zero, []
        for d in range(1, min(x - 3, Dq - 2) + 1):
            M = M + g[:, :, d, :, x]
        for k in range(5):
            e = x + k - 2
            if 1 <= e <= Dq - 2:
                M = M + g[:, :, e, :, x]
            snap.append(M)
        for kd in range(3):
            for kx in range(3):
                s = kx - kd
                m = snap[s + 2]
                last = gl if x + s >= Dq - 1 else zero
                if kd == 0:
                    a = m + last
                elif kd == 1:
                    a = (g0 + m) + last if x + s >= 0 else zero
                else:
                    a = g0 + m if (x + s >= 0 and Dq >= 2) else zero
                A[kd][kx][:, :, :, x] = a
                t, xmax = kd - kx, W - 1 - (1 if kx == 2 else 0)
                v = x + t
                z = dg[v]
                if (kd == 1 or (kd == 2 and Dq >= 2)) and 0 <= v <= xmax:
                    z = z + g[:, :, 0, :, v]
                vl = v + Dq - 1
                if kd <= 1 and Dq >= 2 and 0 <= vl <= xmax:
                    z = z + g[:, :, Dq - 1, :, vl]
                dw = W - 1 - v
                if kx <= 1 and 1 <= dw <= Dq - 2:
                    z = z + g[:, :, dw, :, W - 1]
                Z[kd][kx][:, :, :, x] = z
    return A, Z


def shifted(P, ky, sx):
    """S[b,o,y',x'] = P[b,o,y'-ky+1,x'+sx], zero outside the image."""
    B, O, H, W = P.shape
    S = torch.zeros_like(P)
    for yp in range(H):
        yy = yp - ky + 1
        if not 0 <= yy < H:
            continue
        for xp in range(W):
            xx = xp + sx
            if 0 <= xx < W:
                S[:, :, yp, xp] = P[:, :, yy, xx]
    return S


def decomposed_backward(L, R, Wt, g, chunks=64):
    B, C, H, W = L.shape
    A, Z = reduce_planes(g)
    dL, dR, dW = torch.zeros_like(L), torch.zeros_like(R), torch.zeros_like(Wt)
    rpc = math.ceil(B * H / chunks)
    for h, (planes, feat, dfeat) in enumerate(((A, L, dL), (Z, R, dR))):
        for kd in range(3):
            for kx in range(3):
                sx = 1 - kx if h == 0 else 0
                for ky in range(3):
                    S = shifted(planes[kd][kx], ky, sx)
                    # kernel 2 (vcb_dfeat_kernel): sum over (kd, kx, ky, o)
                    dfeat += torch.einsum("oc,boyx->bcyx", Wt[:, h * C:(h + 1) * C, kd, ky, kx], S)
                    # kernels 3 + 4 (vcb_wgrad_kernel, finalize): per-chunk partials over image rows, added in chunk order
                    Sr = S.permute(0, 2, 1, 3).reshape(B * H, -1, W)
                    Fr = feat.permute(0, 2, 1, 3).reshape(B * H, C, W)
                    acc = torch.zeros_like(Wt[:, :C, 0, 0, 0])
                    for r0 in range(0, B * H, rpc):
                        acc = acc + torch.einsum("rox,rcx->oc", Sr[r0:r0 + rpc], Fr[r0:r0 + rpc])
                    dW[:, h * C:(h + 1) * C, kd, ky, kx] = acc
    return dL, dR, dW


@pytest.mark.parametrize("B,C,H,W,Dq,O", [(2, 3, 4, 9, 5, 4), (1, 2, 3, 4, 6, 3), (1, 2, 2, 12, 1, 2), (1, 1, 3, 7, 7, 2),
                                          (1, 2, 1, 6, 3, 3), (2, 2, 3, 2, 4, 2), (1, 1, 1, 1, 2, 2), (1, 2, 2, 11, 4, 2)])
def test_decomposition_matches_autograd_of_conv3d(B, C, H, W, Dq, O):
    """Covers Dq > W, Dq = 1, Dq = 2, H = 1 and W < 3."""
    torch.manual_seed(B * 1000 + H * 100 + W * 10 + Dq)
    L = torch.randn(B, C, H, W, dtype=torch.float64, requires_grad=True)
    R = torch.randn(B, C, H, W, dtype=torch.float64, requires_grad=True)
    Wt = torch.randn(O, 2 * C, 3, 3, 3, dtype=torch.float64, requires_grad=True)
    out = F.conv3d(so.concat_volume(L, R, Dq), Wt, padding=1)
    g = torch.randn_like(out)
    out.backward(g)
    for chunks in (64, 1):  # one partial per image row, and one partial for everything
        dL, dR, dW = decomposed_backward(L.detach(), R.detach(), Wt.detach(), g, chunks)
        for mine, ref in ((dL, L.grad), (dR, R.grad), (dW, Wt.grad)):
            torch.testing.assert_close(mine, ref, rtol=1e-11, atol=1e-11)


# ------------------------------------------------------------------------------ torch.library registration (fake)
B, C, H, W, Dq = 2, 32, 6, 20, 5


def test_volume_conv_ops_are_registered_with_autograd():
    for name in ("volume_conv", "volume_conv_backward"):
        op = getattr(torch.ops.az_stereo, name).default
        assert op._schema.name == f"az_stereo::{name}" and not op._schema.is_mutable
    from activezero_b200 import _volume_conv_library as vcl

    assert vcl.volume_conv._backward_fn is not None and vcl.volume_conv._setup_context_fn is not None
    assert vcl.volume_conv_backward._backward_fn is None  # once-differentiable backward


def test_volume_conv_fake_kernels_describe_the_outputs():
    ns = torch.ops.az_stereo
    with FakeTensorMode():
        L = torch.empty(B, C, H, W, device="cuda")
        w = torch.empty(32, 64, 3, 3, 3, device="cuda")
        out = ns.volume_conv(L, L, w, Dq)
        assert (tuple(out.shape), out.dtype) == ((B, 32, Dq, H, W), torch.float32)
        grads = ns.volume_conv_backward(torch.empty(B, 32, Dq, H, W, device="cuda"), L, L, w)
        assert [(tuple(t.shape), t.dtype) for t in grads] == [((B, C, H, W), torch.float32)] * 2 + [((32, 64, 3, 3, 3), torch.float32)]


def test_volume_conv_autograd_graph_builds_on_meta_tensors():
    L = torch.empty(B, C, H, W, device="meta", requires_grad=True)
    R = torch.empty(B, C, H, W, device="meta", requires_grad=True)
    w = torch.empty(32, 64, 3, 3, 3, device="meta", requires_grad=True)
    out = torch.ops.az_stereo.volume_conv(L, R, w, Dq)
    grads = torch.autograd.grad(out.sum(), [L, R, w])
    assert [tuple(t.shape) for t in grads] == [tuple(t.shape) for t in (L, R, w)]
