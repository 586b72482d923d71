"""CPU: the fake (meta) kernels of the soft-argmin and fused-upsample operators with 16-bit logits describe what the
CUDA implementation returns (DESIGN.md §4.12): disp, lse and stats are float32, the logits' gradients keep the logits'
dtype.  Fake tensors only, so this runs without a GPU."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import library_ops  # noqa: F401  (importing registers the ops)

B, D, H, W = 2, 24, 8, 12
Dq, Hq, Wq = 6, 2, 3


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_soft_argmin_fakes_with_16_bit_logits(dtype):
    ns = torch.ops.az_stereo
    with FakeTensorMode():
        cost = torch.empty(B, D, H, W, device="cuda", dtype=dtype)
        disp, lse = ns.soft_argmin(cost)
        assert disp.dtype == lse.dtype == torch.float32
        assert tuple(disp.shape) == (B, 1, H, W) and tuple(lse.shape) == (B, 2, H, W)
        g = ns.soft_argmin_backward(cost, disp, lse, torch.empty_like(disp))
        assert g.dtype == dtype and tuple(g.shape) == (B, D, H, W)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("five_d", [False, True])
def test_upsample_soft_argmin_fakes_with_16_bit_logits(dtype, five_d):
    ns = torch.ops.az_stereo
    shape = (B, 1, Dq, Hq, Wq) if five_d else (B, Dq, Hq, Wq)
    with FakeTensorMode():
        low = torch.empty(shape, device="cuda", dtype=dtype)
        disp, stats = ns.upsample_soft_argmin(low, D, H, W)
        assert disp.dtype == stats.dtype == torch.float32
        assert tuple(disp.shape) == (B, 1, H, W) and tuple(stats.shape) == (B, 2, H, W)
        g = ns.upsample_soft_argmin_backward(low, disp, stats, torch.empty_like(disp), D)
        assert g.dtype == dtype and tuple(g.shape) == shape


def test_upsample_soft_argmin_autograd_on_meta_returns_a_bf16_gradient():
    low = torch.empty(B, 1, Dq, Hq, Wq, device="meta", dtype=torch.bfloat16, requires_grad=True)
    disp = library_ops.upsample_soft_argmin(low, (D, H, W))
    assert disp.dtype == torch.float32 and tuple(disp.shape) == (B, 1, H, W)
    (g,) = torch.autograd.grad(disp.sum(), [low])
    assert g.dtype == torch.bfloat16 and tuple(g.shape) == tuple(low.shape)
