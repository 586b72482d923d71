"""CPU: the fake (meta) kernels of the implicit-volume training convolution with 16-bit features describe what the CUDA
implementation returns (DESIGN.md §4.13): the output and the feature gradients have the features' dtype, the weight
gradient the weight's dtype.  Fake and meta tensors only, so this runs without a GPU."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import _lib, library_ops  # noqa: F401  (importing registers the ops)

B, H, W, DQ = 2, 5, 12, 7
DTYPES = [torch.bfloat16, torch.float16]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
def test_volume_conv_fakes_with_16_bit_features(dtype, weight_f32):
    ns = torch.ops.az_stereo
    wdt = torch.float32 if weight_f32 else dtype
    with FakeTensorMode():
        ref = torch.empty(B, 32, H, W, device="cuda", dtype=dtype)
        tgt = torch.empty(B, 32, H, W, device="cuda", dtype=dtype)
        w = torch.empty(32, 64, 3, 3, 3, device="cuda", dtype=wdt)
        out = ns.volume_conv(ref, tgt, w, DQ)
        assert out.dtype == dtype and tuple(out.shape) == (B, 32, DQ, H, W)
        gL, gR, gW = ns.volume_conv_backward(torch.empty_like(out), ref, tgt, w)
        assert gL.dtype == gR.dtype == dtype and gW.dtype == wdt
        assert tuple(gL.shape) == tuple(gR.shape) == (B, 32, H, W) and tuple(gW.shape) == (32, 64, 3, 3, 3)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
def test_volume_conv_autograd_on_meta_keeps_the_dtypes(dtype, weight_f32):
    wdt = torch.float32 if weight_f32 else dtype
    ref = torch.empty(B, 32, H, W, device="meta", dtype=dtype, requires_grad=True)
    tgt = torch.empty(B, 32, H, W, device="meta", dtype=dtype, requires_grad=True)
    w = torch.empty(32, 64, 3, 3, 3, device="meta", dtype=wdt, requires_grad=True)
    out = library_ops.volume_conv(ref, tgt, w, DQ)
    assert out.dtype == dtype and tuple(out.shape) == (B, 32, DQ, H, W)
    gL, gR, gW = torch.autograd.grad(out.sum(), [ref, tgt, w])
    assert gL.dtype == gR.dtype == dtype and gW.dtype == wdt
    assert tuple(gL.shape) == (B, 32, H, W) and tuple(gW.shape) == (32, 64, 3, 3, 3)


def test_volume_conv_bwd_16_is_bound_as_declared():
    assert "az_volume_conv0_bwd_16" in _lib.header_symbols()
    res, args = _lib.SIGNATURES["az_volume_conv0_bwd_16"]
    assert len(args) == 16  # 8 pointers, B C H W Dq, dtype, weight_dtype, stream
    assert _lib.KERNELS_PER_CALL["az_volume_conv0_bwd_16"] == 4
