"""CPU: the fake (meta) kernels of the group-wise correlation volume with 16-bit features describe what the CUDA
implementation returns (DESIGN.md §4.15): the volume and both feature gradients have the features' dtype.  Fake and meta
tensors only, so this runs without a GPU."""
import ctypes

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import _lib, library_ops  # noqa: F401  (importing registers the ops)

B, C, H, W, DQ, G = 2, 16, 5, 12, 7, 4
DTYPES = [torch.bfloat16, torch.float16]


@pytest.mark.parametrize("dtype", DTYPES)
def test_gwc_volume_fakes_with_16_bit_features(dtype):
    ns = torch.ops.az_stereo
    with FakeTensorMode():
        ref = torch.empty(B, C, H, W, device="cuda", dtype=dtype)
        tgt = torch.empty(B, C, H, W, device="cuda", dtype=dtype)
        vol = ns.gwc_volume(ref, tgt, DQ, G)
        assert vol.dtype == dtype and tuple(vol.shape) == (B, G, DQ, H, W)
        gL, gR = ns.gwc_volume_backward(torch.empty_like(vol), ref, tgt)
        assert gL.dtype == gR.dtype == dtype
        assert tuple(gL.shape) == tuple(gR.shape) == (B, C, H, W)


@pytest.mark.parametrize("dtype", DTYPES)
def test_gwc_volume_autograd_on_meta_keeps_the_dtype(dtype):
    ref = torch.empty(B, C, H, W, device="meta", dtype=dtype, requires_grad=True)
    tgt = torch.empty(B, C, H, W, device="meta", dtype=dtype, requires_grad=True)
    vol = library_ops.gwc_volume(ref, tgt, DQ, G)
    assert vol.dtype == dtype and tuple(vol.shape) == (B, G, DQ, H, W)
    gL, gR = torch.autograd.grad(vol.sum(), [ref, tgt])
    assert gL.dtype == gR.dtype == dtype and tuple(gL.shape) == tuple(gR.shape) == (B, C, H, W)


def test_gwc_16_entry_points_are_bound_as_declared():
    symbols = _lib.header_symbols()
    for name, nargs in (("az_gwc_volume_fwd_16", 11), ("az_gwc_volume_bwd_16", 13)):
        assert name in symbols
        res, args = _lib.SIGNATURES[name]
        assert len(args) == nargs  # the fp32 entry's arguments plus the dtype code
        assert args[-2] is ctypes.c_int
        assert _lib.KERNELS_PER_CALL.get(name, 1) == 1
