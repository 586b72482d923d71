"""CPU: the fake (meta) kernels of the concat-volume operators with 16-bit inputs describe what the CUDA
implementation returns (DESIGN.md §4.11): the volume and its gradients keep the features' dtype; the layout follows
``channels_last``.  Fake tensors only, so this runs without a GPU."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from activezero_b200 import library_ops  # noqa: F401  (importing registers the ops)

B, Hq, Wq, Dq = 2, 6, 20, 5


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C", [32, 12, 6])
@pytest.mark.parametrize("channels_last", [False, True])
def test_concat_volume_fakes_keep_the_16_bit_dtype(dtype, C, channels_last):
    ns = torch.ops.az_stereo
    fmt = torch.channels_last_3d if channels_last else torch.contiguous_format
    with FakeTensorMode():
        L = torch.empty(B, C, Hq, Wq, device="cuda", dtype=dtype)
        vol = ns.concat_volume(L, L, Dq, channels_last)
        assert vol.dtype == dtype and tuple(vol.shape) == (B, 2 * C, Dq, Hq, Wq)
        assert vol.is_contiguous(memory_format=fmt)
        g = torch.empty(B, 2 * C, Dq, Hq, Wq, device="cuda", dtype=dtype).contiguous(memory_format=fmt)
        gL, gR = ns.concat_volume_backward(g, C)
        for t in (gL, gR):
            assert t.dtype == dtype and tuple(t.shape) == (B, C, Hq, Wq) and t.is_contiguous()
            assert t.stride() == (C * Hq * Wq, Hq * Wq, Wq, 1)
