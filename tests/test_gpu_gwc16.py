"""GPU: the group-wise correlation volume with bf16 / fp16 features (ops.build_gwc_volume, torch.ops.az_stereo.gwc_volume,
az_gwc_volume_fwd_16 / az_gwc_volume_bwd_16 in csrc/gwc_volume.cu, DESIGN.md §4.15).  The 16-bit operator must equal the
fp32 operator on the widened features followed by .to(dtype), bit for bit, in the forward and in both gradients."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_guard_bands import Guarded  # noqa: E402

if torch.cuda.is_available():
    from activezero_b200 import _lib, library_ops, ops  # noqa: F401  (library_ops registers the torch.ops)
    from activezero_b200.ops import DTYPE16, _ptr, _stream

DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
# (B, C, H, W), Dq, G -- every path of the kernel map (16-bit kernel / what the fp32 entry runs on the widened copy):
SHAPES = [
    ((2, 32, 9, 64), 48, 8),      # cpg 4, W % 8 == 0: planes / systolic (128 threads)
    ((2, 32, 70, 128), 47, 8),    # several rows per CTA, Dq % 4 == 3
    ((1, 16, 1, 520), 50, 4),     # H = 1, W / 4 > 128: systolic with 256 threads, Dq % 4 == 2
    ((1, 16, 5, 60), 13, 16),     # cpg 1, W % 8 == 4: direct backward (fp32: systolic)
    ((1, 16, 7, 36), 13, 8),      # cpg 2, W % 8 == 4
    ((1, 64, 3, 16), 8, 8),       # cpg 8: direct backward in both
    ((1, 64, 9, 256), 24, 8),     # cpg 8, a wide row
    ((1, 8, 3, 1032), 9, 4),      # W > 1024 (W / 4 > 256): direct backward in both
    ((1, 8, 2, 1028), 9, 2),      # W > 1024, W % 8 == 4
    ((1, 8, 4, 24), 30, 2),       # Dq > W
    ((2, 16, 6, 48), 1, 4),       # Dq = 1
    ((1, 24, 4, 37), 6, 8),       # cpg 3, W % 4 != 0: scalar kernels
    ((1, 12, 3, 40), 5, 4),       # cpg 3, W % 8 == 0: scalar kernels
    ((1, 8, 5, 9), 5, 8),         # cpg 1, odd W
    ((8, 32, 136, 240), 48, 8),   # config 2
]


def _inputs(shape, dq, G, dtype, seed, scale=1.0, gscale=1.0):
    torch.manual_seed(seed)
    B, C, H, W = shape
    L = (torch.randn(shape, device=DEV) * scale).to(dtype)
    R = (torch.randn(shape, device=DEV) * scale).to(dtype)
    g = (torch.randn(B, G, dq, H, W, device=DEV) * gscale).to(dtype)
    return L, R, g


def _mine(L, R, g, dq, G, need=(True, True)):
    Lg, Rg = L.clone().requires_grad_(need[0]), R.clone().requires_grad_(need[1])
    vol = ops.build_gwc_volume(Lg, Rg, dq, G)
    vol.backward(g)
    return vol.detach(), Lg.grad, Rg.grad


def _reference(L, R, g, dq, G, need=(True, True)):
    """The fp32 operator on the widened inputs, then .to(dtype)."""
    dt = L.dtype
    Lg, Rg = L.float().requires_grad_(need[0]), R.float().requires_grad_(need[1])
    vol = ops.build_gwc_volume(Lg, Rg, dq, G)
    vol.backward(g.float())
    return vol.detach().to(dt), *(None if t.grad is None else t.grad.to(dt) for t in (Lg, Rg))


def _equal(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, what
    assert torch.equal(a, b), f"{what}: {int((a != b).sum())} elements differ"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,dq,G", SHAPES)
def test_forward_and_backward_equal_fp32_on_widened_inputs(dtype, shape, dq, G):
    L, R, g = _inputs(shape, dq, G, dtype, 80)
    mine, ref = _mine(L, R, g, dq, G), _reference(L, R, g, dq, G)
    for name, a, b in zip(("vol", "gL", "gR"), mine, ref):
        _equal(a, b, name)
    # each one-sided gradient takes the same kernels
    for need in ((True, False), (False, True)):
        one = _mine(L, R, g, dq, G, need)
        for i in (1, 2):
            if need[i - 1]:
                _equal(one[i], mine[i], f"one-sided {need}")
            else:
                assert one[i] is None
    # the library op and its backward op give the same tensors
    _equal(torch.ops.az_stereo.gwc_volume(L, R, dq, G), mine[0], "library op")
    gL, gR = torch.ops.az_stereo.gwc_volume_backward(g, L, R)
    _equal(gL, mine[1], "library gL")
    _equal(gR, mine[2], "library gR")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("offset", [1, 4])
@pytest.mark.parametrize("shape,dq,G", [((2, 32, 9, 64), 48, 8), ((1, 64, 3, 16), 8, 8), ((1, 16, 5, 60), 13, 4)])
def test_misaligned_views_take_a_fallback_and_still_match(dtype, offset, shape, dq, G):
    """A view `offset` elements into its storage: 2 bytes (no 8-byte quads: the scalar kernels) or 8 bytes (quads, but
    no 16-byte bulk copies: the direct backward)."""
    L, R, g = _inputs(shape, dq, G, dtype, 81)

    def shifted(t):
        buf = torch.empty(t.numel() + offset, dtype=dtype, device=DEV)
        v = buf[offset:].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 == 2 * offset
        return v

    Lo, Ro, go = shifted(L), shifted(R), shifted(g)
    ref = _reference(L, R, g, dq, G)
    _equal(torch.ops.az_stereo.gwc_volume(Lo, Ro, dq, G), ref[0], "vol")
    gL, gR = torch.ops.az_stereo.gwc_volume_backward(go, Lo, Ro)
    _equal(gL, ref[1], "gL")
    _equal(gR, ref[2], "gR")


@pytest.mark.parametrize("dtype", DTYPES)
def test_groups_of_one_channel_are_the_rounded_product_of_the_concat_halves(dtype):
    """G = C: vol[b,c,i] = RNE16(L[b,c] * shift_i(R[b,c])), the product of the two halves of the 16-bit concat volume."""
    torch.manual_seed(82)
    B, C, H, W, Dq = 2, 32, 20, 64, 24
    L = torch.randn(B, C, H, W, device=DEV).to(dtype)
    R = torch.randn(B, C, H, W, device=DEV).to(dtype)
    cat = ops.build_concat_volume(L, R, Dq)
    assert cat.dtype == dtype
    _equal(ops.build_gwc_volume(L, R, Dq, C), (cat[:, :C].float() * cat[:, C:].float()).to(dtype), "G = C")


# gscale puts the gradient sums around the fp16 limit (65504): some overflow, some do not
@pytest.mark.parametrize("shape,dq,G,gscale", [((1, 8, 6, 64), 24, 8, 60.0), ((1, 16, 4, 60), 20, 4, 150.0),
                                               ((1, 8, 3, 37), 9, 2, 250.0)])
def test_fp16_results_that_overflow_become_inf_as_to_float16(shape, dq, G, gscale):
    L, R, g = _inputs(shape, dq, G, torch.float16, 83, scale=300.0, gscale=gscale)
    mine, ref = _mine(L, R, g, dq, G), _reference(L, R, g, dq, G)
    for name, a, b in zip(("vol", "gL", "gR"), mine, ref):
        assert bool(torch.isinf(a).any()) and bool(torch.isfinite(a).any()) and not bool(torch.isnan(a).any()), name
        _equal(a, b, name)


@pytest.mark.parametrize("dtype", DTYPES)
def test_two_runs_are_bit_identical(dtype):
    L, R, g = _inputs((2, 32, 40, 240), 48, 8, dtype, 84)
    a, b = _mine(L, R, g, 48, 8), _mine(L, R, g, 48, 8)
    for x, y, name in zip(a, b, ("vol", "gL", "gR")):
        _equal(x, y, name)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,dq,G", [((1, 32, 5, 240), 48, 8), ((2, 8, 3, 36), 13, 4), ((1, 4, 7, 132), 9, 4),
                                        ((1, 16, 2, 520), 50, 4), ((1, 64, 3, 16), 8, 8), ((1, 8, 3, 1028), 9, 4),
                                        ((1, 6, 4, 9), 5, 3), ((3, 8, 5, 60), 7, 2)])
def test_raw_16_bit_calls_write_only_inside_their_outputs(dtype, shape, dq, G):
    B, C, H, W = shape
    L, R, g = _inputs(shape, dq, G, dtype, 85)
    code = DTYPE16[dtype]
    vol = Guarded((B, G, dq, H, W), dtype)
    _lib.call("az_gwc_volume_fwd_16", _ptr(L), _ptr(R), _ptr(vol.t), B, C, H, W, dq, G, code, _stream())
    gL, gR = Guarded(shape, dtype), Guarded(shape, dtype)
    _lib.call("az_gwc_volume_bwd_16", _ptr(g), _ptr(L), _ptr(R), _ptr(gL.t), _ptr(gR.t), B, C, H, W, dq, G, code, _stream())
    torch.cuda.synchronize()
    for buf, name in ((vol, "vol"), (gL, "gL"), (gR, "gR")):
        buf.check(name)
    for a, b, name in zip((vol.t, gL.t, gR.t), _mine(L, R, g, dq, G), ("vol", "gL", "gR")):
        _equal(a, b, name)


# ------------------------------------------------------------------------------------------------ rejections, empty batch
@pytest.mark.parametrize("dtype", DTYPES)
def test_rejections_before_any_launch(dtype):
    other = torch.float16 if dtype == torch.bfloat16 else torch.bfloat16
    L = torch.randn(1, 8, 4, 16, device=DEV).to(dtype)
    g = torch.randn(1, 4, 5, 4, 16, device=DEV).to(dtype)
    n0 = _lib.launch_count
    for a, b in ((L, L.to(other)), (L, L.float()), (L.float(), L), (L, L.cpu()), (L.cpu(), L.cpu())):
        with pytest.raises(ValueError):
            ops.build_gwc_volume(a, b, 5, 4)
        # two CPU tensors never reach the op: the dispatcher has no CPU kernel for it
        with pytest.raises(NotImplementedError if a.is_cpu and b.is_cpu else ValueError):
            torch.ops.az_stereo.gwc_volume(a, b, 5, 4)
    for gbad in (g.float(), g.to(other), g.double(), g.cpu()):  # a gradient of a dtype the forward did not produce
        with pytest.raises(ValueError):
            torch.ops.az_stereo.gwc_volume_backward(gbad, L, L)
        with pytest.raises(ValueError):
            ops.gwc_volume_backward(gbad, L, L)
    with pytest.raises(ValueError):  # and an fp32 forward's backward refuses a 16-bit gradient
        torch.ops.az_stereo.gwc_volume_backward(g, L.float(), L.float())
    assert _lib.launch_count == n0
    lib = _lib.load()
    vol = torch.empty(1, 4, 5, 4, 16, device=DEV, dtype=dtype)
    gL = torch.empty_like(L)
    for dt in (0, 3, -1):
        assert lib.az_gwc_volume_fwd_16(_ptr(L), _ptr(L), _ptr(vol), 1, 8, 4, 16, 5, 4, dt, _stream()) == -1
        assert lib.az_gwc_volume_bwd_16(_ptr(g), _ptr(L), _ptr(L), _ptr(gL), _ptr(gL), 1, 8, 4, 16, 5, 4, dt, _stream()) == -1
    torch.cuda.synchronize()


@pytest.mark.parametrize("dtype", DTYPES)
def test_empty_batch(dtype):
    L = torch.zeros(0, 8, 5, 12, device=DEV, dtype=dtype, requires_grad=True)
    R = torch.zeros(0, 8, 5, 12, device=DEV, dtype=dtype, requires_grad=True)
    n0 = _lib.launch_count
    vol = ops.build_gwc_volume(L, R, 6, 4)
    assert vol.dtype == dtype and vol.shape == (0, 4, 6, 5, 12)
    vol.sum().backward()
    assert L.grad.dtype == R.grad.dtype == dtype and L.grad.shape == L.shape and R.grad.shape == R.shape
    vol2 = torch.ops.az_stereo.gwc_volume(L.detach(), R.detach(), 6, 4)
    assert vol2.dtype == dtype and vol2.shape == (0, 4, 6, 5, 12)
    gL, gR = torch.ops.az_stereo.gwc_volume_backward(vol2, L.detach(), R.detach())
    assert gL.dtype == gR.dtype == dtype and gL.shape == L.shape
    torch.cuda.synchronize()
    assert _lib.launch_count == n0, "an empty batch must not enqueue a kernel"


# ------------------------------------------------------------------------------------------------ custom op
@pytest.mark.parametrize("dtype", DTYPES)
def test_opcheck(dtype):
    torch.manual_seed(86)
    L = torch.randn(2, 16, 5, 24, device=DEV).to(dtype).requires_grad_(True)
    R = torch.randn(2, 16, 5, 24, device=DEV).to(dtype).requires_grad_(True)
    torch.library.opcheck(torch.ops.az_stereo.gwc_volume.default, (L, R, 7, 4),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    g = torch.randn(2, 4, 7, 5, 24, device=DEV).to(dtype)
    torch.library.opcheck(torch.ops.az_stereo.gwc_volume_backward.default, (g, L.detach(), R.detach()),
                          test_utils=("test_schema", "test_faketensor"))


def test_torch_compile_of_a_bf16_step():
    torch.manual_seed(87)
    L = torch.randn(2, 16, 6, 40, device=DEV).to(torch.bfloat16).requires_grad_(True)
    R = torch.randn(2, 16, 6, 40, device=DEV).to(torch.bfloat16).requires_grad_(True)

    def step(L, R):
        return torch.ops.az_stereo.gwc_volume(L, R, 12, 4).float().square().mean()

    eager = step(L, R)
    compiled = torch.compile(step, backend="aot_eager", fullgraph=True)(L, R)
    assert torch.equal(eager, compiled)
    ge = torch.autograd.grad(eager, [L, R])
    gc = torch.autograd.grad(compiled, [L, R])
    for a, b in zip(ge, gc):
        assert a.dtype == torch.bfloat16 and torch.equal(a, b)


def test_bf16_autocast_region():
    """Under autocast ops.build_gwc_volume keeps its fp32 volume (the features are cast to fp32); the library op, which
    has no autocast rule, takes the bf16 features as they are and returns a bf16 volume."""
    L, R, g = _inputs((1, 16, 6, 64), 20, 4, torch.bfloat16, 88)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        vol = ops.build_gwc_volume(L, R, 20, 4)
        vol16 = torch.ops.az_stereo.gwc_volume(L, R, 20, 4)
    assert vol.dtype == torch.float32
    assert torch.equal(vol, ops.build_gwc_volume(L.float(), R.float(), 20, 4))
    _equal(vol16, vol.to(torch.bfloat16), "library op under autocast")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        with torch.autocast("cuda", enabled=False):  # the documented way to a native volume inside an autocast region
            native = ops.build_gwc_volume(L, R, 20, 4)
    _equal(native, vol16, "autocast switched off")
