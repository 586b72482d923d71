"""GPU: PSMNet's disparity heads with native 16-bit logits -- the soft-argmin and the fused upsample + soft-argmin read
bf16 / fp16 logits as they are, return the fp32 operator's disparity on the widened logits and its gradient rounded
once to the logits' dtype, bit for bit (DESIGN.md §4.12); and a PSMNet_3 converted with ``.to(dtype)`` runs end to
end."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_guard_bands import Guarded  # noqa: E402

if torch.cuda.is_available():
    from activezero_b200 import _lib, library_ops, ops
    from activezero_b200.ops import _ptr, _stream
    from benchmarks.psmnet16 import WidenedHeads

DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
CODE = {torch.bfloat16: 1, torch.float16: 2}  # AZ_DTYPE_BF16, AZ_DTYPE_F16
# (B, D, H, W): H*W % 4 == 0 (and % 8 == 0, and not), H*W % 4 != 0, D = 1, D % 8 != 0, D % 16 != 0, B > 1
SA_SHAPES = [(2, 48, 8, 20), (1, 13, 6, 10), (1, 40, 5, 7), (3, 1, 4, 9), (2, 21, 3, 5), (1, 192, 9, 36), (2, 24, 2, 6)]
SCALES = [1.0, 10.0, 1000.0]
# (B, Dq, Hq, Wq) -> (D, H, W): x4 in D and W (upsample4x kernel), x4 in D only (upsample4), another factor (generic);
# W % 4 != 0, Dq = 1
USA_SHAPES = [((2, 12, 6, 10), (48, 24, 40)), ((1, 9, 5, 7), (36, 19, 25)), ((1, 5, 4, 6), (20, 16, 23)),
              ((2, 6, 3, 5), (15, 9, 14)), ((1, 1, 3, 4), (3, 10, 13)), ((1, 48, 8, 15), (192, 32, 60))]


def _logits(shape, dtype, scale, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, device=DEV, generator=g) * scale).to(dtype)


def _offset_view(x):
    """the same values in a contiguous view that starts one element into its storage (a misaligned 16-bit pointer)"""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.is_contiguous() and v.storage_offset() == 1
    return v


def _sa(cost):
    """disp, lse, gcost of the Function layer for `cost` (any dtype), with a fixed upstream gradient"""
    c = cost.detach().clone().requires_grad_(True) if cost.storage_offset() == 0 else cost.detach().requires_grad_(True)
    disp = ops.soft_argmin(c)
    B, _, H, W = disp.shape
    lse = torch.empty((B, 2, H, W), dtype=torch.float32, device=DEV)
    ops.soft_argmin_forward_into(c.detach(), torch.empty_like(disp), lse)
    gd = _logits((B, 1, H, W), torch.float32, 1.0, 99)
    disp.backward(gd)
    return disp.detach(), lse, c.grad


# ------------------------------------------------------------------------------------------------ soft-argmin
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("shape", SA_SHAPES)
def test_soft_argmin_equals_fp32_on_widened_logits(dtype, scale, shape):
    x = _logits(shape, dtype, scale, 1)
    d16, l16, g16 = _sa(x)
    d32, l32, g32 = _sa(x.float())
    assert d16.dtype == torch.float32 and l16.dtype == torch.float32 and g16.dtype == dtype
    assert torch.equal(d16, d32) and torch.equal(l16, l32)
    assert torch.equal(g16, g32.to(dtype))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(2, 48, 8, 20), (1, 13, 6, 10), (1, 40, 5, 7)])
def test_soft_argmin_storage_offset_and_inf_plane(dtype, shape):
    x = _logits(shape, dtype, 10.0, 2)
    x[:, shape[1] // 2] = float("-inf")  # one plane of -inf
    v = _offset_view(x)
    d16, l16, g16 = _sa(v)
    d32, l32, g32 = _sa(x.float())
    assert torch.equal(d16, d32) and torch.equal(l16, l32)
    assert torch.equal(g16, g32.to(dtype))
    assert torch.isfinite(d16).all()


# ------------------------------------------------------------------------------------------------ fused head
def _usa(low, out_size):
    c = low.detach().clone().requires_grad_(True) if low.storage_offset() == 0 else low.detach().requires_grad_(True)
    disp = ops.upsample_soft_argmin(c, out_size)
    B, _, H, W = disp.shape
    stats = torch.empty((B, 2, H, W), dtype=torch.float32, device=DEV)
    Dq, Hq, Wq = c.shape[-3:]
    ops.upsample_soft_argmin_forward_into(c.detach(), torch.empty_like(disp), stats, (B, Dq, Hq, Wq, *out_size))
    disp.backward(_logits((B, 1, H, W), torch.float32, 1.0, 98))
    return disp.detach(), stats, c.grad


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("low,out", USA_SHAPES)
def test_upsample_soft_argmin_equals_fp32_on_widened_logits(dtype, scale, low, out):
    B, Dq, Hq, Wq = low
    x = _logits((B, 1, Dq, Hq, Wq), dtype, scale, 3)
    for xin in (x, _offset_view(x)):
        d16, s16, g16 = _usa(xin, out)
        d32, s32, g32 = _usa(x.float(), out)
        assert d16.dtype == torch.float32 and g16.dtype == dtype
        assert torch.equal(d16, d32) and torch.equal(s16, s32)
        assert torch.equal(g16, g32.to(dtype))


# ------------------------------------------------------------------------------------------------ guard bands (raw ABI)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(1, 7, 3, 5), (2, 21, 9, 36), (1, 33, 5, 130), (1, 17, 3, 6), (2, 19, 4, 10)])
def test_soft_argmin16_writes_stay_inside(dtype, shape):
    B, D, H, W = shape
    cost = _logits(shape, dtype, 3.0, 4)
    disp, lse = Guarded((B, 1, H, W), torch.float32), Guarded((B, 2, H, W), torch.float32)
    _lib.call("az_soft_argmin_fwd_16", _ptr(cost), _ptr(disp.t), _ptr(lse.t), B, D, H, W, CODE[dtype], _stream())
    torch.cuda.synchronize()
    disp.check("disp")
    lse.check("lse")
    gcost = Guarded(shape, dtype)
    gd = _logits((B, 1, H, W), torch.float32, 1.0, 5)
    _lib.call("az_soft_argmin_bwd_16", _ptr(cost), _ptr(disp.t), _ptr(lse.t), _ptr(gd), _ptr(gcost.t), B, D, H, W,
              CODE[dtype], _stream())
    torch.cuda.synchronize()
    gcost.check("gcost")
    assert torch.equal(disp.t, ops.soft_argmin(cost.float()))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("low,out", [((1, 5, 4, 6), (20, 16, 24)), ((2, 12, 9, 15), (48, 36, 60)),
                                     ((1, 3, 2, 3), (9, 7, 10)), ((1, 7, 3, 5), (28, 11, 17))])
def test_upsample_soft_argmin16_writes_stay_inside(dtype, low, out):
    B, Dq, Hq, Wq = low
    D, H, W = out
    lowres = _logits((B, 1, Dq, Hq, Wq), dtype, 3.0, 6)
    disp, stats = Guarded((B, 1, H, W), torch.float32), Guarded((B, 2, H, W), torch.float32)
    _lib.call("az_upsample_soft_argmin_fwd_16", _ptr(lowres), _ptr(disp.t), _ptr(stats.t), B, Dq, Hq, Wq, D, H, W,
              CODE[dtype], _stream())
    torch.cuda.synchronize()
    disp.check("fused disp")
    stats.check("fused stats")
    glow = Guarded((B, 1, Dq, Hq, Wq), dtype)
    ws = Guarded((max(16, _lib.query("az_upsample_soft_argmin_workspace_bytes", B, Dq, H, W, Wq)),), torch.uint8)
    gd = _logits((B, 1, H, W), torch.float32, 1.0, 7)
    _lib.call("az_upsample_soft_argmin_bwd_16", _ptr(lowres), _ptr(disp.t), _ptr(stats.t), _ptr(gd), _ptr(glow.t),
              _ptr(ws.t), B, Dq, Hq, Wq, D, H, W, CODE[dtype], _stream())
    torch.cuda.synchronize()
    glow.check("glow")
    ws.check("fused backward workspace")
    assert torch.equal(disp.t, ops.upsample_soft_argmin(lowres.float(), out))


# ------------------------------------------------------------------------------------------------ rejections, empty batch
@pytest.mark.parametrize("dtype", DTYPES)
def test_rejections_before_any_launch(dtype):
    cost = _logits((1, 8, 4, 8), dtype, 1.0, 8)
    low = _logits((1, 1, 4, 2, 3), dtype, 1.0, 9)
    n0 = _lib.launch_count
    with pytest.raises(ValueError):
        ops.soft_argmin(cost.double())
    with pytest.raises(ValueError):
        ops.upsample_soft_argmin(low.double(), (16, 8, 12))
    with pytest.raises(ValueError):
        library_ops.soft_argmin(cost.double())
    with pytest.raises(ValueError):
        library_ops.upsample_soft_argmin(low.double(), (16, 8, 12))
    disp = torch.zeros((1, 1, 4, 8), device=DEV)
    lse = torch.zeros((1, 2, 4, 8), device=DEV)
    for bad in (torch.bfloat16, torch.float16, torch.float64):
        with pytest.raises(ValueError):
            torch.ops.az_stereo.soft_argmin_backward(cost, disp, lse, disp.to(bad))
        with pytest.raises(ValueError):
            torch.ops.az_stereo.soft_argmin_backward(cost, disp.to(bad), lse, disp)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.soft_argmin_backward(cost, disp, lse.to(bad), disp)
        d8 = torch.zeros((1, 1, 8, 12), device=DEV)
        s8 = torch.zeros((1, 2, 8, 12), device=DEV)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.upsample_soft_argmin_backward(low, d8, s8, d8.to(bad), 16)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.upsample_soft_argmin_backward(low, d8, s8.to(bad), d8, 16)
    assert _lib.launch_count == n0
    lib = _lib.load()
    out = torch.empty((1, 1, 8, 12), device=DEV)
    st = torch.empty((1, 2, 8, 12), device=DEV)
    ws = torch.empty((_lib.query("az_upsample_soft_argmin_workspace_bytes", 1, 4, 8, 12, 3),), dtype=torch.uint8,
                     device=DEV)
    for code in (0, 3, -1):
        assert lib.az_soft_argmin_fwd_16(_ptr(cost), _ptr(disp), _ptr(lse), 1, 8, 4, 8, code, _stream()) == -1
        assert lib.az_soft_argmin_bwd_16(_ptr(cost), _ptr(disp), _ptr(lse), _ptr(disp), _ptr(torch.empty_like(cost)),
                                         1, 8, 4, 8, code, _stream()) == -1
        assert lib.az_upsample_soft_argmin_fwd_16(_ptr(low), _ptr(out), _ptr(st), 1, 4, 2, 3, 16, 8, 12, code,
                                                  _stream()) == -1
        assert lib.az_upsample_soft_argmin_bwd_16(_ptr(low), _ptr(out), _ptr(st), _ptr(out), _ptr(torch.empty_like(low)),
                                                  _ptr(ws), 1, 4, 2, 3, 16, 8, 12, code, _stream()) == -1


@pytest.mark.parametrize("dtype", DTYPES)
def test_empty_batch(dtype):
    cost = torch.empty((0, 8, 4, 8), dtype=dtype, device=DEV, requires_grad=True)
    disp = ops.soft_argmin(cost)
    assert disp.dtype == torch.float32 and tuple(disp.shape) == (0, 1, 4, 8)
    disp.sum().backward()
    assert cost.grad.dtype == dtype and tuple(cost.grad.shape) == (0, 8, 4, 8)
    low = torch.empty((0, 1, 4, 2, 3), dtype=dtype, device=DEV, requires_grad=True)
    d2 = ops.upsample_soft_argmin(low, (16, 8, 12))
    assert d2.dtype == torch.float32 and tuple(d2.shape) == (0, 1, 8, 12)
    d2.sum().backward()
    assert low.grad.dtype == dtype and tuple(low.grad.shape) == tuple(low.shape)


# ------------------------------------------------------------------------------------------------ library ops
@pytest.mark.parametrize("dtype", DTYPES)
def test_library_ops_match_functions_opcheck_and_compile(dtype):
    cost = _logits((2, 21, 6, 10), dtype, 10.0, 10).requires_grad_(True)
    low = _logits((2, 1, 6, 4, 5), dtype, 10.0, 11).requires_grad_(True)
    out = (24, 16, 20)
    d_fn, l_fn, g_fn = _sa(cost)
    disp, lse = torch.ops.az_stereo.soft_argmin(cost)
    assert disp.dtype == lse.dtype == torch.float32 and torch.equal(disp, d_fn) and torch.equal(lse, l_fn)
    gd = _logits(tuple(disp.shape), torch.float32, 1.0, 99)
    gc = torch.ops.az_stereo.soft_argmin_backward(cost, disp, lse, gd)
    assert gc.dtype == dtype and torch.equal(gc, g_fn)
    du_fn, su_fn, gu_fn = _usa(low, out)
    du, su = torch.ops.az_stereo.upsample_soft_argmin(low, *out)
    assert torch.equal(du, du_fn) and torch.equal(su, su_fn)
    gu = torch.ops.az_stereo.upsample_soft_argmin_backward(low, du, su, _logits(tuple(du.shape), torch.float32, 1.0, 98),
                                                           out[0])
    assert gu.dtype == dtype and torch.equal(gu, gu_fn)

    tests = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.az_stereo.soft_argmin.default, (cost,), test_utils=tests)
    torch.library.opcheck(torch.ops.az_stereo.soft_argmin_backward.default, (cost.detach(), disp, lse, gd),
                          test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(torch.ops.az_stereo.upsample_soft_argmin.default, (low, *out), test_utils=tests)
    torch.library.opcheck(torch.ops.az_stereo.upsample_soft_argmin_backward.default,
                          (low.detach(), du, su, torch.ones_like(du), out[0]), test_utils=("test_schema", "test_faketensor"))

    def step(c, lo):
        return library_ops.soft_argmin(c).square().mean() + library_ops.upsample_soft_argmin(lo, out).square().mean()

    eager = step(cost, low)
    compiled = torch.compile(step, backend="aot_eager", fullgraph=True)(cost, low)
    assert torch.allclose(eager, compiled, rtol=1e-6)
    for a, b in zip(torch.autograd.grad(eager, [cost, low]), torch.autograd.grad(compiled, [cost, low])):
        assert a.dtype == dtype and torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ PSMNet_3 in 16 bits
def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def _conditioned_model(x, y):
    """PSMNet_3 with BatchNorm conditioned on (x, y) (momentum 1) and frozen, so that 16-bit activations stay in range"""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    torch.manual_seed(1)
    model = PSMNet(maxdisp=192).cuda().train()
    for m in model.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.momentum = 1.0
    with torch.no_grad():
        model(x, y)
    return model.eval()


def _inputs(B):
    g = torch.Generator(device=DEV).manual_seed(17)
    return torch.rand(B, 3, 256, 512, device=DEV, generator=g), torch.rand(B, 3, 256, 512, device=DEV, generator=g)


@pytest.mark.parametrize("dtype", DTYPES)
def test_psmnet_converted_to_16_bits_eval(dtype):
    x, y = _inputs(1)
    model = _conditioned_model(x, y).to(dtype)
    xh, yh = x.to(dtype), y.to(dtype)
    with torch.no_grad():
        for cl in (False, True):
            model.use_channels_last_3d(cl)
            for fuse in (False, True):
                model.fuse_upsample = fuse
                out = model(xh, yh)
                assert out.dtype == torch.float32 and tuple(out.shape) == (1, 1, 256, 512)
                assert torch.isfinite(out).all(), (cl, fuse)
                with WidenedHeads():
                    ref = model(xh, yh)
                assert torch.equal(out, ref), (cl, fuse)


@pytest.mark.parametrize("dtype", DTYPES)
def test_psmnet_converted_to_16_bits_fused_volume_conv(dtype):
    x, y = _inputs(1)
    model = _conditioned_model(x, y)
    with torch.no_grad():
        ref = model(x, y)
        model.to(dtype)
        xh, yh = x.to(dtype), y.to(dtype)
        for cl in (False, True):
            model.use_channels_last_3d(cl)
            model.fuse_volume_conv = False
            unfused = model(xh, yh)
            model.fuse_volume_conv = True
            fused = model(xh, yh)
            model.fuse_volume_conv = False
            assert model._vc_cache[0][-1] == dtype  # the 16-bit implicit convolution ran
            assert fused.dtype == torch.float32 and torch.isfinite(fused).all()
            assert _rel(fused, ref) <= 3.0 * _rel(unfused, ref) + 1e-4, (cl, _rel(fused, ref), _rel(unfused, ref))


def test_psmnet_bf16_training_step_equals_widened_heads():
    """One config-3 training step of a bf16 PSMNet_3 (256x512, B = 2; BatchNorm conditioned and frozen): native 16-bit
    heads give the loss and predictions of the widened-by-hand dataflow bit for bit; the bf16 parameter gradients are
    equal when that dataflow reproduces its own, else within 3x its run-to-run distance."""
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    model = None
    try:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
        batch = ts.make_batch(2, 256, 512, "cuda", seed=7, T=4)
        model = _conditioned_model(batch["img_sim_L"], batch["img_sim_R"]).train()
        for m in model.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                m.eval()
        model.to(torch.bfloat16)
        b16 = dict(batch, img_sim_L=batch["img_sim_L"].to(torch.bfloat16), img_sim_R=batch["img_sim_R"].to(torch.bfloat16))
        api = ts.az_api()

        def run(widened, fuse):
            model.fuse_upsample = fuse
            model.zero_grad(set_to_none=True)
            preds = []

            def tap(*a):
                preds.extend(model(*a))
                return preds

            if widened:
                with WidenedHeads():
                    loss, _ = ts.sim_step_loss(tap, b16, api)
                    loss.backward()
            else:
                loss, _ = ts.sim_step_loss(tap, b16, api)
                loss.backward()
            grads = [p.grad.detach().clone() for p in model.parameters() if p.grad is not None]
            return loss.detach().clone(), [p.detach().clone() for p in preds], grads

        for fuse in (False, True):
            old, old2, new = run(True, fuse), run(True, fuse), run(False, fuse)
            assert all(p.dtype == torch.float32 for p in new[1])
            assert torch.equal(new[0], old[0]), (fuse, float(new[0]), float(old[0]))
            for a, b in zip(new[1], old[1]):
                assert torch.equal(a, b), fuse
            assert len(new[2]) == len(old[2]) and all(g.dtype == torch.bfloat16 for g in new[2])
            flat = [torch.cat([t.flatten().double() for t in r[2]]) for r in (old, old2, new)]
            run_to_run = _rel(flat[1], flat[0])
            if run_to_run == 0.0:
                for a, b in zip(new[2], old[2]):
                    assert torch.equal(a, b), fuse
            else:
                print(f"fuse_upsample={fuse}: the widened dataflow's gradients differ run to run by {run_to_run:.3e}")
                assert _rel(flat[2], flat[0]) <= 3.0 * run_to_run, (fuse, _rel(flat[2], flat[0]), run_to_run)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev


@pytest.mark.parametrize("dtype", DTYPES)
def test_fuse_volume_conv_train_in_16_bit_model_raises(dtype):
    """The volume-free training convolution stays fp32-only: a 16-bit model with fuse_volume_conv_train raises
    ValueError before any launch of the library."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    torch.manual_seed(1)
    model = PSMNet(maxdisp=192).cuda().train().to(dtype)
    model.fuse_volume_conv_train = True
    x = torch.rand(1, 3, 256, 512, device=DEV).to(dtype)
    n0 = _lib.launch_count
    with pytest.raises(ValueError):
        model(x, x)
    assert _lib.launch_count == n0
