"""GPU: the cost volume kept in 16 bits under torch.autocast -- the bf16 / fp16 concat volume (forward and backward,
NCDHW and channels_last_3d), the implicit first convolution with 16-bit features, their torch.library forms, and
PSMNet_3 under autocast (DESIGN.md §4.11)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import stereo_oracle as so  # noqa: E402  (checker only)
from test_gpu_guard_bands import Guarded  # noqa: E402

if torch.cuda.is_available():
    from activezero_b200 import _lib, library_ops, ops
    from activezero_b200.ops import _ptr, _stream

DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
CODE = {torch.bfloat16: 1, torch.float16: 2}  # AZ_DTYPE_BF16, AZ_DTYPE_F16
CL = torch.channels_last_3d
# (B, C, H, W, Dq): W % 8 == 0 and not, Dq > W, Dq = 1, H = 1, C = 32, C % 8 != 0 (and C % 4 != 0)
CONCAT_SHAPES = [(2, 32, 6, 40, 12), (1, 32, 5, 37, 9), (1, 8, 3, 6, 10), (2, 16, 4, 24, 1), (2, 32, 1, 64, 48),
                 (1, 12, 3, 20, 7), (1, 6, 3, 21, 5), (1, 32, 9, 136, 48), (1, 24, 2, 3, 8)]


def _feat(shape, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, device=DEV, generator=g) * 3).to(dtype)


def _fmt_ok(t, channels_last):
    return t.is_contiguous(memory_format=CL if channels_last else torch.contiguous_format)


# ------------------------------------------------------------------------------------------------ concat forward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("shape", CONCAT_SHAPES)
def test_forward_equals_fp32_volume_rounded(dtype, channels_last, shape):
    B, C, H, W, dq = shape
    Lh, Rh = _feat((B, C, H, W), dtype, 1), _feat((B, C, H, W), dtype, 2)
    vol = ops.build_concat_volume(Lh, Rh, dq, channels_last)
    ref = ops.build_concat_volume(Lh.float(), Rh.float(), dq, channels_last).to(dtype)
    assert vol.dtype == dtype and tuple(vol.shape) == (B, 2 * C, dq, H, W)
    assert _fmt_ok(vol, channels_last)
    assert torch.equal(vol, ref)
    assert torch.equal(vol.float().cpu(), so.concat_volume(Lh.float().cpu(), Rh.float().cpu(), dq))


# ------------------------------------------------------------------------------------------------ concat backward
def _grads(Lh, Rh, dq, channels_last, g, need=(True, True)):
    a, b = Lh.clone().requires_grad_(need[0]), Rh.clone().requires_grad_(need[1])
    ops.build_concat_volume(a, b, dq, channels_last).backward(g)
    return a.grad, b.grad


def _grad_layouts(g):
    """the gradient as NCDHW, channels_last_3d and a non-contiguous view"""
    big = torch.empty(g.shape[:-1] + (2 * g.shape[-1],), dtype=g.dtype, device=g.device)
    big[..., ::2] = g
    return {"ncdhw": g.contiguous(), "channels_last_3d": g.contiguous(memory_format=CL), "strided": big[..., ::2]}


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("shape", CONCAT_SHAPES)
def test_backward_equals_fp32_sums_rounded_once(dtype, channels_last, shape):
    B, C, H, W, dq = shape
    Lh, Rh = _feat((B, C, H, W), dtype, 3), _feat((B, C, H, W), dtype, 4)
    g0 = _feat((B, 2 * C, dq, H, W), dtype, 5)
    for name, g in _grad_layouts(g0).items():
        ref = [t.to(dtype) for t in _grads(Lh.float(), Rh.float(), dq, channels_last, g.float())]
        mine = _grads(Lh, Rh, dq, channels_last, g)
        for a, b in zip(mine, ref):
            assert a.dtype == dtype and a.is_contiguous()
            assert torch.equal(a, b), name
        for need in ((True, False), (False, True)):
            part = _grads(Lh, Rh, dq, channels_last, g, need)
            for k in range(2):
                assert (part[k] is None) != need[k]
                if need[k]:
                    assert torch.equal(part[k], mine[k]), (name, need)


# ------------------------------------------------------------------------------------------------ canary guard bands
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(1, 32, 3, 37, 9), (2, 8, 2, 40, 12), (1, 16, 5, 6, 10), (1, 32, 1, 129, 48)])
def test_concat_writes_stay_inside(dtype, shape):
    B, C, H, W, dq = shape
    Lh, Rh = _feat((B, C, H, W), dtype, 6), _feat((B, C, H, W), dtype, 7)
    g = _feat((B, 2 * C, dq, H, W), dtype, 8)
    for cl in (0, 1):
        vol = Guarded((B, dq, H, W, 2 * C) if cl else (B, 2 * C, dq, H, W), dtype)
        _lib.call("az_concat_volume_fwd_16", _ptr(Lh), _ptr(Rh), _ptr(vol.t), B, C, H, W, dq, cl, _stream())
        gL, gR = Guarded((B, C, H, W), dtype), Guarded((B, C, H, W), dtype)
        gv = g.contiguous(memory_format=CL).permute(0, 2, 3, 4, 1) if cl else g  # the [B][Dq][H][W][2C] storage
        gv = gv.contiguous()
        _lib.call("az_concat_volume_bwd_16", _ptr(gv), _ptr(gL.t), _ptr(gR.t), B, C, H, W, dq, CODE[dtype], cl, _stream())
        torch.cuda.synchronize()
        for buf, name in ((vol, "volume"), (gL, "gL"), (gR, "gR")):
            buf.check(f"{name} (channels_last={cl})")
        v = vol.t.permute(0, 4, 1, 2, 3) if cl else vol.t
        assert torch.equal(v, ops.build_concat_volume(Lh, Rh, dq, bool(cl)))
        ref = _grads(Lh, Rh, dq, False, g)
        assert torch.equal(gL.t, ref[0]) and torch.equal(gR.t, ref[1])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,dq", [((1, 32, 3, 130), 7), ((2, 32, 2, 37), 48), ((1, 32, 2, 60), 56), ((1, 32, 1, 1), 1)])
def test_volume_conv_writes_stay_inside(dtype, shape, dq):
    B, C, H, W = shape
    Lh, Rh = _feat(shape, dtype, 9), _feat(shape, dtype, 10)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05
    wp = Guarded((27 * 3072,), torch.float32)
    _lib.call("az_volume_conv0_pack_16", _ptr(w), _ptr(wp.t), CODE[dtype], _stream())
    out = Guarded((B, 32, dq, H, W), dtype)
    sc, sh = torch.rand(32, device=DEV) + 0.5, torch.randn(32, device=DEV)
    _lib.call("az_volume_conv0_fwd_16", _ptr(Lh), _ptr(Rh), _ptr(wp.t), _ptr(sc), _ptr(sh), _ptr(out.t), B, C, H, W, dq, 1,
              CODE[dtype], _stream())
    torch.cuda.synchronize()
    wp.check("wpacked")
    out.check("out")
    assert torch.equal(wp.t, ops.pack_volume_conv_weight(w, dtype))
    assert torch.equal(out.t, ops.volume_conv0(Lh, Rh, wp.t, dq, sc, sh, relu=True))


# ------------------------------------------------------------------------------------------------ implicit convolution
def _conv_ref64(L, R, w, dq, scale, shift, relu):
    """float64 conv3d of the oracle volume, with the BatchNorm fold and the ReLU."""
    out = F.conv3d(so.concat_volume(L.double().cpu(), R.double().cpu(), dq), w.double().cpu(), padding=1)
    if scale is not None:
        out = out * scale.double().cpu().view(1, -1, 1, 1, 1) + shift.double().cpu().view(1, -1, 1, 1, 1)
    return out.clamp_min(0) if relu else out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,dq", [((1, 32, 5, 37), 12), ((2, 32, 3, 130), 48), ((1, 32, 2, 2), 1), ((1, 32, 3, 131), 56)])
@pytest.mark.parametrize("fold,relu", [(False, False), (True, False), (True, True)])
def test_volume_conv_exact_on_integer_probes(dtype, shape, dq, fold, relu):
    """Small integers with sparse weights: every partial sum is an integer far below 2^24 and every output an integer
    with |v| <= 256, which both 16-bit dtypes hold exactly -- so the output is exact (v2 kernel for Dq <= 55, the
    gather kernel for Dq = 56)."""
    g = torch.Generator(device=DEV).manual_seed(11)
    L = torch.randint(-2, 3, shape, device=DEV, generator=g).to(dtype)
    R = torch.randint(-2, 3, shape, device=DEV, generator=g).to(dtype)
    w = torch.randint(-1, 2, (32, 64, 3, 3, 3), device=DEV, generator=g).float()
    w = w * (torch.rand(w.shape, device=DEV, generator=g) < 0.04)
    scale = torch.randint(1, 3, (32,), device=DEV, generator=g).float() if fold else None
    shift = torch.randint(-3, 4, (32,), device=DEV, generator=g).float() if fold else None
    ref = _conv_ref64(L, R, w, dq, scale, shift, relu)
    assert float(ref.abs().max()) <= 256
    out = ops.volume_conv0(L, R, ops.pack_volume_conv_weight(w, dtype), dq, scale, shift, relu=relu)
    assert out.dtype == dtype and tuple(out.shape) == (shape[0], 32, dq, shape[2], shape[3])
    assert torch.equal(out.double().cpu(), ref)


def _ulp16(x16):
    """spacing of the 16-bit grid at |x16| (float64)"""
    a = x16.abs()
    return (a.view(torch.int16) + 1).view(x16.dtype).double() - a.double()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,dq", [((1, 32, 6, 140), 48), ((2, 32, 3, 37), 9), ((1, 32, 3, 70), 56)])
def test_volume_conv_random_within_one_ulp(dtype, shape, dq):
    """Against the float64 convolution of the 16-bit inputs and the 16-bit-rounded weight, rounded to 16 bits: within one
    16-bit ulp, plus the fp32 accumulation's own error (2^-22 of the sum of |terms|) for outputs near zero."""
    L, R = _feat(shape, dtype, 12), _feat(shape, dtype, 13)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05
    scale, shift = torch.rand(32, device=DEV) + 0.5, torch.randn(32, device=DEV)
    out = ops.volume_conv0(L, R, ops.pack_volume_conv_weight(w, dtype), dq, scale, shift, relu=True)
    w16 = w.to(dtype).float()
    ref = _conv_ref64(L, R, w16, dq, scale, shift, True)
    mag = _conv_ref64(L.abs(), R.abs(), w16.abs(), dq, scale, shift.abs(), False)
    ref16 = ref.to(dtype)
    err = (out.double().cpu() - ref16.double()).abs()
    assert bool((err <= _ulp16(ref16) + 2.0 ** -22 * mag).all()), float(err.max())


# ------------------------------------------------------------------------------------------------ rejections, empty batch
def test_rejections_and_empty_batch():
    Lb = torch.randn(1, 32, 4, 16, device=DEV).bfloat16()
    w = torch.randn(32, 64, 3, 3, 3, device=DEV)
    wp = ops.pack_volume_conv_weight(w, torch.bfloat16)
    bad_pairs = [(Lb, Lb.half()), (Lb, Lb.float()), (Lb.double(), Lb.double()), (Lb, Lb[:, :, :3]), (Lb[0], Lb[0])]
    before = _lib.launch_count
    for a, b in bad_pairs:
        with pytest.raises(ValueError):
            ops.build_concat_volume(a, b, 4)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.concat_volume(a, b, 4, False)
        with pytest.raises(ValueError):
            ops.volume_conv0(a, b, wp, 4)
    with pytest.raises(ValueError):
        ops.pack_volume_conv_weight(w, torch.float64)
    with pytest.raises(ValueError):
        torch.ops.az_stereo.concat_volume_backward(torch.randn(1, 64, 4, 4, 16, device=DEV).double(), 32)
    assert _lib.launch_count == before
    null = ctypes.c_void_p(0)
    lib = _lib.load()
    v = torch.empty(1, 64, 4, 4, 16, device=DEV, dtype=torch.bfloat16)
    assert lib.az_concat_volume_bwd_16(_ptr(v), _ptr(Lb), null, 1, 32, 4, 16, 4, 3, 0, null) == -1       # dtype code
    assert lib.az_concat_volume_fwd_16(_ptr(Lb), _ptr(Lb), _ptr(v), 1, 12, 4, 16, 4, 1, null) == -1     # C % 8, layout
    assert lib.az_volume_conv0_pack_16(_ptr(w), _ptr(wp), 0, null) == -1
    assert lib.az_volume_conv0_fwd_16(_ptr(Lb), _ptr(Lb), _ptr(wp), null, null, _ptr(v), 1, 32, 4, 16, 4, 0, 7, null) == -1
    # B = 0 enqueues nothing
    for dtype in DTYPES:
        E = torch.zeros(0, 32, 5, 12, device=DEV, dtype=dtype, requires_grad=True)
        before = _lib.launch_count
        for cl in (False, True):
            vol = ops.build_concat_volume(E, E, 6, cl)
            assert vol.shape == (0, 64, 6, 5, 12) and vol.dtype == dtype
            vol.float().sum().backward()
        assert E.grad.shape == E.shape and E.grad.dtype == dtype
        out = ops.volume_conv0(E.detach(), E.detach(), wp, 6)
        assert out.shape == (0, 32, 6, 5, 12) and out.dtype == dtype
        torch.cuda.synchronize()
        assert _lib.launch_count == before, "an empty batch must not enqueue a kernel"


# ------------------------------------------------------------------------------------------------ torch.library
@pytest.mark.parametrize("dtype", DTYPES)
def test_library_ops_opcheck_and_compile(dtype):
    L = _feat((2, 16, 5, 24), dtype, 14).requires_grad_(True)
    R = _feat((2, 16, 5, 24), dtype, 15).requires_grad_(True)
    for cl in (False, True):
        torch.library.opcheck(torch.ops.az_stereo.concat_volume.default, (L, R, 7, cl),
                              test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
        g = _feat((2, 32, 7, 5, 24), dtype, 16)
        g = g.contiguous(memory_format=CL) if cl else g
        torch.library.opcheck(torch.ops.az_stereo.concat_volume_backward.default, (g, 16),
                              test_utils=("test_schema", "test_faketensor"))
        vol = torch.ops.az_stereo.concat_volume(L, R, 7, cl)
        assert vol.dtype == dtype and torch.equal(vol, ops.build_concat_volume(L, R, 7, cl))
        gl, gr = torch.ops.az_stereo.concat_volume_backward(g, 16)
        assert gl.dtype == dtype and torch.equal(gl, _grads(L.detach(), R.detach(), 7, cl, g)[0])

        def step(L, R):
            return library_ops.concat_volume(L, R, 7, cl).float().square().mean()

        eager = step(L, R)
        compiled = torch.compile(step, backend="aot_eager", fullgraph=True)(L, R)
        assert torch.allclose(eager, compiled, rtol=1e-6)
        for a, b in zip(torch.autograd.grad(eager, [L, R]), torch.autograd.grad(compiled, [L, R])):
            assert a.dtype == dtype and torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ PSMNet under autocast
def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


@pytest.mark.parametrize("dtype", DTYPES)
def test_psmnet_eval_fused_volume_conv_under_autocast(dtype):
    """fuse_volume_conv=True under autocast runs (it used to raise on the 16-bit features) and is no further from the
    fp32 forward than the unfused autocast forward is (3x, plus a small floor); both layouts."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    torch.manual_seed(1)
    model = PSMNet(maxdisp=192).cuda().train()
    g = torch.Generator(device=DEV).manual_seed(17)
    x, y = torch.rand(1, 3, 256, 512, device=DEV, generator=g), torch.rand(1, 3, 256, 512, device=DEV, generator=g)
    # BatchNorm conditioned on this input (as in test_gpu_volume_conv_train.py), so that fp16 activations stay in range
    for m in model.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.momentum = 1.0
    with torch.no_grad():
        model(x, y)
    model.eval()
    with torch.no_grad():
        ref = model(x, y)
        for cl in (False, True):
            model.use_channels_last_3d(cl)
            with torch.autocast("cuda", dtype=dtype):
                model.fuse_volume_conv = False
                unfused = model(x, y)
                model.fuse_volume_conv = True
                fused = model(x, y)
            model.fuse_volume_conv = False
            assert model._vc_cache[0][-1] == dtype  # the 16-bit implicit convolution ran
            assert torch.isfinite(fused).all()
            assert _rel(fused, ref) <= 3.0 * _rel(unfused, ref) + 1e-4, (cl, _rel(fused, ref), _rel(unfused, ref))
        model.use_channels_last_3d(False)


class _Preds(torch.nn.Module):
    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, *a):
        self.preds = self.net(*a)
        return self.preds


def _previous_dataflow(model):
    """PSMNetBase._forward_features as it was before the native 16-bit volume: the concat volume goes through the fp32
    op inside autocast (16-bit features cast up, fp32 volume, cast down by cuDNN's autocast)."""
    def fwd(ref_feat, tgt_feat):
        H, W = ref_feat.shape[-2:]
        cost = ops.build_concat_volume(ref_feat, tgt_feat, model.maxdisp // 4, channels_last=model.volume_channels_last)
        assert cost.dtype == torch.float32
        cost1, cost2, cost3 = model._aggregate(cost)
        pred3 = model._disparity_head(cost3, H, W)
        pred1 = model._disparity_head(cost1, H, W)
        pred2 = model._disparity_head(cost2, H, W)
        return pred3, pred2, pred1

    return fwd


def test_psmnet_training_step_under_bf16_autocast_is_bit_identical():
    """One config-3 training step of PSMNet_3 at 256x512, B=2, under bf16 autocast, BatchNorm conditioned and frozen as in
    test_gpu_volume_conv_train.py: the native 16-bit volume gives the same loss, predictions and parameter gradients
    as the previous dataflow, bit for bit (fused upsample: torch's trilinear backward uses atomics).  The forward is
    deterministic, so the loss and the predictions are compared exactly.  The gradients are compared exactly when the
    previous dataflow reproduces its own gradients over two runs; where it does not (the feature extractor's bilinear
    upsampling has an atomic backward in torch), the native path must be within 3x the run-to-run distance."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    try:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
        torch.manual_seed(1)
        model = PSMNet(maxdisp=192).cuda().train()
        model.fuse_upsample = True
        batch = ts.make_batch(2, 256, 512, "cuda", seed=7, T=4)
        bns = [m for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
        for m in bns:
            m.momentum = 1.0
        with torch.no_grad():
            model(batch["img_sim_L"], batch["img_sim_R"])
        for m in bns:
            m.eval()
        api = ts.az_api()
        native_fwd = model._forward_features

        def run(previous, channels_last):
            model.use_channels_last_3d(channels_last)
            model._forward_features = _previous_dataflow(model) if previous else native_fwd
            model.zero_grad(set_to_none=True)
            tap = _Preds(model)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss, _ = ts.sim_step_loss(tap, batch, api)
            loss.backward()
            grads = [p.grad.detach().clone() for p in model.parameters() if p.grad is not None]
            return loss.detach().clone(), [p.detach().clone() for p in tap.preds], grads

        for cl in (False, True):
            old, old2, new = run(True, cl), run(True, cl), run(False, cl)
            assert torch.equal(old[0], old2[0]) and all(torch.equal(a, b) for a, b in zip(old[1], old2[1])), cl
            assert torch.equal(new[0], old[0]), (cl, float(new[0]), float(old[0]))
            for a, b in zip(new[1], old[1]):
                assert torch.equal(a, b), cl
            assert len(new[2]) == len(old[2]) == len(old2[2])
            flat = [torch.cat([t.flatten().double() for t in r[2]]) for r in (old, old2, new)]
            run_to_run = _rel(flat[1], flat[0])
            if run_to_run == 0.0:
                for a, b in zip(new[2], old[2]):
                    assert torch.equal(a, b), cl
            else:
                print(f"channels_last={cl}: the previous dataflow's gradients differ run to run by {run_to_run:.3e}")
                assert _rel(flat[2], flat[0]) <= 3.0 * run_to_run, (cl, _rel(flat[2], flat[0]), run_to_run)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev
        model.__dict__.pop("_forward_features", None)
