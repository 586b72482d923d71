"""GPU: the implicit-volume training convolution with bf16 / fp16 tensors (ops.volume_conv, torch.ops.az_stereo.volume_conv,
az_volume_conv0_bwd_16 in csrc/volume_conv_bwd.cu) and PSMNet's fuse_volume_conv_train16 flag (DESIGN.md §4.13).
The 16-bit operator must equal the fp32 operator on the widened features and the dtype-rounded weight, followed by
.to(dtype), bit for bit, in the forward and in every gradient."""
import copy
import itertools

import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_guard_bands import Guarded  # noqa: E402

if torch.cuda.is_available():
    from activezero_b200 import _lib, library_ops, ops
    from activezero_b200.ops import DTYPE16, _ptr, _stream

DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
# ragged shapes: H = 1, W < 3, Dq = 1, Dq > W, Dq = 56 (the first-form forward kernel), rows of several tiles, odd and
# even widths (the 16-bit reduce reads two columns per 4-byte load when W is even)
SHAPES = [((1, 32, 9, 140), 12), ((2, 32, 6, 128), 8), ((1, 32, 5, 37), 48), ((1, 32, 34, 60), 5), ((1, 32, 3, 300), 20),
          ((1, 32, 4, 240), 48), ((1, 32, 1, 126), 3), ((1, 32, 2, 2), 1), ((2, 32, 3, 127), 55), ((1, 32, 2, 131), 56),
          ((1, 32, 3, 258), 56), ((1, 32, 1, 1), 1)]
TRAIN_SHAPE = ((2, 32, 64, 128), 48)


def _inputs(shape, dq, dtype, seed, gscale=1.0):
    torch.manual_seed(seed)
    B = shape[0]
    L = torch.randn(shape, device=DEV).to(dtype)
    R = torch.randn(shape, device=DEV).to(dtype)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05
    g = (torch.randn(B, 32, dq, shape[2], shape[3], device=DEV) * gscale).clamp(-6e4, 6e4).to(dtype)  # finite in fp16
    return L, R, w, g


def _reference(L, R, w, g, dq, weight_dtype, need=(True, True, True)):
    """The fp32 operator on the widened inputs (the weight rounded to the features' dtype first), then .to(dtype)."""
    dt = L.dtype
    ts = [t.float().requires_grad_(n) for t, n in zip((L, R, w.to(dt)), need)]
    out = ops.volume_conv(*ts, dq)
    out.backward(g.float())
    grads = [t.grad for t in ts]
    return out.detach().to(dt), [None if x is None else x.to(dt if i < 2 else weight_dtype) for i, x in enumerate(grads)]


def _mine(L, R, w, g, dq, need=(True, True, True)):
    ts = [t.clone().requires_grad_(n) for t, n in zip((L, R, w), need)]
    out = ops.volume_conv(*ts, dq)
    out.backward(g)
    return out.detach(), [t.grad for t in ts]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
@pytest.mark.parametrize("shape,dq", SHAPES + [TRAIN_SHAPE])
def test_forward_and_backward_equal_fp32_on_widened_inputs(dtype, weight_f32, shape, dq):
    L, R, w, g = _inputs(shape, dq, dtype, 70)
    wt = w if weight_f32 else w.to(dtype)
    wdt = torch.float32 if weight_f32 else dtype
    out, grads = _mine(L, R, wt, g, dq)
    ref_out, ref_grads = _reference(L, R, wt, g, dq, wdt)
    assert out.dtype == dtype and torch.equal(out, ref_out)
    for name, a, b in zip(("gL", "gR", "gW"), grads, ref_grads):
        assert a.dtype == b.dtype and torch.equal(a, b), name
    assert grads[2].dtype == wdt


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
def test_every_needs_input_grad_subset_and_determinism(dtype, weight_f32):
    shape, dq = (2, 32, 7, 130), 24
    L, R, w, g = _inputs(shape, dq, dtype, 71)
    wt = w if weight_f32 else w.to(dtype)
    wdt = torch.float32 if weight_f32 else dtype
    full = _mine(L, R, wt, g, dq)[1]
    again = _mine(L, R, wt, g, dq)[1]
    for a, b in zip(full, again):
        assert torch.equal(a, b), "two calls differ"
    for k in (1, 2):
        for subset in itertools.combinations(range(3), k):
            need = tuple(i in subset for i in range(3))
            mine = _mine(L, R, wt, g, dq, need)[1]
            ref = _reference(L, R, wt, g, dq, wdt, need)[1]
            for i in range(3):
                if need[i]:
                    assert torch.equal(mine[i], full[i]) and torch.equal(mine[i], ref[i]), (subset, i)
                else:
                    assert mine[i] is None and ref[i] is None


@pytest.mark.parametrize("weight_f32", [True, False])
def test_fp16_gradients_that_overflow_become_inf_as_to_float16(weight_f32):
    shape, dq = (1, 32, 6, 96), 48
    L, R, w, g = _inputs(shape, dq, torch.float16, 72, gscale=3e4)
    w = w * 20.0
    wt = w if weight_f32 else w.to(torch.float16)
    wdt = torch.float32 if weight_f32 else torch.float16
    _, grads = _mine(L, R, wt, g, dq)
    _, ref = _reference(L, R, wt, g, dq, wdt)
    assert bool(torch.isinf(grads[0]).any()) and bool(torch.isinf(grads[1]).any())
    assert bool(torch.isfinite(grads[0]).any()) and not bool(torch.isnan(grads[0]).any())
    if not weight_f32:
        assert bool(torch.isinf(grads[2]).any())
    for a, b in zip(grads, ref):
        assert torch.equal(a, b)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
@pytest.mark.parametrize("shape,dq", [((1, 32, 3, 130), 7), ((2, 32, 2, 37), 48), ((1, 32, 5, 254), 3), ((1, 32, 2, 60), 56),
                                      ((1, 32, 1, 1), 1), ((3, 32, 7, 129), 9), ((1, 32, 3, 512), 48)])
def test_raw_backward_writes_stay_inside(dtype, weight_f32, shape, dq):
    """gL, gR, gW and the workspace are windows between 4 KB canary margins; the results equal the autograd path's."""
    B, C, H, W = shape
    L, R, w, g = _inputs(shape, dq, dtype, 73)
    wt = w if weight_f32 else w.to(dtype)
    wdt = torch.float32 if weight_f32 else dtype
    gL, gR, gW = Guarded(shape, dtype), Guarded(shape, dtype), Guarded((32, 64, 3, 3, 3), wdt)
    ws = Guarded((_lib.query("az_volume_conv0_bwd_workspace_bytes", B, H, W, dq),), torch.uint8)
    code = DTYPE16[dtype]
    _lib.call("az_volume_conv0_bwd_16", _ptr(g), _ptr(L), _ptr(R), _ptr(wt), _ptr(gL.t), _ptr(gR.t), _ptr(gW.t),
              _ptr(ws.t), B, C, H, W, dq, code, 0 if weight_f32 else code, _stream())
    torch.cuda.synchronize()
    for buf, name in ((gL, "gL"), (gR, "gR"), (gW, "gW"), (ws, "workspace")):
        buf.check(name)
    for a, b in zip((gL.t, gR.t, gW.t), _mine(L, R, wt, g, dq)[1]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("dtype", DTYPES)
def test_gradient_at_an_odd_element_offset_equals_the_aligned_one(dtype):
    """A grad_out view that starts at an odd element is read with 2-byte loads; the result is the same."""
    shape, dq = (1, 32, 4, 96), 20
    L, R, w, g = _inputs(shape, dq, dtype, 74)
    buf = torch.empty(g.numel() + 1, dtype=dtype, device=DEV)
    g_odd = buf[1:].view(g.shape)
    g_odd.copy_(g)
    assert g_odd.data_ptr() % 4 != 0
    ref = torch.ops.az_stereo.volume_conv_backward(g, L, R, w)
    got = torch.ops.az_stereo.volume_conv_backward(g_odd, L, R, w)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ rejections, empty batch
@pytest.mark.parametrize("dtype", DTYPES)
def test_rejections_before_any_launch(dtype):
    other = torch.float16 if dtype == torch.bfloat16 else torch.bfloat16
    L = torch.randn(1, 32, 4, 16, device=DEV).to(dtype)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV)
    bad = [
        (L, L.to(other), w, 4),                 # features of different dtypes
        (L, L.float(), w, 4),                   # a 16-bit and an fp32 feature
        (L, L, w.to(other), 4),                 # a weight of the other 16-bit dtype
        (L, L, w.double(), 4),                  # a float64 weight
        (L.double(), L.double(), w, 4),         # float64 features
        (L.float(), L.float(), w.to(dtype), 4), # fp32 features with a 16-bit weight
    ]
    g = torch.randn(1, 32, 4, 4, 16, device=DEV)
    n0 = _lib.launch_count
    for args in bad:
        with pytest.raises(ValueError):
            ops.volume_conv(*args)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.volume_conv(*args)
    for gbad in (g, g.to(other), g.double()):   # grad_out of a dtype the forward did not produce
        with pytest.raises(ValueError):
            torch.ops.az_stereo.volume_conv_backward(gbad, L, L, w)
        with pytest.raises(ValueError):
            torch.ops.az_stereo.volume_conv_backward(gbad, L, L, w.to(dtype))
    with pytest.raises(ValueError):             # and an fp32 forward's backward refuses a 16-bit grad_out
        torch.ops.az_stereo.volume_conv_backward(g.to(dtype), L.float(), L.float(), w)
    assert _lib.launch_count == n0
    lib = _lib.load()
    g16 = g.to(dtype)
    gL = torch.empty_like(L)
    gW = torch.empty_like(w)
    ws = torch.empty((_lib.query("az_volume_conv0_bwd_workspace_bytes", 1, 4, 16, 4),), dtype=torch.uint8, device=DEV)
    code, other_code = DTYPE16[dtype], DTYPE16[other]

    def raw(C, dt, wdt):
        return lib.az_volume_conv0_bwd_16(_ptr(g16), _ptr(L), _ptr(L), _ptr(w), _ptr(gL), _ptr(gL), _ptr(gW), _ptr(ws),
                                          1, C, 4, 16, 4, dt, wdt, _stream())

    for dt in (0, 3, -1):
        assert raw(32, dt, 0) == -1
    for wdt in (other_code, 3, -1):
        assert raw(32, code, wdt) == -1
    assert raw(16, code, 0) == -1
    torch.cuda.synchronize()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
def test_empty_batch(dtype, weight_f32):
    L = torch.zeros(0, 32, 5, 12, device=DEV, dtype=dtype, requires_grad=True)
    R = torch.zeros(0, 32, 5, 12, device=DEV, dtype=dtype, requires_grad=True)
    wdt = torch.float32 if weight_f32 else dtype
    w = torch.randn(32, 64, 3, 3, 3, device=DEV).to(wdt).requires_grad_(True)
    n0 = _lib.launch_count
    out = ops.volume_conv(L, R, w, 6)
    assert out.dtype == dtype and out.shape == (0, 32, 6, 5, 12)
    out.sum().backward()
    assert L.grad.dtype == dtype and L.grad.shape == L.shape and R.grad.shape == R.shape
    assert w.grad.dtype == wdt and torch.equal(w.grad, torch.zeros_like(w))
    out2 = torch.ops.az_stereo.volume_conv(L.detach(), R.detach(), w.detach(), 6)
    assert out2.dtype == dtype and out2.shape == (0, 32, 6, 5, 12)
    gW = torch.ops.az_stereo.volume_conv_backward(out2, L.detach(), R.detach(), w.detach())[2]
    assert gW.dtype == wdt and torch.equal(gW, torch.zeros_like(gW))
    torch.cuda.synchronize()
    assert _lib.launch_count == n0, "an empty batch must not enqueue a kernel"


# ------------------------------------------------------------------------------------------------ custom op
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("weight_f32", [True, False])
def test_opcheck_and_torch_compile(dtype, weight_f32):
    torch.manual_seed(75)
    L = torch.randn(2, 32, 5, 24, device=DEV).to(dtype).requires_grad_(True)
    R = torch.randn(2, 32, 5, 24, device=DEV).to(dtype).requires_grad_(True)
    w = (torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05).to(torch.float32 if weight_f32 else dtype).requires_grad_(True)
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.az_stereo.volume_conv.default, (L, R, w, 7), test_utils=checks)
    out = torch.ops.az_stereo.volume_conv(L, R, w, 7)
    torch.library.opcheck(torch.ops.az_stereo.volume_conv_backward.default,
                          (torch.randn_like(out.float()).to(dtype), L.detach(), R.detach(), w.detach()),
                          test_utils=("test_schema", "test_faketensor"))
    assert torch.equal(out, ops.volume_conv(L, R, w, 7))

    def step(L, R, w):
        return library_ops.volume_conv(L, R, w, 7).float().square().mean()

    eager = step(L, R, w)
    compiled = torch.compile(step, backend="aot_eager", fullgraph=True)(L, R, w)
    assert torch.allclose(eager, compiled, rtol=1e-6)
    ge = torch.autograd.grad(eager, [L, R, w])
    gc = torch.autograd.grad(compiled, [L, R, w])
    gf = torch.autograd.grad(ops.volume_conv(L, R, w, 7).float().square().mean(), [L, R, w])
    for a, b, c in zip(ge, gc, gf):
        assert torch.equal(a, b) and torch.equal(a, c)
    assert ge[0].dtype == dtype and ge[2].dtype == w.dtype


# ------------------------------------------------------------------------------------------------ PSMNet_3
def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


class _Preds(torch.nn.Module):
    """Calls the network and keeps its three predictions."""

    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, *a):
        self.preds = self.net(*a)
        return self.preds


def _conditioned_model(batch):
    """PSMNet_3 in train mode with BatchNorm conditioned on the batch (momentum 1) and then frozen (eval statistics)."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    torch.manual_seed(1)
    model = PSMNet(maxdisp=192).cuda().train()
    bns = [m for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
    for m in bns:
        m.momentum = 1.0
    with torch.no_grad():
        model(batch["img_sim_L"], batch["img_sim_R"])
    for m in bns:
        m.eval()
    return model


def _step(model, batch, api, amp_dtype=None):
    from benchmarks import train_step as ts

    model.zero_grad(set_to_none=True)
    tap = _Preds(model)
    if amp_dtype is None:
        loss, _ = ts.sim_step_loss(tap, batch, api)
    else:
        with torch.autocast("cuda", dtype=amp_dtype):
            loss, _ = ts.sim_step_loss(tap, batch, api)
    loss.backward()
    grads = [p.grad.detach().clone() for p in model.parameters() if p.grad is not None]
    return loss.detach().float().clone(), [p.detach().float().clone() for p in tap.preds], grads


def _flat(grads):
    return torch.cat([g.flatten().double() for g in grads])


def test_fp32_model_flag16_equals_fuse_volume_conv_train():
    """Without autocast the 16-bit flag runs the fp32 operator: the loss and predictions are those of
    fuse_volume_conv_train bit for bit, and so are the gradients wherever the step reproduces its own."""
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    try:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
        batch = ts.make_batch(1, 256, 512, "cuda", seed=7, T=4)
        model = _conditioned_model(batch)
        api = ts.az_api()
        model.fuse_volume_conv_train = True
        old, old2 = _step(model, batch, api), _step(model, batch, api)
        model.fuse_volume_conv_train, model.fuse_volume_conv_train16 = False, True
        new = _step(model, batch, api)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev
    assert torch.equal(new[0], old[0])
    for a, b in zip(new[1], old[1]):
        assert torch.equal(a, b)
    run_to_run = _rel(_flat(old2[2]), _flat(old[2]))
    if run_to_run == 0.0:
        for a, b in zip(new[2], old[2]):
            assert torch.equal(a, b)
    else:  # the feature extractor's bilinear upsampling has an atomic backward in torch
        assert _rel(_flat(new[2]), _flat(old[2])) <= 3.0 * run_to_run


@pytest.mark.parametrize("amp_dtype", DTYPES)
def test_autocast_conv_output_dtype_of_each_flag(amp_dtype):
    """Under autocast fuse_volume_conv_train keeps its fp32 convolution; fuse_volume_conv_train16 gives a 16-bit one.
    A converted model with fuse_volume_conv_train16 runs natively and returns a 16-bit weight gradient."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    torch.manual_seed(1)
    model = PSMNet(maxdisp=192).cuda().train()
    seen = []
    model.dres0[0][1].register_forward_hook(lambda m, i, o: seen.append(i[0].dtype))
    x = torch.rand(1, 3, 256, 512, device=DEV)
    for flag16, want in ((False, torch.float32), (True, amp_dtype)):
        model.fuse_volume_conv_train, model.fuse_volume_conv_train16 = not flag16, flag16
        seen.clear()
        with torch.autocast("cuda", dtype=amp_dtype):
            out = model(x, x)
        out[0].float().mean().backward()
        assert seen == [want], (flag16, seen)
    model.zero_grad(set_to_none=True)
    model.to(amp_dtype)
    model.fuse_volume_conv_train, model.fuse_volume_conv_train16 = False, True
    seen.clear()
    out = model(x.to(amp_dtype), x.to(amp_dtype))
    out[0].float().mean().backward()
    assert seen == [amp_dtype]
    assert model.dres0[0][0].weight.grad.dtype == amp_dtype


def test_bf16_autocast_training_step():
    """One config-3 step (256x512, B = 2, BatchNorm conditioned and frozen) under bf16 autocast with
    fuse_volume_conv_train16, with and without channels_last_3d + fuse_upsample: no further from the unfused fp32 step
    than the unfused autocast step of the same configuration is (3x, plus a small floor)."""
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    try:
        batch = ts.make_batch(2, 256, 512, "cuda", seed=7, T=4)
        model = _conditioned_model(batch)
        api = ts.az_api()
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        ref = _step(model, batch, api)
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
        arms = {}
        for cl in (False, True):
            model.use_channels_last_3d(cl)
            model.fuse_upsample = cl
            model.fuse_volume_conv_train16 = False
            unfused = _step(model, batch, api, torch.bfloat16)
            model.fuse_volume_conv_train16 = True
            arms[cl] = (unfused, _step(model, batch, api, torch.bfloat16))
            model.fuse_volume_conv_train16 = False
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    _check_against(ref, arms)


def _check_against(ref, arms):
    for key, (unf, fus) in arms.items():
        d_unf = abs(float(unf[0]) - float(ref[0]))
        assert abs(float(fus[0]) - float(ref[0])) <= 3.0 * d_unf + 1e-5 * abs(float(ref[0])), (key, fus[0], unf[0], ref[0])
        for p, pu, pr in zip(fus[1], unf[1], ref[1]):
            assert _rel(p, pr) <= 3.0 * _rel(pu, pr) + 1e-4, (key, _rel(p, pr), _rel(pu, pr))
        gr = _flat(ref[2])
        assert _rel(_flat(fus[2]), gr) <= 3.0 * _rel(_flat(unf[2]), gr) + 1e-3, (key, _rel(_flat(fus[2]), gr),
                                                                               _rel(_flat(unf[2]), gr))


def test_bf16_model_training_step():
    """The same step for a model converted to bf16: with fuse_volume_conv_train16 no further from the fp32 step than
    the unfused bf16 model is (3x, plus a small floor); every parameter gradient is bf16."""
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    try:
        batch = ts.make_batch(2, 256, 512, "cuda", seed=7, T=4)
        model = _conditioned_model(batch)
        api = ts.az_api()
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        ref = _step(model, batch, api)
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
        m16 = copy.deepcopy(model).to(torch.bfloat16)
        b16 = dict(batch, img_sim_L=batch["img_sim_L"].to(torch.bfloat16), img_sim_R=batch["img_sim_R"].to(torch.bfloat16))
        arms = {}
        for cl in (False, True):
            m16.use_channels_last_3d(cl)
            m16.fuse_upsample = cl
            m16.fuse_volume_conv_train16 = False
            unfused = _step(m16, b16, api)
            m16.fuse_volume_conv_train16 = True
            fused = _step(m16, b16, api)
            m16.fuse_volume_conv_train16 = False
            assert len(fused[2]) == len(ref[2]) and all(g.dtype == torch.bfloat16 for g in fused[2])
            arms[cl] = (unfused, fused)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    _check_against(ref, arms)
