"""GPU: the differentiable first aggregation convolution on the implicit concat volume (ops.volume_conv,
torch.ops.az_stereo.volume_conv; backward in csrc/volume_conv_bwd.cu) and PSMNet's fuse_volume_conv_train flag."""
import ctypes
import itertools

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
SHAPES = [((1, 32, 9, 140), 12), ((2, 32, 6, 128), 8), ((1, 32, 5, 37), 48), ((1, 32, 34, 60), 5), ((1, 32, 3, 300), 20),
          ((1, 32, 4, 240), 48), ((1, 32, 1, 126), 3), ((1, 32, 2, 2), 1), ((2, 32, 3, 127), 55), ((1, 32, 2, 131), 56)]
TRAIN_SHAPE = ((2, 32, 64, 128), 48)  # configs/config.py:93: batch 2 at 256x512, maxdisp 192


def close(a, b, rtol=1e-5, floor=1e-5):
    """|a - b| <= rtol * |b| + floor * max|b| (see tests/test_gpu_parity.py::close for why the floor is there)."""
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    atol = floor * float(b.abs().max()) + 1e-30
    err = (a - b).abs()
    assert bool((err <= atol + rtol * b.abs()).all()), f"max err {float(err.max()):.3e} (atol {atol:.3e})"


def _grads_fused(L, R, w, dq, g):
    Lg, Rg, wg = (t.clone().requires_grad_(True) for t in (L, R, w))
    ops.volume_conv(Lg, Rg, wg, dq).backward(g)
    return Lg.grad, Rg.grad, wg.grad


def _grads_ref64(L, R, w, dq, g, device):
    """float64 autograd of conv3d on the materialised concat volume (the oracle's)."""
    Lg, Rg, wg = (t.detach().to(device, torch.float64).requires_grad_(True) for t in (L, R, w))
    F.conv3d(so.concat_volume(Lg, Rg, dq), wg, padding=1).backward(g.to(device, torch.float64))
    return Lg.grad, Rg.grad, wg.grad


def _inputs(shape, dq, seed):
    torch.manual_seed(seed)
    B, C, H, W = shape
    L, R = torch.randn(shape, device=DEV), torch.randn(shape, device=DEV)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05
    g = torch.randn(B, 32, dq, H, W, device=DEV)
    return L, R, w, g


@pytest.mark.parametrize("shape,dq", SHAPES + [TRAIN_SHAPE])
def test_gradients_match_float64_conv3d_of_materialised_volume(shape, dq):
    """The backward of a linear op does not depend on the TF32 forward: dL, dR, dW against float64 (CPU; on the GPU at
    the training shape, where a float64 CPU convolution takes too long)."""
    L, R, w, g = _inputs(shape, dq, 60)
    mine = _grads_fused(L, R, w, dq, g)
    ref = _grads_ref64(L, R, w, dq, g, "cpu" if shape != TRAIN_SHAPE[0] else DEV)
    for a, b in zip(mine, ref):
        close(a, b)


@pytest.mark.parametrize("shape,dq", [((1, 32, 5, 37), 12), ((2, 32, 4, 40), 8), ((1, 32, 2, 2), 1), ((1, 32, 3, 130), 55),
                                      ((1, 32, 1, 9), 2)])
def test_bit_exact_on_integer_probes(shape, dq):
    """Small integers everywhere: every partial sum of the kernels is an integer below 2^24 (asserted from the
    float64 backward of the absolute values, which bounds every partial sum), so the result is exact."""
    torch.manual_seed(61)
    B, C, H, W = shape
    L = torch.randint(-2, 3, shape, device=DEV).float()
    R = torch.randint(-2, 3, shape, device=DEV).float()
    w = torch.randint(-1, 2, (32, 64, 3, 3, 3), device=DEV).float()
    g = torch.randint(-1, 2, (B, 32, dq, H, W), device=DEV).float()
    bound = _grads_ref64(L.abs(), R.abs(), w.abs(), dq, g.abs(), "cpu")
    assert max(float(t.max()) for t in bound) < 2 ** 24
    for a, b in zip(_grads_fused(L, R, w, dq, g), _grads_ref64(L, R, w, dq, g, "cpu")):
        assert torch.equal(a.double().cpu(), b)


def test_deterministic_and_every_needs_input_grad_subset_agrees():
    (shape, dq) = TRAIN_SHAPE
    L, R, w, g = _inputs(shape, dq, 62)
    full = _grads_fused(L, R, w, dq, g)
    again = _grads_fused(L, R, w, dq, g)
    for a, b in zip(full, again):
        assert torch.equal(a, b), "two calls differ"
    for k in (1, 2):
        for subset in itertools.combinations(range(3), k):
            ts = [t.clone().requires_grad_(i in subset) for i, t in enumerate((L, R, w))]
            ops.volume_conv(*ts, dq).backward(g)
            for i, t in enumerate(ts):
                if i in subset:
                    assert torch.equal(t.grad, full[i]), (subset, i)
                else:
                    assert t.grad is None


def test_empty_batch_enqueues_nothing():
    L = torch.zeros(0, 32, 5, 12, device=DEV, requires_grad=True)
    R = torch.zeros(0, 32, 5, 12, device=DEV, requires_grad=True)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV, requires_grad=True)
    before = _lib.launch_count
    out = ops.volume_conv(L, R, w, 6)
    assert out.shape == (0, 32, 6, 5, 12)
    out.sum().backward()
    assert L.grad.shape == L.shape and R.grad.shape == R.shape and torch.equal(w.grad, torch.zeros_like(w))
    out2 = torch.ops.az_stereo.volume_conv(L.detach(), R.detach(), w.detach(), 6)
    assert out2.shape == (0, 32, 6, 5, 12)
    torch.cuda.synchronize()
    assert _lib.launch_count == before, "an empty batch must not enqueue a kernel"


def test_bad_inputs_are_rejected_before_any_c_abi_call():
    L = torch.randn(1, 32, 4, 16, device=DEV)
    w = torch.randn(32, 64, 3, 3, 3, device=DEV)
    bad = [
        (L.cpu(), L.cpu(), w.cpu(), 4),                             # CPU tensors
        (L.double(), L.double(), w.double(), 4),                    # float64
        (L[:, :16], L[:, :16], w, 4),                               # C != 32
        (L, L[:, :, :3], w, 4),                                     # features of different shapes
        (L[0], L[0], w, 4),                                         # not [B,C,H,W]
        (L, L, w[:, :32], 4),                                       # weight not [32,64,3,3,3]
        (L, L, w.cpu(), 4),                                         # weight on another device
        (L, L, w, 0),                                               # num_disp <= 0
    ]
    before = _lib.launch_count
    for i, args in enumerate(bad):
        with pytest.raises(ValueError):
            ops.volume_conv(*args)
        if i > 0:  # the registered op has CUDA kernels only: the dispatcher refuses all-CPU inputs itself
            with pytest.raises(ValueError):
                torch.ops.az_stereo.volume_conv(*args)
    g = torch.randn(1, 32, 4, 4, 15, device=DEV)  # grad_out of the wrong spatial shape
    with pytest.raises(ValueError):
        torch.ops.az_stereo.volume_conv_backward(g, L, L, w)
    with pytest.raises(ValueError):
        torch.ops.az_stereo.volume_conv_backward(g[:, :16], L, L, w)
    assert _lib.launch_count == before
    null = ctypes.c_void_p(0)
    lib = _lib.load()
    assert lib.az_volume_conv0_bwd(_ptr(g), _ptr(L), _ptr(L), _ptr(w), _ptr(L), null, null, null, 1, 32, 4, 16, 4, null) == -1
    assert lib.az_volume_conv0_bwd(_ptr(g), _ptr(L), _ptr(L), _ptr(w), null, null, null, null, 1, 16, 4, 16, 4, null) == -1


@pytest.mark.parametrize("shape,dq", [((1, 32, 3, 130), 7), ((2, 32, 2, 37), 48), ((1, 32, 5, 254), 3), ((1, 32, 2, 60), 56),
                                      ((1, 32, 1, 1), 1), ((3, 32, 7, 129), 9)])
def test_backward_writes_stay_inside(shape, dq):
    """gL, gR, gW and the workspace are windows between 4 KB canary margins; the results equal the autograd path's."""
    B, C, H, W = shape
    L, R, w, g = _inputs(shape, dq, 63)
    gL, gR, gW = Guarded(shape, torch.float32), Guarded(shape, torch.float32), Guarded((32, 64, 3, 3, 3), torch.float32)
    ws = Guarded((_lib.query("az_volume_conv0_bwd_workspace_bytes", B, H, W, dq),), torch.uint8)
    _lib.call("az_volume_conv0_bwd", _ptr(g), _ptr(L), _ptr(R), _ptr(w), _ptr(gL.t), _ptr(gR.t), _ptr(gW.t), _ptr(ws.t),
              B, C, H, W, dq, _stream())
    torch.cuda.synchronize()
    for buf, name in ((gL, "gL"), (gR, "gR"), (gW, "gW"), (ws, "workspace")):
        buf.check(name)
    for a, b in zip((gL.t, gR.t, gW.t), _grads_fused(L, R, w, dq, g)):
        assert torch.equal(a, b)


def test_opcheck_and_torch_compile():
    torch.manual_seed(64)
    L = torch.randn(2, 32, 5, 24, device=DEV, requires_grad=True)
    R = torch.randn(2, 32, 5, 24, device=DEV, requires_grad=True)
    w = (torch.randn(32, 64, 3, 3, 3, device=DEV) * 0.05).requires_grad_(True)
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.az_stereo.volume_conv.default, (L, R, w, 7), test_utils=checks)

    def step(L, R, w):
        return library_ops.volume_conv(L, R, w, 7).square().mean()

    eager = step(L, R, w)
    compiled = torch.compile(step, backend="aot_eager", fullgraph=True)(L, R, w)
    assert torch.allclose(eager, compiled, rtol=1e-6)
    ge = torch.autograd.grad(eager, [L, R, w])
    gc = torch.autograd.grad(compiled, [L, R, w])
    gf = torch.autograd.grad(ops.volume_conv(L, R, w, 7).square().mean(), [L, R, w])
    for a, b, c in zip(ge, gc, gf):
        assert torch.equal(a, b) and torch.equal(a, c)


# ------------------------------------------------------------------------------ whole network, one config-3 step
def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def test_psmnet_training_step_with_fused_first_conv():
    """One config-3 training step of PSMNet_3 at 256x512, B=2, with BatchNorm conditioned and frozen as in
    test_training_step.py.  The fused step (with and without channels_last_3d) must be no further from the unfused
    fp32 step than the unfused cuDNN-TF32 step is (3x, plus a small floor): loss, predictions, parameter gradients."""
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet
    from benchmarks import train_step as ts

    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    try:
        torch.manual_seed(1)
        model = PSMNet(maxdisp=192).cuda().train()
        batch = ts.make_batch(2, 256, 512, "cuda", seed=7, T=4)
        bns = [m for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
        for m in bns:
            m.momentum = 1.0
        with torch.no_grad():
            model(batch["img_sim_L"], batch["img_sim_R"])
        for m in bns:
            m.eval()
        api = ts.az_api()

        def run(tf32, fused, channels_last):
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
            model.fuse_volume_conv_train = fused
            model.use_channels_last_3d(channels_last)
            model.zero_grad(set_to_none=True)
            tap = _Preds(model)
            loss, _ = ts.sim_step_loss(tap, batch, api)
            loss.backward()
            grads = torch.cat([p.grad.flatten().double() for p in model.parameters() if p.grad is not None])
            return float(loss.detach()), [p.detach().clone() for p in tap.preds], grads

        ref = run(False, False, False)
        tf = run(True, False, False)
        arms = {"fused": run(True, True, False), "fused_channels_last": run(True, True, True)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    loss_tf = abs(tf[0] - ref[0])
    for name, (loss, preds, grads) in arms.items():
        assert abs(loss - ref[0]) <= 3.0 * loss_tf + 1e-6 * abs(ref[0]), (name, loss, ref[0], tf[0])
        for p, p_tf, p_ref in zip(preds, tf[1], ref[1]):
            assert _rel(p, p_ref) <= 3.0 * _rel(p_tf, p_ref) + 1e-5, name
        assert _rel(grads, ref[2]) <= 3.0 * _rel(tf[2], ref[2]) + 1e-4, (name, _rel(grads, ref[2]), _rel(tf[2], ref[2]))


class _Preds(torch.nn.Module):
    """Calls the network and keeps its three predictions."""

    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, *a):
        self.preds = self.net(*a)
        return self.preds
