"""GPU: image gradients of the fused reprojection loss (DESIGN.md §4.14; include/az_stereo.h:
az_reproj_loss_img_bwd) -- against float64 autograd of the oracle's reprojection.py:81-127, the forward and the
disparity gradient untouched, determinism, the empty mask / empty batch, guard bands, rejections, the torch.library
op and the get_reproj_error_patch drop-in."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import stereo_oracle as so  # noqa: E402  (checker only)

if torch.cuda.is_available():
    from activezero_b200 import _lib, library_ops, ops
    from activezero_b200.ops import _ptr, _stream, linspace_table
    from activezero_b200.utils import reprojection as az_rp

DEV = "cuda:0"
GUARD = 4096


def close(a, b, rtol=1e-5, floor=1e-5):
    """|a - b| <= rtol * |b| + floor * max|b| (tests/test_gpu_parity.py::close)."""
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    atol = floor * float(b.abs().max()) + 1e-30
    err = (a - b).abs()
    assert bool((err <= atol + rtol * b.abs()).all()), f"max err {float(err.max()):.3e} (atol {atol:.3e})"


def _case(B, C, H, W, seed, field, masked=True):
    """The fields of tests/test_gpu_round2.py::_patch_case."""
    gen = torch.Generator().manual_seed(seed)
    L = torch.rand(B, C, H, W, generator=gen)
    R = torch.rand(B, C, H, W, generator=gen)
    if field == "random":
        d = torch.rand(B, 1, H, W, generator=gen) * min(64.0, W / 3)
    elif field == "smooth":
        d = (W / 10 + W / 16 * torch.sin(torch.arange(W).float() / 9).view(1, 1, 1, W)
             + 3 * torch.cos(torch.arange(H).float() / 5).view(1, 1, H, 1)).expand(B, 1, H, W).contiguous()
    else:  # samples leaving the image on both sides, boundary cells included
        d = (torch.rand(B, 1, H, W, generator=gen) - 0.5) * 3.0 * W
    m = (torch.rand(B, 1, H, W, generator=gen) > 0.3) if masked else None
    return L, R, d, m


def _kernel_xs(d, sign, W):
    """The kernels' fp32 sample x (common.cuh: sample_pos): f = lin + disp/W, g = 2f - 1, then (g+1)*W - 1 as ONE
    fused multiply-add, as torch's grid_sampler evaluates it, and the halving.  The product of two fp32 values is exact
    in float64, so rounding it minus 1 to fp32 once is the FMA."""
    lin = torch.linspace(0, 1, W, dtype=torch.float32).view(1, 1, W)
    f = lin + (sign * d[:, 0]) / W
    gp1 = (2 * f - 1) + 1
    return (gp1.double() * W - 1).float() * 0.5


def _ref64(L, R, d, m, ps, sign, old=False):
    """float64 autograd of the oracle, on the GPU, sampling at the kernels' fp32 x positions (a float64 disparity
    that reproduces them; fp32 positions are off by up to ulp(W) px, which alone would move the gradients by more
    than the gate at W = 2610).  -> (loss, d loss/d tgt, d loss/d src)."""
    B, C, H, W = L.shape
    xs = _kernel_xs(d, sign, W)
    lin = torch.linspace(0, 1, W).double().view(1, 1, W)
    pred = (-(xs.double() + 0.5 - lin * W))[:, None].to(DEV)
    Lg = L.double().to(DEV).requires_grad_(True)
    Rg = R.double().to(DEV).requires_grad_(True)
    mg = None if m is None else m.to(DEV)
    if old:
        loss, _, _ = so.reproj_error_old(Lg, Rg, pred, mg)
    else:
        loss, _, _ = so.reproj_error_patch(Lg, Rg, pred, mg, ps=ps)
    loss.backward()
    return loss.item(), Lg.grad, Rg.grad


def _fused(L, R, d, m, ps, sign, need=(True, True, False)):
    Lg = L.to(DEV).requires_grad_(need[0])
    Rg = R.to(DEV).requires_grad_(need[1])
    dg = d.to(DEV).requires_grad_(need[2])
    # want_warped: at W = 2610 only the x-tiled kernel (loss + Fold image) stages the rows
    loss, _ = ops.reproj_loss(Lg, Rg, dg, None if m is None else m.to(DEV), ps=ps, sign=sign, want_warped=True)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), Lg.grad, Rg.grad, dg.grad


CASES = [  # (B, C, H, W), ps, field, masked, sign
    ((1, 1, 24, 40), 1, "random", True, -1.0), ((1, 3, 17, 45), 1, "wild", False, 1.0),
    ((1, 1, 24, 40), 3, "random", True, -1.0), ((2, 1, 19, 33), 5, "smooth", True, 1.0),
    ((1, 3, 21, 37), 5, "wild", True, -1.0), ((1, 1, 30, 61), 11, "random", True, -1.0),
    ((2, 1, 23, 50), 11, "wild", False, 1.0), ((1, 3, 16, 29), 13, "smooth", True, -1.0),
    ((1, 1, 20, 31), 15, "random", True, -1.0), ((1, 2, 11, 9), 15, "wild", True, 1.0),
    ((1, 32, 12, 20), 11, "random", True, -1.0), ((1, 1, 7, 5), 11, "wild", True, -1.0),
    ((1, 1, 4, 70), 9, "random", False, -1.0), ((1, 1, 9, 4), 7, "smooth", True, 1.0),
    ((1, 1, 16, 1920), 11, "random", True, -1.0), ((1, 1, 12, 2610), 11, "smooth", True, -1.0),
    ((1, 1, 10, 2610), 11, "wild", False, 1.0),
]


@pytest.mark.parametrize("shape,ps,field,masked,sign", CASES)
def test_image_gradients_match_float64_oracle(shape, ps, field, masked, sign):
    """gtgt and gsrc against float64 autograd of reprojection.py:99-127.  Each image alone, both, with and without
    the disparity: every subset takes the same kernels, so the gradients are bit-identical across subsets."""
    L, R, d, m = _case(*shape, seed=sum(shape) + ps, field=field, masked=masked)
    ref, gL, gR = _ref64(L, R, d, m, ps, sign)
    loss, fL, fR, _ = _fused(L, R, d, m, ps, sign)
    assert abs(loss - ref) <= 1e-5 * abs(ref), (loss, ref)
    close(fL, gL)
    close(fR, gR)
    for need in [(True, False, False), (False, True, True), (True, True, True)]:
        _, aL, aR, ad = _fused(L, R, d, m, ps, sign, need)
        assert (aL is None) != need[0] and (aR is None) != need[1] and (ad is None) != need[2]
        if need[0]:
            assert torch.equal(aL, fL)
        if need[1]:
            assert torch.equal(aR, fR)


@pytest.mark.parametrize("masked", [True, False])
def test_ps1_matches_reproj_error_old(masked):
    """ps = 1 is reprojection.py:81-96 (get_reprojection_error_old)."""
    L, R, d, m = _case(2, 3, 26, 44, seed=3, field="random", masked=masked)
    ref, gL, gR = _ref64(L, R, d, m, 1, -1.0, old=True)
    loss, fL, fR, _ = _fused(L, R, d, m, 1, -1.0)
    assert abs(loss - ref) <= 1e-5 * abs(ref)
    close(fL, gL)
    close(fR, gR)


@pytest.mark.parametrize("ps,shape", [(1, (2, 3, 32, 48)), (5, (1, 2, 33, 71)), (11, (2, 1, 40, 96)),
                                      (11, (1, 1, 20, 2610))])
def test_forward_and_disparity_gradient_untouched(ps, shape):
    """The loss, the warped / Fold image and d loss / d disp are bit-identical whether or not an image requires grad."""
    L, R, d, m = _case(*shape, seed=5, field="random")
    Lg, Rg, mg = L.to(DEV), R.to(DEV), m.to(DEV)
    out = []
    for img_grad in (False, True):
        dg = d.to(DEV).requires_grad_(True)
        Rr = Rg.clone().requires_grad_(img_grad)
        loss, warped = ops.reproj_loss(Lg, Rr, dg, mg, ps=ps, want_warped=True)
        loss.backward()
        out.append((loss.detach(), warped, dg.grad))
    torch.cuda.synchronize()
    for a, b in zip(*out):
        assert torch.equal(a, b)


def test_deterministic_at_config3():
    """Two runs give bit-identical image gradients (fixed-order sums and fixed-point accumulation, no float atomics)."""
    L, R, d, m = _case(2, 1, 256, 512, seed=7, field="random")
    g1 = _fused(L, R, d, m, 11, -1.0, (True, True, True))
    g2 = _fused(L, R, d, m, 11, -1.0, (True, True, True))
    for a, b in zip(g1[1:], g2[1:]):
        assert torch.equal(a, b)


def test_empty_mask_gives_exact_zero_image_gradients_and_nan_loss():
    L, R, d, _ = _case(1, 2, 20, 30, seed=8, field="random")
    m = torch.zeros(1, 1, 20, 30, dtype=torch.bool)
    loss, fL, fR, fd = _fused(L, R, d, m, 5, -1.0, (True, True, True))
    assert loss != loss
    assert bool((fL == 0).all()) and bool((fR == 0).all())
    assert not torch.signbit(fL).any() and not torch.signbit(fR).any()


def test_empty_batch_gives_empty_gradients():
    L = torch.rand(0, 2, 8, 12, device=DEV, requires_grad=True)
    R = torch.rand(0, 2, 8, 12, device=DEV, requires_grad=True)
    d = torch.rand(0, 1, 8, 12, device=DEV, requires_grad=True)
    loss, _ = ops.reproj_loss(L, R, d, None, ps=5)
    loss.backward()
    assert L.grad.shape == L.shape and R.grad.shape == R.shape and d.grad.shape == d.shape


def test_non_finite_inputs_propagate_as_nan():
    L, R, d, m = _case(1, 1, 12, 20, seed=9, field="random", masked=False)
    R[0, 0, 5, 7] = float("nan")
    _, fL, fR, _ = _fused(L, R, d, m, 3, -1.0)
    assert torch.isnan(fR).any() and torch.isnan(fL).any()
    assert not torch.isinf(fR).any()


def _raw(t, s, d, mask, ps, stats, gl, gtgt, gsrc, sign=-1.0, dims=None):
    B, C, H, W = dims or t.shape
    lx, ly = linspace_table(max(W, 1), DEV), linspace_table(max(H, 1), DEV)  # rejected sizes still get tables
    return _lib.load().az_reproj_loss_img_bwd(_ptr(t), _ptr(s), _ptr(d), sign, _ptr(mask), _ptr(lx), _ptr(ly), ps,
                                              _ptr(stats), _ptr(gl), _ptr(gtgt), _ptr(gsrc), B, C, H, W, _stream())


@pytest.mark.parametrize("shape,ps", [((1, 1, 7, 5), 11), ((2, 3, 13, 37), 5), ((1, 2, 9, 261), 15),
                                      ((1, 1, 5, 8193), 3), ((1, 1, 3, 33), 1)])
def test_guard_bands_around_the_raw_call(shape, ps):
    """Every element of gtgt / gsrc is written once (a NaN pre-fill disappears) and nothing outside them is: both
    outputs sit inside larger allocations whose margins hold a canary.  W = 8193 splits gsrc into two column tiles."""
    L, R, d, m = _case(*shape, seed=10, field="wild")
    t, s, dd, mu = L.to(DEV), R.to(DEV), d.to(DEV), m.to(DEV).view(torch.uint8)
    stats = torch.tensor([1.0, float(m.sum())], dtype=torch.float64, device=DEV)
    gl = torch.tensor([0.5], device=DEV)
    n = t.numel()
    bufs = [torch.full((GUARD + n + GUARD,), float("nan"), device=DEV) for _ in range(2)]
    for b in bufs:
        b[:GUARD] = 7.0
        b[GUARD + n:] = 7.0
    gt, gs = (b[GUARD:GUARD + n].view(shape) for b in bufs)
    assert _raw(t, s, dd, mu, ps, stats, gl, gt, gs) == 0
    torch.cuda.synchronize()
    for b in bufs:
        assert bool((b[:GUARD] == 7.0).all()) and bool((b[GUARD + n:] == 7.0).all())
    assert bool(torch.isfinite(gt).all()) and bool(torch.isfinite(gs).all())
    et, es = torch.empty_like(t), torch.empty_like(s)
    ops.reproj_image_backward_into(t, s, dd, mu, stats, gl, -1.0, ps, et, es)
    assert torch.equal(et, gt) and torch.equal(es, gs)


def test_rejections_before_any_launch():
    t = torch.rand(1, 1, 8, 12, device=DEV)
    d = torch.rand(1, 1, 8, 12, device=DEV)
    stats = torch.tensor([1.0, 96.0], dtype=torch.float64, device=DEV)
    gl = torch.ones(1, device=DEV)
    out = torch.empty_like(t)
    null = None
    assert _raw(t, t, d, null, 5, stats, gl, null, null) == 0  # nothing asked for
    assert _raw(t, t, d, null, 4, stats, gl, out, out) == -1   # even ps
    assert _raw(t, t, d, null, 5, null, gl, out, out) == -1    # no stats
    assert _raw(t, t, d, null, 5, stats, null, out, null) == -1
    assert _raw(null, t, d, null, 5, stats, gl, out, null, dims=tuple(t.shape)) == -1
    assert _raw(t, t, d, null, 5, stats, gl, out, out, dims=(0, 1, 8, 12)) == -1
    assert _raw(t, t, d, null, 5, stats, gl, out, out, dims=(1, 1, 8, -1)) == -1
    assert _raw(t, t, d, null, 5, stats, gl, out, out, dims=(70000, 1, 8, 12)) == -1
    img_bwd = torch.ops.az_stereo.reproj_loss_image_backward
    with pytest.raises(ValueError):
        img_bwd(t, t[:, :, :4], d, None, stats, gl, -1.0, 5)
    with pytest.raises(ValueError):
        img_bwd(t, t, d, None, stats.float(), gl, -1.0, 5)
    with pytest.raises(ValueError):
        img_bwd(t, t, d, torch.ones(1, 1, 4, 12, device=DEV), stats, gl, -1.0, 5)
    with pytest.raises(ValueError):
        img_bwd(t, t, d, None, stats, gl, -1.0, 4)
    with pytest.raises(ValueError):
        img_bwd(t.cpu(), t, d, None, stats, gl, -1.0, 5)
    torch.cuda.synchronize()


def test_library_op_opcheck_and_function_layer():
    L, R, d, m = _case(2, 3, 14, 40, seed=11, field="random")
    Lg, Rg, dg, mg = L.to(DEV), R.to(DEV), d.to(DEV), m.to(DEV)
    loss, _, _, stats = torch.ops.az_stereo.reproj_loss(Lg, Rg, dg, mg, 5, -1.0)
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.az_stereo.reproj_loss_image_backward.default,
                          (Lg, Rg, dg, mg, stats, torch.ones((), device=DEV), -1.0, 5), test_utils=checks)
    args = (Lg.clone().requires_grad_(True), Rg.clone().requires_grad_(True), dg.clone().requires_grad_(True), mg, 5, -1.0)
    torch.library.opcheck(torch.ops.az_stereo.reproj_loss.default, args, test_utils=checks)
    # the registered autograd formula equals the Function layer bit for bit (the library op always runs the pass
    # that also writes the Fold image, so the Function layer is asked for it too)
    a = [t.clone().requires_grad_(True) for t in (Lg, Rg, dg)]
    b = [t.clone().requires_grad_(True) for t in (Lg, Rg, dg)]
    ga = torch.autograd.grad(library_ops.reproj_loss(*a, mg, ps=5)[0] * 0.3, a)
    gb = torch.autograd.grad(ops.reproj_loss(*b, mg, ps=5, want_warped=True)[0] * 0.3, b)
    for x, y in zip(ga, gb):
        assert torch.equal(x, y)


def test_torch_compile_fullgraph_forward_and_backward():
    L, R, d, m = _case(1, 2, 20, 48, seed=12, field="smooth")
    Lg, Rg, dg, mg = L.to(DEV), R.to(DEV), d.to(DEV), m.to(DEV)

    def step(a, b, c):
        loss, _ = library_ops.reproj_loss(a, b, c, mg, ps=7)
        return loss * 2.0

    def run(fn):
        ts = [t.clone().requires_grad_(True) for t in (Lg, Rg, dg)]
        out = fn(*ts)
        return (out.detach(), *torch.autograd.grad(out, ts))

    eager = run(step)
    compiled = run(torch.compile(step, backend="aot_eager", fullgraph=True))
    fn_layer = run(lambda a, b, c: ops.reproj_loss(a, b, c, mg, ps=7, want_warped=True)[0] * 2.0)
    for x, y, z in zip(eager, compiled, fn_layer):
        assert torch.equal(x, y) and torch.equal(x, z)


@pytest.mark.parametrize("shape,ps,fold", [((1, 1, 24, 40), 5, True), ((2, 3, 20, 52), 11, True),
                                           ((1, 1, 12, 2610), 11, False), ((1, 1, 12, 2610), 11, True)])
def test_drop_in_with_image_gradient(shape, ps, fold, monkeypatch):
    """get_reproj_error_patch with an image that requires grad takes the fused operator and matches the oracle,
    including RETURN_WARPED_PATCH_IMAGE = False at a width only the x-tiled kernel stages."""
    monkeypatch.setattr(az_rp, "RETURN_WARPED_PATCH_IMAGE", fold)
    L, R, d, m = _case(*shape, seed=13, field="random")
    ref, gL, gR = _ref64(L, R, d, m, ps, -1.0)
    Lg, Rg = L.to(DEV).requires_grad_(True), R.to(DEV).requires_grad_(True)
    loss, vis, mi = az_rp.get_reproj_error_patch(Lg, Rg, d.to(DEV), m.to(DEV), ps=ps)
    loss.backward()
    assert abs(loss.item() - ref) <= 1e-5 * abs(ref)
    close(Lg.grad, gL)
    close(Rg.grad, gR)
    assert (vis is not None) == fold
    assert mi.shape == shape
