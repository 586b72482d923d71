"""The drop-in PSMNet modules: checkpoint compatibility (CPU), plain-torch parts
(CPU) and the whole network (GPU) against outputs captured from the real reference."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from activezero_b200.nets.psmnet import psmnet as az_psm6
from activezero_b200.nets.psmnet import psmnet_3 as az_psm3
from activezero_b200.nets.psmnet.psmnet_submodule import DisparityRegression
from oracle import stereo_oracle as so

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name,mod", [("psmnet", az_psm6), ("psmnet_3", az_psm3)])
def test_state_dict_keys_match_reference(name, mod):
    want = json.load(open(os.path.join(GOLDEN, "psmnet_state_dict_keys.json")))[name]
    got = [[k, list(v.shape)] for k, v in mod.PSMNet(maxdisp=192).state_dict().items()]
    assert got == want


def test_forward_signatures():
    import inspect

    assert list(inspect.signature(az_psm6.PSMNet.forward).parameters) == [
        "self", "img_L", "img_R", "img_L_transformed", "img_R_transformed"]
    assert list(inspect.signature(az_psm3.PSMNet.forward).parameters) == ["self", "img_L", "img_R"]
    assert az_psm3.PSMNet().maxdisp == 192


def test_disparity_regression_api():
    p = torch.softmax(torch.randn(2, 16, 3, 4), 1)
    out = DisparityRegression(16)(p)
    ref = (p * torch.arange(16.0).view(1, 16, 1, 1)).sum(1, keepdim=True)
    assert torch.equal(out, ref)


def test_plain_torch_parts_match_reference_modules():
    """The feature extractor and the 3-D aggregation on the CPU against the CPU outputs of the reference PSMNet_3
    stored in tests/golden/psmnet_inline.npz (built under torch.manual_seed(1), fed torch.rand inputs from the same
    stream; the drop-in consumes the RNG identically, so these are the same weights and images).  The CPU
    convolutions' summation order depends on the thread count, so fp32 rounding is allowed: 1e-5 of each
    tensor's scale."""
    g = np.load(os.path.join(GOLDEN, "psmnet_inline.npz"))
    torch.manual_seed(1)
    net = az_psm3.PSMNet(maxdisp=192).eval()
    img_L, img_R = torch.rand(1, 3, 256, 256), torch.rand(1, 3, 256, 256)
    with torch.no_grad():
        feat_L, feat_R = net.feature_extraction(img_L), net.feature_extraction(img_R)
        vol = so.concat_volume(feat_L, feat_R, 48)
        _, _, cost3 = net._aggregate(vol)
        logits = F.interpolate(cost3, (192, 256, 256), mode="trilinear", align_corners=False)[:, 0]
    ch, rows, C = [3, 17], slice(20, 24), feat_L.shape[1]
    got = {"feat_L": feat_L[:, ch, rows], "feat_R": feat_R[:, ch, rows],
           "vol": vol[:, ch + [C + c for c in ch], :, rows], "logits": logits[:, :, 100:104, 64:96]}
    for name, t in got.items():
        want = g[name]
        np.testing.assert_allclose(t.numpy(), want, rtol=1e-5, atol=1e-5 * np.abs(want).max(), err_msg=name)


@pytest.mark.gpu
def test_psmnet_end_to_end_against_reference_outputs():
    """tests/golden/psmnet_inline.npz was captured from the reference PSMNet_3 built
    under torch.manual_seed(1) and fed torch.rand inputs from the same stream; the
    drop-in consumes the RNG identically, so it is the same network on the same
    images.  cuDNN vs the CPU convolutions differ at ~1e-4 relative."""
    g = np.load(os.path.join(GOLDEN, "psmnet_inline.npz"))
    torch.manual_seed(1)
    net = az_psm3.PSMNet(maxdisp=192).eval()
    img_L, img_R = torch.rand(1, 3, 256, 256), torch.rand(1, 3, 256, 256)
    net = net.cuda()
    feats = []
    net.feature_extraction.register_forward_hook(lambda m, i, o: feats.append(o.detach()))
    vols = []
    net.dres0.register_forward_pre_hook(lambda m, i: vols.append(i[0].detach()))
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            pred = net(img_L.cuda(), img_R.cuda())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    assert pred.shape == (1, 1, 256, 256)
    ch, rows = [3, 17], slice(20, 24)
    fl = feats[0][:, ch, rows].cpu().numpy()
    np.testing.assert_allclose(fl, g["feat_L"], rtol=2e-3, atol=2e-3 * np.abs(g["feat_L"]).max())
    # the volume is an exact rearrangement of the features that entered it
    assert torch.equal(vols[0], so.concat_volume(feats[0], feats[1], 48))
    np.testing.assert_allclose(pred[:, :, 100:104, 64:96].cpu().numpy(), g["pred"], atol=2e-2)


@pytest.mark.gpu
def test_psmnet_train_mode_backward():
    torch.manual_seed(0)
    net = az_psm6.PSMNet(maxdisp=48).cuda().train()
    a = [torch.rand(2, 3, 256, 256, device="cuda") for _ in range(4)]  # BN in the 1x1 SPP branch needs > 1 sample
    p3, p2, p1 = net(*a)
    assert p3.shape == p2.shape == p1.shape == (2, 1, 256, 256)
    (p3.mean() + 0.7 * p2.mean() + 0.5 * p1.mean()).backward()
    g = net.feature_extraction.firstconv[0][0].weight.grad
    assert g is not None and torch.isfinite(g).all() and float(g.abs().max()) > 0
    g3 = net.classif3[2].weight.grad
    assert torch.isfinite(g3).all() and float(g3.abs().max()) > 0


@pytest.mark.gpu
def test_psmnet_channels_last_3d_volume_same_predictions_and_gradients():
    """use_channels_last_3d() changes strides only: same state_dict, same prediction (TF32 off so that the
    different cuDNN algorithms agree to rounding), and training gradients flow through the in-place
    channels_last_3d backward of the volume."""
    torch.manual_seed(3)
    net = az_psm3.PSMNet(maxdisp=96).cuda().eval()
    keys = [(k, tuple(v.shape)) for k, v in net.state_dict().items()]
    x, y = torch.rand(1, 3, 256, 256, device="cuda"), torch.rand(1, 3, 256, 256, device="cuda")  # SPP needs >= 256
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            p0 = net(x, y)
            net.use_channels_last_3d(True)
            vols = []
            h = net.dres0.register_forward_pre_hook(lambda m, i: vols.append(i[0]))
            p1 = net(x, y)
            h.remove()
        assert vols[0].is_contiguous(memory_format=torch.channels_last_3d) and not vols[0].is_contiguous()
        assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == keys
        assert float((p0 - p1).abs().max()) <= 2e-3, float((p0 - p1).abs().max())
        # gradients: channels_last_3d vs NCDHW volume, same network
        grads = []
        for cl in (True, False):
            net.use_channels_last_3d(cl).train()
            net.zero_grad(set_to_none=True)
            torch.manual_seed(5)
            p3, p2, pa = net(torch.cat([x, x * 0.5]), torch.cat([y, y * 0.5]))
            (p3.mean() + 0.7 * p2.mean() + 0.5 * pa.mean()).backward()
            grads.append(net.feature_extraction.firstconv[0][0].weight.grad.clone())
        scale = float(grads[1].abs().max())
        assert scale > 0 and float((grads[0] - grads[1]).abs().max()) <= 2e-2 * scale
    finally:
        torch.backends.cudnn.allow_tf32 = prev
