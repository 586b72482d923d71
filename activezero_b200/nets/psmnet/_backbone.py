"""Plain-torch parts of PSMNet that surround the hot path (2-D feature CNN + SPP,
stacked 3-D hourglass).  They are OUT OF SCOPE for the CUDA work (dense
convolutions stay cuDNN, BASELINE.json north_star) and exist only so that the
drop-in ``PSMNet`` modules have the reference's exact module tree: identical
submodule names, parameter shapes and ``state_dict`` keys, so checkpoints saved
by the reference trainer (``/root/reference/train.py:155-170``) load unchanged.

Layer hyper-parameters follow ``/root/reference/nets/psmnet/psmnet_submodule.py``
(:13-56 helpers, :59-77 residual block, :92-223 feature extractor) and
``/root/reference/nets/psmnet/psmnet.py`` (:11-77 hourglass, :85-117 heads,
:123-142 initialisation).
"""
from __future__ import annotations

import contextlib
import math

import torch
import torch.nn as nn
import torch.nn.functional as F


def convbn(in_planes, out_planes, kernel_size, stride, pad, dilation):
    """Conv2d (no bias) + BatchNorm2d; a dilated conv pads by its dilation."""
    conv = nn.Conv2d(in_planes, out_planes, kernel_size=kernel_size, stride=stride,
                     padding=dilation if dilation > 1 else pad, dilation=dilation, bias=False)
    return nn.Sequential(conv, nn.BatchNorm2d(out_planes))


def conv(in_planes, out_planes, kernel_size, stride, pad, dilation):
    """Conv2d (no bias) alone, wrapped like the reference wraps it."""
    return nn.Sequential(nn.Conv2d(in_planes, out_planes, kernel_size=kernel_size, stride=stride,
                                   padding=dilation if dilation > 1 else pad, dilation=dilation, bias=False))


def convbn_3d(in_planes, out_planes, kernel_size, stride, pad):
    """Conv3d (no bias) + BatchNorm3d."""
    return nn.Sequential(nn.Conv3d(in_planes, out_planes, kernel_size=kernel_size, padding=pad, stride=stride,
                                   bias=False), nn.BatchNorm3d(out_planes))


class BasicBlock(nn.Module):
    """Two 3x3 conv-bn layers with an identity / projected skip (no ReLU after the sum)."""
    expansion = 1

    def __init__(self, inplanes, planes, stride, downsample, pad, dilation):
        super().__init__()
        self.conv1 = nn.Sequential(convbn(inplanes, planes, 3, stride, pad, dilation), nn.ReLU(inplace=True))
        self.conv2 = convbn(planes, planes, 3, 1, pad, dilation)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        y = self.conv2(self.conv1(x))
        skip = x if self.downsample is None else self.downsample(x)
        y += skip
        return y


class FeatureExtractionBase(nn.Module):
    """Shared by the 6-channel (image + adapter output) and 3-channel variants."""

    def __init__(self, in_channels: int):
        super().__init__()
        self.inplanes = 32
        stem = []
        for cin, stride in ((in_channels, 2), (32, 1), (32, 1)):
            stem += [convbn(cin, 32, 3, stride, 1, 1), nn.ReLU(inplace=True)]
        self.firstconv = nn.Sequential(*stem)
        self.layer1 = self._make_layer(BasicBlock, 32, 3, 1, 1, 1)
        self.layer2 = self._make_layer(BasicBlock, 64, 16, 2, 1, 1)
        self.layer3 = self._make_layer(BasicBlock, 128, 3, 1, 1, 1)
        self.layer4 = self._make_layer(BasicBlock, 128, 3, 1, 1, 2)
        for idx, win in ((1, 64), (2, 32), (3, 16), (4, 8)):
            setattr(self, f"branch{idx}", nn.Sequential(nn.AvgPool2d((win, win), stride=(win, win)),
                                                        convbn(128, 32, 1, 1, 0, 1), nn.ReLU(inplace=True)))
        self.lastconv = nn.Sequential(convbn(320, 128, 3, 1, 1, 1), nn.ReLU(inplace=True),
                                      nn.Conv2d(128, 32, kernel_size=1, padding=0, stride=1, bias=False))

    def _make_layer(self, block, planes, blocks, stride, pad, dilation):
        proj = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            proj = nn.Sequential(nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride,
                                           bias=False), nn.BatchNorm2d(planes * block.expansion))
        stack = [block(self.inplanes, planes, stride, proj, pad, dilation)]
        self.inplanes = planes * block.expansion
        stack += [block(self.inplanes, planes, 1, None, pad, dilation) for _ in range(1, blocks)]
        return nn.Sequential(*stack)

    def _features(self, x):
        y = self.layer1(self.firstconv(x))
        raw = self.layer2(y)
        skip = self.layer4(self.layer3(raw))
        size = skip.shape[-2:]
        pooled = [F.interpolate(getattr(self, f"branch{k}")(skip), size, mode="bilinear", align_corners=True)
                  for k in (4, 3, 2, 1)]
        return self.lastconv(torch.cat([raw, skip] + pooled, 1))


class hourglass(nn.Module):
    """3-D encoder/decoder: two stride-2 convs down, two transposed convs up."""

    def __init__(self, inplanes):
        super().__init__()
        c2 = inplanes * 2
        self.conv1 = nn.Sequential(convbn_3d(inplanes, c2, kernel_size=3, stride=2, pad=1), nn.ReLU(inplace=True))
        self.conv2 = convbn_3d(c2, c2, kernel_size=3, stride=1, pad=1)
        self.conv3 = nn.Sequential(convbn_3d(c2, c2, kernel_size=3, stride=2, pad=1), nn.ReLU(inplace=True))
        self.conv4 = nn.Sequential(convbn_3d(c2, c2, kernel_size=3, stride=1, pad=1), nn.ReLU(inplace=True))
        self.conv5 = nn.Sequential(nn.ConvTranspose3d(c2, c2, kernel_size=3, padding=1, output_padding=1, stride=2,
                                                      bias=False), nn.BatchNorm3d(c2))
        self.conv6 = nn.Sequential(nn.ConvTranspose3d(c2, inplanes, kernel_size=3, padding=1, output_padding=1,
                                                      stride=2, bias=False), nn.BatchNorm3d(inplanes))

    def forward(self, x, presqu, postqu):
        pre = self.conv2(self.conv1(x))
        pre = F.relu(pre if postqu is None else pre + postqu, inplace=True)
        mid = self.conv4(self.conv3(pre))
        post = F.relu(self.conv5(mid) + (pre if presqu is None else presqu), inplace=True)
        return self.conv6(post), pre, post


def _head():
    return nn.Sequential(convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True),
                         nn.Conv3d(32, 1, kernel_size=3, padding=1, stride=1, bias=False))


class PSMNetBase(nn.Module):
    """Module tree of the reference PSMNet (psmnet.py:80-142); subclasses give the
    feature extractor and the ``forward`` signature."""

    def __init__(self, feature_extraction: nn.Module, maxdisp: int = 192):
        super().__init__()
        self.maxdisp = maxdisp
        # False = the reference's dataflow (F.interpolate then soft-argmin on the 401 MB logits);
        # True = the fused upsample+soft-argmin kernel (same result to <= 1e-4 px).
        self.fuse_upsample = False
        # False = the reference's NCDHW volume; True = the same volume emitted in torch.channels_last_3d memory
        # format (SURVEY.md §8f rank 2), in which cuDNN runs the 3-D aggregation below without layout passes
        # (2-2.6x faster on B200, benchmarks/agg_layout_probe.py).  Set it with use_channels_last_3d().
        self.volume_channels_last = False
        # True (inference only): dres0's first Conv3d + BatchNorm + ReLU run as ONE tensor-core kernel that gathers the
        # concat volume's values straight from the two feature maps (SURVEY.md §8f rank 2, implicit clause): the
        # [B,64,D/4,H/4,W/4] volume is never written nor re-read.  TF32 operands like cuDNN's default conv path.
        self.fuse_volume_conv = False
        # True: every forward that records gradients (training, or eval with grad enabled) computes dres0's first Conv3d
        # on the implicit volume too (ops.volume_conv: tcgen05 TF32 forward, volume-free fp32 backward); its BatchNorm3d
        # (in the module's own mode) and ReLU stay in torch.  Neither the volume nor its gradient is materialised.
        self.fuse_volume_conv_train = False
        self._vc_cache = None
        self.feature_extraction = feature_extraction
        self.dres0 = nn.Sequential(convbn_3d(64, 32, 3, 1, 1), nn.ReLU(inplace=True),
                                   convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True))
        self.dres1 = nn.Sequential(convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True), convbn_3d(32, 32, 3, 1, 1))
        self.dres2 = hourglass(32)
        self.dres3 = hourglass(32)
        self.dres4 = hourglass(32)
        self.classif1 = _head()
        self.classif2 = _head()
        self.classif3 = _head()
        self._init_weights()

    def _init_weights(self):
        # psmnet.py:123-142: He-normal convs (fan = k*k[*k]*out_channels), unit BN, zero Linear bias
        for m in self.modules():
            if isinstance(m, (nn.Conv2d, nn.Conv3d)):
                fan = m.out_channels
                for k in m.kernel_size:
                    fan *= k
                m.weight.data.normal_(0, math.sqrt(2.0 / fan))
            elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm3d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
            elif isinstance(m, nn.Linear):
                m.bias.data.zero_()

    # -- the part of forward() after feature extraction -------------------------------------
    def use_channels_last_3d(self, enable: bool = True):
        """Emit the cost volume in channels_last_3d and keep the 3-D convolution weights in the same format.
        Shapes, state_dict keys and values are unchanged (checkpoints load either way); only strides differ."""
        self.volume_channels_last = bool(enable)
        fmt = torch.channels_last_3d if enable else torch.contiguous_format
        for m in self.modules():
            if isinstance(m, (nn.Conv3d, nn.ConvTranspose3d)):
                m.weight.data = m.weight.data.contiguous(memory_format=fmt)
        return self

    def _first_conv_implicit(self, ref_feat, tgt_feat):
        """dres0[0] (Conv3d 64->32 + BatchNorm3d, eval statistics) + dres0[1] (ReLU) on the IMPLICIT volume.  16-bit
        features give a 16-bit output, with the weight rounded to their dtype as autocast rounds cuDNN's."""
        from ... import ops

        conv, bn = self.dres0[0][0], self.dres0[0][1]
        key = (conv.weight.data_ptr(), conv.weight._version, str(conv.weight.device), ref_feat.dtype)
        if self._vc_cache is None or self._vc_cache[0] != key:
            self._vc_cache = (key, ops.pack_volume_conv_weight(conv.weight, dtype=ref_feat.dtype))
        # the fold is fp32 (the kernel applies it in fp32); a converted 16-bit model's parameters are widened exactly
        scale = bn.weight.detach().float() * torch.rsqrt(bn.running_var.float() + bn.eps)
        shift = bn.bias.detach().float() - bn.running_mean.float() * scale
        return ops.volume_conv0(ref_feat, tgt_feat, self._vc_cache[1], self.maxdisp // 4, scale, shift, relu=True)

    def _aggregate(self, cost, first=None):
        """psmnet.py:167-181: dres0..4 and the three residual classification heads.  ``first`` = output of
        dres0[0:2] when it was computed on the implicit volume."""
        cost0 = self.dres0(cost) if first is None else self.dres0[3](self.dres0[2](first))
        cost0 = self.dres1(cost0) + cost0
        out1, pre1, post1 = self.dres2(cost0, None, None)
        out1 = out1 + cost0
        out2, pre2, post2 = self.dres3(out1, pre1, post1)
        out2 = out2 + cost0
        out3, pre3, post3 = self.dres4(out2, pre1, post2)
        out3 = out3 + cost0
        cost1 = self.classif1(out1)
        cost2 = self.classif2(out2) + cost1
        cost3 = self.classif3(out3) + cost2
        return cost1, cost2, cost3

    def _disparity_head(self, cost, H, W):
        """psmnet.py:186-217 for one head: trilinear upsample to (maxdisp, 4H, 4W), then the
        fused soft-argmin (replaces softmax + DisparityRegression)."""
        from ... import ops

        if self.fuse_upsample:
            # SURVEY.md §8f rank 1: never materialise the [B,maxdisp,4H,4W] logits
            return ops.upsample_soft_argmin(cost, (self.maxdisp, 4 * H, 4 * W))
        up = F.interpolate(cost, (self.maxdisp, 4 * H, 4 * W), mode="trilinear", align_corners=False)
        return ops.soft_argmin(torch.squeeze(up, 1))

    @staticmethod
    def _native16(ref_feat, tgt_feat):
        """A context in which the volume operators take the features as they are: under torch.autocast with features of
        the autocast dtype (bf16 / fp16; the feature extractor ends in a Conv2d), autocast is switched off around
        the call, so the volume (or the first convolution's output) is produced in 16 bits directly instead of in
        fp32 and cast down by the next convolution.  The concat volume and its gradients are bit-identical to that
        dataflow's (DESIGN.md §4.11).  Otherwise a no-op."""
        if torch.is_autocast_enabled("cuda"):
            dt = torch.get_autocast_dtype("cuda")
            if dt in (torch.bfloat16, torch.float16) and ref_feat.dtype == dt and tgt_feat.dtype == dt:
                return torch.autocast("cuda", enabled=False)
        return contextlib.nullcontext()

    def _forward_features(self, ref_feat, tgt_feat):
        from ... import ops

        H, W = ref_feat.shape[-2:]
        if self.fuse_volume_conv and not self.training and not torch.is_grad_enabled() and ref_feat.shape[1] == 32:
            with self._native16(ref_feat, tgt_feat):
                first = self._first_conv_implicit(ref_feat, tgt_feat)
            if self.volume_channels_last:
                first = first.contiguous(memory_format=torch.channels_last_3d)
            _, _, cost3 = self._aggregate(None, first)
            return self._disparity_head(cost3, H, W)
        if self.fuse_volume_conv_train and torch.is_grad_enabled():
            # dres0[0] = Conv3d + BatchNorm3d, dres0[1] = ReLU
            conv = ops.volume_conv(ref_feat, tgt_feat, self.dres0[0][0].weight, self.maxdisp // 4)
            first = self.dres0[1](self.dres0[0][1](conv))
            if self.volume_channels_last:
                first = first.contiguous(memory_format=torch.channels_last_3d)
            cost1, cost2, cost3 = self._aggregate(None, first)
        else:
            with self._native16(ref_feat, tgt_feat):
                if self.volume_channels_last:
                    cost = ops.build_concat_volume(ref_feat, tgt_feat, self.maxdisp // 4, channels_last=True)
                else:
                    cost = ops.build_concat_volume(ref_feat, tgt_feat, self.maxdisp // 4)  # replaces psmnet.py:151-165
            cost1, cost2, cost3 = self._aggregate(cost)
        pred3 = self._disparity_head(cost3, H, W)
        if self.training:
            pred1 = self._disparity_head(cost1, H, W)
            pred2 = self._disparity_head(cost2, H, W)
            return pred3, pred2, pred1
        return pred3
