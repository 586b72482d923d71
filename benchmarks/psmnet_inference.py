#!/usr/bin/env python
"""Application-level context for the hot path (not a bench line): one PSMNet inference at the
evaluator's shape (test.py:137-146 pads 540x960 to 544x960, batch 1, maxdisp 192) with
  (a) the reference's dataflow re-created with stock torch ops on the GPU (zero-filled volume + 96 slice
      copies, F.interpolate + F.softmax + weighted sum),
  (b) this repository's operators,
  (c) (b) with the trilinear upsample fused into the soft-argmin.
The 2-D/3-D convolutions are identical cuDNN calls in all three; the difference is the hot path.

    python benchmarks/psmnet_inference.py [--batch 1] [--iters 10] [--autocast bf16|fp16]

--autocast runs every arm under torch.autocast with that dtype (the 16-bit volume of DESIGN.md §4.9).
"""
import argparse
import contextlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from activezero_b200 import ops  # noqa: E402
from activezero_b200.nets.psmnet.psmnet_3 import PSMNet  # noqa: E402


def torch_concat_volume(ref, tgt, num_disp):
    """psmnet.py:151-165 with stock torch ops, all on the device (the reference additionally builds the
    zero volume on the HOST and uploads it -- not reproduced here, it would only be slower)."""
    B, C, H, W = ref.shape
    cost = torch.zeros(B, 2 * C, num_disp, H, W, device=ref.device)
    for i in range(num_disp):
        if i > 0:
            cost[:, :C, i, :, i:] = ref[:, :, :, i:]
            cost[:, C:, i, :, i:] = tgt[:, :, :, :-i]
        else:
            cost[:, :C, i] = ref
            cost[:, C:, i] = tgt
    return cost.contiguous()


def torch_soft_argmin(cost):
    p = F.softmax(cost, dim=1)
    d = torch.arange(cost.shape[1], device=cost.device, dtype=torch.float32).view(1, -1, 1, 1)
    return torch.sum(p * d, 1, keepdim=True)


def timed(fn, iters):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--autocast", choices=("bf16", "fp16"), default=None,
                    help="run every arm under torch.autocast with this dtype")
    args = ap.parse_args()
    amp = contextlib.nullcontext() if args.autocast is None else \
        torch.autocast("cuda", dtype=torch.bfloat16 if args.autocast == "bf16" else torch.float16)
    torch.manual_seed(1)
    net = PSMNet(maxdisp=192).cuda().eval()
    x = torch.rand(args.batch, 3, 544, 960, device="cuda")
    y = torch.rand(args.batch, 3, 544, 960, device="cuda")
    res = {}
    with torch.no_grad(), amp:
        res["az_ops_ms"] = timed(lambda: net(x, y), args.iters)
        net.fuse_upsample = True
        res["az_ops_fused_upsample_ms"] = timed(lambda: net(x, y), args.iters)
        # SURVEY.md §8f rank 2: the volume emitted in channels_last_3d (cuDNN then runs the 3-D aggregation without
        # layout passes); with and without the fused upsample
        net.use_channels_last_3d(True)
        res["az_ops_fused_upsample_ndhwc_volume_ms"] = timed(lambda: net(x, y), args.iters)
        net.fuse_upsample = False
        res["az_ops_ndhwc_volume_ms"] = timed(lambda: net(x, y), args.iters)
        net.use_channels_last_3d(False)
        # SURVEY.md §8f rank 2, implicit clause: dres0's first conv + BN + ReLU as the tcgen05 kernel on the implicit
        # volume (the volume is never written); NCDHW aggregation, with and without the fused upsample
        net.fuse_volume_conv = True
        res["az_ops_implicit_volume_conv_ms"] = timed(lambda: net(x, y), args.iters)
        net.fuse_upsample = True
        res["az_ops_implicit_volume_conv_fused_upsample_ms"] = timed(lambda: net(x, y), args.iters)
        net.use_channels_last_3d(True)
        res["az_ops_implicit_volume_conv_fused_upsample_ndhwc_ms"] = timed(lambda: net(x, y), args.iters)
        net.use_channels_last_3d(False)
        net.fuse_upsample = False
        net.fuse_volume_conv = False
        saved = ops.build_concat_volume, ops.soft_argmin
        ops.build_concat_volume, ops.soft_argmin = torch_concat_volume, torch_soft_argmin
        try:
            res["stock_torch_ops_ms"] = timed(lambda: net(x, y), args.iters)
        finally:
            ops.build_concat_volume, ops.soft_argmin = saved
        # the part that is NOT the hot path: feature CNN + 3-D aggregation only
        fl, fr = net.feature_extraction(x), net.feature_extraction(y)
        vol = ops.build_concat_volume(fl, fr, 48)
        res["convs_only_ms"] = timed(lambda: (net.feature_extraction(x), net.feature_extraction(y), net._aggregate(vol)),
                                     args.iters)
    res.update(batch=args.batch, shape="544x960", maxdisp=192, autocast=args.autocast,
               hot_path_ms={k.replace("_ms", ""): res[k] - res["convs_only_ms"] for k in
                            ("stock_torch_ops_ms", "az_ops_ms", "az_ops_fused_upsample_ms")})
    print(json.dumps(res))


if __name__ == "__main__":
    main()
