#!/usr/bin/env python
"""Patch reprojection loss (ps = 11) with image gradients: forward + backward to tgt, src and disp, two arms timed in
one process (DESIGN.md §4.14):

    fused    ops.reproj_loss: the fused forward, the disparity gradient, and the image gradients recomputed from the
             inputs (az_reproj_loss_img_bwd, no [B,K,H,W] tensor)
    unfold   the reference's dataflow (reprojection.py:99-118) as the drop-in composed it before: Unfold of both
             images, this library's warp kernel on the C*ps*ps unfolded planes, the boolean-mask gathers and mse_loss

CUDA events around forward + backward, arms alternated within an iteration, median over --iters after --warmup;
torch.cuda.max_memory_allocated over one forward + backward per arm, reported above what was allocated before it
(the inputs).  Workloads: config 3's loss (B = 2, 1x256x512, random mask), one 544x960 frame, and a feature-metric
loss on [2,32,64,128] features.

    python benchmarks/reproj_image_grad.py --out profiles/r3_reproj_image_grad.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

PS = 11
WORKLOADS = {"config3_2x1x256x512": (2, 1, 256, 512), "frame_1x1x544x960": (1, 1, 544, 960),
             "features_2x32x64x128": (2, 32, 64, 128)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def fused(L, R, d, m):
    from activezero_b200 import ops

    return ops.reproj_loss(L, R, d, m, ps=PS, sign=-1.0)[0]


def unfold(L, R, d, m):
    from activezero_b200 import ops

    B, C, H, W = L.shape
    u = torch.nn.Unfold(kernel_size=(PS, PS), padding=(PS - 1) // 2)
    Lu = u(L).reshape(B, -1, H, W)
    Ru = u(R).reshape(B, -1, H, W)
    Wu = ops.warp(Ru, -d)
    sel = m.repeat(1, Lu.shape[1], 1, 1)
    return F.mse_loss(Wu[sel], Lu[sel])


ARMS = {"fused": fused, "unfold": unfold}


def inputs(B, C, H, W):
    gen = torch.Generator().manual_seed(0)
    L = torch.rand(B, C, H, W, generator=gen).cuda().requires_grad_(True)
    R = torch.rand(B, C, H, W, generator=gen).cuda().requires_grad_(True)
    d = (torch.rand(B, 1, H, W, generator=gen) * min(64.0, W / 3)).cuda().requires_grad_(True)
    m = (torch.rand(B, 1, H, W, generator=gen) > 0.3).cuda()
    return L, R, d, m


def bench(shape, iters, warmup):
    L, R, d, m = inputs(*shape)
    ts = (L, R, d)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    times = {k: [] for k in ARMS}
    for it in range(warmup + iters):
        for name, fn in ARMS.items():
            for t in ts:
                t.grad = None
            e0, e1 = ev(), ev()
            e0.record()
            fn(L, R, d, m).backward()
            e1.record()
            torch.cuda.synchronize()
            if it >= warmup:
                times[name].append(e0.elapsed_time(e1))
    res, grads = {}, {}
    for name, fn in ARMS.items():
        for t in ts:
            t.grad = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        loss = fn(L, R, d, m)
        loss.backward()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        grads[name] = (loss.detach().double(), *(t.grad.double() for t in ts))
        del loss
        res[name] = {"fwd_bwd_ms": statistics.median(times[name]), "fwd_bwd_ms_min": min(times[name]),
                     "fwd_bwd_ms_max": max(times[name]), "peak_above_inputs_MB": (peak - base) / 2**20}
    res["unfold_over_fused_time"] = res["unfold"]["fwd_bwd_ms"] / res["fused"]["fwd_bwd_ms"]
    res["unfold_over_fused_memory"] = res["unfold"]["peak_above_inputs_MB"] / max(res["fused"]["peak_above_inputs_MB"], 1e-9)
    res["fused_vs_unfold_rel_maxdiff"] = {
        k: float((a - b).abs().max() / b.abs().max()) for k, a, b in zip(("loss", "dtgt", "dsrc", "ddisp"), grads["fused"], grads["unfold"])}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("reproj_image_grad.py measures on a CUDA device; none found")
    result = {"what": f"patch reprojection loss, ps = {PS}, forward + backward to tgt, src and disp per arm: median ms "
                      f"of {args.iters} after {args.warmup} warm-up iterations, arms alternated; peak memory above the "
                      "inputs over one forward + backward",
              "card (name, power limit, max SM clock)": card(), "torch": torch.__version__, "workloads": {}}
    for name, shape in WORKLOADS.items():
        result["workloads"][name] = {"shape": list(shape), **bench(shape, args.iters, args.warmup)}
        print(name, json.dumps(result["workloads"][name]), flush=True)
    text = json.dumps(result, indent=2)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
