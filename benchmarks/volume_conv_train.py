#!/usr/bin/env python
"""dres0[0]'s Conv3d(64, 32, 3, pad 1) on the concat volume, forward + backward, three arms timed in one process:

    fused        ops.volume_conv: tcgen05 TF32 forward on the implicit volume, volume-free fp32 backward
    ncdhw        concat_volume (this library's kernels, forward and backward) + cuDNN conv3d, NCDHW
    ndhwc        concat_volume(channels_last=True) + cuDNN conv3d on channels_last_3d volume and weight

CUDA events around the forward and around the backward of every iteration, arms alternated within an iteration,
median over --iters after --warmup; torch.cuda.max_memory_allocated over one forward + backward per arm (inputs
included).  cuDNN runs with torch's defaults (TF32 convolutions allowed).  The sizes are the training crop
(256x512, B=2, maxdisp 192: features 64x128, Dq=48) and the eval size (544x960: 136x240, Dq=48).

    python benchmarks/volume_conv_train.py --out profiles/r3_volume_conv_train.json
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

SHAPES = [(2, 64, 128, 48), (2, 136, 240, 48)]  # (B, H/4, W/4, maxdisp/4)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def arms(w):
    from activezero_b200 import ops

    w_cl = w.detach().contiguous(memory_format=torch.channels_last_3d).requires_grad_(True)
    return {
        "fused": (lambda L, R, dq: ops.volume_conv(L, R, w, dq), w),
        "ncdhw": (lambda L, R, dq: F.conv3d(ops.build_concat_volume(L, R, dq), w, padding=1), w),
        "ndhwc": (lambda L, R, dq: F.conv3d(ops.build_concat_volume(L, R, dq, channels_last=True), w_cl, padding=1), w_cl),
    }


def bench_shape(B, H, W, dq, iters, warmup):
    torch.manual_seed(0)
    L = torch.randn(B, 32, H, W, device="cuda", requires_grad=True)
    R = torch.randn(B, 32, H, W, device="cuda", requires_grad=True)
    w = (torch.randn(32, 64, 3, 3, 3, device="cuda") * 0.05).requires_grad_(True)
    g = torch.randn(B, 32, dq, H, W, device="cuda")
    fns = arms(w)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    times = {k: ([], []) for k in fns}
    for it in range(warmup + iters):
        for name, (fn, wt) in fns.items():
            L.grad = R.grad = wt.grad = None
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            out = fn(L, R, dq)
            e1.record()
            out.backward(g)
            e2.record()
            torch.cuda.synchronize()
            if it >= warmup:
                times[name][0].append(e0.elapsed_time(e1))
                times[name][1].append(e1.elapsed_time(e2))
            del out
    res, grads = {}, {}
    for name, (fn, wt) in fns.items():
        L.grad = R.grad = wt.grad = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = fn(L, R, dq)
        out.backward(g)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        grads[name] = (L.grad.clone(), R.grad.clone(), wt.grad.clone())
        del out
        fwd, bwd = statistics.median(times[name][0]), statistics.median(times[name][1])
        res[name] = {"fwd_ms": fwd, "bwd_ms": bwd, "fwd_bwd_ms": fwd + bwd,
                     "fwd_ms_min": min(times[name][0]), "bwd_ms_min": min(times[name][1]),
                     "max_memory_allocated_MB": peak / 2**20, "peak_above_inputs_MB": (peak - base) / 2**20}
    # the fused gradients against the NCDHW arm's (cuDNN TF32): relative max difference per gradient
    res["fused_vs_ncdhw_grad_rel_maxdiff"] = {
        k: float((a - b).abs().max() / b.abs().max()) for k, a, b in zip(("dL", "dR", "dW"), grads["fused"], grads["ncdhw"])}
    return res


def profile_fused(B, H, W, dq, n=5):
    from torch.profiler import ProfilerActivity, profile

    from activezero_b200 import ops

    L = torch.randn(B, 32, H, W, device="cuda", requires_grad=True)
    R = torch.randn(B, 32, H, W, device="cuda", requires_grad=True)
    w = (torch.randn(32, 64, 3, 3, 3, device="cuda") * 0.05).requires_grad_(True)
    g = torch.randn(B, 32, dq, H, W, device="cuda")
    ops.volume_conv(L, R, w, dq).backward(g)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            ops.volume_conv(L, R, w, dq).backward(g)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
        if t > 0:
            out[e.key[:80]] = round(t / n / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the JSON result here")
    ap.add_argument("--profile", action="store_true",
                    help="after the timed runs: device time per kernel of the fused arm (torch.profiler, 5 iterations)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("volume_conv_train.py measures on a CUDA device; none found")
    result = {"what": "dres0[0] Conv3d(64,32,3,pad 1) on the concat volume: forward + backward per arm, median ms "
                      f"of {args.iters} after {args.warmup} warm-up iterations, arms alternated",
              "card (name, power limit, max SM clock)": card(), "torch": torch.__version__,
              "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32, "shapes": {}}
    for B, H, W, dq in SHAPES:
        result["shapes"][f"B{B}_{H}x{W}_Dq{dq}"] = bench_shape(B, H, W, dq, args.iters, args.warmup)
    if args.profile:
        result["fused_kernel_ms_per_iteration"] = {f"B{B}_{H}x{W}_Dq{dq}": profile_fused(B, H, W, dq) for B, H, W, dq in SHAPES}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
