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

With --dtype bf16|fp16 the features are 16-bit and the weight is an fp32 master weight, as in autocast training, and the
arms are the 16-bit dataflows of that layer (DESIGN.md §4.13):

    fused16            ops.volume_conv on the 16-bit features outside autocast (16-bit output and feature gradients)
    fused_fp32_island  ops.volume_conv called under autocast: the features are cast to fp32, the output is fp32
    ncdhw16            native 16-bit concat volume + cuDNN's conv3d under autocast (16-bit), NCDHW
    ndhwc16            the same in channels_last_3d (volume and weight)

grad_out has the dtype of each arm's output.  --profile then reports the kernels of fused16 and, beside them, those of
fused_fp32_island (the fp32 reduce), with the reduce's GB/s on the bytes it must move (g in, 18 fp32 planes out).

    python benchmarks/volume_conv_train.py --dtype bf16 --profile --out profiles/r3_volume_conv_train_bf16.json
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


def arms16(w, dtype):
    from activezero_b200 import ops

    w_cl = w.detach().contiguous(memory_format=torch.channels_last_3d).requires_grad_(True)

    def amp():
        return torch.autocast("cuda", dtype=dtype)

    def island(L, R, dq):
        with amp():
            return ops.volume_conv(L, R, w, dq)

    def cudnn(L, R, dq, channels_last):
        vol = ops.build_concat_volume(L, R, dq, channels_last=channels_last)  # 16-bit features in, 16-bit volume out
        with amp():
            return F.conv3d(vol, w_cl if channels_last else w, padding=1)

    return {
        "fused16": (lambda L, R, dq: ops.volume_conv(L, R, w, dq), w),
        "fused_fp32_island": (island, w),
        "ncdhw16": (lambda L, R, dq: cudnn(L, R, dq, False), w),
        "ndhwc16": (lambda L, R, dq: cudnn(L, R, dq, True), w_cl),
    }


def inputs(B, H, W, dq, dtype):
    torch.manual_seed(0)
    L = torch.randn(B, 32, H, W, device="cuda").to(dtype).requires_grad_(True)
    R = torch.randn(B, 32, H, W, device="cuda").to(dtype).requires_grad_(True)
    w = (torch.randn(32, 64, 3, 3, 3, device="cuda") * 0.05).requires_grad_(True)
    g = torch.randn(B, 32, dq, H, W, device="cuda")
    return L, R, w, g


def bench_shape(B, H, W, dq, iters, warmup, dtype=None):
    L, R, w, g = inputs(B, H, W, dq, dtype or torch.float32)
    fns = arms(w) if dtype is None else arms16(w, dtype)
    gs = {torch.float32: g} if dtype is None else {torch.float32: g, dtype: g.to(dtype)}
    del g
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    times = {k: ([], []) for k in fns}
    for it in range(warmup + iters):
        for name, (fn, wt) in fns.items():
            L.grad = R.grad = wt.grad = None
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            out = fn(L, R, dq)
            e1.record()
            out.backward(gs[out.dtype])
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
        out_dtype = str(out.dtype)
        out.backward(gs[out.dtype])
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        grads[name] = (L.grad.clone(), R.grad.clone(), wt.grad.clone())
        del out
        fwd, bwd = statistics.median(times[name][0]), statistics.median(times[name][1])
        res[name] = {"fwd_ms": fwd, "bwd_ms": bwd, "fwd_bwd_ms": fwd + bwd, "output_dtype": out_dtype,
                     "fwd_ms_min": min(times[name][0]), "bwd_ms_min": min(times[name][1]),
                     "max_memory_allocated_MB": peak / 2**20, "peak_above_inputs_MB": (peak - base) / 2**20}
    # the fused gradients against the NCDHW arm's (cuDNN): relative max difference per gradient
    fused, ncdhw = ("fused", "ncdhw") if dtype is None else ("fused16", "ncdhw16")
    res[f"{fused}_vs_{ncdhw}_grad_rel_maxdiff"] = {
        k: float((a.double() - b.double()).abs().max() / b.double().abs().max())
        for k, a, b in zip(("dL", "dR", "dW"), grads[fused], grads[ncdhw])}
    return res


def profile_arm(B, H, W, dq, dtype=None, arm="fused", n=5):
    from torch.profiler import ProfilerActivity, profile

    L, R, w, g = inputs(B, H, W, dq, dtype or torch.float32)
    fn = (arms(w) if dtype is None else arms16(w, dtype))[arm][0]
    g = g.to(fn(L, R, dq).dtype)
    fn(L, R, dq).backward(g)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn(L, R, dq).backward(g)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
        if t > 0:
            out[e.key[:80]] = round(t / n / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def reduce_side_by_side(B, H, W, dq, dtype):
    """The kernels of fused16 and of fused_fp32_island; the reduce's ms and GB/s on g in + 18 fp32 planes out."""
    k16 = profile_arm(B, H, W, dq, dtype, "fused16")
    k32 = profile_arm(B, H, W, dq, dtype, "fused_fp32_island")
    planes = 18 * B * 32 * H * W * 4
    n = B * 32 * dq * H * W

    def red(kernels, elem):
        ms = sum(v for k, v in kernels.items() if "vcb_reduce" in k)
        return {"ms": ms, "bytes_MB": (n * elem + planes) / 1e6, "GB_per_s": (n * elem + planes) / (ms * 1e6) if ms else None}

    return {"fused16_kernels_ms": k16, "fused_fp32_island_kernels_ms": k32,
            "reduce": {"16-bit": red(k16, 2), "fp32": red(k32, 4)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the JSON result here")
    ap.add_argument("--profile", action="store_true",
                    help="after the timed runs: device time per kernel of the fused arm (torch.profiler, 5 iterations)")
    ap.add_argument("--dtype", choices=("bf16", "fp16"), default=None,
                    help="16-bit features and the 16-bit dataflows of the layer (see the module docstring)")
    args = ap.parse_args()
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}.get(args.dtype)
    if not torch.cuda.is_available():
        raise SystemExit("volume_conv_train.py measures on a CUDA device; none found")
    result = {"what": "dres0[0] Conv3d(64,32,3,pad 1) on the concat volume: forward + backward per arm, median ms "
                      f"of {args.iters} after {args.warmup} warm-up iterations, arms alternated",
              "card (name, power limit, max SM clock)": card(), "torch": torch.__version__,
              "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32, "dtype": args.dtype or "fp32", "shapes": {}}
    for B, H, W, dq in SHAPES:
        result["shapes"][f"B{B}_{H}x{W}_Dq{dq}"] = bench_shape(B, H, W, dq, args.iters, args.warmup, dtype)
    if args.profile and dtype is None:
        result["fused_kernel_ms_per_iteration"] = {f"B{B}_{H}x{W}_Dq{dq}": profile_arm(B, H, W, dq) for B, H, W, dq in SHAPES}
    elif args.profile:
        result["kernel_ms_per_iteration"] = {f"B{B}_{H}x{W}_Dq{dq}": reduce_side_by_side(B, H, W, dq, dtype)
                                             for B, H, W, dq in SHAPES}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
