#!/usr/bin/env python
"""Group-wise correlation volume with 16-bit features: three arms timed in one process (DESIGN.md §4.15):

    native   ops.build_gwc_volume on two bf16 / fp16 features outside autocast (az_gwc_volume_fwd_16 / _bwd_16): the
             volume and the feature gradients in the features' dtype
    island   today's autocast dataflow: the fp32 operator on the widened features, then .to(dtype) (what the next
             Conv3d reads); its backward widens the 16-bit gradient, runs the fp32 backward and rounds the gradients
    fp32     the fp32 operator alone on fp32 features

Per arm: forward, backward and forward + backward times (CUDA events, median after warm-up; arms alternated within an
iteration, the whole measurement repeated once to show the spread), the operator's algorithmic bytes
(forward s*(2*C*HW + G*Dq*HW)*B, backward s*(G*Dq*HW + 4*C*HW)*B, s the element size: the 16-bit size for the native
and island arms, whose problem is the 16-bit one) and their fraction of a device-to-device copy measured in the same
run, and torch.cuda.max_memory_allocated over one forward + backward above what was allocated before it (the inputs).
Workloads: config 2 (B = 8, C = 32, G = 8, 136x240, Dq = 48; the 16-bit volume is 200 MB and streams from HBM) and the
training crop (B = 2, 64x128, Dq = 48; every tensor fits the 126 MB L2).

    python benchmarks/gwc16.py --dtype bf16 --out profiles/r3_gwc16.json
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

DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
WORKLOADS = {"config2_B8_136x240": dict(B=8, C=32, G=8, H=136, W=240, Dq=48, l2_resident=False),
             "train_crop_B2_64x128": dict(B=2, C=32, G=8, H=64, W=128, Dq=48, l2_resident=True)}
ARMS = ("native", "island", "fp32")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def copy_peak_Bps(iters=20):
    """Device-to-device copy of 1 GiB: bytes read + written over the median time."""
    n = 1 << 28
    src = torch.empty(n, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    ts = []
    for i in range(iters + 3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(e0.elapsed_time(e1))
    del src, dst
    torch.cuda.empty_cache()
    return 2.0 * 4 * n / (statistics.median(ts) * 1e-3)


def algorithmic_bytes(w, s):
    HW = w["H"] * w["W"]
    fwd = s * w["B"] * (2 * w["C"] * HW + w["G"] * w["Dq"] * HW)
    bwd = s * w["B"] * (w["G"] * w["Dq"] * HW + 4 * w["C"] * HW)
    return fwd, bwd


def make_arms(w, dtype):
    from activezero_b200 import ops

    gen = torch.Generator().manual_seed(0)
    B, C, G, H, W, Dq = (w[k] for k in ("B", "C", "G", "H", "W", "Dq"))
    L32 = torch.randn(B, C, H, W, generator=gen).cuda()
    R32 = torch.randn(B, C, H, W, generator=gen).cuda()
    g32 = torch.randn(B, G, Dq, H, W, generator=gen).cuda()
    L16, R16, g16 = L32.to(dtype), R32.to(dtype), g32.to(dtype)
    L32, R32, g32 = L16.float(), R16.float(), g16.float()  # the same values in every arm

    def fwd(arm):
        if arm == "native":
            return ops.build_gwc_volume(L16, R16, Dq, G)
        if arm == "island":
            return ops.build_gwc_volume(L16.float(), R16.float(), Dq, G).to(dtype)
        return ops.build_gwc_volume(L32, R32, Dq, G)

    def bwd(arm):
        if arm == "native":
            return ops.gwc_volume_backward(g16, L16, R16)
        if arm == "island":
            gL, gR = ops.gwc_volume_backward(g16.float(), L16.float(), R16.float())
            return gL.to(dtype), gR.to(dtype)
        return ops.gwc_volume_backward(g32, L32, R32)

    def fwd_bwd(arm):
        a, b = (L32, R32) if arm == "fp32" else (L16, R16)
        a, b = a.detach().requires_grad_(True), b.detach().requires_grad_(True)
        if arm == "island":
            vol = ops.build_gwc_volume(a.float(), b.float(), Dq, G).to(dtype)
        else:
            vol = ops.build_gwc_volume(a, b, Dq, G)
        vol.backward(g32 if arm == "fp32" else g16)
        return vol, a.grad, b.grad

    return fwd, bwd, fwd_bwd


def bench(w, dtype, iters, warmup):
    fwd, bwd, fwd_bwd = make_arms(w, dtype)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    times = {a: {"fwd": [], "bwd": [], "fwd_bwd": []} for a in ARMS}
    for it in range(warmup + iters):
        for kind, fn in (("fwd", fwd), ("bwd", bwd), ("fwd_bwd", fwd_bwd)):
            for arm in ARMS:
                with torch.no_grad() if kind != "fwd_bwd" else torch.enable_grad():
                    e0, e1 = ev(), ev()
                    e0.record()
                    out = fn(arm)
                    e1.record()
                    torch.cuda.synchronize()
                del out
                if it >= warmup:
                    times[arm][kind].append(e0.elapsed_time(e1))
    res = {}
    outs = {}
    for arm in ARMS:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        vol, gL, gR = fwd_bwd(arm)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        outs[arm] = (vol.detach(), gL, gR)
        res[arm] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in times[arm].items()}
        res[arm]["peak_above_inputs_MB"] = (peak - base) / 2**20
        del vol, gL, gR
    res["native_equals_island"] = all(torch.equal(a, b) for a, b in zip(outs["native"], outs["island"]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtype", choices=sorted(DTYPES), default="bf16")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=2, help="whole measurement repeated to show the spread")
    ap.add_argument("--out", default=None, help="write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gwc16.py measures on a CUDA device; none found")
    dtype = DTYPES[args.dtype]
    peak = copy_peak_Bps()
    result = {"what": f"gwc volume, {args.dtype} features, three arms (native, island, fp32): median ms of {args.iters} "
                      f"after {args.warmup} warm-up iterations, arms alternated; fwd = forward, bwd = backward from a "
                      "given gradient, fwd_bwd = forward + autograd backward; peak memory above the inputs over one "
                      "forward + backward; fractions against the device-to-device copy measured in the same run",
              "card (name, power limit, max SM clock)": card(), "torch": torch.__version__, "dtype": args.dtype,
              "copy_peak_GBps": peak / 1e9, "workloads": {}}
    for name, w in WORKLOADS.items():
        runs = []
        for _ in range(args.repeats):
            r = bench(w, dtype, args.iters, args.warmup)
            for arm in ARMS:
                s = 4 if arm == "fp32" else torch.empty((), dtype=dtype).element_size()
                fb, bb = algorithmic_bytes(w, s)
                d = r[arm]
                d["algorithmic_bytes"] = {"fwd": fb, "bwd": bb, "fwd_bwd": fb + bb}
                d["fraction_of_copy_peak"] = {k: d["algorithmic_bytes"][k] / (d[k]["median_ms"] * 1e-3) / peak
                                              for k in ("fwd", "bwd", "fwd_bwd")}
            for k in ("fwd", "bwd", "fwd_bwd"):
                r[f"island_over_native_{k}"] = r["island"][k]["median_ms"] / r["native"][k]["median_ms"]
            r["island_over_native_memory"] = r["island"]["peak_above_inputs_MB"] / max(r["native"]["peak_above_inputs_MB"], 1e-9)
            runs.append(r)
        result["workloads"][name] = {**w, "runs": runs}
        print(name, json.dumps({k: v for k, v in runs[0].items() if k.startswith("island_over")}), flush=True)
    text = json.dumps(result, indent=2)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
