#!/usr/bin/env python
"""PSMNet's disparity heads with native 16-bit logits (DESIGN.md §4.12).

Operators at B = 8, 544x960, D = 192 (the logits, 1.6-3.2 GB, are far beyond the 126 MB L2 in every arm):
  soft-argmin forward, forward with lse, and backward, in four arms: fp32 logits, bf16 native, fp16 native, and bf16
  widened by hand (``cost.float()`` before the fp32 operator, the gradient cast back after it);
  the fused upsample + soft-argmin head ([8,1,48,136,240] -> (192,544,960)) forward (with stats) and backward, fp32
  against bf16.
Each arm reports its median time over several windows (arms alternated, every shape warmed up first, CUDA events) and
the achieved GB/s on its algorithmic bytes (N = B*D*H*W logits):
  fp32: forward 4N, backward 8N (read logits, write gradient);  native 16-bit: 2N and 4N;
  widened: forward 10N (cast reads 2N, writes 4N, kernel reads 4N), backward 14N (kernel reads 4N, writes 4N, the
  narrowing cast reads 4N and writes 2N).
The disparity, lse and gdisp planes (N/D each) are left out of the byte counts.  The fused head's bytes (P = B*H*W
output pixels, L = B*Dq*Hq*Wq low-res logits of e bytes): forward e*L + 12P (disp and stats written), backward
e*L + 16P (disp, stats, gdisp read) + 8*Dq*P (fp32 workspace plane G written and read) + 8*Dq*B*H*Wq (plane T written
and read) + e*L (glow written).

Whole network: PSMNet_3 eval at 544x960, B = 1, channels_last_3d, with fuse_upsample and fuse_volume_conv off and on,
five arms: fp32 model, fp32 model under bf16 autocast, bf16 model, fp16 model, bf16 model with widened heads.
BatchNorm is conditioned on the input first (momentum 1, then frozen) so that the 16-bit models stay finite.

    python benchmarks/psmnet16.py [--iters 10] [--reps 5] [--out profiles/x.json]
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from activezero_b200 import ops  # noqa: E402
from activezero_b200.nets.psmnet.psmnet_3 import PSMNet  # noqa: E402


def card():
    """device name, power limit and max SM clock, queried read-only"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f"unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": out}


def time_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def race(arms, iters, reps):
    """arms: name -> fn.  Warm every arm, then `reps` windows of `iters` calls with the arms alternated; median ms."""
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t[k].append(time_ms(fn, iters))
    return {k: {"median_ms": statistics.median(v), "windows_ms": [round(x, 4) for x in v]} for k, v in t.items()}


def soft_argmin_ops(iters, reps):
    B, D, H, W = 8, 192, 544, 960
    N = B * D * H * W
    g = torch.Generator(device="cuda").manual_seed(0)
    x32 = torch.randn((B, D, H, W), device="cuda", generator=g) * 10
    xs = {"fp32": x32, "bf16": x32.to(torch.bfloat16), "fp16": x32.to(torch.float16)}
    disp = torch.empty((B, 1, H, W), device="cuda")
    lse = torch.empty((B, 2, H, W), device="cuda")
    gd = torch.randn((B, 1, H, W), device="cuda", generator=g)
    grads = {k: torch.empty_like(v) for k, v in xs.items()}

    def fwd(k, with_lse):
        return lambda: ops.soft_argmin_forward_into(xs[k], disp, lse if with_lse else None)

    def bwd(k):
        return lambda: ops.soft_argmin_backward_into(xs[k], disp, lse, gd, grads[k])

    def widened_fwd(with_lse):
        return lambda: ops.soft_argmin_forward_into(xs["bf16"].float(), disp, lse if with_lse else None)

    def widened_bwd():  # the saved fp32 logits are read; the fp32 gradient is narrowed by autograd's cast
        g32 = torch.empty_like(x32)
        ops.soft_argmin_backward_into(x32, disp, lse, gd, g32)
        return g32.to(torch.bfloat16)

    res = {}
    nbytes = {"fwd": {"fp32": 4 * N, "bf16": 2 * N, "fp16": 2 * N, "bf16_widened": 10 * N},
              "bwd": {"fp32": 8 * N, "bf16": 4 * N, "fp16": 4 * N, "bf16_widened": 14 * N}}
    for name, arms, kind in (
            ("forward", {"fp32": fwd("fp32", False), "bf16": fwd("bf16", False), "fp16": fwd("fp16", False),
                         "bf16_widened": widened_fwd(False)}, "fwd"),
            ("forward_with_lse", {"fp32": fwd("fp32", True), "bf16": fwd("bf16", True), "fp16": fwd("fp16", True),
                                  "bf16_widened": widened_fwd(True)}, "fwd"),
            ("backward", {"fp32": bwd("fp32"), "bf16": bwd("bf16"), "fp16": bwd("fp16"), "bf16_widened": widened_bwd},
             "bwd")):
        if kind == "bwd":
            ops.soft_argmin_forward_into(x32, disp, lse)
        r = race(arms, iters, reps)
        for k, v in r.items():
            v["bytes"] = nbytes[kind][k]
            v["GB_per_s"] = round(nbytes[kind][k] / (v["median_ms"] * 1e-3) / 1e9, 1)
            v["ratio_to_fp32"] = round(v["median_ms"] / r["fp32"]["median_ms"], 3)
        res[name] = r
    return {"shape": [B, D, H, W], "logits_N": N, **res}


def fused_head_ops(iters, reps):
    B, Dq, Hq, Wq = 8, 48, 136, 240
    D, H, W = 192, 544, 960
    g = torch.Generator(device="cuda").manual_seed(1)
    x32 = torch.randn((B, 1, Dq, Hq, Wq), device="cuda", generator=g) * 10
    xs = {"fp32": x32, "bf16": x32.to(torch.bfloat16)}
    dims = (B, Dq, Hq, Wq, D, H, W)
    disp = torch.empty((B, 1, H, W), device="cuda")
    stats = torch.empty((B, 2, H, W), device="cuda")
    gd = torch.randn((B, 1, H, W), device="cuda", generator=g)
    grads = {k: torch.empty_like(v) for k, v in xs.items()}
    fw = race({k: (lambda k=k: ops.upsample_soft_argmin_forward_into(xs[k], disp, stats, dims)) for k in xs}, iters, reps)
    ops.upsample_soft_argmin_forward_into(x32, disp, stats, dims)
    bw = race({k: (lambda k=k: ops.upsample_soft_argmin_backward_into(xs[k], disp, stats, gd, grads[k], dims))
               for k in xs}, iters, reps)
    P, L = B * H * W, B * Dq * Hq * Wq
    for r, nbytes in ((fw, lambda e: e * L + 12 * P), (bw, lambda e: 2 * e * L + 16 * P + 8 * Dq * P + 8 * Dq * B * H * Wq)):
        for k, v in r.items():
            v["bytes"] = nbytes(xs[k].element_size())
            v["GB_per_s"] = round(v["bytes"] / (v["median_ms"] * 1e-3) / 1e9, 1)
            v["ratio_to_fp32"] = round(v["median_ms"] / r["fp32"]["median_ms"], 3)
    return {"lowres": [B, 1, Dq, Hq, Wq], "out": [D, H, W], "forward_with_stats": fw, "backward": bw}


class WidenedHeads:
    """ops.soft_argmin / ops.upsample_soft_argmin replaced by the fp32 operator on widened logits (the workaround a 16-bit
    model needed before the native heads); the tests compare the native heads against this dataflow."""

    def __enter__(self):
        self.sa, self.usa = ops.soft_argmin, ops.upsample_soft_argmin
        ops.soft_argmin = lambda c: self.sa(c.float())
        ops.upsample_soft_argmin = lambda lo, size: self.usa(lo.float(), size)

    def __exit__(self, *exc):
        ops.soft_argmin, ops.upsample_soft_argmin = self.sa, self.usa


def network(iters, reps):
    torch.manual_seed(1)
    g = torch.Generator(device="cuda").manual_seed(17)
    x, y = torch.rand(1, 3, 544, 960, device="cuda", generator=g), torch.rand(1, 3, 544, 960, device="cuda", generator=g)
    m32 = PSMNet(maxdisp=192).cuda().train()
    for m in m32.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.momentum = 1.0
    with torch.no_grad():
        m32(x, y)
    m32.eval()
    models = {"fp32": m32, "bf16": copy.deepcopy(m32).to(torch.bfloat16), "fp16": copy.deepcopy(m32).to(torch.float16)}
    xs = {torch.float32: (x, y), torch.bfloat16: (x.bfloat16(), y.bfloat16()), torch.float16: (x.half(), y.half())}

    def run(model, dtype, autocast=False, widened=False):
        a, b = xs[dtype]

        def fn():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                if widened:
                    with WidenedHeads():
                        return model(a, b)
                return model(a, b)
        return fn

    out = []
    for fuse_up in (False, True):
        for fuse_vc in (False, True):
            for m in models.values():
                m.use_channels_last_3d(True)
                m.fuse_upsample, m.fuse_volume_conv = fuse_up, fuse_vc
            arms = {"fp32": run(models["fp32"], torch.float32),
                    "fp32_bf16_autocast": run(models["fp32"], torch.float32, autocast=True),
                    "bf16": run(models["bf16"], torch.bfloat16), "fp16": run(models["fp16"], torch.float16),
                    "bf16_widened_heads": run(models["bf16"], torch.bfloat16, widened=True)}
            finite = {k: bool(torch.isfinite(fn()).all()) for k, fn in arms.items()}
            r = race(arms, iters, reps)
            for k in r:
                r[k]["output_finite"] = finite[k]
            out.append({"channels_last_3d": True, "fuse_upsample": fuse_up, "fuse_volume_conv": fuse_vc, "arms": r})
    return {"input": [1, 3, 544, 960], "configs": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-network", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("psmnet16.py measures on a CUDA device; none is available")
    torch.backends.cudnn.benchmark = True
    res = {"card": card(), "iters": a.iters, "reps": a.reps, "soft_argmin": soft_argmin_ops(a.iters, a.reps)}
    torch.cuda.empty_cache()
    res["fused_head"] = fused_head_ops(a.iters, a.reps)
    torch.cuda.empty_cache()
    if not a.skip_network:
        res["network_544x960_b1"] = network(a.iters, a.reps)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
