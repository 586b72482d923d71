#!/usr/bin/env python
"""The concat volume under torch.autocast (DESIGN.md §4.11): the previous dataflow against the native 16-bit volume.

  previous: 16-bit features -> the fp32 op (custom_fwd casts them up) -> fp32 volume -> autocast casts it to 16 bits
            for cuDNN's dres0[0];  backward: cuDNN's 16-bit gvol -> fp32 copy -> fp32 concat backward -> cast down
  native  : 16-bit features -> 16-bit volume -> cuDNN;  backward: 16-bit gvol -> 16-bit concat backward

Volume + dres0[0] (Conv3d 64->32, 3x3x3), forward and forward+backward, NCDHW and channels_last_3d, B = 2 at 64x128
and B = 1, 4 at 136x240 (quarter resolution of 256x512 and 544x960; Dq = 48), with CUDA events on warm shapes, the
two arms alternated; peak memory above the inputs.  Then PSMNet_3 eval at 544x960 under autocast with
fuse_volume_conv (the 16-bit implicit first convolution) against the unfused autocast forward.

    python benchmarks/autocast_volume.py [--dtype bf16|fp16] [--iters 20] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from activezero_b200 import ops  # noqa: E402
from activezero_b200.nets.psmnet.psmnet_3 import PSMNet  # noqa: E402

DQ = 48
SHAPES = [(2, 64, 128), (1, 136, 240), (4, 136, 240)]
CL = torch.channels_last_3d


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f"unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": out}


def time_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def peak_mb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def layer_arms(B, Hq, Wq, dtype, channels_last, iters):
    torch.manual_seed(0)
    conv = torch.nn.Conv3d(64, 32, 3, 1, 1, bias=False).cuda()
    if channels_last:
        conv.weight.data = conv.weight.data.contiguous(memory_format=CL)
    L = torch.randn(B, 32, Hq, Wq, device="cuda").to(dtype).requires_grad_(True)
    R = torch.randn(B, 32, Hq, Wq, device="cuda").to(dtype).requires_grad_(True)
    gout = torch.randn(B, 32, DQ, Hq, Wq, device="cuda").to(dtype)
    if channels_last:
        gout = gout.contiguous(memory_format=CL)

    def previous():
        with torch.autocast("cuda", dtype=dtype):
            return conv(ops.build_concat_volume(L, R, DQ, channels_last))

    def native():
        with torch.autocast("cuda", dtype=dtype, enabled=False):
            vol = ops.build_concat_volume(L, R, DQ, channels_last)
        with torch.autocast("cuda", dtype=dtype):
            return conv(vol)

    arms = {"previous": previous, "native": native}
    res = {}
    with torch.no_grad():
        outs = {k: f() for k, f in arms.items()}
    res["forward_outputs_equal"] = bool(torch.equal(outs["previous"], outs["native"]))
    grads = {}
    for k, f in arms.items():
        L.grad = R.grad = conv.weight.grad = None
        f().backward(gout)
        grads[k] = (L.grad.clone(), R.grad.clone())
    res["feature_grads_equal"] = all(torch.equal(a, b) for a, b in zip(grads["previous"], grads["native"]))
    del outs, grads

    def fwd(f):
        with torch.no_grad():
            f()

    def fwd_bwd(f):
        L.grad = R.grad = conv.weight.grad = None
        f().backward(gout)

    for mode, run in (("forward", fwd), ("forward_backward", fwd_bwd)):
        for f in arms.values():  # warm: cuDNN picks its algorithms per shape
            for _ in range(3):
                run(f)
        t = {k: [] for k in arms}
        for _ in range(3):  # alternate the arms; report the median of three windows
            for k, f in arms.items():
                t[k].append(time_ms(lambda: run(f), iters))
        for k, f in arms.items():
            res[f"{mode}_{k}_ms"] = sorted(t[k])[1]
            res[f"{mode}_{k}_peak_mb"] = peak_mb(lambda: run(f))
        res[f"{mode}_speedup"] = res[f"{mode}_previous_ms"] / res[f"{mode}_native_ms"]
    return res


def network_arms(dtype, iters):
    torch.manual_seed(1)
    net = PSMNet(maxdisp=192).cuda().eval()
    x = torch.rand(1, 3, 544, 960, device="cuda")
    y = torch.rand(1, 3, 544, 960, device="cuda")
    res = {}
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        for cl in (False, True):
            net.use_channels_last_3d(cl)
            tag = "channels_last_3d" if cl else "ncdhw"
            t = {"unfused": [], "fuse_volume_conv": []}
            for fused in (False, True):
                net.fuse_volume_conv = fused
                for _ in range(3):
                    net(x, y)
            for _ in range(3):
                for fused, k in ((False, "unfused"), (True, "fuse_volume_conv")):
                    net.fuse_volume_conv = fused
                    t[k].append(time_ms(lambda: net(x, y), iters))
            for k in t:
                res[f"psmnet_544x960_{tag}_{k}_ms"] = sorted(t[k])[1]
            net.fuse_volume_conv = False
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtype", choices=("bf16", "fp16"), default="bf16")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autocast_volume.py measures on a CUDA device; none found")
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    res = {"what": "concat volume + dres0[0] under torch.autocast: previous dataflow vs native 16-bit volume",
           "dtype": args.dtype, "Dq": DQ, "C": 32, "iters_per_window": args.iters, **card(), "layer": []}
    for B, Hq, Wq in SHAPES:
        for cl in (False, True):
            row = {"B": B, "Hq": Hq, "Wq": Wq, "layout": "channels_last_3d" if cl else "ncdhw"}
            row.update(layer_arms(B, Hq, Wq, dtype, cl, args.iters))
            res["layer"].append(row)
            print(json.dumps(row), flush=True)
    res["network"] = network_arms(dtype, max(3, args.iters // 4))
    print(json.dumps(res["network"]), flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
