#!/usr/bin/env python
"""Synthetic-data training-step harness for BASELINE configs 3 and 4 (a CALLER of the
hot path: the reference's trainer itself is out of scope, SURVEY.md §2 row 7).

Config 3 -- PSMNet training step at a 256x512 crop with backward through the cost volume and
the IR reprojection loss, DDP on N GPUs.  Config 4 -- the mixed-domain step: the supervised
sim step plus the real step whose IR patterns are extracted ON THE GPU from synthetic T-frame
IR sequences (tools/temporal_ir.py on the reference side is an offline CPU script).

The step functions restate `/root/reference/train.py:220-432` + `utils/losses.py:7-15,74-160`
on synthetic tensors and take the operator set as an argument, so tests can run the very same
step once with this repository's CUDA operators and once with the oracle's torch restatements
(stock torch on the GPU) and compare losses and parameter gradients.

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 benchmarks/train_step.py --steps 10
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

MAX_DISP, PATCH = 192, 11  # configs/config.py:8, :41


def az_api():
    """The drop-in operator set (this repository)."""
    from activezero_b200.tools.temporal_ir import extract_temporal_ir_pattern
    from activezero_b200.utils.reprojection import get_reproj_error_patch
    from activezero_b200.utils.warp_ops import apply_disparity_cu

    return types.SimpleNamespace(name="activezero_b200", get_reproj_error_patch=get_reproj_error_patch,
                                 apply_disparity_cu=apply_disparity_cu, temporal_ir=extract_temporal_ir_pattern)


def make_batch(B, H, W, device, seed, T=4):
    """Synthetic stand-in for one MessyTable sample batch (SURVEY.md §8d configs 3/4)."""
    g = torch.Generator().manual_seed(seed)
    mean, std = 0.45, 0.224  # dataset_utils.py:76-81 style normalisation
    b = {
        "img_sim_L": (torch.rand(B, 3, H, W, generator=g) - mean) / std,
        "img_sim_R": (torch.rand(B, 3, H, W, generator=g) - mean) / std,
        "img_real_L": (torch.rand(B, 3, H, W, generator=g) - mean) / std,
        "img_real_R": (torch.rand(B, 3, H, W, generator=g) - mean) / std,
        "disp_R": torch.rand(B, 1, H, W, generator=g) * 79.0 + 1.0,  # GT disparity in the right view, U(1,80)
        "sim_pat_L": (torch.rand(B, 1, H, W, generator=g) > 0.5).float(),
        "sim_pat_R": (torch.rand(B, 1, H, W, generator=g) > 0.5).float(),
    }
    # real domain: T-frame IR sequences with an emitter ramp on a dot pattern (config 4)
    for side in ("L", "R"):
        base = torch.randint(0, 256, (B, 1, H, W), generator=g).float() * 0.5
        dots = (torch.rand(B, 1, H, W, generator=g) < 0.1).float()
        ramp = torch.arange(T).view(1, T, 1, 1).float()
        noise = torch.randint(0, 6, (B, T, H, W), generator=g).float()
        b[f"real_seq_{side}"] = (base + ramp * dots * 10.0 + noise).clamp(0, 255).to(torch.uint8)
    return {k: v.to(device) for k, v in b.items()}


def psmnet_disp(preds, disp_gt, mask):
    """utils/losses.py:7-15."""
    p3, p2, p1 = preds
    return (0.5 * F.smooth_l1_loss(p1[mask], disp_gt[mask], reduction="mean")
            + 0.7 * F.smooth_l1_loss(p2[mask], disp_gt[mask], reduction="mean")
            + F.smooth_l1_loss(p3[mask], disp_gt[mask], reduction="mean"))


def sim_step_loss(model, batch, api):
    """train.py:255-293 + losses.py:81-98 (onSim): GT brought to the left view by the integer
    scatter warp, mask 0 < gt < MAX_DISP, smooth-L1 on three heads + patch reprojection loss."""
    disp_r = batch["disp_R"].contiguous()
    disp_gt_l = api.apply_disparity_cu(disp_r, disp_r.type(torch.int).contiguous())
    mask = (disp_gt_l < MAX_DISP) * (disp_gt_l > 0)
    preds = model(batch["img_sim_L"], batch["img_sim_R"])
    loss_disp = psmnet_disp(preds, disp_gt_l, mask)
    loss_reproj, _, _ = api.get_reproj_error_patch(input_L=batch["sim_pat_L"], input_R=batch["sim_pat_R"],
                                                   pred_disp_l=preds[0], mask=mask, ps=PATCH)
    return loss_disp + 1.0 * loss_reproj, {"disp": loss_disp.detach(), "reproject": loss_reproj.detach()}


def real_step_loss(model, batch, api):
    """train.py:369-432 + losses.py:88-91 (real domain): reprojection only, no mask; the IR
    patterns come from the temporal sequences (tools/temporal_ir.py:93-114)."""
    pat_L = api.temporal_ir(batch["real_seq_L"]).unsqueeze(1).float()
    pat_R = api.temporal_ir(batch["real_seq_R"]).unsqueeze(1).float()
    preds = model(batch["img_real_L"], batch["img_real_R"])
    loss_reproj, _, _ = api.get_reproj_error_patch(input_L=pat_L, input_R=pat_R, pred_disp_l=preds[0], ps=PATCH)
    return 1.0 * loss_reproj, {"reproject": loss_reproj.detach()}


def main():
    from activezero_b200 import dist_util
    from activezero_b200.nets.psmnet.psmnet_3 import PSMNet

    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=2)  # configs/config.py:93, per GPU
    ap.add_argument("--height", type=int, default=256)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--no-real", action="store_true", help="config 3 only (skip the real-domain step)")
    ap.add_argument("--channels-last-3d", action="store_true",
                    help="emit the cost volume in channels_last_3d (SURVEY 8f rank 2, layout clause)")
    ap.add_argument("--fuse-upsample", action="store_true",
                    help="use the fused trilinear-upsample + soft-argmin kernel for the three heads (SURVEY §8f-1)")
    ap.add_argument("--fuse-volume-conv", action="store_true",
                    help="dres0's first Conv3d on the implicit volume in training too (PSMNet.fuse_volume_conv_train)")
    ap.add_argument("--profile", action="store_true", help="after the timed region: kernel-time shares via torch.profiler")
    args = ap.parse_args()

    rank, world, local = dist_util.env_rank_world()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist_util.init_from_env("nccl", dev)
    torch.manual_seed(1)  # cfg.SOLVER.SEED, configs/config.py:100
    model = PSMNet(maxdisp=MAX_DISP).to(dev)
    model.fuse_upsample = args.fuse_upsample
    model.fuse_volume_conv_train = args.fuse_volume_conv
    if args.channels_last_3d:
        model.use_channels_last_3d(True)
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local])
    opt = torch.optim.Adam(model.parameters(), lr=2e-4, betas=(0.9, 0.999))  # configs/config.py:88
    api = az_api()
    model.train()
    batch = make_batch(args.batch, args.height, args.width, dev, 100 + rank, T=args.frames)

    def one_iteration():
        loss, vals = sim_step_loss(model, batch, api)
        opt.zero_grad()
        loss.backward()
        opt.step()
        if not args.no_real:
            loss_r, _ = real_step_loss(model, batch, api)
            opt.zero_grad()
            loss_r.backward()
            opt.step()
        return loss.detach()

    for _ in range(args.warmup):
        one_iteration()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist_util.barrier()
    torch.cuda.synchronize()
    start.record()
    for _ in range(args.steps):
        last = one_iteration()
    stop.record()
    dist_util.barrier()
    torch.cuda.synchronize()
    (ms,) = dist_util.max_over_ranks([start.elapsed_time(stop)], dev)

    # where the device time goes (rank 0, two more iterations under torch.profiler / CUPTI): this library's kernels
    # (the hot path), NCCL (DDP's gradient all-reduce: 2 x 20.9 MB per iteration, SURVEY 2c) and everything else
    # (cuDNN / torch).  A number measured under the profiler is not a throughput; only the SHARES are reported.
    shares = None
    if args.profile:
        from torch.profiler import ProfilerActivity, profile

        dist_util.barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                one_iteration()
            torch.cuda.synchronize()
        az = nccl = other = 0.0
        for e in prof.key_averages():
            t = float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
            name = e.key
            if "az::" in name or name.startswith("void az") or "az_" in name:
                az += t
            elif "nccl" in name.lower():
                nccl += t
            else:
                other += t
        tot = az + nccl + other
        shares = {"hot_path_kernels_ms_per_iter": az / 2e3, "nccl_ms_per_iter": nccl / 2e3, "other_ms_per_iter": other / 2e3,
                  "hot_path_share_of_kernel_time": az / tot if tot else None, "nccl_share_of_kernel_time": nccl / tot if tot else None,
                  "note": "kernel time summed over streams (NCCL overlaps the backward): nccl_ms is its busy time, the EXPOSED "
                          "part is what the iteration time grows by from 1 GPU to N (see the efficiency table)"}
    if rank == 0:
        print(json.dumps({
            "metric": "training pairs/s (sim step + real step per iteration)" if not args.no_real else "training pairs/s (sim step)",
            "value": world * args.batch * args.steps / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "ms_per_iteration": ms / args.steps, "scaling": "weak",
            "config": {"workload": f"config{'3' if args.no_real else '4'}: PSMNet_3 train step {args.height}x{args.width}, "
                                   f"D={MAX_DISP}, batch {args.batch}/GPU, patch reproj ps={PATCH}, T={args.frames}",
                       "ddp": world > 1, "fuse_upsample": args.fuse_upsample, "fuse_volume_conv": args.fuse_volume_conv,
                       "channels_last_3d": args.channels_last_3d},
            "device_time_shares_rank0": shares,
            "final_loss": float(last)}), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
