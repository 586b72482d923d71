#!/usr/bin/env python
"""bench.py -- the stereo hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): stereo pairs/s for costvol + dispreg + reproj at 544x960,
D = 192, and the fraction of the HBM roofline the dominant kernel reaches.

A *step* is one pass of the forward hot path over one batch of B = 8 synthetic
stereo pairs (BASELINE config 2, "PSMNet inference at 544x960, D=192, batch 8"):
  1. concat cost volume      [8,32,136,240] x2 -> [8,64,48,136,240]   (a1)
  2. soft-argmin             [8,192,544,960] logits -> [8,1,544,960]  (a4)
  3. patch reprojection loss (ps = 11, masked MSE) of the IR patterns warped by
     the predicted disparity, + the Fold visualisation image            (a7)
Weak scaling: every rank processes its own batch of 8 pairs; no collective on
the data path (SURVEY.md §8e).  `value` times the step with inputs resident in
HBM; `e2e` times the same calls with every input copied from pinned host memory
and the results (disparity + loss) copied back inside the timed region.

`--impl reference` times the reference's CPU implementation of the same step
(the torch restatement in oracle/, all host threads) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "stereo pairs/s, costvol+dispreg+reproj @544x960 D=192"
UNIT = "pairs/s"
B, C, H, W, D, PS = 8, 32, 544, 960, 192, 11
HQ, WQ, DQ = H // 4, W // 4, D // 4
WORKLOAD = (f"config2: PSMNet inference hot path fwd, batch {B} x {H}x{W}, D={D}: concat volume "
            f"[{B},{2 * C},{DQ},{HQ},{WQ}] + soft-argmin [{B},{D},{H},{W}] + patch reprojection loss ps={PS} (+fold image); "
            f"logits = trilinear upsample of random [{DQ},{HQ},{WQ}] logits as psmnet.py:186-197 produces them")

# identical in both arms (the driver compares the dicts): what one step processes and how it is sharded
CONFIG = {"workload": WORKLOAD, "pairs_per_gpu_per_step": B, "sharding": "batch (pairs) per rank, no data-path collective",
          "l2": "inputs larger than L2: 6.5 GB streamed per step vs 126 MB L2"}
NOMINAL_HBM_GBS = 8000.0  # the ~8 TB/s the north star quotes (DGX figure; HGX B200: 7.7 TB/s)

# algorithmic bytes per launch (SURVEY.md §8d formulas x B pairs), fp32
ALGO_BYTES = {
    "concat_volume_fwd": 4 * (2 * C * HQ * WQ + 2 * C * DQ * HQ * WQ) * B,
    "soft_argmin_fwd": 4 * (D * H * W + H * W) * B,
    "reproj_patch_loss+fold_fwd": (4 * (2 * 1 * H * W + H * W) + H * W + 4 * H * W) * B,  # + fold image out
}


# training hot path per pair (SURVEY.md §8d): concat fwd+bwd, 3 x soft-argmin fwd+bwd, patch reprojection fwd+bwd
TRAIN_B, TRAIN_STEPS = 2, 10
TRAIN_BATCHES = (2, 8)   # the reference's per-GPU batch (configs/config.py:93) and the bench batch
STOCK_B = 2
TRAIN_BYTES_PER_PAIR = (2 * 4 * (2 * C * HQ * WQ + 2 * C * DQ * HQ * WQ) + 3 * (4 * (D * H * W + H * W) + 4 * (2 * D * H * W + 2 * H * W))
                        + 4 * 3 * H * W + H * W + 4 * H * W)
BOUND = {"concat_volume_fwd": "hbm", "soft_argmin_fwd": "hbm", "reproj_patch_loss+fold_fwd": "lsu (shared-memory wavefronts)"}
NUM_SMS = 148
FUSED_EX2 = (2 * (DQ - 1) + 4) * H * W * B   # ex2 per launch of the fused upsample + soft-argmin kernel
_VOL, _FEAT, _LOG, _IMG = 4 * 2 * C * DQ * HQ * WQ, 4 * 2 * C * HQ * WQ, 4 * D * H * W, 4 * H * W
TRAIN_PHASE_BYTES = {"concat_fwd": _VOL + _FEAT, "concat_bwd": _VOL + _FEAT, "soft_argmin_fwd_x3": 3 * (_LOG + 3 * _IMG),
                     "soft_argmin_bwd_x3": 3 * (2 * _LOG + 4 * _IMG)}  # per pair


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _traffic():
    """dram bytes per launch from the committed ncu --set full capture, if any."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            pass
    return {}


# ----------------------------------------------------------------------------------------------
# clocks sampled DURING the timed regions
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    BAD = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
           "hw_power_brake_slowdown": 0x80}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._active = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception as e:  # pragma: no cover
            self._nv, self.error = None, repr(e)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                    for name, bit in {**self.BAD, **self.NOTE}.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        self._active.set()

    def pause(self):
        self._active.clear()

    def result(self):
        self._stop.set()
        if self._nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": int(statistics.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's torch restatement on the host cores
# ----------------------------------------------------------------------------------------------
def cpu_reference_step(inputs, so):
    """One pass of the same forward step for `inputs` (a 1-pair sample), stock torch on CPU."""
    L, R, cost, pat_L, pat_R, mask = inputs
    vol = so.concat_volume(L, R, DQ)
    disp = so.soft_argmin(cost)
    loss, vis, _ = so.reproj_error_patch(pat_L, pat_R, disp, mask, ps=PS)
    return vol, disp, loss, vis


def stock_torch_step(L, R, cost, pat_L, pat_R, mask):
    """The reference's dataflow with stock torch operators on whatever device the inputs live on
    (psmnet.py:151-165, :200-201 + psmnet_submodule.py:80-89, utils/reprojection.py:13-35 and :99-127)."""
    import torch.nn.functional as F

    nb, c, hq, wq = L.shape
    vol = torch.zeros(nb, 2 * c, DQ, hq, wq, device=L.device)
    for i in range(DQ):
        if i > 0:
            vol[:, :c, i, :, i:] = L[:, :, :, i:]
            vol[:, c:, i, :, i:] = R[:, :, :, :-i]
        else:
            vol[:, :c, i] = L
            vol[:, c:, i] = R
    prob = F.softmax(cost, dim=1)
    disp = torch.sum(prob * torch.arange(D, device=cost.device, dtype=torch.float32).view(1, D, 1, 1), 1, keepdim=True)
    bs, ch, h, w = pat_L.shape
    unfold = torch.nn.Unfold(kernel_size=(PS, PS), padding=(PS - 1) // 2)
    Lu = unfold(pat_L).reshape(bs, -1, h, w)
    Ru = unfold(pat_R).reshape(bs, -1, h, w)
    xb = torch.linspace(0, 1, w, device=L.device).repeat(bs, h, 1)
    yb = torch.linspace(0, 1, h, device=L.device).repeat(bs, w, 1).transpose(1, 2)
    flow = torch.stack((xb + (-disp[:, 0]) / w, yb), dim=3)
    Wu = F.grid_sample(Ru, 2 * flow - 1, mode="bilinear", padding_mode="zeros", align_corners=False)
    sel = mask.repeat(1, Lu.shape[1], 1, 1)
    loss = F.mse_loss(Wu[sel], Lu[sel])
    fold = torch.nn.Fold(output_size=(h, w), kernel_size=(PS, PS), padding=(PS - 1) // 2)
    vis = fold(Wu.reshape(bs, -1, h * w))
    return vol, disp, loss, vis


def time_stock_torch_gpu(L, R, cost, pat_L, pat_R, mask, steps=5):
    with torch.no_grad():
        for _ in range(2):
            stock_torch_step(L, R, cost, pat_L, pat_R, mask)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(steps):
            out = stock_torch_step(L, R, cost, pat_L, pat_R, mask)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        loss = float(out[2])
        del out
    torch.cuda.empty_cache()
    nb = L.shape[0]
    return {"note": "informational: the same forward step with STOCK torch operators on this B200 (the reference's own "
                    "dataflow; the reference hard-codes .cuda(), so this is its execution target)",
            "pairs_per_step": nb, "ms_per_step": ms, "value": nb / (ms * 1e-3), "unit": UNIT, "loss_check": loss}


def make_inputs(nb, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    L = torch.randn(nb, C, HQ, WQ, generator=g)
    R = torch.randn(nb, C, HQ, WQ, generator=g)
    # The logits PSMNet feeds to softmax are ALWAYS the trilinear upsample of the [1,D/4,H/4,W/4] output of the
    # 3-D aggregation (nets/psmnet/psmnet.py:186-197), so the synthetic logits are built the same way from
    # random low-resolution logits: spatially smooth, like the disparity map regressed from them.
    cost = torch.empty(nb, D, H, W)
    for b in range(nb):  # generated per pair to bound the temporary
        low = torch.randn(1, 1, DQ, HQ, WQ, generator=g) * 4.0
        cost[b] = torch.nn.functional.interpolate(low, size=(D, H, W), mode="trilinear", align_corners=False)[0, 0]
    pat_L = (torch.rand(nb, 1, H, W, generator=g) > 0.5).float()
    pat_R = (torch.rand(nb, 1, H, W, generator=g) > 0.5).float()
    mask = torch.rand(nb, 1, H, W, generator=g) > 0.2
    ts = [L, R, cost, pat_L, pat_R, mask]
    if pin:
        ts = [t.pin_memory() for t in ts]
    if device != "cpu":
        ts = [t.to(device) for t in ts]
    return ts


VOLUME_SAMPLE = 1 << 22  # cost-volume elements --dump-outputs keeps (16 MB of the 3.3 GB volume)


def dump_outputs(out_dir, outputs):
    """Write what one step returns to its caller as float32 <name>.npy files in `out_dir`: the disparity, the loss and
    the fold image whole, and of the cost volume the VOLUME_SAMPLE elements at flat indices drawn from a generator
    seeded with 0, in increasing index order (50 MB in all at B = 8)."""
    import numpy as np

    vol, disp, loss, vis = outputs
    idx = torch.randint(vol.numel(), (VOLUME_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    arrays = {"cost_volume_sample": vol.reshape(-1)[idx.to(vol.device)], "disparity": disp, "loss": loss,
              "fold_image": vis}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def time_cpu_reference(steps, warmup):
    from oracle import stereo_oracle as so

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    inputs = make_inputs(1, 1234)
    with torch.no_grad():
        for _ in range(warmup):
            cpu_reference_step(inputs, so)
        t0 = time.perf_counter()
        for _ in range(steps):
            cpu_reference_step(inputs, so)
        dt = time.perf_counter() - t0
    return steps * 1 / dt, dt / steps * 1e3, cores


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)  # each step is a bounded 1-pair sample (~1 s)
    pairs_s, ms, cores = time_cpu_reference(steps, warmup)
    sample = f"1 pair of the {B}-pair batch per step, {steps} timed steps after {warmup} warm-up, torch {torch.__version__} CPU"
    line = {
        "impl": "reference", "metric": METRIC, "value": pairs_s, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": CONFIG, "sample": sample,
        "note": "the reference runs this path on CUDA (hard-coded .cuda()); this arm is its torch code on the host cores, "
                "as the tier contract asks -- the same-GPU comparison is the B200 arm's variant_stock_torch_gpu",
        "cpu_baseline": {"value": pairs_s, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": pairs_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    from activezero_b200 import _lib, dist_util, ops
    from activezero_b200.utils import reprojection as az_rp

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_util.init_from_env("nccl", dev)
    _lib.load()
    # weak scaling: the job is world*B pairs, rank r owns pairs [first, first+B)
    first_pair, n_pairs = dist_util.shard_pairs(world * B, rank, world)
    assert n_pairs == B

    host = make_inputs(n_pairs, 1000 + first_pair, pin=True)
    L, R, cost, pat_L, pat_R, mask = [t.to(dev, non_blocking=True) for t in host]
    torch.cuda.synchronize()
    # Order inside a step (the three calls are independent except disp -> loss): the volume's 3.3 GB store stream is
    # followed by the compute-bound patch kernel, so the write-back of its last dirty L2 lines drains under a kernel
    # that does not need HBM; with the soft-argmin behind it (round 1's order) that kernel's read stream paid for the
    # drain (0.494 ms in the step against 0.459 ms alone).
    names = ["soft_argmin_fwd", "concat_volume_fwd", "reproj_patch_loss+fold_fwd"]

    def step(Ld, Rd, costd, pLd, pRd, md, evs=None):
        if evs is not None:
            evs[0].record()
        disp = ops.soft_argmin(costd)
        if evs is not None:
            evs[1].record()
        vol = ops.build_concat_volume(Ld, Rd, DQ)
        if evs is not None:
            evs[2].record()
        loss, vis = ops.reproj_loss(pLd, pRd, disp, md, ps=PS, sign=-1.0, want_warped=True)
        if evs is not None:
            evs[3].record()
        return vol, disp, loss, vis

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    with torch.no_grad():
        for _ in range(args.warmup):
            out = step(L, R, cost, pat_L, pat_R, mask)
        del out
        # ---- per-kernel CUDA events for the roofline: K eager steps, the three calls bracketed by events ----
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for k in range(args.steps):
            out = step(L, R, cost, pat_L, pat_R, mask, evs[k])
        e1.record()
        barrier()
        ms_eager = e0.elapsed_time(e1)
        del out
        # ---- device-resident timing (value): the step captured ONCE in a CUDA graph (the calls only enqueue on the
        # caller's stream: no allocation, no sync, no host readback), then exactly K replays between the barriers.
        # One graph launch per step keeps eight ranks' Python launch paths (4 host CPUs each) off the critical path;
        # the eager figure above is reported next to it.
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(L, R, cost, pat_L, pat_R, mask)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        launches0 = _lib.kernel_launches
        with torch.cuda.graph(graph):
            gout = step(L, R, cost, pat_L, pat_R, mask)
        launches_per_step = _lib.kernel_launches - launches0
        for _ in range(2):
            graph.replay()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        clocks.start()
        start.record()
        for k in range(args.steps):
            graph.replay()
        stop.record()
        barrier()
        clocks.pause()
        launches = launches_per_step * args.steps
        ms_total = start.elapsed_time(stop)
        loss_graph = float(gout[2])
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, gout)
        del gout, graph

        # ---- end to end: pinned host -> device, compute, results back, every step ----
        e2e_steps = max(1, min(args.steps, 10))
        res_disp = torch.empty((B, 1, H, W), dtype=torch.float32).pin_memory()
        res_loss = torch.empty((), dtype=torch.float32).pin_memory()
        h2d = sum(t.numel() * t.element_size() for t in host)
        d2h = res_disp.numel() * 4 + 4

        # The step is pipelined over two streams: the 3.2 GB of logits are shipped pair by pair on a copy stream
        # (one cudaMemcpyAsync per tensor per pair) while the compute stream runs the soft-argmin of the pairs that
        # have landed; the small inputs go first, the batch-level calls (volume, patch loss over the whole batch,
        # as the reference computes its masked mean) follow the last pair, and the results return on the copy stream.
        copy_stream = torch.cuda.Stream(device=dev)
        dev_in = [torch.empty_like(t, device=dev) for t in host]
        disp_buf = torch.empty((n_pairs, 1, H, W), dtype=torch.float32, device=dev)
        pair_ready = [torch.cuda.Event() for _ in range(n_pairs)]
        small_ready, done_ev, reuse_ev = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()

        def e2e_step():
            comp = torch.cuda.current_stream()
            copy_stream.wait_event(reuse_ev)  # the previous step no longer reads the staging buffers
            with torch.cuda.stream(copy_stream):
                for k in (0, 1, 3, 4, 5):
                    dev_in[k].copy_(host[k], non_blocking=True)
                small_ready.record(copy_stream)
                for j in range(n_pairs):
                    dev_in[2][j].copy_(host[2][j], non_blocking=True)
                    pair_ready[j].record(copy_stream)
            comp.wait_event(small_ready)
            vol = ops.build_concat_volume(dev_in[0], dev_in[1], DQ)
            for j in range(n_pairs):
                comp.wait_event(pair_ready[j])
                disp_buf[j:j + 1] = ops.soft_argmin(dev_in[2][j:j + 1])
            loss, vis, _ = az_rp.get_reproj_error_patch(dev_in[3], dev_in[4], disp_buf, dev_in[5], ps=PS)
            done_ev.record(comp)
            reuse_ev.record(comp)
            copy_stream.wait_event(done_ev)
            with torch.cuda.stream(copy_stream):
                res_disp.copy_(disp_buf, non_blocking=True)
                res_loss.copy_(loss, non_blocking=True)
            comp.wait_stream(copy_stream)
            return vol, vis

        def az_call(dv):
            # the call a user makes: the reference-named functions of the drop-in modules
            vol = ops.build_concat_volume(dv[0], dv[1], DQ)
            disp = ops.soft_argmin(dv[2])
            loss, vis, _ = az_rp.get_reproj_error_patch(dv[3], dv[4], disp, dv[5], ps=PS)
            return vol, disp, loss, vis

        reuse_ev.record(torch.cuda.current_stream())
        for _ in range(2):
            e2e_step()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        clocks.start()
        s2.record()
        for _ in range(e2e_steps):
            e2e_step()
        e2.record()
        barrier()
        clocks.pause()
        ms_e2e = s2.elapsed_time(e2)
        loss_val = float(res_loss)
        # the host link alone: the same pinned buffers, H2D only, all ranks at once (barrier on both sides)
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        h0.record()
        for _ in range(3):
            for k in range(len(host)):
                dev_in[k].copy_(host[k], non_blocking=True)
        h1.record()
        barrier()
        ms_h2d = h0.elapsed_time(h1) / 3

        # ---- informational variant (SURVEY.md §8f-1): the same step when the soft-argmin is fed by the
        # LOW-RESOLUTION logits and fused with the trilinear upsample, i.e. the [B,192,544,960] tensor is
        # never materialised (nor shipped over PCIe).  Not part of `value` / `e2e`.
        low_host = (torch.randn(n_pairs, 1, DQ, HQ, WQ, generator=torch.Generator().manual_seed(7 + first_pair)) * 4.0).pin_memory()
        low_dev = low_host.to(dev)

        fk = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]

        def fused_step(Ld, Rd, lowd, pLd, pRd, md, ev=None):
            vol = ops.build_concat_volume(Ld, Rd, DQ)
            if ev is not None:
                ev[0].record()
            disp = ops.upsample_soft_argmin(lowd, (D, H, W))
            if ev is not None:
                ev[1].record()
            loss, vis = ops.reproj_loss(pLd, pRd, disp, md, ps=PS, sign=-1.0, want_warped=True)
            return vol, disp, loss, vis

        def fused_e2e_step():
            dv = [host[0].to(dev, non_blocking=True), host[1].to(dev, non_blocking=True),
                  low_host.to(dev, non_blocking=True)] + [t.to(dev, non_blocking=True) for t in host[3:]]
            _, disp, loss, _ = fused_step(*dv)
            res_disp.copy_(disp, non_blocking=True)
            res_loss.copy_(loss, non_blocking=True)

        for _ in range(3):
            fused_step(L, R, low_dev, pat_L, pat_R, mask)
            fused_e2e_step()
        f0, f1, f2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        barrier()
        f0.record()
        for k in range(args.steps):
            fused_step(L, R, low_dev, pat_L, pat_R, mask, fk[k])
        f1.record()
        for _ in range(e2e_steps):
            fused_e2e_step()
        f2.record()
        barrier()
        ms_fused, ms_fused_e2e = f0.elapsed_time(f1), f1.elapsed_time(f2)
        ms_fused_k = statistics.fmean(a_.elapsed_time(b_) for a_, b_ in fk)
        h2d_fused = h2d - host[2].numel() * 4 + low_host.numel() * 4

        # ---- informational variant: the TRAINING hot path (BASELINE target "fwd/bwd"), forward and backward of
        # concat volume + three soft-argmin heads (psmnet.py:200-217) + patch reprojection loss on the last head,
        # at the same frame size, device-resident, at the reference's per-GPU batch (2) and at the bench batch (8).
        # The upstream gradients of the volume and of the three heads are synthetic tensors (in the network they
        # come from dres0 and the smooth-L1 loss).  Each phase is bracketed by CUDA events.
        del low_dev
        ms_train = float("nan")
        train_rows = {}
        if not args.no_train_variant:
            phases = ["concat_fwd", "soft_argmin_fwd_x3", "reproj_patch_fwd", "reproj_patch_bwd", "soft_argmin_bwd_x3", "concat_bwd"]
            for tb in TRAIN_BATCHES:
                with torch.enable_grad():
                    Lt, Rt = L[:tb].clone().requires_grad_(True), R[:tb].clone().requires_grad_(True)
                    heads = [cost[:tb].clone().requires_grad_(True) for _ in range(3)]
                    gvol = torch.randn(tb, 2 * C, DQ, HQ, WQ, device=dev)
                    gheads = [torch.randn(tb, 1, H, W, device=dev) for _ in range(3)]
                    tev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)] for _ in range(TRAIN_STEPS)]

                    def train_step(ev=None):
                        def mark(i_):
                            if ev is not None:
                                ev[i_].record()
                        for t in [Lt, Rt] + heads:
                            t.grad = None
                        mark(0)
                        vol = ops.build_concat_volume(Lt, Rt, DQ)
                        mark(1)
                        d1, d2, d3 = (ops.soft_argmin(c_) for c_ in heads)
                        mark(2)
                        loss, _, _ = az_rp.get_reproj_error_patch(pat_L[:tb], pat_R[:tb], d3, mask[:tb], ps=PS)
                        mark(3)
                        gd3, = torch.autograd.grad(loss, d3)
                        mark(4)
                        torch.autograd.backward([d1, d2, d3], [gheads[0], gheads[1], gheads[2] + gd3])
                        mark(5)
                        vol.backward(gvol)
                        mark(6)

                    for _ in range(3):
                        train_step()
                    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    barrier()
                    t0.record()
                    for k in range(TRAIN_STEPS):
                        train_step(tev[k])
                    t1.record()
                    barrier()
                    ms_tb = t0.elapsed_time(t1)
                    train_rows[tb] = {"ms_total": ms_tb, "phases": {
                        n_: statistics.fmean(tev[k][i_].elapsed_time(tev[k][i_ + 1]) for k in range(TRAIN_STEPS))
                        for i_, n_ in enumerate(phases)}}
                    if tb == TRAIN_B:
                        ms_train = ms_tb
                    del Lt, Rt, heads, gvol, gheads

        # ---- informational: the SAME forward step with stock torch operators on this GPU (the reference's own
        # dataflow: zero volume + 96 slice copies, softmax + regression, Unfold + grid_sample + boolean gathers + Fold),
        # STOCK_B pairs.  This, not the CPU arm, is the like-for-like baseline: the reference runs on CUDA.
        stock = None
        if world == 1 and not args.no_stock_variant:
            stock = time_stock_torch_gpu(L[:STOCK_B], R[:STOCK_B], cost[:STOCK_B], pat_L[:STOCK_B], pat_R[:STOCK_B],
                                         mask[:STOCK_B])

        # ---- informational: SURVEY §8f-2, the first aggregation convolution (Conv3d 64 -> 32, 3x3x3 on the concat volume,
        # psmnet.py:165-168) on the IMPLICIT volume -- the one tensor-core kernel of the library (tcgen05 TF32, TMEM) --
        # against volume + cuDNN on the same 2 pairs.  Not part of value / e2e.
        vconv = None
        if world == 1 and not args.no_stock_variant:
            import torch.nn.functional as F_

            VB = 2
            wconv = torch.randn(32, 64, 3, 3, 3, device=dev) * 0.05
            wp = ops.pack_volume_conv_weight(wconv)
            Lv, Rv = L[:VB].contiguous(), R[:VB].contiguous()

            def _time(fn, n=10):
                for _ in range(3):
                    fn()
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a_.record()
                for _ in range(n):
                    fn()
                b_.record()
                torch.cuda.synchronize()
                return a_.elapsed_time(b_) / n

            ms_v = _time(lambda: ops.volume_conv0(Lv, Rv, wp, DQ))
            ms_lib = _time(lambda: F_.conv3d(ops.build_concat_volume(Lv, Rv, DQ, channels_last=True), wconv.contiguous(
                memory_format=torch.channels_last_3d), padding=1))
            flop_nominal = 2.0 * VB * DQ * HQ * WQ * 32 * 64 * 27
            vconv = {"note": "informational: first aggregation convolution on the implicit volume (tcgen05 TF32, fp32 accumulation "
                             "in tensor memory; the right half of the volume is shift-invariant in x - d and computed once per "
                             "row, so about half of the nominal FLOPs are executed) vs this repo's channels_last_3d volume + "
                             "cuDNN conv3d (TF32) on the same pairs",
                     "pairs": VB, "ms": ms_v, "ms_volume_plus_cudnn": ms_lib, "speedup": ms_lib / ms_v,
                     "roofline": {"bound": "tensor", "achieved": flop_nominal / (ms_v * 1e-3) / 1e12, "unit": "TFLOP/s (nominal FLOPs)",
                                  "peak": 1125.0, "peak_source": "nominal dense TF32 = half of the 2.25 PFLOP/s bf16 figure",
                                  "frac": flop_nominal / (ms_v * 1e-3) / 1e12 / 1125.0}}
            del wconv, wp, Lv, Rv

        # ---- informational: the same K steps software-pipelined across batches over two streams -- the patch loss of
        # batch i (compute-bound, bands sized for 48 SMs: AZ_PATCH_SMS) runs UNDER the concat volume of batch i and the
        # soft-argmin of batch i+1 (HBM-bound), which it cannot do inside one step (DESIGN.md section 4.10;
        # benchmarks/sm_partition_pipeline.py also runs it on green-context SM partitions).  Every kernel of the K
        # steps, the last loss included, lies inside the timed region.  Not part of value / e2e.
        pipe = None
        if world == 1 and not args.no_stock_variant:
            try:
                s_patch, s_hbm = torch.cuda.Stream(device=dev, priority=-1), torch.cuda.Stream(device=dev)
                keep = [None]

                def _pipe(n):
                    for _ in range(n):
                        with torch.cuda.stream(s_hbm):
                            d_ = ops.soft_argmin(cost)
                            ready = torch.cuda.Event()
                            ready.record(s_hbm)
                            v_ = ops.build_concat_volume(L, R, DQ)
                            del v_
                        d_.record_stream(s_patch)  # allocated on s_hbm, read on s_patch: the allocator recycles the
                        with torch.cuda.stream(s_patch):  # block only after s_patch has passed this point (no growth)
                            s_patch.wait_event(ready)
                            keep[0] = ops.reproj_loss(pat_L, pat_R, d_, mask, ps=PS, sign=-1.0, want_warped=True)

                os.environ["AZ_PATCH_SMS"] = "48"
                s_hbm.wait_stream(torch.cuda.current_stream())
                s_patch.wait_stream(torch.cuda.current_stream())
                _pipe(max(3, args.warmup))
                torch.cuda.synchronize()
                p0, ph, pp = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                p0.record(s_hbm)
                _pipe(args.steps)
                ph.record(s_hbm)
                pp.record(s_patch)
                torch.cuda.synchronize()
                ms_pipe = max(p0.elapsed_time(ph), p0.elapsed_time(pp)) / args.steps
                pipe = {"note": "informational: K steps pipelined across batches over two streams (eager launches): patch loss "
                                "of batch i, bands sized for 48 SMs, under the concat volume of batch i and the soft-argmin of "
                                "batch i+1; all work of the K steps inside the timed region",
                        "ms_per_step": ms_pipe, "value": B / (ms_pipe * 1e-3), "unit": UNIT,
                        "speedup_vs_eager_sequential": ms_eager / args.steps / ms_pipe,
                        "loss": float(keep[0][0]),
                        "pipeline_frac": sum(ALGO_BYTES.values()) / (ms_pipe * 1e-3) / 1e9 / _peaks()[0]}
                keep[0] = None
            except Exception as e:  # informational only: never take the bench line down
                pipe = {"error": repr(e)}
            finally:
                os.environ.pop("AZ_PATCH_SMS", None)

    ms_total, ms_e2e, ms_fused, ms_fused_e2e, ms_train, ms_h2d, ms_fused_k, ms_eager = dist_util.max_over_ranks(
        [ms_total, ms_e2e, ms_fused, ms_fused_e2e, ms_train, ms_h2d, ms_fused_k, ms_eager], dev)

    if rank == 0:
        per_kernel = {}
        for i, n in enumerate(names):
            per_kernel[n] = statistics.fmean(evs[k][i].elapsed_time(evs[k][i + 1]) for k in range(args.steps))
        peak, peak_src = _peaks()
        traffic = _traffic()
        clk = clocks.result()
        sm_hz = (clk.get("sm_mhz") or 1965) * 1e6
        kernels = []
        for n in names:
            gbs = ALGO_BYTES[n] / (per_kernel[n] * 1e-3) / 1e9
            tr = traffic.get(n)
            row = {"kernel": n, "ms": per_kernel[n], "share": per_kernel[n] / sum(per_kernel.values()), "bound": BOUND[n],
                   "algo_bytes": ALGO_BYTES[n], "achieved_gbs": gbs}
            if BOUND[n] == "hbm":
                row.update({"frac": gbs / peak, "frac_nominal": gbs / NOMINAL_HBM_GBS,
                            "traffic": tr.get("dram_bytes") if isinstance(tr, dict) else tr})
            else:
                # not an HBM kernel (121 taps per pixel out of shared memory): placed on the LSU roofline -- shared-memory
                # wavefronts per launch from the committed ncu capture / (1 wavefront per clock per SM at the sampled clock)
                wf = tr.get("smem_wavefronts") if isinstance(tr, dict) else None
                row.update({"frac": None, "hbm_frac_for_reference_only": gbs / peak})
                if wf:
                    ach = wf / (per_kernel[n] * 1e-3)
                    row.update({"achieved": ach, "peak": NUM_SMS * sm_hz, "unit": "shared-memory wavefronts/s",
                                "frac": ach / (NUM_SMS * sm_hz), "wavefronts_per_launch": wf,
                                "wavefronts_ideal_per_launch": tr.get("smem_wavefronts_ideal"),
                                "source": tr.get("source")})
            kernels.append(row)
        # the roofline object is an HBM roofline: it describes the slowest of the HBM-bound kernels; the
        # patch kernel (121 taps per pixel out of shared memory, ~9 MB of compulsory traffic per pair) is
        # listed with its share in `kernels` and cannot be placed on a bandwidth roofline meaningfully
        dom = max((k for k in kernels if k["bound"] == "hbm"), key=lambda k: k["ms"])
        line = {
            "metric": METRIC, "value": world * B * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "launch": "one CUDA-graph replay per step (captured once; 3 C-ABI calls, %d kernels + 1 memset)" % launches_per_step,
            "ms_per_step_eager": ms_eager / args.steps, "value_eager": world * B * args.steps / (ms_eager * 1e-3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": CONFIG,
            "clocks": clk,
            "e2e": {"value": world * B * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps,
                    "api": "ops.build_concat_volume + ops.soft_argmin + utils.reprojection.get_reproj_error_patch",
                    "pipeline": "two streams: per-pair cudaMemcpyAsync of the logits overlapped with the soft-argmin of the "
                                "pairs already on the device; D2H of the results on the copy stream",
                    "h2d_only_ms": ms_h2d, "h2d_gbs_per_rank": h2d / (ms_h2d * 1e-3) / 1e9,
                    "h2d_share_of_step": ms_h2d / (ms_e2e / e2e_steps),
                    "limiter": "host->device copy of the 3.2 GB of logits per step (PCIe / host memory system; slowest rank reported)"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": peak,
                         "unit": "GB/s", "frac": dom["frac"], "traffic": dom["traffic"], "peak_source": peak_src,
                         "peak_nominal": NOMINAL_HBM_GBS, "frac_nominal": dom["achieved_gbs"] / NOMINAL_HBM_GBS,
                         "selection": "slowest HBM-bound kernel of the step (see kernels[] for all shares)",
                         "hbm_bound_share_of_step": sum(k["share"] for k in kernels if k["bound"] == "hbm"),
                         "pipeline_frac": sum(ALGO_BYTES.values()) / (ms_total / args.steps * 1e-3) / 1e9 / peak,
                         "pipeline_frac_nominal": sum(ALGO_BYTES.values()) / (ms_total / args.steps * 1e-3) / 1e9 / NOMINAL_HBM_GBS},
            "kernels": kernels,
            "variant_fused_upsample": {
                "note": "informational, SURVEY §8f-1: soft-argmin fused with the trilinear upsample reads the "
                        "[B,1,48,136,240] low-res logits; not the BASELINE config, not part of value/e2e",
                "value": world * B * args.steps / (ms_fused * 1e-3), "ms_per_step": ms_fused / args.steps,
                "e2e_value": world * B * e2e_steps / (ms_fused_e2e * 1e-3), "h2d_bytes_per_step": h2d_fused, "unit": UNIT,
                # the fused kernel reads 64x fewer bytes than the plain soft-argmin and is bounded by the MUFU (ex2) unit:
                # 2 ex2 per pixel and depth interval (geometric progression inside an interval) + 4 at the ends
                "fused_soft_argmin_kernel": {
                    "ms": ms_fused_k, "bound": "mufu", "ex2_per_launch": FUSED_EX2, "achieved": FUSED_EX2 / (ms_fused_k * 1e-3),
                    "peak": NUM_SMS * 16 * sm_hz, "unit": "ex2/s", "frac": FUSED_EX2 / (ms_fused_k * 1e-3) / (NUM_SMS * 16 * sm_hz),
                    "peak_source": "148 SMs x 16 MUFU lanes per clock x sampled SM clock"}},
            "loss_check": loss_val, "loss_check_graph": loss_graph,
        }
        if not args.no_train_variant:
            pairs_s = world * TRAIN_B * TRAIN_STEPS / (ms_train * 1e-3)
            line["variant_train_fwd_bwd"] = {
                "note": "informational: training hot path at the same frame size -- concat volume fwd+bwd, three "
                        "soft-argmin heads fwd+bwd, patch reprojection loss (ps=11, with Fold image) fwd+bwd; "
                        "synthetic upstream gradients; not part of value/e2e; rank 0's phases, slowest rank's total",
                "value": pairs_s, "unit": UNIT, "pairs_per_gpu_per_step": TRAIN_B, "steps": TRAIN_STEPS,
                "ms_per_step": ms_train / TRAIN_STEPS, "algo_bytes_per_pair": TRAIN_BYTES_PER_PAIR,
                "hbm_frac": pairs_s / world * TRAIN_BYTES_PER_PAIR / 1e9 / peak,
                "hbm_frac_nominal": pairs_s / world * TRAIN_BYTES_PER_PAIR / 1e9 / NOMINAL_HBM_GBS,
                "by_batch": {str(tb): {
                    "ms_per_step": r_["ms_total"] / TRAIN_STEPS, "pairs_per_s_per_gpu": tb * TRAIN_STEPS / (r_["ms_total"] * 1e-3),
                    "hbm_frac": tb * TRAIN_STEPS / (r_["ms_total"] * 1e-3) * TRAIN_BYTES_PER_PAIR / 1e9 / peak,
                    "phases_ms": r_["phases"],
                    "phases_hbm_frac": {n_: TRAIN_PHASE_BYTES[n_] * tb / (ms_ * 1e-3) / 1e9 / peak for n_, ms_ in r_["phases"].items()
                                        if n_ in TRAIN_PHASE_BYTES}} for tb, r_ in train_rows.items()}}
        if stock is not None:
            stock["speedup_of_value_per_pair"] = (line["value"] / world) / stock["value"]
            line["variant_stock_torch_gpu"] = stock
        if vconv is not None:
            line["variant_implicit_volume_conv"] = vconv
        if pipe is not None:
            line["variant_batch_pipelined"] = pipe
        if world == 1 and not args.no_cpu_baseline:
            pairs_s, _, cores = time_cpu_reference(12, 1)  # ~10 s of CPU work on the box's host cores
            line["cpu_baseline"] = {"value": pairs_s, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "1 pair of the 8-pair batch per step, 12 timed steps after 1 warm-up"}
        emit(line)
    else:
        clocks.result()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version
    banner to stdout when the communicator is created), so fd 1 is pointed at stderr for the whole run
    and the JSON line is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-variant", action="store_true")
    ap.add_argument("--no-stock-variant", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="B200 arm: after the timed steps, write the outputs of the last one as DIR/<name>.npy "
                         "(rank 0's batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        args.warmup = max(args.warmup, 3)  # timing rule: at least 3 warm-up steps
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
