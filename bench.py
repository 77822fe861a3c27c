#!/usr/bin/env python
"""Benchmark of the B-mode renderer hot path (BASELINE.json metric: frames/s and Gsamples/s, forward+backward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--poses P] [--dump-outputs DIR]

Workload (SURVEY.md 8d config 3, the batched pose sweep, with config 2's loss): P probe
poses per GPU x 128 rays x 512 samples over one synthetic MRI-shaped 256^3 impedance
volume, trilinear sampler, one step = render forward -> MSE against target frames ->
backward to d loss/d source and d loss/d directions of every pose.  Poses shard across
ranks with a full volume replica each and no data-path collective (weak scaling).

One JSON line on stdout (rank 0).  `value` is device-timed with everything resident in HBM;
`e2e` goes through the public API with the step's poses arriving from pinned host memory
and the loss + pose gradients read back to the host inside the timed region (the volume and
the target frames are uploaded once: they are the scene and the dataset of a pose-recovery
run, the poses are what changes per step).

Besides the headline (weak scaling: 1024 poses PER GPU) the line carries, at every N:
  `strong`       BASELINE config 3 as worded -- 1024 poses in total, sharded over the N ranks;
  `config4`      the MLP -> render -> MSE training step (4096 frames per step in total, sharded) with the NCCL all-reduce
                 of the weight gradients INSIDE the timed region, and the fused Adam update;
  `nccl_parity`  a small scene rendered rank-sharded: gathered frames and all-reduced weight gradients against the full
                 batch computed on rank 0 alone;
  `config5`      (N = 1) the 512^3 / 512 x 2048 stress case on >= 1024 poses spread over the sphere.
Every timed loop of these records runs `--steps` steps.  `--dump-outputs DIR` writes what the last timed headline step
returned (loss.npy, grad_sources.npy, grad_directions.npy; with N ranks, every rank's shard concatenated in rank order,
one loss per rank); the scene and poses are seeded, so two builds given the same arguments can be compared output for output.
`--impl reference` times the UNMODIFIED reference (oracle/_ref archive or /root/reference) on the host cores: all 128 rays of
a pose at the first 128 samples, forward + backward, plus one full config-1 frame (forward).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

# stdout carries exactly one JSON line: NCCL's banner ("NCCL version ...", printed to its debug file -- stdout by default --
# when the box sets NCCL_DEBUG) and any other NCCL log go to stderr.  Set before torch / NCCL read the environment.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bmode_frames_per_s_fwd_bwd"
UNIT = "frames/s"
N_RAYS, N_SAMPLES, VOL_N = 128, 512, 256
ALPHA = 1e-4
OPENING_ANGLE = math.radians(60.0)     # pose_sweep's fan aperture
BYTES_PER_SAMPLE_FWD = 36      # SURVEY.md 8(d): 8 trilinear gathers x 4 B + 4 B frame write
BYTES_PER_SAMPLE_BWD = 36      # re-gather 8 x 4 B + read d loss/d frame 4 B (pose gradients only)
BYTES_PER_SAMPLE_FUSED = 36    # fused step: 8 gathers x 4 B + 4 B target read (frames are not written)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 100 ms while the GPU is under the benchmark load."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.mark = index, [], None, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def begin_region(self):
        self.mark = len(self.rows)

    def count(self):
        return len(self.rows) - self.mark

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.mark:]:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(P, layout):
    """DRAM bytes per launch of the fused kernel from the committed ncu capture, if it is the same workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            entries = json.load(f)["render_bwd_kernel_fused_mse"]
        for t in (entries if isinstance(entries, list) else [entries]):
            if (t["poses"], t["rays"], t["samples"], t["layout"]) == (P, N_RAYS, N_SAMPLES, layout):
                return t["bytes_per_launch"]
    except Exception:
        pass
    return None


def ncu_counter(P, layout, key):
    """Another per-launch counter of the committed ncu capture (same file as ncu_traffic)."""
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            entries = json.load(f)["render_bwd_kernel_fused_mse"]
        for t in (entries if isinstance(entries, list) else [entries]):
            if (t["poses"], t["rays"], t["samples"], t["layout"]) == (P, N_RAYS, N_SAMPLES, layout):
                return t.get(key)
    except Exception:
        pass
    return None


def build_scene(device, n_poses, seed, return_params=False):
    from diffus_b200.phantoms import intensity_to_impedance, mri_phantom, pose_sweep
    vol = intensity_to_impedance(mri_phantom(VOL_N, "t1", seed=0))
    sources, dirs, median, hint = pose_sweep(n_poses, N_RAYS, VOL_N, seed=seed, return_params=True)
    if return_params:
        return vol, sources, dirs, median, hint
    return vol, sources, dirs


def headline_config(P, world, layout):
    """The `config` object: identical in both arms (the reference arm times a bounded sample OF THIS workload)."""
    return {
        "workload": f"config3 pose sweep fwd+bwd: {P} poses/GPU x {N_RAYS} rays x {N_SAMPLES} samples, "
                    f"{VOL_N}^3 MRI-shaped impedance volume, trilinear, MSE vs target frames, "
                    "gradients to every pose's source and directions",
        "poses_per_gpu": P, "rays": N_RAYS, "samples": N_SAMPLES, "volume": f"{VOL_N}^3 f32",
        "volume_layout": layout, "parallelism": f"pose-sharded x{world}, volume replicated",
        "l2": "no explicit flush: inputs exceed L2 -- every step streams its own 268 MB of target frames per "
              "1024 poses (>> 126 MB L2, marked evict-first); the 64 MiB volume is meant to stay L2-resident",
    }


def timed_steps(fn, warmup, steps, barrier):
    """CUDA-event time of `steps` back-to-back calls of fn after `warmup` calls, bracketed by barriers (ms per step)."""
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


DUMP_BYTES = 60 * 1000 ** 2      # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(out_dir, outputs):
    """Write the tensors a caller of the timed step receives as ``out_dir/<name>.npy`` (float32; float64 stays float64), so
    that two builds can be compared output for output.  If they exceed DUMP_BYTES in all, every array keeps the same fixed, seeded
    sample of rows along its first (pose) axis."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name, t in outputs.items():
        t = t.detach()
        arrays[name] = (t if t.dtype == torch.float64 else t.float()).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES and a.ndim > 0:
            keep = max(1, a.shape[0] * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def gather_ranks(t, world):
    """Every rank's tensor of the same shape, concatenated along dim 0 in rank order (a collective: all ranks call it)."""
    if world == 1:
        return t
    import torch.distributed as dist
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t.contiguous())
    return torch.cat(parts)


def max_over_ranks(values, dev, world):
    import torch.distributed as dist
    t = torch.tensor(values, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def strong_scaling_record(dev, rank, world, barrier, layout, steps):
    """BASELINE config 3 as worded: 1024 poses IN TOTAL, sharded over the ranks (each rank: its contiguous block)."""
    from diffus_b200 import PreparedVolume, ops, render_frames
    from diffus_b200 import distributed as D
    from diffus_b200._lib import SAMPLER_TRILINEAR
    from diffus_b200.graphs import GraphedPoseStep
    total = 1024
    vol_h, src_h, dir_h = build_scene(dev, total, seed=1000)
    sl = D.pose_shard(total, rank, world)
    pv = PreparedVolume(vol_h.to(dev), layout)
    src, dirs = src_h[sl].to(dev).contiguous(), dir_h[sl].to(dev).contiguous()
    with torch.no_grad():
        target = render_frames(pv, src + torch.tensor([1.5, 0.0, -1.0], device=dev), dirs, N_SAMPLES, ALPHA, 0, sampler="trilinear")
    dims = list(pv.volume.shape)

    def eager():
        ops.render_mse_impl(pv.volume, pv.bricks, dims, src, dirs, target, N_SAMPLES, 0, ALPHA, SAMPLER_TRILINEAR, False, False, True, False)
    ms_eager = timed_steps(eager, 5, steps, barrier)
    g = GraphedPoseStep(pv, target, N_RAYS, N_SAMPLES, ALPHA)
    g.sources.copy_(src)
    g.directions.copy_(dirs)
    ms_graph = timed_steps(g.graph.replay, 5, steps, barrier)
    ms_eager, ms_graph = max_over_ranks([ms_eager, ms_graph], dev, world)
    return {"what": "config 3 strong scaling: 1024 poses in total, contiguous pose blocks per rank, fused fwd+MSE+bwd step, no collective "
                    "on the path; max over ranks of the CUDA-event time",
            "poses_total": total, "poses_per_gpu": sl.stop - sl.start, "ms_per_step_op_calls": ms_eager, "ms_per_step_cuda_graph": ms_graph,
            "frames_per_s_op_calls": total / (ms_eager * 1e-3), "frames_per_s_cuda_graph": total / (ms_graph * 1e-3)}


def config4_record(dev, rank, world, barrier, steps):
    """BASELINE config 4: MLP over a T2-shaped 256^3 volume -> 4096 frames per step IN TOTAL (sharded) -> MSE ->
    weight gradients -> NCCL all-reduce -> Adam, everything inside the timed region (FusedTrainer.step)."""
    from diffus_b200 import ImpedanceEstimator, PreparedVolume, render_frames
    from diffus_b200 import distributed as D
    from diffus_b200.phantoms import mri_phantom, pose_sweep
    from diffus_b200.training import FusedTrainer
    total = 4096
    torch.manual_seed(0)
    model = ImpedanceEstimator(1)
    with torch.no_grad():
        model.model[4].bias.fill_(1.5)
        model.model[4].weight.mul_(0.3)
    model = model.to(dev)
    mri = (mri_phantom(VOL_N, "t2") / 1000.0).to(dev)
    s_h, d_h = pose_sweep(total, N_RAYS, VOL_N, seed=2)
    sl = D.pose_shard(total, rank, world)
    s, d = s_h[sl].to(dev).contiguous(), d_h[sl].to(dev).contiguous()
    out = {"what": "config 4 training step: MLP(256^3) -> frames -> MSE -> d/dweights -> NCCL all-reduce (4.6 KB flat buffer) -> fused Adam; "
                   "4096 frames per step in total, sharded; CUDA-event time of FusedTrainer.step, max over ranks",
           "frames_total": total, "frames_per_gpu": sl.stop - sl.start}
    # target frames: the same scene through a SECOND seeded MLP (SURVEY 8(d) config 4) -- a rescaled copy of the first one
    # would leave every reflection coefficient, hence the loss, unchanged
    torch.manual_seed(1)
    model_tgt = ImpedanceEstimator(1)
    with torch.no_grad():
        model_tgt.model[4].bias.fill_(1.5)
        model_tgt.model[4].weight.mul_(0.3)
        z_tgt = model_tgt.to(dev).impedance_volume(mri, None, 1e6, 400.0)
    for sampler in ("trilinear", "nearest"):
        with torch.no_grad():
            tgt = render_frames(PreparedVolume(z_tgt), s, d, N_SAMPLES, ALPHA, sampler=sampler)
        tr = FusedTrainer(model, mri, lr=1e-4, sampler=sampler, out_scale=1e6, gather=os.environ.get("DIFFUS_CONFIG4_GATHER", "auto"))
        n_total = total * N_RAYS * N_SAMPLES
        last = [None]

        def step():
            last[0] = tr.step(s, d, tgt, N_SAMPLES, ALPHA, n_total=n_total)      # (a view of the trainer's persistent loss slot)
        step()
        loss_first = float(last[0])                      # read back before the next step overwrites the slot; untimed
        ms = timed_steps(step, 3, steps, barrier)
        (ms,) = max_over_ranks([ms], dev, world)
        out[sampler] = {"ms_per_step": ms, "frames_per_s": total / (ms * 1e-3), "gsamples_per_s": n_total / (ms * 1e-3) / 1e9,
                        "loss_first": loss_first, "loss_last": float(last[0]), "adam_steps": 1 + 3 + steps}
        del tr, tgt
    return out


def nccl_parity_record(dev, rank, world):
    """A small scene rendered rank-sharded through NCCL against the full batch on rank 0 alone: gathered frames must be
    bit-equal, the all-reduced weight gradients and the loss must agree to rounding (the volume scatter uses atomics)."""
    import copy
    import torch.distributed as dist
    from diffus_b200 import ImpedanceEstimator, render_frames
    from diffus_b200 import distributed as D
    from diffus_b200.phantoms import mri_phantom, pose_sweep
    from diffus_b200.training import FusedTrainer
    P, R, S, n = 8 * max(world, 1) + 3, 6, 48, 24                 # ragged on purpose when world > 1
    torch.manual_seed(7)
    model = ImpedanceEstimator(1)
    with torch.no_grad():
        model.model[4].bias.fill_(1.5)
        model.model[4].weight.mul_(0.3)
    mri = (mri_phantom(n, "t2", seed=2) / 1000.0).to(dev)
    s_h, d_h = pose_sweep(P, R, n, seed=9)
    tgt_h = 0.01 * torch.randn((P, R, S), generator=torch.Generator().manual_seed(3))
    sl = D.pose_shard(P, rank, world)
    tr = FusedTrainer(copy.deepcopy(model).to(dev), mri, lr=1e-3, sampler="trilinear", out_scale=1e6)
    z = tr.forward_volume().clone()
    from diffus_b200 import ops
    z_lin = z if tr.gather == "texture" else ops.from_bricks(z, [n, n, n])       # (texture gathers: the volume is in torch order)
    frames_local = render_frames(z_lin, s_h[sl].to(dev), d_h[sl].to(dev), S, 1e-3, sampler="trilinear")
    frames = D.gather_frames(frames_local)                          # ragged shards: sizes are exchanged first
    loss = tr.step(s_h[sl].to(dev).contiguous(), d_h[sl].to(dev).contiguous(), tgt_h[sl].to(dev).contiguous(), S, 1e-3,
                   n_total=P * R * S)
    grads = tr.grads.clone()
    rec = None
    if rank == 0:
        full = FusedTrainer(copy.deepcopy(model).to(dev), mri, lr=1e-3, sampler="trilinear", out_scale=1e6)
        frames_full = render_frames(z_lin, s_h.to(dev), d_h.to(dev), S, 1e-3, sampler="trilinear")
        # rank 0 alone on the whole batch: temporarily a world of one (no collective is issued)
        saved = D.world
        D.world = lambda: (0, 1)
        try:
            loss_full = full.step(s_h.to(dev), d_h.to(dev), tgt_h.to(dev), S, 1e-3, n_total=P * R * S)
        finally:
            D.world = saved
        gerr = float((grads - full.grads).abs().max() / full.grads.abs().max())
        lerr = float(abs(loss.item() - loss_full.item()) / abs(loss_full.item()))
        rec = {"what": f"{P} poses x {R} rays x {S} samples on a {n}^3 volume, ragged pose shards over {world} rank(s): gathered frames "
                       "vs the full batch on rank 0 (bit-equal), all-reduced MLP weight gradients and loss vs the full batch",
               "frames_bit_equal": bool(torch.equal(frames, frames_full)), "weight_grad_max_rel_err": gerr, "loss_rel_err": lerr,
               "ok": bool(torch.equal(frames, frames_full)) and gerr <= 1e-4 and lerr <= 1e-5}
    if world > 1:
        dist.barrier()
    return rec


def config5_record(dev, poses, layout, steps):
    """BASELINE config 5 on one GPU: 512^3 volume (512 MiB: four times the L2), 512 rays x 2048 samples, `poses` poses spread
    over the sphere, fused fwd + MSE + bwd (pose gradients).  BASELINE's 4096 poses are `4096 / poses` such launches."""
    from diffus_b200 import PreparedVolume, ops, render_frames
    from diffus_b200._lib import SAMPLER_TRILINEAR
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n, R, S = 512, 512, 2048
    pv = PreparedVolume(layered_phantom(n, 0).to(dev), layout)
    s_h, d_h = pose_sweep(poses, R, n, seed=3)
    s, d = s_h.to(dev), d_h.to(dev)
    with torch.no_grad():
        tgt = render_frames(pv, s + torch.tensor([1.5, 0.0, -1.0], device=dev), d, S, ALPHA, sampler="trilinear")
    dims = [n, n, n]

    def step():
        ops.render_mse_impl(pv.volume, pv.bricks, dims, s, d, tgt, S, 0, ALPHA, SAMPLER_TRILINEAR, False, False, True, False)
    ms = timed_steps(step, 2, steps, torch.cuda.synchronize)
    samples = poses * R * S
    peak, _ = load_peaks()
    gs = samples / (ms * 1e-3) / 1e9
    rec = {"what": f"config 5: {n}^3 volume ({layout}), {R} rays x {S} samples, {poses} poses over the sphere, fused fwd+MSE+bwd with pose "
                   "gradients: ONE launch, one CTA per ray walking its four 512-column passes together (one warp each; no forward pre-pass)",
           "poses": poses, "ms_per_step": ms, "gsamples_per_s": gs, "frames_per_s": poses / (ms * 1e-3),
           "ms_for_4096_poses": ms * 4096 / poses, "bytes_per_sample": BYTES_PER_SAMPLE_FUSED,
           "hbm_frac_at_36B": gs * BYTES_PER_SAMPLE_FUSED / peak}
    try:
        hbm = ops.gather_probe(2048, device=dev)
        rec["hbm_random_sector_roof"] = {"sectors_per_s": hbm["sectors_per_s"], "buffer_mib": 2048}
    except Exception as exc:
        rec["hbm_random_sector_roof"] = {"error": str(exc)}
    return rec


def run_ours(args):
    import torch.distributed as dist
    from diffus_b200 import PreparedVolume, ops, render_frames, render_mse_loss
    from diffus_b200.graphs import GraphedFanPoseStep, GraphedPoseStep
    from diffus_b200._lib import SAMPLER_TRILINEAR

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout must carry exactly one JSON line, and NCCL prints its banner ("NCCL version ...") to stdout when the
        # communicator is created: point fd 1 at stderr while the process group comes up (eagerly, plus one collective)
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    P = args.poses
    vol_h, src_h, dir_h, med_h, hint_h = build_scene(dev, P, seed=1000 + rank, return_params=True)   # every rank: its own pose shard
    vol = PreparedVolume(vol_h.to(dev), args.layout) if args.layout != "linear" else vol_h.to(dev)
    src_pin, dir_pin = src_h.pin_memory(), dir_h.pin_memory()
    src_d, dir_d = src_h.to(dev), dir_h.to(dev)
    with torch.no_grad():
        shift = torch.tensor([1.5, 0.0, -1.0], device=dev)
        target = render_frames(vol, src_d + shift, dir_d, N_SAMPLES, ALPHA, 0, sampler="trilinear")
    samples_per_step = P * N_RAYS * N_SAMPLES
    bricks = vol.bricks if isinstance(vol, PreparedVolume) else None
    vol_t = vol.volume if isinstance(vol, PreparedVolume) else vol
    dims = list(vol_t.shape)

    # ---- device-resident step: the fused forward + MSE + backward op (what autograd calls) ----
    def step_device(ev=None):
        if ev:
            ev[0].record()
        loss, _, _, gs, gd = ops.render_mse_impl(vol_t, bricks, dims, src_d, dir_d, target, N_SAMPLES, 0, ALPHA,
                                                 SAMPLER_TRILINEAR, False, False, True, False)
        if ev:
            ev[1].record()
        return loss, gs, gd

    # ---- end-to-end step through the public API: host poses in, loss + gradients out ----
    out_src = torch.empty((P, 3), dtype=torch.float32).pin_memory()
    out_dir = torch.empty((P, N_RAYS, 3), dtype=torch.float32).pin_memory()
    out_loss = torch.empty((), dtype=torch.float32).pin_memory()

    # A pose sweep repeats the same shapes every step: the user-facing call for that is a CUDA-graph wrapper of the
    # fused step (diffus_b200.graphs); eager autograd costs more.  "fan" (default) drives the step with the
    # pose PARAMETERS north_star names -- source, median direction, in-plane hint, aperture (9 floats per pose in, 9
    # gradient floats + the loss out; the fans are built and their gradient folded back on the device) -- "graph" and
    # "eager" pass explicit (P,R,3) direction tensors like the reference's plot_beam_frame.
    gstep = fstep = None
    poses_pin = torch.stack([src_h, med_h, hint_h]).contiguous().pin_memory()       # (3, P, 3): one H2D copy per step
    out_pin = torch.empty((9 * P + 1,), dtype=torch.float32).pin_memory()            # gradients + loss: one D2H copy
    if args.e2e == "graph":
        gstep = GraphedPoseStep(vol, target, N_RAYS, N_SAMPLES, ALPHA)
    elif args.e2e == "fan":
        fstep = GraphedFanPoseStep(vol, target, N_RAYS, N_SAMPLES, OPENING_ANGLE, ALPHA)

    def step_e2e():
        if fstep is not None:
            out_pin.copy_(fstep.packed(poses_pin), non_blocking=True)   # pose parameters in, gradients + loss out
        elif gstep is not None:
            loss, gs, gd = gstep(src_pin, dir_pin)              # H2D of the poses into the graph's static inputs
            out_loss.copy_(loss, non_blocking=True)
            out_src.copy_(gs, non_blocking=True)
            out_dir.copy_(gd, non_blocking=True)
        else:
            s = src_pin.to(dev, non_blocking=True).requires_grad_(True)
            d = dir_pin.to(dev, non_blocking=True).requires_grad_(True)
            loss = render_mse_loss(vol, s, d, target, N_SAMPLES, ALPHA, 0, sampler="trilinear")
            loss.backward()
            out_loss.copy_(loss.detach(), non_blocking=True)
            out_src.copy_(s.grad, non_blocking=True)
            out_dir.copy_(d.grad, non_blocking=True)
        torch.cuda.current_stream().synchronize()        # the caller needs the numbers on the host
        return out_loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = max(args.warmup, 3), args.steps
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                  # nvidia-smi needs a moment to come up: start before the warm-up
    for _ in range(W):
        step_device()
    barrier()
    sampler.begin_region()
    launches0 = ops.launch_count()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(K):
        loss, gs, gd = step_device(evs[i])
    t1.record()
    barrier()
    launches = ops.launch_count() - launches0
    ms_total = t0.elapsed_time(t1)
    step_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)     # the fused kernel (+ 2 tiny reductions)

    for _ in range(W):
        step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        step_e2e()
    e1.record()
    barrier()
    e2e_ms_total = e0.elapsed_time(e1)
    if rank == 0:
        # a short run can end before nvidia-smi delivers a sample: keep the same load on (untimed) until it has
        t_hold = time.perf_counter()
        while sampler.proc is not None and sampler.count() < 3 and time.perf_counter() - t_hold < 4.0:
            for _ in range(20):
                step_device()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    ms_total, e2e_ms_total, step_ms = max_over_ranks([ms_total, e2e_ms_total, step_ms], dev, world)
    ms_per_step = ms_total / K
    frames_per_s = world * P / (ms_per_step * 1e-3)
    e2e_frames_per_s = world * P / (e2e_ms_total / K * 1e-3)
    loss_value, loss_e2e = float(loss), (float(out_pin[-1]) if args.e2e == "fan" else float(out_loss))
    if args.dump_outputs:
        # the last timed step's tensors (render_mse_impl allocates fresh outputs on every call); every rank's shard
        outs = {name: gather_ranks(t, world) for name, t in (("loss", loss), ("grad_sources", gs), ("grad_directions", gd))}
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)

    # ---- the other records: every rank takes part (collectives inside), rank 0 reports; a failure never costs the headline ----
    del target, fstep, gstep
    extras = {}
    if not args.no_extras:
        for name, fn in (("strong", lambda: strong_scaling_record(dev, rank, world, barrier, args.layout, K)),
                         ("config4", lambda: config4_record(dev, rank, world, barrier, K)),
                         ("nccl_parity", lambda: nccl_parity_record(dev, rank, world))):
            try:
                extras[name] = fn()
            except Exception as exc:                        # noqa: BLE001
                extras[name] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()
        if world == 1 and args.config5_poses > 0:
            try:
                extras["config5"] = config5_record(dev, args.config5_poses, args.layout, K)
            except Exception as exc:                        # noqa: BLE001
                extras["config5"] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = load_peaks()
        dom = f"render_bwd_kernel<trilinear, {args.layout}, pose_grad, LOSS_MSE> (fused forward + MSE + backward)"
        dom_bytes = samples_per_step * BYTES_PER_SAMPLE_FUSED
        achieved = dom_bytes / (step_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": frames_per_s, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "gsamples_per_s": world * samples_per_step / (ms_per_step * 1e-3) / 1e9,
            "config": headline_config(P, world, args.layout),
            "e2e": {"value": e2e_frames_per_s, "unit": UNIT,
                    "h2d_bytes_per_step": int(poses_pin.numel() * 4) if args.e2e == "fan"
                                          else int(src_pin.numel() * 4 + dir_pin.numel() * 4),
                    "d2h_bytes_per_step": int(out_pin.numel() * 4) if args.e2e == "fan"
                                          else int(out_src.numel() * 4 + out_dir.numel() * 4 + 4),
                    "ms_per_step": e2e_ms_total / K,
                    "api": {"fan": "GraphedFanPoseStep (CUDA-graph replay: fans from pose parameters -> fused step -> gradient "
                                   "folded back onto the pose parameters)",
                            "graph": "GraphedPoseStep (CUDA-graph replay of the fused step, explicit (P,R,3) directions)",
                            "eager": "render_mse_loss + loss.backward() (eager autograd, explicit directions)"}[args.e2e],
                    "note": "public API call per step; pose parameters (fan: source, median direction, in-plane hint; else "
                            "source + explicit directions) from pinned host memory each step, loss and pose gradients copied "
                            "back to pinned host memory, stream synchronised every step; volume and target frames resident.  "
                            "The explicit-direction forms (--e2e graph / eager, the reference's plot_beam_frame signature) move "
                            "1.57 MB each way per step, ~0.12 ms of PCIe that the 36 KB pose-parameter form does not pay"},
            "gpu_launches": launches,
            "kernels_ms": {"fused_step(render_bwd_kernel+reduce_rays_and_sum)": step_ms},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(P, args.layout), "peak_source": peak_src,
                         "bytes_per_sample": BYTES_PER_SAMPLE_FUSED,
                         "bytes_note": "SURVEY 8(d) counts 72 B/sample for forward+backward done as two passes "
                                       "(2 x (8 gathers x 4 B + 4 B)); the fused kernel gathers once and reads the "
                                       "target once, so its own algorithmic traffic is 36 B/sample.  The volume is L2-resident "
                                       "by design (DRAM is ~9 % busy, L2 19 %, L1/texture 46 %): no memory roof is near -- the "
                                       "kernel is bound by its issue slots (65 % busy at 16 resident warps per SM, 5.44 warp "
                                       "instructions per sample) and the latency of its texture gathers, see gather_roof and "
                                       "profiles/r2_fused_kernel_final.md",
                         "binding_unit": "issue slots / texture-gather latency (ncu: issue active 65 %, long_scoreboard 25 %)",
                         "frac_vs_two_pass_bytes": samples_per_step * 72 / (step_ms * 1e-3) / 1e9 / peak},
            "clocks": clocks,
            "loss": loss_value,
            "loss_e2e": loss_e2e,
        }
        line.update(extras)
        # SURVEY 8(d): the L2 gather roof from our own microbenchmark (random 32-byte sectors over a 64 MiB buffer), and
        # the same over 512 MiB (HBM random sectors: what a volume copy that does not fit L2 would run at)
        try:
            l2 = ops.gather_probe(64, device=dev)
            hbm = ops.gather_probe(512, device=dev)
            l1_miss_sectors = ncu_counter(P, args.layout, "l2_read_sectors_per_launch")
            roof = {"what": "random 32-byte-sector reads, 8 loads in flight per thread, 148 x 8 x 256 threads",
                    "l2_resident_64MiB": {"sectors_per_s": l2["sectors_per_s"], "gb_per_s": l2["gb_per_s"]},
                    "hbm_512MiB": {"sectors_per_s": hbm["sectors_per_s"], "gb_per_s": hbm["gb_per_s"]}}
            if l1_miss_sectors:
                rate = l1_miss_sectors / (step_ms * 1e-3)
                roof["kernel_l2_sector_reads_per_s"] = rate
                roof["frac_of_l2_gather_roof"] = rate / l2["sectors_per_s"]
                roof["note"] = ("the kernel's L2 -> L1 sector reads per launch are the ncu count "
                                "(lts__t_sectors_srcunit_tex_op_read) of the committed capture; the rest of its gather sectors "
                                "hit L1 and never reach L2")
            line["roofline"]["gather_roof"] = roof
        except Exception as exc:                       # the probe must never take the headline number down with it
            line["roofline"]["gather_roof"] = {"error": str(exc)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline(args.cpu_rays)
            except Exception as exc:                    # noqa: BLE001
                line["cpu_baseline"] = {"error": f"{type(exc).__name__}: {exc}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference on the host cores (oracle/reference_loader.py: /root/reference or the staged archive);
# the oracle's literal dense-solve port stands in only if neither exists (kind "port").
# ---------------------------------------------------------------------------------------------------------------------
CPU_SAMPLES = 128          # depth of the bounded CPU sample: the first 128 of the 512 samples of every ray
# 128 -> 512 samples: the reference's own forward (compute_echo_traces, 128 rays) measured 1.25 s at S = 128 and 68.0 s at
# S = 512 on 8 cores (SURVEY.md section 6) -- x54.4; its flop count grows as S^4 (x256).  The smaller factor is used.
CPU_DEPTH_FACTOR = 68.0 / 1.25


def cpu_scene():
    """All 128 rays of one pose of the workload, truncated to the first CPU_SAMPLES samples: the echo at depth k depends on
    the samples up to k only, so these ARE the first 128 columns of the workload's frame."""
    from oracle import port
    vol, src, dirs = build_scene(None, 1, seed=1000)
    d, s = dirs[0].contiguous(), src[0]
    with torch.no_grad():
        _, _, _, target = port.plot_beam_frame(vol, s + torch.tensor([1.5, 0.0, -1.0]), d, CPU_SAMPLES, ALPHA,
                                               sampler="trilinear", propagation="closed_form")
    return vol, s, d, target.float()


def cpu_sample_step(vol, src, dirs, target):
    """One bounded sample of the workload on the CPU: forward + MSE + backward to the pose through the reference's own
    ``UltrasoundRenderer.plot_beam_frame`` (its dense per-depth solves, torch autograd) with the trilinear sampler of its
    notebooks installed -- the only form in which the reference has pose gradients.  Returns (loss, kind)."""
    from oracle import port
    from oracle import reference_loader as RL
    s = src.clone().requires_grad_(True)
    d = dirs.clone().requires_grad_(True)
    ref = RL.load()
    if ref is not None:
        ren = ref.renderer.UltrasoundRenderer(CPU_SAMPLES, ALPHA)
        with RL.trilinear_sampler_installed(ref), RL.quiet():
            _, _, _, f = ren.plot_beam_frame(volume=vol, source=s, directions=d, plot=False, artifacts=False, start=0)
        kind = "reference"
    else:
        _, _, _, f = port.plot_beam_frame(vol, s, d, CPU_SAMPLES, ALPHA, sampler="trilinear", propagation="dense")
        kind = "port"
    loss = torch.nn.functional.mse_loss(f, target)
    loss.backward()
    return float(loss.detach()), kind


def sample_text(kind, dt):
    how = ("the UNMODIFIED reference (UltrasoundRenderer.plot_beam_frame: dense per-depth solves, its notebooks' trilinear sampler, "
           "torch autograd)" if kind == "reference" else "the oracle's literal port of the reference's dense per-depth solves + torch autograd")
    return (f"all {N_RAYS} rays of one pose of the workload truncated to the first {CPU_SAMPLES} of {N_SAMPLES} samples, forward + MSE + "
            f"backward to the pose, by {how}: {dt:.1f} s; the full depth does not run (about 190 GB of autograd state), so "
            f"frames/s = 1 / (time x {CPU_DEPTH_FACTOR:.1f}), the factor being the reference's own measured forward-time ratio between "
            f"{CPU_SAMPLES} and {N_SAMPLES} samples (its flop count, S^4, would give x256)")


def cpu_record(dt, kind):
    return {"value": 1.0 / (dt * CPU_DEPTH_FACTOR), "unit": UNIT, "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(),
            "kind": kind, "sample": sample_text(kind, dt), "sample_seconds": dt,
            "extrapolation": {"from_samples": CPU_SAMPLES, "to_samples": N_SAMPLES, "factor": CPU_DEPTH_FACTOR}}


def cpu_baseline(_unused=None):
    vol, s, d, target = cpu_scene()
    t = time.perf_counter()
    _, kind = cpu_sample_step(vol, s, d, target)
    return cpu_record(time.perf_counter() - t, kind)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if os.environ.get("OMP_NUM_THREADS") and not os.environ.get("DIFFUS_REF_CHILD"):
        # torchrun pins OMP_NUM_THREADS=1; the reference arm is entitled to every host thread, and
        # torch.set_num_threads() after start-up makes the batched LAPACK solves crawl, so re-exec clean
        env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS")}
        env["DIFFUS_REF_CHILD"] = "1"
        out = subprocess.run([sys.executable, os.path.abspath(__file__), *sys.argv[1:]], env=env, capture_output=True, text=True)
        sys.stdout.write(out.stdout)
        sys.stderr.write(out.stderr[-2000:])
        sys.stdout.flush()
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    K, W = args.steps, args.warmup
    vol, s, d, target = cpu_scene()
    kind = "reference"
    for _ in range(min(W, 1)):
        _, kind = cpu_sample_step(vol, s, d, target)
    # every step is a bounded sample; the whole arm is bounded too (the GPU arm's default K is sized for a
    # 1 ms step, the CPU sample takes seconds): stop after K steps or ~100 s, whichever comes first
    t = time.perf_counter()
    done = 0
    while done < K and (done == 0 or time.perf_counter() - t < 100.0):
        _, kind = cpu_sample_step(vol, s, d, target)
        done += 1
    dt = (time.perf_counter() - t) / done
    rec = cpu_record(dt, kind)
    line = {
        "impl": "reference", "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world,
        "steps": done, "steps_requested": K, "warmup": min(W, 1), "ms_per_step": dt * CPU_DEPTH_FACTOR * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(args.poses, world, args.layout),
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_cpu_config1 and kind == "reference":
        # BASELINE config 1 exactly as the reference runs it: ONE full 128 x 512 frame, nearest sampler, forward only (measured, no factor)
        from diffus_b200.phantoms import config1_pose, layered_phantom
        from oracle import reference_loader as RL
        ref = RL.load()
        v1 = layered_phantom(VOL_N, seed=0)
        s1, d1 = config1_pose(VOL_N, N_RAYS)
        t = time.perf_counter()
        with RL.quiet(), torch.no_grad():
            ref.renderer.UltrasoundRenderer(N_SAMPLES, ALPHA).plot_beam_frame(volume=v1, source=s1, directions=d1, plot=False, artifacts=False)
        t1 = time.perf_counter() - t
        line["config1_forward"] = {"what": "BASELINE config 1 by the unmodified reference: one full 128 x 512 frame, nearest sampler, forward "
                                           "only, measured (no extrapolation)", "s_per_frame": t1, "frames_per_s": 1.0 / t1}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--poses", type=int, default=1024, help="poses per GPU per step")
    ap.add_argument("--layout", default="texture", choices=["linear", "brick", "quad", "texture"])
    ap.add_argument("--cpu-rays", type=int, default=128, help="(kept for compatibility; the CPU sample is all 128 rays at 128 samples)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip the strong / config4 / nccl_parity / config5 records")
    ap.add_argument("--config5-poses", type=int, default=1024, help="poses of the 512^3 stress record (N = 1 only; 0 = skip)")
    ap.add_argument("--no-cpu-config1", action="store_true", help="reference arm: skip the full config-1 frame (~75 s on 8 cores)")
    ap.add_argument("--e2e", default="fan", choices=["fan", "graph", "eager"], help="public API used by the end-to-end loop")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and pose gradients of the last timed step (all ranks', in rank order) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
