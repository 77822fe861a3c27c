#!/usr/bin/env python
"""Secondary measurements for the BASELINE.json configs the headline bench does not cover (1 GPU).

    python benchmarks/run_configs.py [--configs 1,2,3f,4,5] [--iters 20]

Prints one JSON line per config: CUDA-event time per call, Gsamples/s, frames/s and the fraction of the
measured HBM copy peak at SURVEY 8(d)'s algorithmic bytes per sample.  The driver's contract lives in
bench.py; this script only feeds the tables in DESIGN.md.
"""
import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1,2,3f,4,5")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--layout", default="auto", choices=["auto", "brick", "quad", "texture"], help="packed layout of the pose-sweep volumes")
    args = ap.parse_args()
    from diffus_b200 import ImpedanceEstimator, PreparedVolume, UltrasoundRenderer, render_frames, render_mse_loss
    from diffus_b200.phantoms import config1_pose, intensity_to_impedance, layered_phantom, mri_phantom, pose_sweep
    from diffus_b200.training import TrainingVolume, mlp_render_mse_loss
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    import torch.distributed as dist
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:                          # torchrun: only config 4 has a collective (the weight-gradient all-reduce)
        dist.init_process_group("nccl", device_id=dev)
    want = args.configs.split(",")

    def report(name, ms, samples, frames, bytes_per_sample, extra=None):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, samples, frames = t.item(), samples * world, frames * world
            name = f"[{world} GPUs, poses sharded, max over ranks] " + name
            if rank != 0:
                return
        gs = samples / (ms * 1e-3) / 1e9
        line = {"config": name, "ms": ms, "gsamples_per_s": gs, "frames_per_s": frames / (ms * 1e-3),
                "bytes_per_sample": bytes_per_sample, "hbm_frac": gs * bytes_per_sample / peak}
        line.update(extra or {})
        print(json.dumps(line), flush=True)

    if "1" in want or "2" in want:
        vol = layered_phantom(256, 0).to(dev)
        src, dirs = config1_pose(256, 128)
        src, dirs = src.to(dev), dirs.to(dev)
        ren = UltrasoundRenderer(512, 1e-4)
        if "1" in want:
            ms = timed(lambda: ren.plot_beam_frame(vol, src, dirs, plot=False, return_indices=False), args.iters)
            report("1: single frame 128x512 forward, nearest, plot_beam_frame (host call included)", ms, 65536, 1, 8)
            ms = timed(lambda: ren.plot_beam_frame(vol, src, dirs, plot=False), args.iters)
            report("1: same with the x,y,z int64 index outputs", ms, 65536, 1, 32)
        if "2" in want:
            with torch.no_grad():
                tgt = render_frames(vol, (src + torch.tensor([1.5, 0.0, -1.0], device=dev)).reshape(1, 3), dirs, 512, 1e-4,
                                    sampler="trilinear")

            def step():
                s = src.clone().requires_grad_(True)
                d = dirs.clone().requires_grad_(True)
                render_mse_loss(vol, s.reshape(1, 3), d, tgt, 512, 1e-4).backward()
                return s.grad, d.grad
            ms = timed(step, args.iters)
            report("2: single frame fwd+bwd (pose-recovery step), fused kernel through autograd", ms, 65536, 1, 36)
            from diffus_b200 import ops
            s1, d1 = src.reshape(1, 3).contiguous(), dirs.contiguous()
            ms = timed(lambda: ops.render_mse_impl(vol, None, [256, 256, 256], s1, d1, tgt, 512, 0, 1e-4, 1, False, False,
                                                   True, False), args.iters)
            report("2: same, raw op call (no autograd bookkeeping)", ms, 65536, 1, 36)
            from diffus_b200.graphs import GraphedPoseStep
            gstep = GraphedPoseStep(vol, tgt, 128, 512, 1e-4)
            ms = timed(lambda: gstep(s1, d1), args.iters)
            report("2: same as a GraphedPoseStep (CUDA graph replay incl. copying the new pose in)", ms, 65536, 1, 36)
    if "3f" in want:
        vol = PreparedVolume(intensity_to_impedance(mri_phantom(256, "t1")).to(dev), args.layout)
        s, d = pose_sweep(1024, 128, 256, seed=1)
        s, d = s.to(dev), d.to(dev)
        for sampler, b in (("trilinear", 36), ("nearest", 8)):
            with torch.no_grad():
                ms = timed(lambda: render_frames(vol, s, d, 512, 1e-4, sampler=sampler), args.iters)
            report(f"3: pose sweep forward only, 1024 poses, {sampler}, {vol.layout} layout", ms, 1024 * 65536, 1024, b)
    if "4" in want:
        torch.manual_seed(0)
        model = ImpedanceEstimator(1).to(dev)
        with torch.no_grad():
            model.model[4].bias.fill_(1.5)
            model.model[4].weight.mul_(0.3)
        mri = (mri_phantom(256, "t2") / 1000.0).to(dev)
        P = 4096
        s, d = pose_sweep(P, 128, 256, seed=2 + rank)
        s, d = s.to(dev), d.to(dev)
        from diffus_b200 import distributed as D
        with torch.no_grad():
            tgt = render_frames(PreparedVolume(model.impedance_volume(mri, None, 1e6, 400.0) * 1.01), s, d, 512, 1e-4,
                                sampler="trilinear")

        tv = TrainingVolume(mri)

        def step(sampler="trilinear"):
            model.zero_grad(set_to_none=True)
            mlp_render_mse_loss(model, tv, s, d, tgt, 512, 1e-4, out_scale=1e6, sampler=sampler).backward()
            D.allreduce_module_grads(model, average=True)          # one 4.6 KB flat all-reduce (no-op on 1 GPU)
        ms_near = timed(lambda: step("nearest"), max(3, args.iters // 4))
        report("4: MLP(256^3) -> 4096 frames -> MSE -> d/dweights, NEAREST sampler (the reference's own training form)",
               ms_near, P * 65536, P, 12)
        ms = timed(step, max(3, args.iters // 4))
        from diffus_b200 import ops
        from diffus_b200.impedance import pack_params
        pk = pack_params(model).detach()
        gz = torch.randn(mri.numel(), device=dev)
        paths = (("cuda cores", ops.MLP_PATH_CUDA_CORES), ("piecewise-linear table", ops.MLP_PATH_PIECEWISE))
        for name, path in paths:
            with ops.mlp_path(path):
                t_ms = timed(lambda: ops.mlp_fwd_impl(pk, mri.reshape(-1), None, 1e6, 400.0), args.iters)
                b_ms = timed(lambda: ops.mlp_bwd_impl(pk, mri.reshape(-1), None, gz, 1e6), max(3, args.iters // 4))
            print(json.dumps({"config": f"4: MLP forward over 256^3 voxels, {name}", "ms": t_ms,
                              "gvoxels_per_s": mri.numel() / (t_ms * 1e-3) / 1e9,
                              "tflops_layer2": mri.numel() * 2048 / (t_ms * 1e-3) / 1e12,
                              "hbm_gb_per_s": mri.numel() * 8 / (t_ms * 1e-3) / 1e9}), flush=True)
            print(json.dumps({"config": f"4: MLP weight gradient over 256^3 voxels (dense d loss / d Z), {name}", "ms": b_ms,
                              "gvoxels_per_s": mri.numel() / (b_ms * 1e-3) / 1e9,
                              "tflops_layer2": mri.numel() * 6144 / (b_ms * 1e-3) / 1e12,
                              "hbm_gb_per_s": mri.numel() * 8 / (b_ms * 1e-3) / 1e9}), flush=True)
        bwd_ms = timed(lambda: ops.mlp_bwd_impl(pk, mri.reshape(-1), None, gz, 1e6), max(3, args.iters // 4))
        fwd_ms = timed(lambda: ops.mlp_fwd_impl(pk, mri.reshape(-1), None, 1e6, 400.0), args.iters)
        report("4: MLP(256^3) -> 4096 frames -> MSE -> d/dweights (one training step, 1 GPU)", ms, P * 65536, P, 68,
               {"mlp_fwd_ms": fwd_ms, "mlp_bwd_dense_ms": bwd_ms})
    if "5" in want:
        vol = PreparedVolume(layered_phantom(512, 0).to(dev))
        P = 64
        s, d = pose_sweep(P, 512, 512, seed=3)
        s, d = s.to(dev), d.to(dev)
        with torch.no_grad():
            tgt = render_frames(vol, s + 1.0, d, 2048, 1e-4, sampler="trilinear")

        def step():
            ss = s.clone().requires_grad_(True)
            dd = d.clone().requires_grad_(True)
            render_mse_loss(vol, ss, dd, tgt, 2048, 1e-4).backward()
        ms = timed(step, max(3, args.iters // 4))
        report(f"5: 512^3 volume, 512 rays x 2048 samples, {P} poses fwd+bwd (per-pose time x 4096 = full config)", ms,
               P * 512 * 2048, P, 36, {"ms_for_4096_poses": ms * 4096 / P})


if __name__ == "__main__":
    main()
    import torch.distributed as _d
    if _d.is_initialized():
        _d.destroy_process_group()
