"""Array probes on the B200, on the bench's workload (1024 poses x 128 rays x 512 samples, 256^3 MRI-shaped volume, TEXTURE
layout): the fused MSE step and the Gauss-Newton system with a sector probe, a convex probe (radius 20 voxels) and a linear probe
(width 60 voxels), alternated in one process and timed with CUDA events, and the probe-ray kernels' own time.  Optionally
(--lm) Levenberg-Marquardt from perturbed linear-probe poses on the smooth test scene and on the bench's scene, with the
protocol of profiles/r3_gauss_newton.md (1 voxel + 1 degree, targets rendered at the true poses).  Prints the card's name and
power limit with the numbers; writes one JSON record with --out.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks", "experiments"))

import torch  # noqa: E402

from gauss_newton_step import ALPHA, ANGLE, N_RAYS, N_SAMPLES, card, scene  # noqa: E402

PROBES = {"sector": {}, "convex": dict(radius=20.0), "linear": dict(width=60.0)}


def rays(probe, s, m, h):
    from diffus_b200 import fan_directions, probe_rays
    if probe == "sector":
        return s, fan_directions(m, h, ANGLE, N_RAYS)
    return probe_rays(probe, s, m, h, N_RAYS, opening_angle=ANGLE, **PROBES[probe])


def timed(fns, reps, per):
    times = {k: [] for k in fns}
    for _ in range(3):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(per):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / per)
    return {k: {"median_ms": sorted(v)[len(v) // 2], "min_ms": min(v)} for k, v in times.items()}


def step_costs(P, reps, per, dev):
    from diffus_b200 import ops, render_frames
    from diffus_b200._lib import SAMPLER_TRILINEAR
    vol, s, _, m, h = scene(P, 1000, dev)
    vt, bricks, dims = vol.volume, vol.bricks, list(vol.volume.shape)
    fused, gn, gen = {}, {}, {}
    for probe in PROBES:
        src, dirs = (t.detach().contiguous() for t in rays(probe, s, m, h))
        with torch.no_grad():
            tgt = render_frames(vol, *rays(probe, s + torch.tensor([1.5, 0.0, -1.0], device=dev), m, h), N_SAMPLES, ALPHA,
                                sampler="trilinear")
        outs = dict(loss_out=torch.empty(P, device=dev), jtj_out=torch.empty((P, 6, 6), device=dev),
                    jtr_out=torch.empty((P, 6), device=dev))
        fused[probe] = (lambda src=src, dirs=dirs, tgt=tgt: ops.render_mse_impl(
            vt, bricks, dims, src, dirs, tgt, N_SAMPLES, 0, ALPHA, SAMPLER_TRILINEAR, False, False, True, False))
        gn[probe] = (lambda src=src, dirs=dirs, tgt=tgt, outs=outs: ops.render_gauss_newton_impl(
            vt, bricks, dims, src, dirs, tgt, N_SAMPLES, 0, ALPHA, **outs))
        if probe != "sector":
            kid, angle, rho, w = ops.probe_args(probe, ANGLE, PROBES[probe].get("radius", 0.0), PROBES[probe].get("width"))
            g = torch.randn((P, N_RAYS, 3), device=dev)
            gen[probe + "_rays"] = (lambda kid=kid, angle=angle, rho=rho, w=w: ops.probe_rays_fwd(kid, s, m, h, N_RAYS, angle, rho, w))
            gen[probe + "_rays_backward"] = (lambda kid=kid, angle=angle, rho=rho, w=w, g=g: ops.probe_rays_bwd(
                kid, s, m, h, g, g, N_RAYS, angle, rho, w))
        else:
            gen["sector_fan_directions"] = lambda: ops.fan_directions_fwd(m, h, ANGLE, N_RAYS)
    return {"fused_mse_step": timed(fused, reps, per), "gauss_newton_system": timed(gn, reps, per),
            "ray_generation": timed(gen, reps, per * 10)}


def lm_linear(vol, P, n, iters, dev, seed=8):
    from diffus_b200 import recover_poses, render_frames
    from diffus_b200.phantoms import pose_sweep
    from diffus_b200.pose_recovery import apply_fan_twist, fan_frame_angle
    src, _, med, hint = pose_sweep(P, n_rays=N_RAYS, n=n, seed=seed, return_params=True)
    src, med, hint = src.to(dev), med.to(dev), hint.to(dev)
    with torch.no_grad():
        targets = render_frames(vol, *rays("linear", src, med, hint), N_SAMPLES, ALPHA, sampler="trilinear")
    g = torch.Generator().manual_seed(0)
    u = torch.randn((P, 6), generator=g)
    u[:, :3] = u[:, :3] / u[:, :3].norm(dim=-1, keepdim=True)
    u[:, 3:] = u[:, 3:] / u[:, 3:].norm(dim=-1, keepdim=True) * math.radians(1.0)
    s0, m0, h0 = apply_fan_twist(src, med, hint, u.to(dev))
    (s1, m1, h1), hist = recover_poses(vol, targets, s0, m0, h0, ANGLE, N_RAYS, N_SAMPLES, ALPHA, iterations=iters, probe="linear",
                                       width=PROBES["linear"]["width"])
    pos = (s1 - src).norm(dim=-1).cpu()
    ang = torch.rad2deg(fan_frame_angle(m1, h1, med, hint)).cpu()
    q = lambda t, p: float(t.quantile(p))
    return {"poses": P, "iterations": iters, "loss_median_start": float(hist[0].median()), "loss_median_end": float(hist[-1].median()),
            "position_err_voxel": {"median": q(pos, 0.5), "p95": q(pos, 0.95), "max": float(pos.max())},
            "angle_err_deg": {"median": q(ang, 0.5), "p95": q(ang, 0.95), "max": float(ang.max())}}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--poses", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--per", type=int, default=20)
    ap.add_argument("--lm", action="store_true")
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    rec = {"card": card(), "workload": f"{args.poses} poses x {N_RAYS} rays x {N_SAMPLES} samples, 256^3 TEXTURE",
           "probes": PROBES, "costs": step_costs(args.poses, args.reps, args.per, dev)}
    if args.lm:
        from diffus_b200 import PreparedVolume
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from test_gpu_array_probes import _smooth_phantom
        rec["lm_linear_smooth_scene"] = lm_linear(PreparedVolume(_smooth_phantom(64).to(dev), "texture"), 32, 64, 10, dev)
        vol, _, _, _, _ = scene(1, 0, dev)
        rec["lm_linear_bench_scene"] = lm_linear(vol, 256, 256, 20, dev, seed=1000)
    print(json.dumps(rec, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
