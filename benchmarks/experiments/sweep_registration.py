"""Tracked-sweep registration on the B200: (a) the cost of ONE sweep system (``render_gauss_newton_sweep``) against the per-pose
systems (``render_gauss_newton``), alternated in one process, for 256 and 1024 poses x 128 rays x 512 samples on the 256^3
MRI-shaped volume (TEXTURE layout); (b) convergence of ``register_sweep`` against per-pose ``recover_poses`` from the same starts:
gauss_newton_step.py's scene (256 poses of bench's sweep, seed 2000, targets at the true poses), all poses moved by ONE shared
twist of 1, 2 and 4 voxels and degrees about the origin centroid.  Prints the card name and power limit with the numbers; writes
one JSON record with --out.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import math
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

import torch  # noqa: E402

import gauss_newton_step as gns  # noqa: E402


def cost(P, reps, per, dev):
    """Median ms per call of the per-pose systems and of the sweep system, in alternating blocks of `per` calls."""
    from diffus_b200 import ops, render_frames
    vol, src, dirs, _, _ = gns.scene(P, 1000, dev)
    with torch.no_grad():
        target = render_frames(vol, src + torch.tensor([1.5, 0.0, -1.0], device=dev), dirs, gns.N_SAMPLES, gns.ALPHA,
                               sampler="trilinear")
    bricks, vt = vol.bricks, vol.volume
    dims = list(vt.shape)
    per_pose = dict(loss_out=torch.empty(P, device=dev), jtj_out=torch.empty((P, 6, 6), device=dev),
                    jtr_out=torch.empty((P, 6), device=dev))
    f64 = dict(dtype=torch.float64, device=dev)
    sweep = dict(loss_out=torch.empty((), **f64), jtj_out=torch.empty((6, 6), **f64), jtr_out=torch.empty((6,), **f64))
    pivot = src.double().mean(0)

    def gn():
        ops.render_gauss_newton_impl(vt, bricks, dims, src, dirs, target, gns.N_SAMPLES, 0, gns.ALPHA, **per_pose)

    def gn_sweep():
        ops.render_gauss_newton_sweep_impl(vt, bricks, dims, src, dirs, target, gns.N_SAMPLES, 0, gns.ALPHA, pivot, **sweep)

    fns = {"per_pose_systems": gn, "sweep_system": gn_sweep}
    for _ in range(3):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(per):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / per)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    row = {"poses": P, "ms_median": med, "ms_min": {k: min(v) for k, v in times.items()},
           "ratio_sweep_over_per_pose": med["sweep_system"] / med["per_pose_systems"]}
    print(json.dumps(row), flush=True)
    return row


def rotation_angle_deg(r):
    return math.degrees(math.acos(max(-1.0, min(1.0, (float(r.trace()) - 1.0) / 2.0))))


def convergence(P, dev, perturbations, iterations):
    from diffus_b200 import fan_directions, recover_poses, register_sweep, render_frames
    from diffus_b200.pose_recovery import apply_rigid_transform, compose_sweep_twist
    vol, src, _, med, hint = gns.scene(P, 2000, dev)
    with torch.no_grad():
        targets = render_frames(vol, src, fan_directions(med, hint, gns.ANGLE, gns.N_RAYS), gns.N_SAMPLES, gns.ALPHA,
                                sampler="trilinear")
    centroid = src.double().mean(0)
    eye, zero = torch.eye(3, dtype=torch.float64, device=dev), torch.zeros(3, dtype=torch.float64, device=dev)
    rows = []
    for vox, deg in perturbations:
        g = torch.Generator().manual_seed(int(100 * vox + deg))
        u = torch.randn(6, generator=g, dtype=torch.float64)
        u[:3] *= vox / u[:3].norm()
        u[3:] *= math.radians(deg) / u[3:].norm()
        r0, t0 = compose_sweep_twist(eye, zero, u.to(dev), centroid)
        start = tuple(x.float() for x in apply_rigid_transform(r0, t0, src, med, hint))
        row = {"perturbation": {"voxels": vox, "degrees": deg}}
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        (rot, trans), poses, hist = register_sweep(vol, targets, *start, gns.ANGLE, gns.N_RAYS, gns.N_SAMPLES, gns.ALPHA,
                                                   iterations=iterations)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - h0) * 1e3
        # the registered sweep as a transform of the TRUE sweep: (rot r0, rot t0 + trans)
        r_err = rot @ r0
        t_err = rot @ t0 + trans
        pos, ang = gns.pose_errors(*poses, src, med, hint)
        row["register_sweep"] = {
            "transform_rotation_error_deg": rotation_angle_deg(r_err.cpu()),
            "transform_translation_error_at_centroid_voxel": float((r_err @ centroid + t_err - centroid).norm()),
            "p95_position_error_voxel": float(torch.quantile(pos, 0.95)), "p95_angle_error_deg": float(torch.quantile(ang, 0.95)),
            "max_position_error_voxel": float(pos.max()), "max_angle_error_deg": float(ang.max()),
            "loss_first_last": [float(hist[0]), float(hist[-1])], "wall_ms": wall}
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        poses, phist = recover_poses(vol, targets, *start, gns.ANGLE, gns.N_RAYS, gns.N_SAMPLES, gns.ALPHA, iterations=iterations)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - h0) * 1e3
        pos, ang = gns.pose_errors(*poses, src, med, hint)
        row["recover_poses"] = {
            "p95_position_error_voxel": float(torch.quantile(pos, 0.95)), "p95_angle_error_deg": float(torch.quantile(ang, 0.95)),
            "max_position_error_voxel": float(pos.max()), "max_angle_error_deg": float(ang.max()),
            "loss_sum_first_last": [float(phist[0].double().sum()), float(phist[-1].double().sum())], "wall_ms": wall}
        print(json.dumps(row), flush=True)
        rows.append(row)
    return {"poses": P, "iterations": iterations, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cost-poses", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--per", type=int, default=10)
    ap.add_argument("--conv-poses", type=int, default=256)
    ap.add_argument("--iterations", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    rec = {"card": gns.card()}
    print(rec["card"], flush=True)
    rec["cost"] = [cost(P, args.reps, args.per, dev) for P in args.cost_poses]
    rec["convergence"] = convergence(args.conv_poses, dev, [(1.0, 1.0), (2.0, 2.0), (4.0, 4.0)], args.iterations)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
