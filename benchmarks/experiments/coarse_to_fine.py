"""Coarse-to-fine pose recovery on the B200: (a) the cost of the 3-D Gaussian blur (``smooth_volume``) at 256^3 and 512^3
against the same three separable passes in torch (``F.pad(mode='replicate')`` + ``F.conv3d`` with 1-D kernels); (b) convergence
of Levenberg-Marquardt from blurred to sharp volumes against single-level LM on gauss_newton_step.py's bench scene and
perturbation protocol.  Prints the card name and power limit with the numbers; writes one JSON record with --out.  Needs a CUDA
device (no CPU fallback)."""
import argparse
import json
import math
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import gauss_newton_step as gns  # noqa: E402

HBM_TBPS = 7.7        # HGX B200 data sheet, one GPU


def torch_blur(v, w, r):
    """The same filter in torch: replicate-pad one axis, correlate with the 1-D kernel along it; p2, then p1, then p0."""
    x = v[None, None]
    x = F.conv3d(F.pad(x, (r, r, 0, 0, 0, 0), mode="replicate"), w.view(1, 1, 1, 1, -1))
    x = F.conv3d(F.pad(x, (0, 0, r, r, 0, 0), mode="replicate"), w.view(1, 1, 1, -1, 1))
    x = F.conv3d(F.pad(x, (0, 0, 0, 0, r, r), mode="replicate"), w.view(1, 1, -1, 1, 1))
    return x[0, 0]


def blur_cost(sizes, sigmas, reps, per, dev):
    """Median ms per call of smooth_volume and of torch_blur, alternating blocks of `per` calls after a warm-up of both."""
    from diffus_b200 import smooth_volume
    from oracle import smoothing
    torch.backends.cudnn.allow_tf32 = False           # fp32 arithmetic in the baseline too
    rows = []
    for n in sizes:
        v = 1.48e6 + 2.2e5 * torch.rand((n, n, n), device=dev, generator=torch.Generator(device=dev).manual_seed(n))
        for sigma in sigmas:
            r = smoothing.gaussian_radius(sigma)
            w = torch.tensor(smoothing.gaussian_weights(sigma), dtype=torch.float32, device=dev)
            fns = {"smooth_volume": lambda: smooth_volume(v, sigma), "torch_conv3d": lambda: torch_blur(v, w, r)}
            for f in fns.values():
                f(), f()
            torch.cuda.synchronize()
            diff = float((fns["smooth_volume"]() - fns["torch_conv3d"]()).abs().max() / v.abs().max())
            times = {k: [] for k in fns}
            for _ in range(reps):
                for name, f in fns.items():
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(per):
                        f()
                    b.record()
                    b.synchronize()
                    times[name].append(a.elapsed_time(b) / per)
            med = {k: statistics.median(t) for k, t in times.items()}
            nbytes = 3 * 8 * n ** 3                   # three passes, each reads and writes 4 B per voxel
            row = {"n": n, "sigma": sigma, "radius": r, "ms_median": med, "ms_min": {k: min(t) for k, t in times.items()},
                   "gb_per_s": {k: nbytes / (ms * 1e-3) / 1e9 for k, ms in med.items()},
                   "share_of_hbm_peak": {k: nbytes / (ms * 1e-3) / (HBM_TBPS * 1e12) for k, ms in med.items()},
                   "max_abs_diff_over_max": diff}
            rows.append(row)
            print(json.dumps(row), flush=True)
        del v
        torch.cuda.empty_cache()
    return rows


def run_schedule(vol, targets, truth, start, sigmas, iters, tol, damping=1e-3):
    """recover_poses_coarse_to_fine's levels, driven one iteration at a time so that the pose error is observable after every
    iteration.  Device time of each blur and each LM iteration from CUDA events; the host-clock set-up of a level (packed copy,
    graph capture, the start poses' system) separately."""
    from diffus_b200 import PreparedVolume, smooth_volume
    from diffus_b200.graphs import GraphedFanGaussNewtonStep
    src, med, hint = truth
    poses = start
    base, layout = vol.volume, vol.layout
    levels, pos_all, ang_all, t_cum, blur_cum = [], [], [], [], []
    t = b_ms = 0.0
    for li, (sigma, k) in enumerate(zip(sigmas, iters)):
        blur_ms = 0.0
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        if sigma == 0.0:
            level = vol
        else:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            blurred = smooth_volume(base, sigma)
            b.record()
            b.synchronize()
            blur_ms = a.elapsed_time(b)
            level = PreparedVolume(blurred, layout)
        step = GraphedFanGaussNewtonStep(level, targets, gns.N_RAYS, gns.N_SAMPLES, gns.ANGLE, gns.ALPHA)
        step.reset(*poses, damping)
        torch.cuda.synchronize()
        setup_ms = (time.perf_counter() - h0) * 1e3 - blur_ms
        t += blur_ms
        b_ms += blur_ms
        it_ms = []
        for i in range(k + 1):
            if i:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step()
                b.record()
                b.synchronize()
                it_ms.append(a.elapsed_time(b))
                t += it_ms[-1]
            if i or li == 0:
                p, q = gns.pose_errors(step.sources, step.median, step.hint, src, med, hint)
                pos_all.append(p)
                ang_all.append(q)
                t_cum.append(t)
                blur_cum.append(b_ms)
        poses = (step.sources.clone(), step.median.clone(), step.hint.clone())
        levels.append({"sigma": sigma, "iterations": k, "blur_ms": blur_ms, "setup_ms_host": setup_ms,
                       "ms_per_iteration": statistics.mean(it_ms) if it_ms else None,
                       "p95_position_error_voxel": float(torch.quantile(pos_all[-1], 0.95)),
                       "p95_angle_error_deg": float(torch.quantile(ang_all[-1], 0.95))})
        del step
        if level is not vol:
            level.close()
    pos, ang = torch.stack(pos_all).cpu(), torch.stack(ang_all).cpu()
    kk = gns.reached(pos, ang, *tol)
    return poses, {"sigmas": list(sigmas), "iterations": list(iters), "levels": levels,
                   "iterations_to_tolerance": kk, "ms_to_tolerance": None if kk is None else t_cum[kk],
                   "blur_ms_inside": None if kk is None else blur_cum[kk],
                   "device_ms_total": t, "setup_ms_host_total": sum(lv["setup_ms_host"] for lv in levels),
                   "final_p95_position_error_voxel": float(torch.quantile(pos[-1], 0.95)),
                   "final_p95_angle_error_deg": float(torch.quantile(ang[-1], 0.95)),
                   "final_max_position_error_voxel": float(pos[-1].max()), "final_max_angle_error_deg": float(ang[-1].max())}


def convergence(P, dev, perturbations, schedules, tol):
    from diffus_b200 import fan_directions, recover_poses_coarse_to_fine, render_frames
    from diffus_b200.pose_recovery import apply_fan_twist
    vol, src, _, med, hint = gns.scene(P, 2000, dev)
    with torch.no_grad():
        targets = render_frames(vol, src, fan_directions(med, hint, gns.ANGLE, gns.N_RAYS), gns.N_SAMPLES, gns.ALPHA,
                                sampler="trilinear")
    rows = []
    for vox, deg in perturbations:
        g = torch.Generator().manual_seed(int(100 * vox + deg))        # gauss_newton_step.py's start poses
        u = torch.randn((P, 6), generator=g)
        u[:, :3] *= vox / u[:, :3].norm(dim=-1, keepdim=True)
        u[:, 3:] *= math.radians(deg) / u[:, 3:].norm(dim=-1, keepdim=True)
        start = apply_fan_twist(src, med, hint, u.to(dev))
        row = {"perturbation": {"voxels": vox, "degrees": deg}, "schedules": []}
        for sigmas, iters in schedules:
            poses, rec = run_schedule(vol, targets, (src, med, hint), start, sigmas, iters, tol)
            # the public function end to end (host clock, synchronised), and that it lands on the same poses
            torch.cuda.synchronize()
            h0 = time.perf_counter()
            got, _ = recover_poses_coarse_to_fine(vol, targets, *start, gns.ANGLE, gns.N_RAYS, gns.N_SAMPLES, gns.ALPHA,
                                                  sigmas=sigmas, iterations=list(iters))
            torch.cuda.synchronize()
            rec["public_function_wall_ms"] = (time.perf_counter() - h0) * 1e3
            rec["public_function_same_poses"] = all(torch.equal(x, y) for x, y in zip(got, poses))
            row["schedules"].append(rec)
            print(json.dumps({"perturbation": row["perturbation"], **rec}), flush=True)
        rows.append(row)
    return {"poses": P, "tolerance": {"p95_position_voxel": tol[0], "p95_angle_deg": tol[1]}, "rows": rows}


SCHEDULES = [((0.0,), (15,)), ((0.0,), (20,)), ((2.0, 1.0, 0.0), (5, 5, 5)), ((4.0, 2.0, 1.0, 0.0), (5, 5, 5, 5)),
             ((8.0, 4.0, 2.0, 1.0, 0.0), (4, 4, 4, 4, 4))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--sigmas", type=float, nargs="+", default=[1.0, 2.0, 4.0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--per", type=int, default=10)
    ap.add_argument("--conv-poses", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    rec = {"card": gns.card()}
    print(rec["card"], flush=True)
    rec["blur_cost"] = blur_cost(args.sizes, args.sigmas, args.reps, args.per, dev)
    rec["convergence"] = convergence(args.conv_poses, dev, [(1.0, 1.0), (2.0, 2.0), (4.0, 4.0)], SCHEDULES, (0.05, 0.05))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
