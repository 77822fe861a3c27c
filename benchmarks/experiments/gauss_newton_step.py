"""Gauss-Newton pose recovery on the B200: (a) the cost of one Gauss-Newton system against the fused MSE pose step, alternated in
one process, on the bench's workload (1024 poses x 128 rays x 512 samples, 256^3 MRI-shaped volume, TEXTURE layout); (b) how many
Levenberg-Marquardt iterations and how many Adam steps through GraphedFanPoseStep reach the same pose error from the same
perturbed start poses (targets rendered at the true poses).  Prints the card name and power limit with the numbers; writes one
JSON record with --out.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_RAYS, N_SAMPLES, VOL_N, ALPHA = 128, 512, 256, 1e-4      # bench.py's workload
ANGLE = math.radians(60.0)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # the numbers still stand with the card's name
        q = f"unavailable ({e})"
    return f"{name}, power limit / max SM clock: {q}"


def scene(P, seed, dev, layout="texture"):
    from diffus_b200 import PreparedVolume
    from diffus_b200.phantoms import intensity_to_impedance, mri_phantom, pose_sweep
    vol = PreparedVolume(intensity_to_impedance(mri_phantom(VOL_N, "t1", seed=0)).to(dev), layout)
    s, d, m, h = pose_sweep(P, N_RAYS, VOL_N, seed=seed, return_params=True)
    return vol, s.to(dev), d.to(dev), m.to(dev), h.to(dev)


def cost_of_one_system(P, reps, per, dev):
    """Median time per call of the fused MSE step and of the Gauss-Newton system, in alternating blocks of `per` calls."""
    from diffus_b200 import ops, render_frames
    from diffus_b200._lib import SAMPLER_TRILINEAR
    vol, src, dirs, _, _ = scene(P, 1000, dev)
    with torch.no_grad():
        target = render_frames(vol, src + torch.tensor([1.5, 0.0, -1.0], device=dev), dirs, N_SAMPLES, ALPHA, sampler="trilinear")
    bricks, vt = vol.bricks, vol.volume
    dims = list(vt.shape)
    outs = dict(loss_out=torch.empty(P, device=dev), jtj_out=torch.empty((P, 6, 6), device=dev), jtr_out=torch.empty((P, 6), device=dev))

    def fused():
        ops.render_mse_impl(vt, bricks, dims, src, dirs, target, N_SAMPLES, 0, ALPHA, SAMPLER_TRILINEAR, False, False, True, False)

    def gn():
        ops.render_gauss_newton_impl(vt, bricks, dims, src, dirs, target, N_SAMPLES, 0, ALPHA, **outs)
    times = {"fused_mse_step": [], "gauss_newton_system": []}
    for _ in range(3):                          # warm-up of both shapes
        fused(), gn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, fn in (("fused_mse_step", fused), ("gauss_newton_system", gn)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(per):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / per)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"poses": P, "ms_median": med, "ms_min": {k: min(v) for k, v in times.items()},
            "ratio_gn_over_fused": med["gauss_newton_system"] / med["fused_mse_step"]}


def pose_errors(s, m, h, s_true, m_true, h_true):
    from diffus_b200.pose_recovery import fan_frame_angle
    return (s - s_true).norm(dim=-1), torch.rad2deg(fan_frame_angle(m, h, m_true, h_true)).float()


def reached(pos, ang, tol_pos, tol_ang):
    """First row (iteration) at which 95 % of the poses are within both tolerances, or None."""
    q_pos = torch.quantile(pos, 0.95, dim=1)
    q_ang = torch.quantile(ang, 0.95, dim=1)
    ok = ((q_pos <= tol_pos) & (q_ang <= tol_ang)).nonzero()
    return int(ok[0]) if len(ok) else None


def convergence(P, dev, perturbations, lm_iters, adam_steps, lrs, tol_pos, tol_ang):
    from diffus_b200 import fan_directions, render_frames
    from diffus_b200.graphs import GraphedFanGaussNewtonStep, GraphedFanPoseStep
    from diffus_b200.pose_recovery import apply_fan_twist
    vol, src, _, med, hint = scene(P, 2000, dev)
    with torch.no_grad():
        targets = render_frames(vol, src, fan_directions(med, hint, ANGLE, N_RAYS), N_SAMPLES, ALPHA, sampler="trilinear")
    lm = GraphedFanGaussNewtonStep(vol, targets, N_RAYS, N_SAMPLES, ANGLE, ALPHA)
    adam = GraphedFanPoseStep(vol, targets, N_RAYS, N_SAMPLES, ANGLE, ALPHA)
    rows = []
    for vox, deg in perturbations:
        g = torch.Generator().manual_seed(int(100 * vox + deg))
        u = torch.randn((P, 6), generator=g)
        u[:, :3] *= vox / u[:, :3].norm(dim=-1, keepdim=True)
        u[:, 3:] *= math.radians(deg) / u[:, 3:].norm(dim=-1, keepdim=True)
        s0, m0, h0 = apply_fan_twist(src, med, hint, u.to(dev))
        row = {"perturbation": {"voxels": vox, "degrees": deg}}
        # LM: errors recorded on the device after every iteration; the time per iteration from a second, unobserved run
        lm.reset(s0, m0, h0)
        errs = [pose_errors(lm.sources, lm.median, lm.hint, src, med, hint)]
        for _ in range(lm_iters):
            lm()
            errs.append(pose_errors(lm.sources, lm.median, lm.hint, src, med, hint))
        pos, ang = torch.stack([e[0] for e in errs]).cpu(), torch.stack([e[1] for e in errs]).cpu()
        lm.reset(s0, m0, h0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(lm_iters):
            lm()
        b.record()
        b.synchronize()
        ms_it = a.elapsed_time(b) / lm_iters
        k = reached(pos, ang, tol_pos, tol_ang)
        row["lm"] = {"ms_per_iteration": ms_it, "iterations_to_tolerance": k, "ms_to_tolerance": None if k is None else k * ms_it,
                     "p95_position_error_voxel": [float(x) for x in torch.quantile(pos, 0.95, dim=1)],
                     "p95_angle_error_deg": [float(x) for x in torch.quantile(ang, 0.95, dim=1)]}
        best = None
        for lr_s, lr_a in lrs:
            s, m, h = (t.clone().requires_grad_(True) for t in (s0, m0, h0))
            opt = torch.optim.Adam([{"params": [s], "lr": lr_s}, {"params": [m, h], "lr": lr_a}])
            errs = [pose_errors(s.detach(), m.detach(), h.detach(), src, med, hint)]
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(adam_steps):
                _, gs, gm, gh = adam(s.detach(), m.detach(), h.detach())
                s.grad, m.grad, h.grad = gs.clone(), gm.clone(), gh.clone()
                opt.step()
                errs.append(pose_errors(s.detach(), m.detach(), h.detach(), src, med, hint))
            b.record()
            b.synchronize()
            ms_step = a.elapsed_time(b) / adam_steps          # (includes the on-device error bookkeeping: an upper bound)
            pos, ang = torch.stack([e[0] for e in errs]).cpu(), torch.stack([e[1] for e in errs]).cpu()
            k = reached(pos, ang, tol_pos, tol_ang)
            rec = {"lr_source": lr_s, "lr_direction": lr_a, "ms_per_step": ms_step, "steps_to_tolerance": k,
                   "ms_to_tolerance": None if k is None else k * ms_step,
                   "final_p95_position_error_voxel": float(torch.quantile(pos[-1], 0.95)),
                   "final_p95_angle_error_deg": float(torch.quantile(ang[-1], 0.95))}
            if best is None or (k is not None and (best["steps_to_tolerance"] is None or k < best["steps_to_tolerance"])):
                best = rec
        row["adam_best_lr"] = best
        rows.append(row)
        print(json.dumps(row), flush=True)
    return {"poses": P, "tolerance": {"p95_position_voxel": tol_pos, "p95_angle_deg": tol_ang}, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--poses", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--per", type=int, default=20)
    ap.add_argument("--conv-poses", type=int, default=256)
    ap.add_argument("--lm-iters", type=int, default=15)
    ap.add_argument("--adam-steps", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    rec = {"card": card()}
    print(rec["card"], flush=True)
    rec["cost"] = cost_of_one_system(args.poses, args.reps, args.per, dev)
    print(json.dumps(rec["cost"]), flush=True)
    rec["convergence"] = convergence(args.conv_poses, dev, [(1.0, 1.0), (2.0, 2.0), (4.0, 4.0)], args.lm_iters, args.adam_steps,
                                     [(0.05, 1e-3), (0.1, 2e-3), (0.2, 4e-3)], 0.05, 0.05)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
