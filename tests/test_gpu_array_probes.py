"""GPU: one origin per ray (linear and convex array probes) through the render kernels, the fused step, Gauss-Newton, the
probe-ray kernels, the graphed steps and Levenberg-Marquardt -- against the per-pose path (bit for bit where the rays are the
same) and against the float64 oracle where they are not."""
import math

import numpy as np
import pytest
import torch

from conftest import assert_frame_close, assert_grad_close, oracle_grads

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _geometry(n, P, R, step, seed, spread=0.0):
    """Poses outside a corner aiming at the centre; ``spread`` > 0 moves every ray's origin by up to that many voxels."""
    g = torch.Generator().manual_seed(seed)
    src = torch.tensor([[3.0, 2.0, 4.0], [n * 0.5, n * 0.3, 1.5], [n - 3.5, n * 0.6, n - 4.0]])[:P]
    aim = torch.tensor([n * 0.5] * 3) - src
    d = aim[:, None, :] / aim.norm(dim=-1)[:, None, None] + 0.25 * torch.randn((P, R, 3), generator=g)
    dirs = (d / d.norm(dim=-1, keepdim=True) * step).contiguous()
    origins = (src[:, None, :] + spread * (2 * torch.rand((P, R, 3), generator=g) - 1)).contiguous()
    return src.contiguous(), origins, dirs


LAYOUTS = [None, "brick", "quad", "texture"]


def _vol(v, layout):
    from diffus_b200 import PreparedVolume
    return PreparedVolume(v, layout) if layout else v


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("start", [0, 9])
def test_broadcast_sources_render_bit_identical(layout, sampler, start):
    from diffus_b200 import render_frames
    from diffus_b200.phantoms import layered_phantom
    n, P, R, S = 40, 3, 8, 140
    v = layered_phantom(n, seed=2).to(dev())
    src, _, dirs = _geometry(n, P, R, 0.3, 1)
    src, dirs = src.to(dev()), dirs.to(dev())
    vv = _vol(v, layout)
    a = render_frames(vv, src, dirs, S, 1e-3, start, sampler=sampler)
    b = render_frames(vv, src[:, None, :].expand(-1, R, -1).contiguous(), dirs, S, 1e-3, start, sampler=sampler)
    assert torch.equal(a, b)


# one pass, WIDE (257..512), one CTA per ray (513..2048), multi-pass (> 2048)
@pytest.mark.parametrize("S,step", [(200, 0.2), (450, 0.08), (1100, 0.03), (2300, 0.015)])
@pytest.mark.parametrize("start", [0, 6])
@pytest.mark.parametrize("layout", [None, "texture"])
def test_broadcast_sources_fused_step_bit_identical(S, step, start, layout):
    from diffus_b200 import render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    n, P, R = 36, 3, 5
    v = layered_phantom(n, seed=3).to(dev())
    src, _, dirs = _geometry(n, P, R, step, S)
    src, dirs = src.to(dev()), dirs.to(dev())
    with torch.no_grad():
        target = render_frames(v, src + 0.5, dirs, S, 7e-4, start, sampler="trilinear")
    out = []
    for per_ray in (False, True):
        vol = v.clone().requires_grad_(True)
        s = (src[:, None, :].expand(-1, R, -1).contiguous() if per_ray else src.clone()).requires_grad_(True)
        d = dirs.clone().requires_grad_(True)
        loss = render_mse_loss(_vol(vol, layout) if layout else vol, s, d, target, S, 7e-4, start)
        loss.backward()
        out.append((loss.detach(), s.grad, d.grad, vol.grad if not layout else None))
    (l0, s0, d0, v0), (l1, s1, d1, v1) = out
    assert s1.shape == (P, R, 3)
    assert torch.equal(l0, l1) and torch.equal(d0, d1)
    if v0 is not None:
        torch.testing.assert_close(v1, v0, rtol=1e-6, atol=1e-6 * float(v0.abs().max()))   # atomics: order may differ
    torch.testing.assert_close(s1.sum(1), s0, rtol=1e-5, atol=1e-6 * float(s0.abs().max()))


@pytest.mark.parametrize("S,step,start,layout", [(160, 0.25, 0, None), (300, 0.1, 4, "brick"), (900, 0.04, 0, "texture"),
                                                 (2200, 0.015, 3, "quad")])
def test_distinct_origins_against_oracle(S, step, start, layout):
    from diffus_b200 import ops, render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    from oracle import port, probes
    n, P, R, alpha = 32, 3, 4, 7e-4
    vol = layered_phantom(n, seed=4)
    _, org, dirs = _geometry(n, P, R, step, 40 + S, spread=3.0)
    with torch.no_grad():
        target = render_frames(vol.to(dev()), org.to(dev()) + 0.4, dirs.to(dev()), S, alpha, start, sampler="trilinear").cpu()
    frames64 = torch.stack([probes.plot_beam_frame(vol.double(), org[p].double(), dirs[p].double(), S, alpha, start,
                                                 sampler="trilinear")[3] for p in range(P)])
    v = vol.to(dev())
    frame = render_frames(_vol(v, layout), org.to(dev()), dirs.to(dev()), S, alpha, start, sampler="trilinear")
    assert_frame_close(frame.cpu().numpy(), frames64.numpy(), "per-ray frame")

    def fn(vv, oo, dd):
        f = torch.stack([probes.plot_beam_frame(vv, oo[p], dd[p], S, alpha, start, sampler="trilinear")[3] for p in range(P)])
        return (f - target.to(f.dtype)).square().mean()
    (gv64, go64, gd64), noise, _ = oracle_grads(fn, vol, org, dirs)
    vg = v.clone().requires_grad_(True)
    o = org.to(dev()).requires_grad_(True)
    d = dirs.to(dev()).requires_grad_(True)
    loss = render_mse_loss(_vol(vg, layout) if layout else vg, o, d, target.to(dev()), S, alpha, start)
    loss.backward()
    np.testing.assert_allclose(loss.item(), float(fn(vol.double(), org.double(), dirs.double())), rtol=1e-5)
    assert o.grad.shape == (P, R, 3)
    assert_grad_close(o.grad.cpu().numpy(), go64.numpy(), "d/d origins", noise=noise[1])
    assert_grad_close(d.grad.cpu().numpy(), gd64.numpy(), "d/d directions", noise=noise[2])
    if not layout:
        assert_grad_close(vg.grad.cpu().numpy(), gv64.numpy(), "d/d volume", noise=noise[0])
    # ray_indices and trace_values: bit-exact against the port
    x, y, z = ops.ray_indices([n] * 3, org.to(dev()), dirs.to(dev()), S, start)
    tv = ops.trace_values(v, None, [n] * 3, org.to(dev()), dirs.to(dev()), S, 0)
    for p in range(P):
        xo, yo, zo, _ = probes.plot_beam_frame(vol, org[p], dirs[p], S, alpha, start, sampler="nearest")
        assert torch.equal(x[p].cpu(), xo) and torch.equal(y[p].cpu(), yo) and torch.equal(z[p].cpu(), zo)
        pts = probes.ray_points(org[p], dirs[p], S)
        assert torch.equal(tv[p].cpu(), port.sample_nearest(vol, pts)[3])


def test_trace_values_backward_per_ray_origins():
    from diffus_b200 import ops
    from diffus_b200.phantoms import layered_phantom
    from oracle import port, probes
    n, P, R, S = 24, 2, 5, 60
    vol = layered_phantom(n, seed=6)
    _, org, dirs = _geometry(n, P, R, 0.3, 5, spread=2.0)
    g = torch.randn((P, R, S), generator=torch.Generator().manual_seed(1))
    o = org.to(dev()).requires_grad_(True)
    d = dirs.to(dev()).requires_grad_(True)
    v = vol.to(dev())
    out = ops.TraceValuesFunction.apply(v, None, [n] * 3, o, d, S, 1, False)
    (out * g.to(dev())).sum().backward()

    def fn(vv, oo, dd):
        return sum((port.sample_trilinear(vv, probes.ray_points(oo[p], dd[p], S))[3] * g[p].to(vv.dtype)).sum() for p in range(P))
    (_, go, gd), noise, _ = oracle_grads(fn, vol, org, dirs)
    assert_grad_close(o.grad.cpu().numpy(), go.numpy(), "trace d/d origins", noise=noise[1])
    assert_grad_close(d.grad.cpu().numpy(), gd.numpy(), "trace d/d directions", noise=noise[2])


GN_CASES = [(300, 0, None, False, 0.07), (512, 0, "texture", True, 0.07), (385, 37, "brick", False, 0.07),
            (130, 3, "quad", False, 0.2), (1100, 0, "quad", False, 0.025), (1537, 11, "texture", False, 0.017),
            (2048, 0, "brick", True, 0.0165), (2600, 5, None, False, 0.013)]


@pytest.mark.parametrize("S,start,layout,shared,step", GN_CASES)
def test_gauss_newton_distinct_origins_vs_oracle(S, start, layout, shared, step):
    from diffus_b200 import render_frames, render_gauss_newton, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    from oracle import probes
    n, P, R, alpha = 36, 3, 4, 7e-4
    vol = layered_phantom(n, seed=7)
    _, org, dirs = _geometry(n, P, R, step, S + start, spread=4.0)
    if shared:
        dirs = dirs[0].contiguous()
    with torch.no_grad():
        target = render_frames(vol.to(dev()), org.to(dev()) + 0.6, dirs.to(dev()), S, alpha, start, sampler="trilinear")
    out = {dt: probes.pose_gauss_newton(vol.to(dt), org.to(dt), dirs.to(dt), target.cpu().to(dt), S, alpha, start)
           for dt in (torch.float64, torch.float32)}
    l64, jtj64, jtr64, _ = out[torch.float64]
    n_jtj = float((out[torch.float32][1].double() - jtj64).abs().max())
    n_jtr = float((out[torch.float32][2].double() - jtr64).abs().max())
    v = vol.to(dev())
    vv = _vol(v, layout)
    o, d = org.to(dev()), dirs.to(dev())
    loss, jtj, jtr = render_gauss_newton(vv, o, d, target, S, alpha, start)
    what = f"S={S} start={start} {layout} shared={shared}"
    np.testing.assert_allclose(loss.cpu().numpy(), l64.numpy(), rtol=1e-4, err_msg=what)
    assert_grad_close(jtr.cpu().numpy(), jtr64.numpy(), what + " Jtr", noise=n_jtr)
    assert_grad_close(jtj.cpu().numpy(), jtj64.numpy(), what + " JtJ", noise=n_jtj)
    l2, jtj2, jtr2 = render_gauss_newton(vv, o, d, target, S, alpha, start)
    assert torch.equal(loss, l2) and torch.equal(jtj, jtj2) and torch.equal(jtr, jtr2)     # run to run
    # (2/n) Jtr = the fused gradient in twist coordinates about the pivot
    oo = o.clone().requires_grad_(True)
    dd = (d if d.dim() == 3 else d.unsqueeze(0).expand(P, -1, -1)).contiguous().clone().requires_grad_(True)
    render_mse_loss(vv, oo, dd, target, S, alpha, start).backward()
    piv = o.double().mean(1, keepdim=True)
    gs, gdd = oo.grad.double(), dd.grad.double()
    g_v = gs.sum(1)
    g_w = torch.linalg.cross(o.double() - piv, gs, dim=-1).sum(1) + torch.linalg.cross(dd.detach().double(), gdd, dim=-1).sum(1)
    want = torch.cat([g_v, g_w], -1)
    n_el = target.numel()
    assert_grad_close((2.0 / n_el * jtr.double()).cpu().numpy(), want.cpu().numpy(), what + " 2 Jtr / n vs fused", rtol=1e-3)


@pytest.mark.parametrize("kind,kw", [("convex", dict(opening_angle=1.0, radius=20.0)), ("convex", dict(opening_angle=0.7)),
                                     ("linear", dict(width=60.0)), ("linear", dict(width=0.5))])
@pytest.mark.parametrize("R", [1, 33, 128])
def test_probe_rays_forward_and_backward(kind, kw, R):
    from diffus_b200 import probe_rays
    from oracle import probes
    g = torch.Generator().manual_seed(R)
    P = 5
    c, m, h = torch.randn((P, 3), generator=g) * 30, torch.randn((P, 3), generator=g) * 2, torch.randn((P, 3), generator=g)
    cd, md, hd = (t.to(dev()).requires_grad_(True) for t in (c, m, h))
    o, d = probe_rays(kind, cd, md, hd, R, **kw)
    o64, d64 = probes.probe_rays(kind, c.double(), m.double(), h.double(), R, **kw)
    assert o.shape == d.shape == (P, R, 3) and o.dtype == torch.float32
    np.testing.assert_allclose(d.detach().cpu().numpy(), d64.float().numpy(), rtol=0, atol=2e-7)
    np.testing.assert_allclose(o.detach().cpu().numpy(), o64.float().numpy(), rtol=0,
                               atol=float(o64.abs().max()) * 2 ** -23)
    wo, wd = torch.randn((P, R, 3), generator=g), torch.randn((P, R, 3), generator=g)
    ((o * wo.to(dev())).sum() + (d * wd.to(dev())).sum()).backward()
    c64, m64, h64 = (t.double().requires_grad_(True) for t in (c, m, h))
    o64, d64 = probes.probe_rays(kind, c64, m64, h64, R, **kw)
    ((o64 * wo.double()).sum() + (d64 * wd.double()).sum()).backward()
    assert_grad_close(cd.grad.cpu().numpy(), c64.grad.numpy(), "d/d centre", rtol=1e-5)
    assert_grad_close(md.grad.cpu().numpy(), m64.grad.numpy(), "d/d median", rtol=1e-5)
    assert_grad_close(hd.grad.cpu().numpy(), h64.grad.numpy(), "d/d hint", rtol=1e-5)


def test_convex_radius_zero_is_the_sector_probe():
    from diffus_b200 import fan_directions, probe_rays, render_frames
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n, P, R, S, angle = 48, 6, 32, 120, math.radians(55.0)
    src, _, med, hint = pose_sweep(P, n_rays=R, n=n, seed=2, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    o, d = probe_rays("convex", src, med, hint, R, opening_angle=angle)
    fan = fan_directions(med, hint, angle, R)
    assert torch.equal(d, fan) and torch.equal(o, src[:, None, :].expand(-1, R, -1))
    v = layered_phantom(n, seed=1).to(dev())
    for sampler in ("nearest", "trilinear"):
        assert torch.equal(render_frames(v, o, d, S, 1e-3, sampler=sampler), render_frames(v, src, fan, S, 1e-3, sampler=sampler))


def _smooth_phantom(n, seed=0):
    from diffus_b200.phantoms import layered_phantom
    v = layered_phantom(n, seed=seed, noise=0.0)[None, None]
    for _ in range(3):
        v = torch.nn.functional.avg_pool3d(torch.nn.functional.pad(v, (1, 1, 1, 1, 1, 1), mode="replicate"), 3, stride=1)
    return v[0, 0].contiguous()


PROBES = [("convex", dict(radius=8.0)), ("linear", dict(width=20.0))]


@pytest.mark.parametrize("probe,kw", PROBES)
def test_graphed_array_probe_step_matches_eager(probe, kw):
    from diffus_b200 import PreparedVolume, probe_rays, render_frames, render_mse_loss
    from diffus_b200.graphs import GraphedFanPoseStep
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n, P, R, S, angle = 32, 5, 16, 96, math.radians(50.0)
    pv = PreparedVolume(layered_phantom(n, seed=1).to(dev()), "brick")
    src, _, med, hint = pose_sweep(P, R, n, seed=3, opening_angle=angle, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    with torch.no_grad():
        target = render_frames(pv, *probe_rays(probe, src + 0.6, med, hint, R, opening_angle=angle, **kw), S, 1e-3,
                               sampler="trilinear")
    step = GraphedFanPoseStep(pv, target, R, S, angle, 1e-3, probe=probe, **kw)
    for shift in (0.0, 0.3):
        s = (src + shift).clone().requires_grad_(True)
        m = med.clone().requires_grad_(True)
        h = hint.clone().requires_grad_(True)
        loss = render_mse_loss(pv, *probe_rays(probe, s, m, h, R, opening_angle=angle, **kw), target, S, 1e-3)
        loss.backward()
        gl, gs, gm, gh = step(s.detach(), m.detach(), h.detach())
        torch.cuda.synchronize()
        assert gl.item() == loss.item()
        assert torch.equal(gs, s.grad) and torch.equal(gm, m.grad) and torch.equal(gh, h.grad)
        again = [t.clone() for t in step(s.detach(), m.detach(), h.detach())]
        assert all(torch.equal(a, b) for a, b in zip(again, (gl, gs, gm, gh)))


@pytest.mark.parametrize("probe,kw", PROBES)
def test_levenberg_marquardt_recovers_perturbed_array_probes(probe, kw):
    """The scene and tolerances of test_levenberg_marquardt_recovers_perturbed_poses, with array probes."""
    from diffus_b200 import PreparedVolume, probe_rays, recover_poses, render_frames
    from diffus_b200.graphs import GraphedFanGaussNewtonStep
    from diffus_b200.phantoms import pose_sweep
    from diffus_b200.pose_recovery import apply_fan_twist, fan_frame_angle
    n, P, R, S, angle = 64, 32, 32, 96, math.radians(60.0)
    vol = PreparedVolume(_smooth_phantom(n).to(dev()), "texture")
    src, _, med, hint = pose_sweep(P, n_rays=R, n=n, seed=8, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    with torch.no_grad():
        targets = render_frames(vol, *probe_rays(probe, src, med, hint, R, opening_angle=angle, **kw), S, 5e-3, sampler="trilinear")
    g = torch.Generator().manual_seed(0)
    u = torch.randn((P, 6), generator=g)
    u[:, :3] = u[:, :3] / u[:, :3].norm(dim=-1, keepdim=True) * 1.0
    u[:, 3:] = u[:, 3:] / u[:, 3:].norm(dim=-1, keepdim=True) * math.radians(1.0)
    s0, m0, h0 = apply_fan_twist(src, med, hint, u.to(dev()))
    K = 10
    (s1, m1, h1), hist = recover_poses(vol, targets, s0, m0, h0, angle, R, S, 5e-3, iterations=K, probe=probe, **kw)
    hist = hist.cpu()
    assert (hist[1:] <= hist[:-1]).all()
    pos_err = (s1 - src).norm(dim=-1).cpu()
    ang_err = torch.rad2deg(fan_frame_angle(m1, h1, med, hint)).cpu()
    print(f"LM {probe} K={K}: loss {hist[0].median():.3e} -> {hist[-1].median():.3e}; position error max {pos_err.max():.2e} "
          f"voxel; angle error max {ang_err.max():.2e} deg")
    assert float(pos_err.max()) < 1e-3 and float(ang_err.max()) < 1e-3
    # two graphs from the same start replay bit-identically
    a = GraphedFanGaussNewtonStep(vol, targets, R, S, angle, 5e-3, probe=probe, **kw)
    b = GraphedFanGaussNewtonStep(vol, targets, R, S, angle, 5e-3, probe=probe, **kw)
    for st in (a, b):
        st.reset(s0, m0, h0)
        for _ in range(3):
            st()
    assert torch.equal(a.poses, b.poses) and torch.equal(a.loss, b.loss)
