"""GPU: the Gauss-Newton system of a whole tracked sweep (one twist shared by every pose, about one pivot) against the float64
forward-mode oracle of ``test_sweep_registration.py``, against the per-pose kernel, against the fused MSE step's gradient,
its NaN rule, determinism, CUDA-graph capture with the pivot read on the device, and Levenberg-Marquardt sweep registration."""
import math

import numpy as np
import pytest
import torch

from conftest import assert_grad_close
from test_sweep_registration import lever_map, mapped_pose_systems, sweep_gauss_newton

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _geometry(n, P, R, seed, step, shared):
    g = torch.Generator().manual_seed(seed)
    sources = torch.tensor([[3.0, 2.0, 4.0], [n * 0.5, n * 0.3, 1.5], [n - 3.5, n * 0.6, n - 4.0]])[:P]
    aim = torch.tensor([n * 0.5, n * 0.5, n * 0.5]) - sources
    d = aim[:, None, :] / aim.norm(dim=-1)[:, None, None] + 0.25 * torch.randn((P, R, 3), generator=g)
    dirs = d / d.norm(dim=-1, keepdim=True) * step
    return sources.contiguous(), (dirs[0] if shared else dirs).contiguous()


def _oracle(vol, sources, dirs, target, S, alpha, start, pivot):
    """fp64 oracle plus its own fp32 drift (the float32-noise rule of conftest.oracle_grads applied to JtJ and Jtr)."""
    out = {dt: sweep_gauss_newton(vol.to(dt), sources.to(dt), dirs.to(dt), target.to(dt), S, alpha, start, pivot)
           for dt in (torch.float64, torch.float32)}
    l64, jtj64, jtr64 = out[torch.float64]
    _, jtj32, jtr32 = out[torch.float32]
    return l64, jtj64, jtr64, float((jtj32.double() - jtj64).abs().max()), float((jtr32.double() - jtr64).abs().max())


def _check(loss, jtj, jtr, ref, what):
    l64, jtj64, jtr64, n_jtj, n_jtr = ref
    assert loss.dtype == jtj.dtype == jtr.dtype == torch.float64
    assert loss.shape == () and jtj.shape == (6, 6) and jtr.shape == (6,)
    np.testing.assert_allclose(loss.item(), l64.item(), rtol=1e-4, err_msg=what)
    assert_grad_close(jtr.cpu().numpy(), jtr64.numpy(), what + " Jtr", noise=n_jtr)
    assert_grad_close(jtj.cpu().numpy(), jtj64.numpy(), what + " JtJ", noise=n_jtj)
    assert torch.equal(jtj, jtj.T)


CASES = [  # (S, start, layout, shared, step, pivot): one pass / 513..2048 / > 2048 columns, every layout, crops, own and shared
    (300, 0, None, False, 0.07, None), (512, 0, "texture", True, 0.07, (20.0, 15.0, 9.0)),
    (385, 37, "brick", False, 0.07, None), (130, 3, "quad", False, 0.2, (5.0, 30.0, 12.0)),
    (1100, 0, "quad", False, 0.025, None), (1537, 11, "texture", False, 0.017, (18.0, 18.0, 18.0)),
    (2048, 0, "brick", True, 0.0165, None), (2600, 5, None, False, 0.013, (1.0, 2.0, 3.0)),
]


@pytest.mark.parametrize("S,start,layout,shared,step,pivot", CASES)
def test_sweep_system_vs_oracle(S, start, layout, shared, step, pivot):
    from diffus_b200 import PreparedVolume, render_frames, render_gauss_newton_sweep
    from diffus_b200.phantoms import layered_phantom
    n, P, R, alpha = 36, 3, 4, 7e-4
    vol = layered_phantom(n, seed=7)
    sources, dirs = _geometry(n, P, R, S + start, step, shared)
    with torch.no_grad():
        target = render_frames(vol.to(dev()), sources.to(dev()) + 0.6, dirs.to(dev()), S, alpha, start, sampler="trilinear")
    piv = None if pivot is None else torch.tensor(pivot, dtype=torch.float64)
    ref = _oracle(vol, sources, dirs, target.cpu(), S, alpha, start, piv)
    v = vol.to(dev())
    vv = PreparedVolume(v, layout) if layout else v
    out = render_gauss_newton_sweep(vv, sources.to(dev()), dirs.to(dev()), target, S, alpha, start,
                                    pivot=None if piv is None else piv.to(dev()))
    _check(*out, ref, f"S={S} start={start} {layout} shared={shared} pivot={pivot}")


def test_sweep_median_tie_vs_oracle():
    """The geometry of test_gauss_newton_median_tie_vs_oracle: start > 0 with most rays' first kept coefficient exactly 0."""
    from diffus_b200 import render_frames, render_gauss_newton_sweep
    from diffus_b200.phantoms import layered_phantom
    n, P, R, S, start = 24, 2, 6, 120, 4
    vol = layered_phantom(n, seed=5)
    g = torch.Generator().manual_seed(9)
    sources = torch.tensor([[-6.0, -6.0, -6.0], [-5.0, -7.0, -6.5]])
    aim = torch.tensor([n * 0.5, n * 0.5, n * 0.5]) - sources
    d = aim[:, None, :] / aim.norm(dim=-1)[:, None, None] + 0.2 * torch.randn((P, R, 3), generator=g)
    dirs = (d / d.norm(dim=-1, keepdim=True) * 0.4).contiguous()
    with torch.no_grad():
        target = render_frames(vol.to(dev()), sources.to(dev()) + 0.3, dirs.to(dev()), S, 1e-3, start, sampler="trilinear")
    from oracle import port
    z = port.sample_trilinear(vol, port.ray_points(sources[0], dirs[0], S))[3]
    r1 = port.reflection_coeff(z[:, start], z[:, start + 1])
    assert int((r1 == r1.median()).sum()) >= 2, "the case is meant to hold a tie"
    for pivot in (None, torch.tensor([4.0, 8.0, 2.0], dtype=torch.float64)):
        ref = _oracle(vol, sources, dirs, target.cpu(), S, 1e-3, start, pivot)
        out = render_gauss_newton_sweep(vol.to(dev()), sources.to(dev()), dirs.to(dev()), target, S, 1e-3, start,
                                        pivot=None if pivot is None else pivot.to(dev()))
        _check(*out, ref, f"tie pivot={pivot}")


PROBES = [("convex", dict(opening_angle=1.0, radius=6.0)), ("linear", dict(width=12.0))]


def _array_scene(probe, kw, n, P, R, S, seed):
    from diffus_b200 import probe_rays, render_frames
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    vol = layered_phantom(n, seed=seed)
    src, _, med, hint = pose_sweep(P, n_rays=R, n=n, seed=seed, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    with torch.no_grad():
        org, dirs = probe_rays(probe, src, med, hint, R, **kw)
        step = 0.35
        target = render_frames(vol.to(dev()), org + 0.4, dirs * step, S, 1e-3, sampler="trilinear")
    return vol, org.contiguous(), (dirs * step).contiguous(), target


@pytest.mark.parametrize("probe,kw", PROBES)
@pytest.mark.parametrize("start", [0, 3])
def test_sweep_array_probes_vs_oracle(probe, kw, start):
    from diffus_b200 import render_gauss_newton_sweep
    n, P, R, S = 32, 3, 6, 160
    vol, org, dirs, target = _array_scene(probe, kw, n, P, R, S, 4)
    target = target[..., start:].contiguous()
    ref = _oracle(vol, org.cpu(), dirs.cpu(), target.cpu(), S, 1e-3, start, None)
    out = render_gauss_newton_sweep(vol.to(dev()), org, dirs, target, S, 1e-3, start)
    _check(*out, ref, f"{probe} start={start}")


@pytest.mark.parametrize("kind", ["own", "shared", "convex", "linear"])
def test_sweep_system_is_the_sum_of_lever_mapped_pose_systems(kind):
    """sum_p A_p^T (JtJ_p, Jtr_p) of render_gauss_newton, A_p = [[I, -[o_p]x], [0, I]], o_p = the pose's own pivot - c."""
    from diffus_b200 import render_frames, render_gauss_newton, render_gauss_newton_sweep
    from diffus_b200.phantoms import layered_phantom
    n, P, R, S = 36, 3, 5, 700
    if kind in ("convex", "linear"):
        probe, kw = PROBES[0] if kind == "convex" else PROBES[1]
        vol, src, dirs, target = _array_scene(probe, kw, n, P, R, S, 2)
        vol = vol.to(dev())
        own = src.double().mean(1)
    else:
        vol = layered_phantom(n, seed=2).to(dev())
        src, dirs = _geometry(n, P, R, 3, 0.04, kind == "shared")
        src, dirs = src.to(dev()), dirs.to(dev())
        with torch.no_grad():
            target = render_frames(vol, src + 0.5, dirs, S, 1e-3, sampler="trilinear")
        own = src.double()
    pivot = own.mean(0) + torch.tensor([3.0, -2.0, 5.0], dtype=torch.float64, device=dev())
    loss, jtj, jtr = render_gauss_newton_sweep(vol, src, dirs, target, S, 1e-3, pivot=pivot)
    l_p, jtj_p, jtr_p = render_gauss_newton(vol, src, dirs, target, S, 1e-3)
    want_jtj, want_jtr = mapped_pose_systems(jtj_p.cpu(), jtr_p.cpu(), own.cpu(), pivot.cpu())
    np.testing.assert_allclose(loss.item(), l_p.double().sum().item(), rtol=1e-5)
    assert_grad_close(jtj.cpu().numpy(), want_jtj.numpy(), f"{kind} JtJ", rtol=1e-3)
    assert_grad_close(jtr.cpu().numpy(), want_jtr.numpy(), f"{kind} Jtr", rtol=1e-3)


def test_one_sector_pose_is_its_own_system():
    """P = 1, one source, no pivot given: the pivot is the source, the lever is exactly 0 and the system is the pose's own (the
    rotational tangent rounds in another order: (k d) x g instead of k (d x g))."""
    from diffus_b200 import render_frames, render_gauss_newton, render_gauss_newton_sweep
    from diffus_b200.phantoms import layered_phantom
    n, R, S = 36, 16, 400
    vol = layered_phantom(n, seed=6).to(dev())
    src, dirs = _geometry(n, 1, R, 5, 0.07, False)
    src, dirs = src.to(dev()), dirs.to(dev())
    with torch.no_grad():
        target = render_frames(vol, src + 0.4, dirs, S, 1e-3, sampler="trilinear")
    loss, jtj, jtr = render_gauss_newton_sweep(vol, src, dirs, target, S, 1e-3)
    l1, jtj1, jtr1 = render_gauss_newton(vol, src, dirs, target, S, 1e-3)
    np.testing.assert_allclose(loss.item(), l1.item(), rtol=1e-5)
    for got, want in ((jtj, jtj1[0]), (jtr, jtr1[0])):
        w = want.double().cpu().numpy()
        np.testing.assert_allclose(got.cpu().numpy(), w, rtol=1e-5, atol=1e-5 * np.abs(w).max())


@pytest.mark.parametrize("probe,kw", [("sector", {})] + PROBES)
def test_jtr_is_the_fused_mse_gradient_of_a_shared_twist(probe, kw):
    """(2/n) Jtr equals the autograd gradient of render_mse_loss w.r.t. ONE twist of every pose's parameters about the pivot
    (apply_probe_twist at xi = 0)."""
    from diffus_b200 import fan_directions, probe_rays, render_frames, render_gauss_newton_sweep, render_mse_loss
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    from diffus_b200.pose_recovery import apply_probe_twist
    n, P, R, S, angle = 40, 6, 16, 300, math.radians(50.0)
    vol = layered_phantom(n, seed=3).to(dev())
    src, _, med, hint = pose_sweep(P, n_rays=R, n=n, seed=5, opening_angle=angle, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())

    def rays(s, m, h):
        if probe == "sector":
            return s, fan_directions(m, h, angle, R) * 0.15
        o, d = probe_rays(probe, s, m, h, R, **kw)
        return o, d * 0.15
    with torch.no_grad():
        target = render_frames(vol, *rays(src + 0.5, med, hint), S, 1e-3, sampler="trilinear")
        o0, d0 = rays(src, med, hint)
    pivot = o0.reshape(-1, 3).double().mean(0)
    loss, _, jtr = render_gauss_newton_sweep(vol, o0, d0, target, S, 1e-3, pivot=pivot)
    xi = torch.zeros((1, 6), device=dev(), requires_grad=True)
    s, m, h = apply_probe_twist(src, med, hint, xi, pivot[None])
    mse = render_mse_loss(vol, *rays(s, m, h), target, S, 1e-3)
    mse.backward()
    nel = target.numel()
    np.testing.assert_allclose(loss.item() / nel, mse.item(), rtol=1e-5)
    g = xi.grad[0].double()
    torch.testing.assert_close((2.0 / nel) * jtr, g, rtol=2e-3, atol=2e-4 * float(g.abs().max()))


def test_zero_impedance_block_outputs_are_finite():
    from diffus_b200 import render_frames, render_gauss_newton_sweep
    from diffus_b200.phantoms import layered_phantom
    n, P, R = 36, 3, 12
    clean = layered_phantom(n, seed=11)
    holed = clean.clone()
    holed[15:21, 15:21, 15:21] = 0.0
    for S, step in ((400, 0.09), (1100, 0.033)):
        src, dirs = _geometry(n, P, R, S, step, False)
        src, dirs = src.to(dev()), dirs.to(dev())
        target = render_frames(clean.to(dev()), src + 0.4, dirs, S, 8e-4, sampler="trilinear")
        frame = render_frames(holed.to(dev()), src, dirs, S, 8e-4, sampler="trilinear")
        assert (frame[..., -1] == 0).any(), "some ray is meant to cross the block"
        loss, jtj, jtr = render_gauss_newton_sweep(holed.to(dev()), src, dirs, target, S, 8e-4)
        assert torch.isfinite(loss) and torch.isfinite(jtj).all() and torch.isfinite(jtr).all()


def test_two_calls_bit_identical_and_graph_replay_reads_the_pivot():
    from diffus_b200 import PreparedVolume, ops, render_frames
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n, S, P = 48, 600, 300                   # 4800 rays: several ranges in the two-stage sums
    vol = layered_phantom(n, seed=1).to(dev())
    pv = PreparedVolume(vol, "texture")
    sources, dirs = pose_sweep(P, n_rays=16, n=n, seed=4)
    sources, dirs = sources.to(dev()), (dirs * 0.2).to(dev())
    target = render_frames(vol, sources + 0.3, dirs, S, 1e-3, 20, sampler="trilinear")
    pivot = torch.tensor([20.0, 24.0, 26.0], dtype=torch.float64, device=dev())

    def call(piv, **out):
        return ops.render_gauss_newton_sweep_impl(vol, pv.bricks, list(vol.shape), sources, dirs, target, S, 20, 1e-3, piv, **out)
    a, b = call(None), call(None)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    c = call(pivot)
    assert not torch.equal(a[1], c[1])
    bufs = dict(loss_out=torch.zeros((), dtype=torch.float64, device=dev()),
                jtj_out=torch.zeros((6, 6), dtype=torch.float64, device=dev()),
                jtr_out=torch.zeros((6,), dtype=torch.float64, device=dev()))
    static_pivot = torch.zeros(3, dtype=torch.float64, device=dev())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call(static_pivot, **bufs)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call(static_pivot, **bufs)
    static_pivot.copy_(pivot)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(bufs["loss_out"], c[0]) and torch.equal(bufs["jtj_out"], c[1]) and torch.equal(bufs["jtr_out"], c[2])


def smooth_phantom(n, seed=0):
    """test_gpu_gauss_newton.py's smooth_phantom: layered_phantom without noise, blurred by three 3^3 box filters."""
    from diffus_b200.phantoms import layered_phantom
    v = layered_phantom(n, seed=seed, noise=0.0)[None, None]
    for _ in range(3):
        v = torch.nn.functional.avg_pool3d(torch.nn.functional.pad(v, (1, 1, 1, 1, 1, 1), mode="replicate"), 3, stride=1)
    return v[0, 0].contiguous()


@pytest.mark.parametrize("probe,kw", [("sector", {}), ("convex", dict(radius=8.0)), ("linear", dict(width=20.0))])
def test_register_sweep_recovers_a_shared_transform(probe, kw):
    from diffus_b200 import PreparedVolume, fan_directions, probe_rays, register_sweep, render_frames
    from diffus_b200.phantoms import pose_sweep
    from diffus_b200.pose_recovery import apply_rigid_transform, compose_sweep_twist, fan_frame_angle
    n, P, R, S, angle = 64, 32, 32, 96, math.radians(60.0)
    vol = PreparedVolume(smooth_phantom(n).to(dev()), "texture")
    src, _, med, hint = pose_sweep(P, n_rays=R, n=n, seed=8, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    with torch.no_grad():
        if probe == "sector":
            targets = render_frames(vol, src, fan_directions(med, hint, angle, R), S, 5e-3, sampler="trilinear")
        else:
            targets = render_frames(vol, *probe_rays(probe, src, med, hint, R, opening_angle=angle, **kw), S, 5e-3,
                                    sampler="trilinear")
    g = torch.Generator().manual_seed(1)
    u = torch.randn(6, generator=g, dtype=torch.float64)
    u[:3] *= 2.0 / u[:3].norm()                                     # 2 voxels
    u[3:] *= math.radians(2.0) / u[3:].norm()                       # and 2 degrees, about the centroid
    eye, zero = torch.eye(3, dtype=torch.float64, device=dev()), torch.zeros(3, dtype=torch.float64, device=dev())
    r0, t0 = compose_sweep_twist(eye, zero, u.to(dev()), src.double().mean(0))
    s0, m0, h0 = (x.float() for x in apply_rigid_transform(r0, t0, src, med, hint))
    K = 10
    (rot, trans), (s1, m1, h1), hist = register_sweep(vol, targets, s0, m0, h0, angle, R, S, 5e-3, iterations=K, probe=probe, **kw)
    hist = hist.cpu()
    assert hist.dtype == torch.float64 and hist.shape == (K + 1,)
    assert (hist[1:] <= hist[:-1]).all(), "the accept / reject rule never lets the loss grow"
    pos_err = (s1 - src).norm(dim=-1).cpu()
    ang_err = torch.rad2deg(fan_frame_angle(m1, h1, med, hint)).cpu()
    print(f"sweep LM {probe} K={K}: loss {hist[0]:.3e} -> {hist[-1]:.3e}; position error max {pos_err.max():.2e} voxel, "
          f"angle error max {ang_err.max():.2e} deg")
    assert float(pos_err.max()) < 1e-3 and float(ang_err.max()) < 1e-3
    # (R, t) maps the start sweep onto the returned one (the poses are that transform of the start, rounded once)
    for got, want in zip((s1, m1, h1), apply_rigid_transform(rot, trans, s0, m0, h0)):
        torch.testing.assert_close(got, want.float(), rtol=0, atol=1e-5 * float(want.abs().max()))
    assert rot.dtype == trans.dtype == torch.float64
    torch.testing.assert_close(rot @ rot.T, eye, rtol=0, atol=1e-12)
