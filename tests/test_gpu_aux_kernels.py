"""GPU: the small kernels around the march (csrc/aux_kernels.cu) against the float64 oracle.

* the start > 0 median select (radix select + tie count) at R across the CTA, warp and shared-memory boundaries, with
  coefficient sets chosen for the radix key (negatives, signed zeros, low-byte differences, ties, NaN);
* the median backward and the gradient sets of the fused step and the autograd backward with start > 0, including the
  calls that ask for no gradient at all (loss only);
* trace_values forward / backward, sample_points, ray_indices and the per-pose reduction of the source gradient.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import assert_frame_close, assert_grad_close, oracle_grads

pytestmark = pytest.mark.gpu

LAYOUTS = [None, "brick", "quad", "texture"]
POSE_KINDS = ["f32", "f64", "per_ray"]


def dev():
    return torch.device("cuda:0")


def _vol(v, layout):
    from diffus_b200 import PreparedVolume
    return PreparedVolume(v, layout) if layout else v


def _close(vv):
    from diffus_b200 import PreparedVolume
    if isinstance(vv, PreparedVolume):
        vv.close()


def _oracle_frame(vol, src, dirs, S, alpha, start, sampler):
    """float64-or-whatever-dtype oracle frame of one pose; (R,3) ``src`` means one origin per ray."""
    from oracle import port, probes
    if src.dim() == 2:
        return probes.plot_beam_frame(vol, src, dirs, S, alpha, start, sampler=sampler)[3]
    return port.plot_beam_frame(vol, src, dirs, S, alpha, start, sampler=sampler)[3]


# ---------------------------------------------------------------------------------------
# a. the median select
# ---------------------------------------------------------------------------------------
def _pair_scene(pairs, n=48, stride=2):
    """A volume and one origin per ray (direction +axis 2, start = 1) such that samples k = 1, 2 of ray (p, r) are exactly the
    voxels holding ``pairs[p, r] = (z0, z1)``, and samples k = 3.. are the voxels after them (left at 1).  Integer
    coordinates: the nearest and the trilinear sampler both return the stored values bit for bit."""
    P, R, _ = pairs.shape
    per_line = n // stride
    slot = torch.arange(P * R)
    assert P * R <= n * n * per_line
    i, j, c = slot // (n * per_line), (slot // per_line) % n, stride * (slot % per_line)
    vol = torch.ones((n, n, n), dtype=torch.float32)
    vol[i, j, c] = pairs[..., 0].reshape(-1)
    vol[i, j, c + 1] = pairs[..., 1].reshape(-1)
    origins = torch.stack([i, j, c - 1], -1).float().view(P, R, 3).contiguous()
    dirs = torch.tensor([0.0, 0.0, 1.0]).expand(P, R, 3).contiguous()
    return vol, origins, dirs


def _coeff_pairs(kind, R, g):
    """(R, 2) float32 impedance pairs whose first reflection coefficients form one of the radix-key test sets."""
    if kind == "negative":                          # all negative, distinct
        r = -(0.01 + 0.89 * torch.rand(R, generator=g, dtype=torch.float64))
    elif kind == "mixed":                           # both signs, +0 and -0, one value repeated on a quarter of the rays
        r = 1.8 * torch.rand(R, generator=g, dtype=torch.float64) - 0.9
    elif kind == "lowbyte":                         # z1 a few ulps apart: the coefficients differ in the key's low byte
        z1 = torch.full((R,), 1.857, dtype=torch.float32)
        z1 = z1 + torch.randint(0, 48, (R,), generator=g).float() * float(torch.finfo(torch.float32).eps)
        return torch.stack([torch.ones(R), z1], -1)
    else:
        raise ValueError(kind)
    z = torch.stack([torch.ones(R, dtype=torch.float64), (1 + r) / (1 - r)], -1).float()
    if kind == "mixed":
        z[0::4] = torch.tensor([2.0, 2.0])           # r = +0
        z[1::4] = torch.tensor([-3.0, -3.0])         # r = 0 / -6 = -0
        z[2::4] = torch.tensor([1.0, 1.5])           # one value on many rays
    return z


def _device_median_check(frame, pairs):
    """Column 1 of a start = 1, alpha = 0 frame is the pose's median itself.  Every ray of a pose must carry the same value,
    and it must be the float32 lower median of the pose's coefficients (torch.median), identified among the pose's
    distinct coefficients; NaN where the median is NaN."""
    r32 = (pairs[..., 1] - pairs[..., 0]) / (pairs[..., 0] + pairs[..., 1])
    col = frame[:, :, 1].cpu()
    for p in range(pairs.shape[0]):
        want = torch.median(r32[p])
        got = col[p]
        if torch.isnan(want):
            assert torch.isnan(got).all() or (got == 0).all(), f"pose {p}: NaN median, got {got[:4]}"
            continue
        assert (got == got[0]).all(), f"pose {p}: rays disagree on the median"
        vals = torch.unique(r32[p])
        pick = vals[(vals.double() - float(got[0])).abs().argmin()]
        assert pick == want, f"pose {p}: column 1 {float(got[0])!r} is the coefficient {float(pick)!r}, lower median {float(want)!r}"


MEDIAN_R = [1, 2, 3, 31, 32, 33, 255, 256, 257, 1000, 10240, 10241]
SETS = ["negative", "mixed", "lowbyte"]


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("R", MEDIAN_R)
def test_median_select(R, sampler):
    """Three poses, each with another coefficient set (so a pose-index mistake shows), R on both sides of one warp, one
    256-thread CTA and the 40 KB shared-memory opt-in; the layout rotates with R."""
    from diffus_b200 import render_frames
    g = torch.Generator().manual_seed(R)
    k = MEDIAN_R.index(R)
    sets = SETS[k % 3:] + SETS[:k % 3]
    pairs = torch.stack([_coeff_pairs(s, R, g) for s in sets])
    vol, org, dirs = _pair_scene(pairs)
    layout = LAYOUTS[k % 4]
    vv = _vol(vol.to(dev()), layout)
    frame = render_frames(vv, org.to(dev()), dirs.to(dev()), 3, 0.0, 1, sampler=sampler)
    _close(vv)
    _device_median_check(frame, pairs)
    want = torch.stack([_oracle_frame(vol.double(), org[p].double(), dirs[p].double(), 3, 0.0, 1, sampler) for p in range(3)])
    assert_frame_close(frame.cpu().numpy(), want.numpy(), f"median R={R} {layout}")


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("R", [5, 40, 300])
def test_median_nan_stays_in_its_pose(R, sampler):
    """A zero-impedance block at the first interface of some rays of pose 1: 0/0 makes its median NaN, which zeroes the rest
    of that pose's frame (the echo's NaN rule); poses 0 and 2, in the same launch, keep their frames."""
    from diffus_b200 import render_frames
    g = torch.Generator().manual_seed(7 + R)
    pairs = torch.stack([_coeff_pairs(s, R, g) for s in SETS])
    pairs[1, 1::3] = 0.0
    vol, org, dirs = _pair_scene(pairs, stride=4)
    n = vol.shape[0]
    i, j, c = org[..., 0].long(), org[..., 1].long(), org[..., 2].long() + 1
    vol[i, j, c + 2] = 1.6                          # a later interface with an echo of its own
    vol[i, j, c + 3] = 0.7
    assert int(c.max()) + 3 < n
    S, start = 5, 1
    frame = render_frames(vol.to(dev()), org.to(dev()), dirs.to(dev()), S, 0.0, start, sampler=sampler).cpu()
    want = torch.stack([_oracle_frame(vol.double(), org[p].double(), dirs[p].double(), S, 0.0, start, sampler) for p in range(3)])
    assert (want[1, :, 1:] == 0).all() and (want[[0, 2], :, 2:] != 0).any()
    assert (frame[1] == 0).all(), "a NaN median must zero the whole frame of its pose"
    assert_frame_close(frame.numpy(), want.numpy(), f"NaN median R={R}")
    _device_median_check(frame, pairs)


# ---------------------------------------------------------------------------------------
# b. the median backward and the gradient sets with start > 0
# ---------------------------------------------------------------------------------------
TIE_N, TIE_P, TIE_R, TIE_S, TIE_START, TIE_ALPHA = 20, 3, 13, 24, 4, 0.05


def _tie_scene(kind):
    """A volume that varies along axis 0 only, and per pose 8 rays with the same source x and the same direction x, integer
    y and z steps from integer y and z: their first coefficients are bit-identical under both samplers, in the kernels and in
    the oracle at either precision (exactly equal ties, 8 of 13, so the median is theirs).  Three more rays have their own x
    slope; two leave through the x = 0 face before ``start``, so both of their samples clamp to the border: r = 0 exactly."""
    g = torch.Generator().manual_seed(11)
    i = torch.arange(TIE_N, dtype=torch.float64)
    prof = 1.5 + 0.4 * torch.tanh((i - 9) / 1.5) + 0.15 * torch.sin(1.3 * i) + 0.2 * (i > 13)
    vol = prof.view(-1, 1, 1).expand(TIE_N, TIE_N, TIE_N).float().contiguous()
    src = torch.tensor([[2.0, 10.0, 8.0], [2.5, 10.0, 9.0], [3.25, 9.0, 10.0]])
    steps = torch.tensor([[0, 0], [1, 0], [-1, 0], [0, 1], [0, -1], [1, 1], [-1, 1], [1, -1]], dtype=torch.float32)
    d = torch.empty((TIE_P, TIE_R, 3))
    for p in range(TIE_P):
        d[p, :8, 0] = 0.55 + 0.05 * p
        d[p, :8, 1:] = steps[torch.randperm(8, generator=g)]
        d[p, 8:11, 0] = 0.3 + 0.5 * torch.rand(3, generator=g)
        d[p, 11:, 0] = -2.5
        d[p, 8:, 1:] = 0.3 * torch.randn((TIE_R - 8, 2), generator=g)
    if kind == "per_ray":                           # own origins, differing off axis 0 by whole voxels
        org = src[:, None, :].expand(-1, TIE_R, -1).clone()
        org[..., 1:] += torch.randint(-2, 3, (TIE_P, TIE_R, 2), generator=g).float()
        return vol, org.contiguous(), d.contiguous()
    dt = torch.float64 if kind == "f64" else torch.float32
    return vol, src.to(dt), d.to(dt)


_TIE_ORACLE = {}


def _tie_oracle(kind, sampler):
    """Frames, target, loss and float64 gradients (with the oracle's own float32 noise) of the tie scene."""
    key = (kind, sampler)
    if key not in _TIE_ORACLE:
        vol, src, dirs = _tie_scene(kind)
        with torch.no_grad():
            f = torch.stack([_oracle_frame(vol.double(), src[p].double(), dirs[p].double(), TIE_S, TIE_ALPHA, TIE_START, sampler)
                             for p in range(TIE_P)])
        # the residual sits mostly in column 1, the median's own column, so the gradient is mostly the median backward's
        g = torch.Generator().manual_seed(3)
        peak = float(f.abs().max())
        target = f + 1e-3 * peak * torch.randn(f.shape, generator=g, dtype=torch.float64)
        target[..., 1] += 0.2 * peak
        target = target.float()

        def fn(vv, ss, dd):
            if sampler == "nearest":                # no pose derivative; the points exactly as the kernels form them
                ss, dd = src, dirs
            fr = torch.stack([_oracle_frame(vv, ss[p], dd[p], TIE_S, TIE_ALPHA, TIE_START, sampler) for p in range(TIE_P)])
            return (fr - target.to(fr.dtype)).square().mean(), fr
        (gv, gs, gd), noise, frames = oracle_grads(fn, vol, src, dirs)
        loss = float(fn(vol.double(), src.double(), dirs.double())[0])
        _TIE_ORACLE[key] = dict(vol=vol, src=src, dirs=dirs, target=target, frames=frames.detach(), loss=loss, gv=gv, gs=gs,
                                gd=gd, noise=noise)
    return _TIE_ORACLE[key]


GRAD_SETS = ["none", "volume", "poses", "both"]


def _check_grads(o, vg, s, d, want_vol, want_pose, sampler, what):
    if want_vol:
        assert_grad_close(vg.grad.cpu().numpy(), o["gv"].numpy(), what + " d/d volume", noise=o["noise"][0])
    if want_pose and sampler == "trilinear":
        assert s.grad.dtype == o["src"].dtype and d.grad.dtype == o["dirs"].dtype
        assert_grad_close(s.grad.cpu().numpy(), o["gs"].numpy(), what + " d/d sources", noise=o["noise"][1])
        assert_grad_close(d.grad.cpu().numpy(), o["gd"].numpy(), what + " d/d directions", noise=o["noise"][2])
    elif want_pose:                                 # the nearest sampler has no pose derivative
        assert s.grad is None and d.grad is None


@pytest.mark.parametrize("kind", POSE_KINDS)
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("grads", GRAD_SETS)
def test_median_backward_gradient_sets(grads, sampler, layout, kind):
    """Every gradient set of the fused step (eager and under no_grad) and of render_frames + backward, with start > 0 and a
    median that 8 rays tie for (torch spreads its gradient evenly over them).  A call that ends up with no gradient at all --
    nothing requested, or only the poses of the nearest sampler -- must still give the loss, bit for bit the loss of the
    call with every gradient wherever both run the same kernel."""
    from diffus_b200 import render_frames, render_mse_loss
    o = _tie_oracle(kind, sampler)
    want_vol, want_pose = grads in ("volume", "both"), grads in ("poses", "both")
    target = o["target"].to(dev())
    what = f"{grads} {sampler} {layout} {kind}"
    args = (TIE_S, TIE_ALPHA, TIE_START)

    def inputs(vol_grad, pose_grad):
        vg = o["vol"].to(dev()).requires_grad_(vol_grad)
        s = o["src"].to(dev()).requires_grad_(pose_grad)
        d = o["dirs"].to(dev()).requires_grad_(pose_grad)
        return vg, s, d

    # fused step, eager
    vg, s, d = inputs(want_vol, want_pose)
    vv = _vol(vg, layout)
    loss, frame = render_mse_loss(vv, s, d, target, *args, sampler=sampler, return_frame=True)
    assert_frame_close(frame.cpu().numpy(), o["frames"].numpy(), what + " fused frame")
    np.testing.assert_allclose(loss.item(), o["loss"], rtol=2e-5, err_msg=what)
    if loss.requires_grad:
        loss.backward()
    _check_grads(o, vg, s, d, want_vol, want_pose, sampler, what + " fused")
    # the same call with every gradient, and with none under no_grad: the same loss, bit for bit
    va, sa, da = inputs(True, True)
    vf = _vol(va, layout)
    full = render_mse_loss(vf, sa, da, target, *args, sampler=sampler)
    _close(vf)
    with torch.no_grad():
        quiet = render_mse_loss(vv, s, d, target, *args, sampler=sampler)
    # bit for bit where the same kernel runs (float64 poses, the nearest sampler); the float32 one-pass kernels with and
    # without a pose gradient are different instantiations and agree to a few ulp
    same_kernel = kind == "f64" or sampler == "nearest" or want_pose
    tol = 0.0 if same_kernel else 4 * 2.0 ** -23 * abs(full.item())
    assert abs(loss.item() - full.item()) <= tol, f"{what}: loss {loss.item()!r} vs {full.item()!r} with every gradient"
    assert torch.equal(quiet, loss.detach()), f"{what}: no_grad loss {quiet.item()!r} vs {loss.item()!r}"
    _close(vv)
    # render_frames + backward (the unfused render backward, then the median backward)
    vg, s, d = inputs(want_vol, want_pose)
    vv = _vol(vg, layout)
    frame = render_frames(vv, s, d, *args, sampler=sampler)
    assert_frame_close(frame.detach().cpu().numpy(), o["frames"].numpy(), what + " frame")
    if frame.requires_grad:
        (frame - target).square().mean().backward()
    _check_grads(o, vg, s, d, want_vol, want_pose, sampler, what + " render_frames")
    _close(vv)


@pytest.mark.parametrize("layout", [None, "texture"])
def test_graphed_pose_step_nearest_start(layout):
    """GraphedPoseStep with the nearest sampler asks the library for the loss alone (no pose derivative exists)."""
    from diffus_b200 import render_mse_loss
    from diffus_b200.graphs import GraphedPoseStep
    o = _tie_oracle("f32", "nearest")
    v = o["vol"].to(dev())
    vv = _vol(v, layout)
    target = o["target"].to(dev())
    step = GraphedPoseStep(vv, target, TIE_R, TIE_S, TIE_ALPHA, TIE_START, sampler="nearest")
    for shift in (0.0, 0.0, 1.0):
        src = o["src"].to(dev()) + shift
        loss, _, _ = step(src, o["dirs"].to(dev()))
        eager = render_mse_loss(vv, src, o["dirs"].to(dev()), target, TIE_S, TIE_ALPHA, TIE_START, sampler="nearest")
        torch.cuda.synchronize()
        assert torch.equal(loss, eager), f"graphed {loss.item()!r} vs eager {eager.item()!r}"
        if shift == 0.0:
            np.testing.assert_allclose(loss.item(), o["loss"], rtol=2e-5)
    _close(vv)


# ---------------------------------------------------------------------------------------
# c. trace_values forward and backward
# ---------------------------------------------------------------------------------------
TV_DIMS = (9, 12, 7)


def _edge_rays(kind):
    """3 poses x 7 rays (21: not a multiple of the backward's 4 rays per CTA) from integer sources: unit steps along +-each
    axis (samples on integer coordinates, through 0 and n - 1 and out of every face) and one dyadic oblique ray -- exact in
    float32 and float64 alike."""
    src = torch.tensor([[4.0, 6.0, 3.0], [0.0, 11.0, 6.0], [8.0, 0.0, 0.0]])
    base = torch.tensor([[1.0, 0, 0], [-1.0, 0, 0], [0, 1.0, 0], [0, -1.0, 0], [0, 0, 1.0], [0, 0, -1.0],
                         [0.3125, -0.46875, 0.21875]])
    dirs = torch.stack([base * (0.5 if p == 1 else 1.0) for p in range(3)])
    dirs[2, 6] = torch.tensor([0.25, 0.625, 0.5])
    if kind == "per_ray":
        org = src[:, None, :].expand(-1, 7, -1).clone()
        org[:, 6] += torch.tensor([0.5, -0.25, 0.75])
        return org.contiguous(), dirs.contiguous()
    dt = torch.float64 if kind in ("f64", "f64_product_f32") else torch.float32
    return src.to(dt), dirs.to(dt)


def _tv_points(ss, dd, S, kind):
    from oracle import port, probes
    if kind == "per_ray":
        return torch.stack([probes.ray_points(ss[p], dd[p], S) for p in range(ss.shape[0])])
    if kind == "f64_product_f32":                   # float32 product, float64 sum
        dd = dd.float()
    return torch.stack([port.ray_points(ss[p], dd[p], S) for p in range(ss.shape[0])])


@pytest.mark.parametrize("kind", ["f32", "f64", "f64_product_f32", "per_ray"])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_trace_values_forward_backward(sampler, layout, kind):
    from diffus_b200 import ops
    from diffus_b200.phantoms import layered_phantom
    from oracle import port
    sid = 0 if sampler == "nearest" else 1
    pf32 = kind == "f64_product_f32"
    vol = (layered_phantom(12, seed=5)[:TV_DIMS[0], :, :TV_DIMS[1] - 5] + 0.3).contiguous()
    assert tuple(vol.shape) == TV_DIMS
    src, dirs = _edge_rays(kind)
    v = vol.to(dev())
    vv = _vol(v, layout)
    bricks = vv.bricks if layout else None
    sample = port.sample_nearest if sampler == "nearest" else port.sample_trilinear
    for S in (2, 31, 32, 33, 100):
        what = f"{sampler} {layout} {kind} S={S}"
        out = ops.trace_values(v, bricks, list(TV_DIMS), src.to(dev()), dirs.to(dev()), S, sid, pf32).cpu()
        pts = _tv_points(src, dirs, S, kind)
        if sampler == "nearest":
            assert torch.equal(out, sample(vol, pts)[3]), what
        else:
            assert_frame_close(out.numpy(), sample(vol.double(), pts)[3].numpy(), what)
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(S))

        def fn(vq, sq, dq):
            if sampler == "nearest":
                sq, dq = src, dirs
            return (sample(vq, _tv_points(sq, dq, S, kind))[3] * g.to(vq.dtype)).sum()
        (gv, gs, gd), noise, _ = oracle_grads(fn, vol, src, dirs)
        for vol_grad, pose_grad in ((True, True), (True, False), (False, True)):
            vg = v.clone().requires_grad_(vol_grad)
            s = src.to(dev()).requires_grad_(pose_grad)
            d = dirs.to(dev()).requires_grad_(pose_grad)
            res = ops.TraceValuesFunction.apply(vg, bricks, list(TV_DIMS), s, d, S, sid, pf32)
            if not res.requires_grad:
                continue
            (res * g.to(dev())).sum().backward()
            sub = f"{what} vol={vol_grad} pose={pose_grad}"
            if vol_grad:
                assert_grad_close(vg.grad.cpu().numpy(), gv.numpy(), sub + " d/d volume", noise=noise[0])
            if pose_grad and sampler == "trilinear":
                assert_grad_close(s.grad.cpu().numpy(), gs.numpy(), sub + " d/d sources", noise=noise[1])
                assert_grad_close(d.grad.cpu().numpy(), gd.numpy(), sub + " d/d directions", noise=noise[2])
            elif pose_grad:
                assert s.grad is None and d.grad is None
    _close(vv)


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_trace_ray_and_simulate_rays(sampler):
    """The public wrappers: one pose, float64 source with float32 directions (float32 product, float64 sum)."""
    from diffus_b200 import UltrasoundRenderer
    from diffus_b200.phantoms import layered_phantom
    from oracle import port
    vol = layered_phantom(16, seed=2) + 0.3
    src = torch.tensor([7.0, 0.5, 8.0], dtype=torch.float64)
    dirs = torch.tensor([[0.0, 1.0, 0.0], [0.375, 0.75, -0.25], [-0.5, 0.625, 0.5], [0.0, -1.0, 0.0], [1.0, 0.0, 0.0]])
    S = 33
    v = vol.to(dev()).requires_grad_(True)
    s = src.to(dev()).requires_grad_(True)
    d = dirs.to(dev()).requires_grad_(True)
    ren = UltrasoundRenderer(S, 0.1)
    x, y, z, val = ren.trace_ray(v, s, d, S, sampler=sampler)
    pts = port.ray_points(src, dirs, S)
    xo, yo, zo = port.nearest_indices(vol.shape, pts)
    assert torch.equal(x.cpu(), xo) and torch.equal(y.cpu(), yo) and torch.equal(z.cpu(), zo)
    g = torch.randn((5, S), generator=torch.Generator().manual_seed(0))
    sample = port.sample_nearest if sampler == "nearest" else port.sample_trilinear

    def fn(vq, sq, dq):
        return (sample(vq, port.ray_points(sq, dq.float(), S) if sampler == "trilinear" else pts)[3] * g.to(vq.dtype)).sum()
    (gv, gs, gd), noise, _ = oracle_grads(fn, vol, src, dirs)
    (val * g.to(dev())).sum().backward()
    assert_grad_close(v.grad.cpu().numpy(), gv.numpy(), "trace_ray d/d volume", noise=noise[0])
    if sampler == "trilinear":
        assert s.grad.dtype == torch.float64 and d.grad.dtype == torch.float32
        assert_grad_close(s.grad.cpu().numpy(), gs.numpy(), "trace_ray d/d source", noise=noise[1])
        assert_grad_close(d.grad.cpu().numpy(), gd.numpy(), "trace_ray d/d directions", noise=noise[2])
    with torch.no_grad():
        _, _, _, refl = ren.simulate_rays(v, s, d, S, sampler=sampler)
        z1 = ren.simulate_rays(v, s, d, S, MRI=True, sampler=sampler)
    assert torch.equal(z1, val.detach()[:, :-1])
    want = port.reflection_coeff(val.detach()[:, :-1], val.detach()[:, 1:])
    assert torch.equal(refl, want)


# ---------------------------------------------------------------------------------------
# d. sample_points and ray_indices
# ---------------------------------------------------------------------------------------
def _edge_points(n_pts, dims, g):
    """Points in and far outside the volume, with exact .5 ties (round half to even), -0.5, integer coordinates and values
    beyond the int32 range (the conversion saturates)."""
    hi = torch.tensor(dims, dtype=torch.float32)
    pts = torch.rand((n_pts, 3), generator=g) * (hi + 8) - 4
    special = torch.tensor([-0.5, 0.5, 1.5, 2.5, -1.5, 0.0, -0.0, 3.0, 1e6, -1e6, 3e9, -3e9, 4.5, 5.5])
    m = min(n_pts, 4 * len(special))
    pick = torch.randint(0, len(special), (m, 3), generator=g)
    pts[:m] = special[pick]
    ties = torch.randint(-2, 20, (n_pts // 5, 3), generator=g).float() + 0.5
    pts[m:m + ties.shape[0]] = ties[:max(0, n_pts - m)]
    return pts.contiguous()


@pytest.mark.parametrize("n_pts", [1, 255, 256, 257, 148 * 16 * 256 + 1])
@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_sample_points(n_pts, sampler):
    from diffus_b200 import ops
    from diffus_b200.phantoms import layered_phantom
    from oracle import port
    dims = (13, 10, 17)
    vol = layered_phantom(17, seed=3)[:13, :10, :].contiguous() + 0.2
    pts = _edge_points(n_pts, dims, torch.Generator().manual_seed(n_pts))
    sid = 0 if sampler == "nearest" else 1
    x, y, z, val = ops.sample_points(vol.to(dev()), pts.to(dev()), sid)
    xo, yo, zo = port.nearest_indices(dims, pts)
    assert torch.equal(x.cpu(), xo) and torch.equal(y.cpu(), yo) and torch.equal(z.cpu(), zo)
    if sampler == "nearest":
        assert torch.equal(val.cpu(), port.sample_nearest(vol, pts)[3])
    else:
        assert_frame_close(val.cpu().numpy(), port.sample_trilinear(vol.double(), pts.double())[3].numpy(), "sample_points")


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_sample_points_abi_every_layout(sampler):
    """diffus_sample_points reads every layout the renderer can gather from; an unknown layout tag and a QUAD buffer off its
    16-byte alignment are rejected with their error codes."""
    from diffus_b200 import _lib, ops
    from diffus_b200.phantoms import layered_phantom
    from oracle import port
    lib = _lib.load()
    dims = (11, 14, 9)
    vol = layered_phantom(14, seed=4)[:11, :, :9].contiguous() + 0.2
    pts = _edge_points(3001, dims, torch.Generator().manual_seed(5))
    v, p = vol.to(dev()), pts.to(dev())
    sid = 0 if sampler == "nearest" else 1
    tex = ops.VolumeTexture(v)
    quads, bricks = ops.to_quads(v), ops.to_bricks(v)
    data = {_lib.LAYOUT_LINEAR: v.data_ptr(), _lib.LAYOUT_BRICK: bricks.data_ptr(), _lib.LAYOUT_QUAD: quads.data_ptr(),
            _lib.LAYOUT_TEXTURE: tex.texture}
    want_idx = port.nearest_indices(dims, pts)
    want = port.sample_nearest(vol, pts)[3] if sampler == "nearest" else port.sample_trilinear(vol.double(), pts.double())[3]

    def call(layout, ptr):
        dv = _lib.DiffusVolume()
        dv.data = ptr
        dv.dim[0], dv.dim[1], dv.dim[2] = dims
        dv.layout = layout
        val = torch.full((pts.shape[0],), float("nan"), device=dev())
        idx = torch.full((3, pts.shape[0]), -1, dtype=torch.int64, device=dev())
        rc = lib.diffus_sample_points(C.byref(dv), p.data_ptr(), pts.shape[0], sid, val.data_ptr(), idx[0].data_ptr(),
                                      idx[1].data_ptr(), idx[2].data_ptr(), ops._stream(dev()))
        return rc, val, idx
    for layout, ptr in data.items():
        rc, val, idx = call(layout, ptr)
        assert rc == 0, f"layout {layout}: {lib.diffus_error_string(rc).decode()}"
        assert all(torch.equal(idx[a].cpu(), want_idx[a]) for a in range(3)), f"layout {layout} indices"
        if sampler == "nearest":
            assert torch.equal(val.cpu(), want), f"layout {layout}"
        else:
            assert_frame_close(val.cpu().numpy(), want.numpy(), f"sample_points layout {layout}")
    assert call(7, v.data_ptr())[0] == -3                               # DIFFUS_E_ENUM
    assert call(_lib.LAYOUT_QUAD, quads.data_ptr() + 4)[0] == -5        # DIFFUS_E_UNSUPPORTED: float4 loads
    torch.cuda.synchronize()
    tex.close()


@pytest.mark.parametrize("kind", ["f32", "f64", "f64_product_f32", "per_ray"])
@pytest.mark.parametrize("start", [0, 5])
def test_ray_indices_bit_exact(kind, start):
    from diffus_b200 import ops
    g = torch.Generator().manual_seed(2)
    P, R, S, dims = 4, 37, 70, [15, 22, 11]
    src = (torch.rand((P, 3), generator=g) * 10 + 2).double()
    dirs = torch.randn((P, R, 3), generator=g, dtype=torch.float64) * 0.37
    dirs[:, :4] = torch.tensor([0.5, -0.25, 0.125], dtype=torch.float64)        # samples on the .5 ties
    src[0] = torch.tensor([3.0, 4.0, 5.0], dtype=torch.float64)
    if kind == "per_ray":
        src = (src[:, None, :] + torch.rand((P, R, 3), generator=g, dtype=torch.float64)).float().contiguous()
        dirs = dirs.float()
    elif kind == "f32":
        src, dirs = src.float(), dirs.float()
    pf32 = kind == "f64_product_f32"
    x, y, z = ops.ray_indices(dims, src.to(dev()), dirs.to(dev()), S, start, pf32)
    pts = _tv_points(src, dirs, S, kind)
    from oracle import port
    xo, yo, zo = port.nearest_indices(dims, pts)
    for got, want in ((x, xo), (y, yo), (z, zo)):
        assert torch.equal(got.cpu(), want[..., start:])


# ---------------------------------------------------------------------------------------
# e. the per-pose reduction of the source gradient
# ---------------------------------------------------------------------------------------
def _reduce_check(got, partial, what):
    """(P,3) per-pose sums against the float64 sum of the (P,R,3) per-ray partials the same kernel wrote with one origin per
    ray: each lane adds ceil(R/32) partials, then five shuffle levels -- a float32 rounding budget of that many terms."""
    R = partial.shape[1]
    want = partial.double().sum(1)
    budget = (-(-R // 32) + 6) * 2.0 ** -24 * partial.double().abs().sum(1) + 1e-30
    err = (got.double() - want).abs()
    assert (err <= 2 * budget).all(), f"{what}: max err / budget {float((err / budget).max()):.2f}"
    assert want.abs().max() > 0


def _reduce_geometry(P, R, n, g):
    src = torch.tensor([n * 0.5, 1.0, n * 0.5]) + torch.rand((P, 3), generator=g) * 4 - 2
    d = torch.tensor([0.0, 1.0, 0.0]) + 0.4 * (torch.rand((P, R, 3), generator=g) - 0.5)
    return src.contiguous(), (d / d.norm(dim=-1, keepdim=True) * 0.45).contiguous()


@pytest.mark.parametrize("R", [1, 31, 32, 33, 1000])
def test_reduce_rays(R):
    """Per-pose d/d sources of trace_values_bwd and of the unfused render backward (start > 0) = the sum of what the same
    kernels write with one origin per ray."""
    from diffus_b200 import ops, render_frames
    from diffus_b200.phantoms import layered_phantom
    n, P, S = 32, 3, 40
    g = torch.Generator().manual_seed(R)
    v = layered_phantom(n, seed=1).to(dev())
    src, dirs = _reduce_geometry(P, R, n, g)
    src, dirs = src.to(dev()), dirs.to(dev())
    per_ray = src[:, None, :].expand(-1, R, -1).contiguous()
    gv = torch.randn((P, R, S), generator=g).to(dev())
    _, gs, _ = ops.trace_values_bwd(gv, v, None, [n] * 3, src, dirs, S, 1, False, False, True)
    _, gr, _ = ops.trace_values_bwd(gv, v, None, [n] * 3, per_ray, dirs, S, 1, False, False, True)
    assert gs.shape == (P, 3) and gr.shape == (P, R, 3)
    _reduce_check(gs.cpu(), gr.cpu(), f"trace_values_bwd R={R}")
    out = []
    for s in (src, per_ray):
        s = s.clone().requires_grad_(True)
        f = render_frames(v, s, dirs, S, 1e-2, 3, sampler="trilinear")
        (f * gv[..., 3:]).sum().backward()
        out.append(s.grad)
    _reduce_check(out[0].cpu(), out[1].cpu(), f"render backward R={R}")


def test_reduce_rays_beyond_fused_reduction():
    """P R > 2^18 rays: the fused step's source gradient leaves the one-launch reduction for reduce_rays."""
    from diffus_b200 import render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    n, P, R, S = 32, 64, 4097, 8
    assert P * R > 1 << 18
    g = torch.Generator().manual_seed(9)
    v = layered_phantom(n, seed=2).to(dev())
    src, dirs = _reduce_geometry(P, R, n, g)
    src, dirs = src.to(dev()), dirs.to(dev())
    with torch.no_grad():
        target = render_frames(v, src + 0.3, dirs, S, 1e-2, sampler="trilinear")
    out = []
    for s in (src, src[:, None, :].expand(-1, R, -1).contiguous()):
        s = s.clone().requires_grad_(True)
        loss = render_mse_loss(v, s, dirs, target, S, 1e-2)
        loss.backward()
        out.append((loss.detach(), s.grad))
    (l0, g0), (l1, g1) = out
    assert torch.equal(l0, l1)
    _reduce_check(g0.cpu(), g1.cpu(), "fused step P R > 2^18")
