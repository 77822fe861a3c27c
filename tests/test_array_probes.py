"""CPU: linear and convex array probes -- the float64 oracle geometry against explicit loops and the sector fan, the twists
about the pivot, the C ABI's rejection of bad arguments for the per-ray pose tag and the probe entry points, and the keyword
validation of the pose-recovery drivers."""
import ctypes as C
import math

import numpy as np
import pytest
import torch


def _params(P, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((P, 3), generator=g) * 10.0, torch.randn((P, 3), generator=g) * 2.0, torch.randn((P, 3), generator=g))


@pytest.mark.parametrize("R", [1, 2, 7, 64])
def test_oracle_convex_against_loops_and_the_fan(R):
    from diffus_b200.phantoms import fan_directions
    from oracle import probes
    c, m, h = _params(3, R)
    angle, rho = 1.1, 20.0
    o, d = probes.convex_rays(c, m, h, angle, R, rho)
    for p in range(3):
        mv = [float(x) for x in m[p]]
        nm = math.sqrt(sum(x * x for x in mv))
        mh = [x / nm for x in mv]
        hv = [float(x) for x in h[p]]
        hm = sum(a * b for a, b in zip(hv, mh))
        uv = [a - hm * b for a, b in zip(hv, mh)]
        nu = math.sqrt(sum(x * x for x in uv))
        uh = [x / nu for x in uv]
        for i in range(R):
            a = -angle / 2 if R == 1 else (angle / 2 if i == R - 1 else -angle / 2 + i * angle / (R - 1))
            for k in range(3):
                dk = math.cos(a) * mh[k] + math.sin(a) * uh[k]
                assert abs(float(d[p, i, k]) - dk) < 1e-12
                assert abs(float(o[p, i, k]) - (float(c[p, k]) + rho * dk)) < 1e-11
    o0, d0 = probes.convex_rays(c, m, h, angle, R, 0.0)
    assert torch.equal(o0, c.double().unsqueeze(1).expand(-1, R, -1))          # rho = 0: every ray leaves the centre
    np.testing.assert_allclose(d0.float().numpy(), fan_directions(m, h, angle, R).numpy(), rtol=0, atol=2e-7)


@pytest.mark.parametrize("R", [2, 5, 128])
def test_oracle_linear_elements_equally_spaced_on_u(R):
    from oracle import probes
    c, m, h = _params(4, 100 + R)
    w = 60.0
    o, d = probes.linear_rays(c, m, h, w, R)
    mh, uh = probes.frame(m, h)
    assert torch.allclose(d, mh.unsqueeze(1).expand(-1, R, -1), rtol=0, atol=0)
    step = o[:, 1:] - o[:, :-1]
    np.testing.assert_allclose(step.numpy(), (w / (R - 1) * uh).unsqueeze(1).expand(-1, R - 1, -1).numpy(), rtol=0, atol=1e-12)
    np.testing.assert_allclose(o.mean(1).numpy(), c.double().numpy(), atol=1e-12)           # centred on the centre
    assert float((o - c.double().unsqueeze(1)).mul(mh.unsqueeze(1)).sum(-1).abs().max()) < 1e-12   # the array is normal to m^
    np.testing.assert_allclose((o[:, -1] - o[:, 0]).norm(dim=-1).numpy(), w, rtol=1e-14)


@pytest.mark.parametrize("kind", ["convex", "linear"])
def test_probe_twist_commutes_with_the_geometry(kind):
    """Origins of the twisted parameters == the twisted origins about their pivot, in float64."""
    from diffus_b200.pose_recovery import apply_pose_twist, apply_probe_twist, probe_pivot
    from oracle import probes
    c, m, h = _params(5, 3)
    kw = dict(opening_angle=0.9, radius=20.0) if kind == "convex" else dict(width=60.0)
    o, d = probes.probe_rays(kind, c.double(), m.double(), h.double(), 16, **kw)
    g = torch.Generator().manual_seed(4)
    delta = torch.cat([torch.randn((5, 3), generator=g), 0.3 * torch.randn((5, 3), generator=g)], -1).double()
    o_want, d_want = apply_pose_twist(o, d, delta)
    c2, m2, h2 = apply_probe_twist(c.double(), m.double(), h.double(), delta, probe_pivot(o))
    o_got, d_got = probes.probe_rays(kind, c2, m2, h2, 16, **kw)
    np.testing.assert_allclose(o_got.numpy(), o_want.numpy(), rtol=0, atol=1e-11)
    np.testing.assert_allclose(d_got.numpy(), d_want.numpy(), rtol=0, atol=1e-13)


def test_pose_twist_per_ray_with_equal_origins_is_the_per_pose_twist():
    from diffus_b200.pose_recovery import apply_pose_twist
    g = torch.Generator().manual_seed(5)
    P, R = 6, 9
    src = torch.randn((P, 3), generator=g) * 30.0
    dirs = torch.randn((P, R, 3), generator=g)
    delta = torch.randn((P, 6), generator=g) * 0.5
    s1, d1 = apply_pose_twist(src, dirs, delta)
    s2, d2 = apply_pose_twist(src.unsqueeze(1).expand(-1, R, -1).contiguous(), dirs, delta)
    assert s2.dtype == torch.float32 and s2.shape == (P, R, 3)
    assert torch.equal(s2, s1.unsqueeze(1).expand(-1, R, -1)) and torch.equal(d2, d1)


@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()
    return _lib.load()


def _render_args(tag):
    from diffus_b200._lib import DiffusRenderArgs
    a = DiffusRenderArgs()
    a.volume.data = 0x1000
    a.volume.dim[0] = a.volume.dim[1] = a.volume.dim[2] = 8
    a.sources = a.directions = a.frame = 0x1000
    a.n_poses, a.n_rays, a.n_samples = 2, 4, 16
    a.sampler = 1
    a.pose_dtype = tag
    return a


def test_abi_per_ray_tag(lib):
    from diffus_b200._lib import POSE_F32_PER_RAY, DiffusGaussNewtonArgs, DiffusRenderBwdArgs
    assert POSE_F32_PER_RAY == 2
    a = _render_args(3)
    assert lib.diffus_render_forward(C.byref(a), None) == -3                  # tags beyond 2 are unknown
    assert lib.diffus_ray_indices(C.byref(a), 0x1000, 0x1000, 0x1000, None) == -3
    assert lib.diffus_trace_values(C.byref(a), 0x1000, None) == -3
    b = DiffusRenderBwdArgs()
    b.fwd = a
    b.grad_frame = 0x1000
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == -3
    assert lib.diffus_render_backward(C.byref(b), None) == -3
    a = _render_args(POSE_F32_PER_RAY)
    a.sources = None
    assert lib.diffus_render_forward(C.byref(a), None) == -1
    a = _render_args(POSE_F32_PER_RAY)
    a.n_rays = 0
    assert lib.diffus_render_forward(C.byref(a), None) == -2
    assert lib.diffus_trace_values(C.byref(a), 0x1000, None) == -2
    a = _render_args(POSE_F32_PER_RAY)
    a.n_samples = 4000
    b.fwd = a
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) in (0, 1)
    # the per-ray backward writes grad_sources itself: no source partials in the workspace
    b.grad_sources, b.grad_directions = 0x1000, 0x1000
    with_src = lib.diffus_render_bwd_workspace_bytes(C.byref(b))
    b.fwd.pose_dtype = 0
    assert with_src < lib.diffus_render_bwd_workspace_bytes(C.byref(b))
    assert lib.diffus_trace_values_backward(C.byref(_render_args(POSE_F32_PER_RAY)), None, None, 0x1000, 0x1000, None, 0, None) == -1
    # Gauss-Newton: the pivots take workspace; float64 poses stay unsupported
    g = DiffusGaussNewtonArgs()
    g.fwd = _render_args(POSE_F32_PER_RAY)
    g.target = g.loss = g.jtr = g.jtj = 0x1000
    per_ray = lib.diffus_render_gauss_newton_workspace_bytes(C.byref(g))
    g.fwd.pose_dtype = 0
    assert per_ray > lib.diffus_render_gauss_newton_workspace_bytes(C.byref(g))
    g.fwd.pose_dtype = 1
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -5
    g.fwd.pose_dtype = POSE_F32_PER_RAY
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -4                 # valid up to the missing workspace


def test_abi_probe_rays_rejects_bad_arguments(lib):
    p = 0x1000
    f, bwd = lib.diffus_probe_rays, lib.diffus_probe_rays_backward
    assert f(0, None, p, p, 1, 4, 0.5, 1.0, 0.0, p, p, None) == -1
    assert f(1, p, p, p, 1, 4, 0.0, 0.0, 10.0, p, None, None) == -1
    assert f(0, p, p, p, 0, 4, 0.5, 1.0, 0.0, p, p, None) == -2
    assert f(0, p, p, p, 1, 0, 0.5, 1.0, 0.0, p, p, None) == -2
    assert f(0, p, p, p, 1, 4, 0.5, -1.0, 0.0, p, p, None) == -2                  # negative radius
    assert f(0, p, p, p, 1, 4, 0.5, math.inf, 0.0, p, p, None) == -2
    assert f(0, p, p, p, 1, 4, math.nan, 1.0, 0.0, p, p, None) == -2
    assert f(1, p, p, p, 1, 4, 0.0, 0.0, 0.0, p, p, None) == -2                   # width <= 0
    assert f(1, p, p, p, 1, 4, 0.0, 0.0, -3.0, p, p, None) == -2
    assert f(1, p, p, p, 1, 4, 0.0, 0.0, math.nan, p, p, None) == -2
    assert f(2, p, p, p, 1, 4, 0.5, 1.0, 1.0, p, p, None) == -3                   # unknown kind
    assert f(-1, p, p, p, 1, 4, 0.5, 1.0, 1.0, p, p, None) == -3
    assert bwd(0, p, p, p, None, p, 1, 4, 0.5, 1.0, 0.0, p, p, p, None) == -1
    assert bwd(0, p, p, p, p, p, 1, 4, 0.5, 1.0, 0.0, p, p, None, None) == -1
    assert bwd(1, p, p, p, p, p, 1, 4, 0.0, 0.0, 0.0, p, p, p, None) == -2
    assert bwd(0, p, p, p, p, p, 1, 4, 0.5, -0.5, 0.0, p, p, p, None) == -2
    assert bwd(5, p, p, p, p, p, 1, 4, 0.5, 1.0, 1.0, p, p, p, None) == -3


def test_python_rejects_float64_per_ray_sources():
    from diffus_b200 import ops
    from diffus_b200._lib import DiffusError
    vol = torch.zeros((4, 4, 4))
    with pytest.raises(DiffusError, match="float32"):
        ops._check_inputs(vol, None, [4, 4, 4], torch.zeros((2, 3, 3), dtype=torch.float64),
                          torch.zeros((2, 3, 3), dtype=torch.float64))
    with pytest.raises(DiffusError, match="R"):
        ops._check_inputs(vol, None, [4, 4, 4], torch.zeros((2, 5, 3)), torch.zeros((2, 3, 3)))
    ops._check_inputs(vol, None, [4, 4, 4], torch.zeros((2, 3, 3)), torch.zeros((3, 3)))
    with pytest.raises(ValueError, match="kind"):
        ops.probe_args("phased", 1.0, 0.0, None)
    with pytest.raises(ValueError, match="opening_angle"):
        ops.probe_args("convex", None, 1.0, None)
    with pytest.raises(ValueError, match="width"):
        ops.probe_args("linear", None, 0.0, None)


@pytest.mark.parametrize("kw,match", [
    (dict(probe="phased"), "probe must be"),
    (dict(probe="sector", radius=3.0), "only apply"),
    (dict(probe="sector", width=10.0), "only apply"),
    (dict(probe="convex", radius=-1.0), "radius >= 0"),
    (dict(probe="convex", radius=math.nan), "radius >= 0"),
    (dict(probe="convex", width=4.0), "not width"),
    (dict(probe="linear"), "width > 0"),
    (dict(probe="linear", width=0.0), "width > 0"),
    (dict(probe="linear", width=math.inf), "width > 0"),
    (dict(probe="linear", width=5.0, radius=2.0), "not radius"),
])
def test_recover_poses_probe_keywords(kw, match):
    """Rejected on the host before any device work (the tensors here are CPU tensors)."""
    from diffus_b200 import recover_poses, recover_poses_coarse_to_fine
    z = torch.zeros((1, 3))
    with pytest.raises(ValueError, match=match):
        recover_poses(torch.zeros((4, 4, 4)), torch.zeros((1, 2, 8)), z, z, z, 1.0, 2, 8, **kw)
    with pytest.raises(ValueError, match=match):
        recover_poses_coarse_to_fine(torch.zeros((4, 4, 4)), torch.zeros((1, 2, 8)), z, z, z, 1.0, 2, 8, **kw)


def test_probe_keywords_accept_the_valid_forms():
    from diffus_b200.pose_recovery import probe_keywords
    assert probe_keywords("sector", None, None) == ("sector", 0.0, None)
    assert probe_keywords("convex", None, None) == ("convex", 0.0, None)
    assert probe_keywords("convex", 20, None) == ("convex", 20.0, None)
    assert probe_keywords("linear", None, 60) == ("linear", 0.0, 60.0)


@pytest.mark.parametrize("sampler,start", [("nearest", 0), ("trilinear", 0), ("trilinear", 5)])
def test_oracle_per_ray_frame_with_equal_origins_is_the_port_frame(sampler, start):
    """The per-ray restatement of plot_beam_frame reduces to oracle.port's when every ray leaves the same source."""
    from diffus_b200.phantoms import layered_phantom
    from oracle import port, probes
    vol = layered_phantom(20, seed=3).double()
    g = torch.Generator().manual_seed(6)
    src = torch.tensor([2.0, 3.0, 1.5], dtype=torch.float64)
    d = torch.randn((5, 3), generator=g, dtype=torch.float64) * 0.3 + torch.tensor([0.5, 0.5, 0.5], dtype=torch.float64)
    want = port.plot_beam_frame(vol, src, d, 40, 1e-2, start, sampler=sampler)
    got = probes.plot_beam_frame(vol, src.expand(5, 3), d, 40, 1e-2, start, sampler=sampler)
    for a, b in zip(got, want):
        assert torch.equal(a, b)


def test_oracle_per_ray_gauss_newton_with_equal_origins_is_the_pose_oracle():
    """Equal origins: the pivot is the source, so the per-ray Gauss-Newton oracle is oracle.gauss_newton's."""
    from diffus_b200.phantoms import layered_phantom
    from oracle import gauss_newton, probes
    vol = layered_phantom(16, seed=2).double()
    g = torch.Generator().manual_seed(7)
    src = torch.tensor([[2.0, 3.0, 1.5], [12.0, 1.0, 3.0]], dtype=torch.float64)
    d = (torch.randn((2, 4, 3), generator=g, dtype=torch.float64) * 0.2 + 0.4)
    target = torch.randn((2, 4, 27), generator=g, dtype=torch.float64) * 1e-2
    want = gauss_newton.pose_gauss_newton(vol, src, d, target, 30, 1e-2, 3)
    got = probes.pose_gauss_newton(vol, src.unsqueeze(1).expand(-1, 4, -1).contiguous(), d, target, 30, 1e-2, 3)
    for a, b in zip(got, want):
        np.testing.assert_allclose(a.numpy(), b.numpy(), rtol=1e-12, atol=1e-15)
