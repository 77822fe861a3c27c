"""CPU: the Gauss-Newton oracle (forward-mode autograd through the port), the pose twist, and the C-ABI argument checks of
``diffus_render_gauss_newton`` (no device needed)."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "diffus_b200.h")


def _tiny_case(shared=False, start=0):
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n = 20
    vol = layered_phantom(n, seed=3)
    sources, dirs = pose_sweep(2, n_rays=4, n=n, seed=1)
    if shared:
        dirs = dirs[0]
    S = 40
    g = torch.Generator().manual_seed(2)
    target = 0.01 * torch.randn((2, 4, S - start), generator=g)
    return vol.double(), sources, dirs, target, S, 0.01, start


@pytest.mark.parametrize("shared,start", [(False, 0), (True, 3)])
def test_oracle_jacobian_matches_central_differences(shared, start):
    from diffus_b200.pose_recovery import apply_pose_twist
    from oracle import gauss_newton, port
    vol, sources, dirs, target, S, alpha, start = _tiny_case(shared, start)
    loss, jtj, jtr, frames = gauss_newton.pose_gauss_newton(vol, sources, dirs, target, S, alpha, start)
    h = 1e-6
    for p in range(sources.shape[0]):
        d = dirs[p] if dirs.dim() == 3 else dirs

        def frame(xi):
            s2, d2 = apply_pose_twist(sources[p:p + 1].double(), d.double().unsqueeze(0), xi.unsqueeze(0))
            return port.plot_beam_frame(vol, s2[0], d2[0], S, alpha, start=start, sampler="trilinear")[3].reshape(-1)
        cols = []
        for j in range(6):
            e = torch.zeros(6, dtype=torch.float64)
            e[j] = h
            cols.append((frame(e) - frame(-e)) / (2 * h))
        J = torch.stack(cols, dim=-1)
        res = frame(torch.zeros(6, dtype=torch.float64)) - target[p].reshape(-1).double()
        np.testing.assert_allclose(loss[p].item(), float((res * res).sum()), rtol=1e-12)
        np.testing.assert_allclose(jtr[p].numpy(), (J.T @ res).numpy(), rtol=1e-6, atol=1e-9 * float(jtr[p].abs().max()))
        np.testing.assert_allclose(jtj[p].numpy(), (J.T @ J).numpy(), rtol=1e-6, atol=1e-9 * float(jtj[p].abs().max()))


def twist_gradient(grad_sources, grad_dirs, dirs):
    """The MSE gradient w.r.t. (sources, directions) in twist coordinates: g_v = dL/ds, g_w = sum_i d_i x dL/dd_i."""
    if dirs.dim() == 2:
        dirs = dirs.unsqueeze(0).expand_as(grad_dirs)
    return torch.cat([grad_sources, torch.linalg.cross(dirs, grad_dirs, dim=-1).sum(1)], dim=-1)


@pytest.mark.parametrize("shared,start", [(False, 0), (True, 3)])
def test_oracle_jtr_is_the_reverse_mode_mse_gradient_in_twist_coordinates(shared, start):
    from oracle import gauss_newton, port
    vol, sources, dirs, target, S, alpha, start = _tiny_case(shared, start)
    loss, jtj, jtr, _ = gauss_newton.pose_gauss_newton(vol, sources, dirs, target, S, alpha, start)
    s = sources.double().requires_grad_(True)
    d = dirs.double()
    d_per_pose = (d if d.dim() == 3 else d.unsqueeze(0).expand(2, -1, -1)).clone().requires_grad_(True)
    frames = torch.stack([port.plot_beam_frame(vol, s[p], d_per_pose[p], S, alpha, start=start, sampler="trilinear")[3]
                          for p in range(2)])
    mse = (frames - target.double()).square().mean()
    mse.backward()
    n = frames.numel()
    np.testing.assert_allclose(loss.sum().item() / n, mse.item(), rtol=1e-12)
    g = twist_gradient(s.grad, d_per_pose.grad, d_per_pose.detach())
    np.testing.assert_allclose((2.0 / n) * jtr.numpy(), g.numpy(), rtol=1e-9, atol=1e-12 * float(g.abs().max()))


def test_oracle_jtj_is_symmetric_positive_semidefinite():
    from oracle import gauss_newton
    vol, sources, dirs, target, S, alpha, start = _tiny_case()
    _, jtj, _, _ = gauss_newton.pose_gauss_newton(vol, sources, dirs, target, S, alpha, start)
    torch.testing.assert_close(jtj, jtj.transpose(-1, -2), rtol=0, atol=0)
    ev = torch.linalg.eigvalsh(jtj)
    assert (ev >= -1e-10 * ev.abs().amax(-1, keepdim=True)).all()


def test_pose_twist_identity_rotation_and_composition():
    from scipy.spatial.transform import Rotation
    from diffus_b200.pose_recovery import apply_fan_twist, apply_pose_twist
    g = torch.Generator().manual_seed(0)
    src = torch.randn((3, 3), generator=g, dtype=torch.float64)
    dirs = torch.randn((3, 5, 3), generator=g, dtype=torch.float64)
    shared = dirs[0]
    s0, d0 = apply_pose_twist(src, dirs, torch.zeros((3, 6), dtype=torch.float64))
    assert torch.equal(s0, src) and torch.equal(d0, dirs)
    s1, d1 = apply_pose_twist(src, shared, torch.zeros((3, 6), dtype=torch.float64))
    assert d1.shape == (3, 5, 3) and torch.equal(d1[2], shared)
    # a rotation vector rotates like scipy's, for small angles (series branch) and large ones
    for scale in (1e-6, 3e-5, 0.02, 1.3):
        delta = torch.randn((3, 6), generator=g, dtype=torch.float64) * scale
        s2, d2 = apply_pose_twist(src, dirs, delta)
        torch.testing.assert_close(s2, src + delta[:, :3], rtol=0, atol=0)
        for p in range(3):
            want = Rotation.from_rotvec(delta[p, 3:].numpy()).apply(dirs[p].numpy())
            np.testing.assert_allclose(d2[p].numpy(), want, rtol=1e-12, atol=1e-14)
    # two small twists compose to the twist of the composed rotation, and to their sum up to second order
    w1 = torch.tensor([[1e-3, -2e-3, 5e-4]], dtype=torch.float64)
    w2 = torch.tensor([[-7e-4, 1e-3, 2e-3]], dtype=torch.float64)
    z = torch.zeros((1, 3), dtype=torch.float64)
    _, a = apply_pose_twist(src[:1], dirs[:1], torch.cat([z, w1], -1))
    _, ab = apply_pose_twist(src[:1], a, torch.cat([z, w2], -1))
    comp = (Rotation.from_rotvec(w2[0].numpy()) * Rotation.from_rotvec(w1[0].numpy())).as_rotvec()
    _, direct = apply_pose_twist(src[:1], dirs[:1], torch.cat([z, torch.tensor(comp)[None]], -1))
    np.testing.assert_allclose(ab.numpy(), direct.numpy(), rtol=1e-12, atol=1e-14)
    _, summed = apply_pose_twist(src[:1], dirs[:1], torch.cat([z, w1 + w2], -1))
    assert float((ab - summed).abs().max()) < 1e-5 * float(dirs[:1].abs().max())
    # the fan of rotated fan parameters is the rotated fan
    from diffus_b200.phantoms import fan_directions
    med, hint = torch.randn((3, 3), generator=g), torch.randn((3, 3), generator=g)
    delta = torch.randn((3, 6), generator=g, dtype=torch.float64) * 0.1
    _, m2, h2 = apply_fan_twist(src, med.double(), hint.double(), delta)
    _, want = apply_pose_twist(src, fan_directions(med, hint, math.radians(60), 7).double(), delta)
    np.testing.assert_allclose(fan_directions(m2, h2, math.radians(60), 7).numpy(), want.float().numpy(), atol=2e-7)


@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()                       # nvcc cross-compiles without a GPU
    return _lib.load()


def test_gauss_newton_struct_layout_matches_header(lib):
    from diffus_b200._lib import DiffusGaussNewtonArgs
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef struct DiffusGaussNewtonArgs \{(.*?)\} DiffusGaussNewtonArgs;", text, flags=re.S).group(1)
    fields = [re.split(r"[\s\*]+", f.strip())[-1] for f in body.split(";") if f.strip()]
    assert fields == [f[0] for f in DiffusGaussNewtonArgs._fields_]


def test_gauss_newton_argument_validation_without_a_device(lib):
    from diffus_b200._lib import DiffusGaussNewtonArgs
    g = DiffusGaussNewtonArgs()
    assert lib.diffus_render_gauss_newton(None, None) == -1
    assert lib.diffus_render_gauss_newton_workspace_bytes(None) == 0
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -1              # NULL volume
    a = g.fwd
    a.volume.data = 0x1000
    a.volume.dim[0] = a.volume.dim[1] = a.volume.dim[2] = 8
    a.sources = a.directions = 0x1000
    a.n_poses, a.n_rays, a.n_samples, a.sampler = 2, 4, 16, 1
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -1              # NULL target / outputs
    g.target, g.loss, g.jtr = 0x1000, 0x2000, 0x3000
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -1              # NULL jtj
    g.jtj = 0x4000
    a.sampler = 0
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -5              # nearest: no pose derivative
    a.sampler, a.pose_dtype = 1, 1
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -5              # float64 poses
    a.pose_dtype = 0
    need = lib.diffus_render_gauss_newton_workspace_bytes(C.byref(g))
    assert need >= 2 * 4 * 32 * 4
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -4              # no workspace
    a.start = 3
    assert lib.diffus_render_gauss_newton_workspace_bytes(C.byref(g)) > need   # median, ties and its tangent
    g.workspace, g.workspace_bytes = 0x5000, need
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -4              # too small for start > 0
    a.start = 15
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -2              # start > S-2
    a.start, a.sampler = 0, 5
    assert lib.diffus_render_gauss_newton(C.byref(g), None) == -3              # unknown sampler
