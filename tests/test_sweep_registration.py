"""CPU: the float64 oracle of a tracked sweep's ONE Gauss-Newton system (a twist shared by every pose, about one pivot), the
transform algebra of sweep registration against scipy, the host-side argument checks of ``render_gauss_newton_sweep`` and
``register_sweep``, and the C-ABI checks of ``diffus_render_gauss_newton_sweep`` (no device needed).

:func:`sweep_gauss_newton` is the reference the GPU tests (``test_gpu_sweep_registration.py``) compare against.  Like
:func:`oracle.gauss_newton.pose_gauss_newton` it restates none of the kernel's formulas: the Jacobian is taken by torch
forward-mode autograd through the port's ``plot_beam_frame`` of every pose moved by the shared twist."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "diffus_b200.h")


def sweep_gauss_newton(volume, sources, directions, target, num_samples, attenuation_coeff=0.5, start=0, pivot=None):
    """The sweep's system in the dtype of ``volume``: ``J = d frame / d xi`` at ``xi = 0`` for ONE twist ``xi = (v, w)`` about
    ``pivot`` c moving every pose, ``s -> c + v + Rot(w) (s - c)``, ``d -> Rot(w) d`` (``apply_probe_twist`` with the origins
    as centres and the directions as orientation vectors), through :func:`oracle.port.plot_beam_frame` ((P,3) sources) or
    :func:`oracle.probes.plot_beam_frame` ((P,R,3) origins), trilinear.  ``pivot`` None: the float64 mean of all ray origins.
    Returns ``loss ()``, ``JtJ (6,6)``, ``Jtr (6,)`` summed over all poses."""
    import torch.autograd.forward_ad as fwAD
    from diffus_b200.pose_recovery import apply_probe_twist
    from oracle import port, probes
    dt = volume.dtype
    per_ray = sources.dim() == 3
    if pivot is None:
        pivot = sources.double().reshape(-1, 3).mean(0)
    c = pivot.to(dt).reshape(1, 3)
    eye = torch.eye(6, dtype=dt)
    loss, jtj, jtr = torch.zeros((), dtype=dt), torch.zeros((6, 6), dtype=dt), torch.zeros((6,), dtype=dt)
    for p in range(sources.shape[0]):
        org = sources[p].to(dt).reshape(-1, 3)
        dirs = (directions[p] if directions.dim() == 3 else directions).to(dt)
        cols = []
        for j in range(6):
            with fwAD.dual_level():
                xi = fwAD.make_dual(torch.zeros((1, 6), dtype=dt), eye[j:j + 1])
                o2, d2, _ = apply_probe_twist(org, dirs, dirs, xi, c)
                if per_ray:
                    f = probes.plot_beam_frame(volume, o2, d2, num_samples, attenuation_coeff, start, sampler="trilinear")[3]
                else:
                    f = port.plot_beam_frame(volume, o2[0], d2, num_samples, attenuation_coeff, start=start, sampler="trilinear")[3]
                f, t = fwAD.unpack_dual(f)
            cols.append(t.reshape(-1))
        J = torch.stack(cols, dim=-1)
        res = f.reshape(-1) - target[p].reshape(-1).to(dt)
        loss = loss + (res * res).sum()
        jtj = jtj + J.T @ J
        jtr = jtr + J.T @ res
    return loss, jtj, jtr


def lever_map(o):
    """``A = [[I, -[o]x], [0, I]]``: the pose's own twist (about c + o) of the shared twist (about c)."""
    a = torch.eye(6, dtype=torch.float64)
    ox = torch.tensor([[0.0, -o[2], o[1]], [o[2], 0.0, -o[0]], [-o[1], o[0], 0.0]], dtype=torch.float64)
    a[:3, 3:] = -ox
    return a


def mapped_pose_systems(jtj_p, jtr_p, own_pivots, pivot):
    """``sum_p A_p^T JtJ_p A_p`` and ``sum_p A_p^T Jtr_p`` with ``o_p`` = the pose's own pivot - ``pivot``."""
    jtj, jtr = torch.zeros((6, 6), dtype=torch.float64), torch.zeros((6,), dtype=torch.float64)
    for p in range(jtj_p.shape[0]):
        a = lever_map((own_pivots[p].double() - pivot.double()).tolist())
        jtj = jtj + a.T @ jtj_p[p].double() @ a
        jtr = jtr + a.T @ jtr_p[p].double()
    return jtj, jtr


def _tiny_sweep(kind, start):
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n, P, R, S = 20, 3, 4, 40
    vol = layered_phantom(n, seed=3).double()
    sources, dirs = pose_sweep(P, n_rays=R, n=n, seed=1)
    g = torch.Generator().manual_seed(2)
    if kind == "shared":
        dirs = dirs[0]
    if kind == "per_ray":
        sources = (sources[:, None, :] + 2.0 * (2 * torch.rand((P, R, 3), generator=g) - 1)).contiguous()
    target = 0.01 * torch.randn((P, R, S - start), generator=g)
    return vol, sources, dirs, target, S, 0.01, start


@pytest.mark.parametrize("kind,start", [("own", 0), ("shared", 3), ("per_ray", 0), ("per_ray", 5)])
def test_sweep_oracle_is_the_sum_of_lever_mapped_pose_systems(kind, start):
    from oracle import gauss_newton, probes
    vol, sources, dirs, target, S, alpha, start = _tiny_sweep(kind, start)
    pivot = torch.tensor([9.5, 7.25, 11.0], dtype=torch.float64)
    loss, jtj, jtr = sweep_gauss_newton(vol, sources, dirs, target, S, alpha, start, pivot)
    if kind == "per_ray":
        l_p, jtj_p, jtr_p, _ = probes.pose_gauss_newton(vol, sources, dirs, target, S, alpha, start)
        own = sources.double().mean(1)
    else:
        l_p, jtj_p, jtr_p, _ = gauss_newton.pose_gauss_newton(vol, sources, dirs, target, S, alpha, start)
        own = sources.double()
    want_jtj, want_jtr = mapped_pose_systems(jtj_p, jtr_p, own, pivot)
    np.testing.assert_allclose(loss.item(), l_p.sum().item(), rtol=1e-12)
    np.testing.assert_allclose(jtj.numpy(), want_jtj.numpy(), rtol=1e-10, atol=1e-10 * float(want_jtj.abs().max()))
    np.testing.assert_allclose(jtr.numpy(), want_jtr.numpy(), rtol=1e-10, atol=1e-10 * float(want_jtr.abs().max()))
    # the default pivot is the mean of all ray origins; a sector pose's R rays share its source
    _, jtj0, _ = sweep_gauss_newton(vol, sources, dirs, target, S, alpha, start)
    want0, _ = mapped_pose_systems(jtj_p, jtr_p, own, sources.double().reshape(-1, 3).mean(0))
    np.testing.assert_allclose(jtj0.numpy(), want0.numpy(), rtol=1e-10, atol=1e-10 * float(want0.abs().max()))


def test_rotation_and_composition_match_scipy():
    from scipy.spatial.transform import Rotation
    from diffus_b200.pose_recovery import apply_rigid_transform, compose_sweep_twist, rotation_matrix
    g = torch.Generator().manual_seed(0)
    for scale in (1e-7, 3e-5, 0.02, 1.3, 3.0):
        w = torch.randn(3, generator=g, dtype=torch.float64) * scale
        np.testing.assert_allclose(rotation_matrix(w).numpy(), Rotation.from_rotvec(w.numpy()).as_matrix(), rtol=0, atol=1e-15)
    rot = torch.tensor(Rotation.from_rotvec([0.3, -0.2, 0.5]).as_matrix())
    trans = torch.tensor([4.0, -2.0, 7.5], dtype=torch.float64)
    pivot = torch.tensor([10.0, 20.0, 30.0], dtype=torch.float64)
    delta = torch.tensor([0.5, -1.0, 2.0, 0.02, -0.04, 0.01], dtype=torch.float64)
    r2, t2 = compose_sweep_twist(rot, trans, delta, pivot)
    w = Rotation.from_rotvec(delta[3:].numpy())
    np.testing.assert_allclose(r2.numpy(), (w * Rotation.from_matrix(rot.numpy())).as_matrix(), rtol=0, atol=1e-15)
    np.testing.assert_allclose(t2.numpy(), pivot.numpy() + delta[:3].numpy() + w.apply(trans.numpy() - pivot.numpy()), rtol=1e-14)
    # the composed transform on points = the twist about the pivot after the first transform
    x = torch.randn((5, 3), generator=g, dtype=torch.float64) * 20
    m, h = torch.randn((5, 3), generator=g, dtype=torch.float64), torch.randn((5, 3), generator=g, dtype=torch.float64)
    s1, m1, h1 = apply_rigid_transform(rot, trans, x, m, h)
    s2, m2, h2 = apply_rigid_transform(r2, t2, x, m, h)
    np.testing.assert_allclose(s2.numpy(), pivot.numpy() + delta[:3].numpy() + w.apply((s1 - pivot).numpy()), rtol=1e-14, atol=1e-12)
    np.testing.assert_allclose(m2.numpy(), w.apply(m1.numpy()), rtol=1e-14, atol=1e-14)
    np.testing.assert_allclose(h2.numpy(), w.apply(h1.numpy()), rtol=1e-14, atol=1e-14)
    # the identity transform returns the float32 start poses exactly once rounded
    eye, zero = torch.eye(3, dtype=torch.float64), torch.zeros(3, dtype=torch.float64)
    xf = x.float()
    assert torch.equal(apply_rigid_transform(eye, zero, xf, xf, xf)[0].float(), xf)
    # fans of transformed parameters are the transformed fans (rigidity of the fan generator)
    from diffus_b200.phantoms import fan_directions
    fan = fan_directions(m.float(), h.float(), math.radians(60), 7).double().reshape(-1, 3)
    got = fan_directions(m2.float(), h2.float(), math.radians(60), 7).double().reshape(-1, 3)
    np.testing.assert_allclose(got.numpy(), Rotation.from_matrix(r2.numpy()).apply(fan.numpy()), atol=3e-7)


def test_host_argument_checks():
    from diffus_b200 import register_sweep, render_gauss_newton_sweep
    from diffus_b200._lib import DiffusError
    P, R, S = 2, 4, 30
    vol = torch.zeros((8, 8, 8))
    src, dirs = torch.zeros((P, 3)), torch.zeros((P, R, 3))
    tgt = torch.zeros((P, R, S))
    with pytest.raises(DiffusError, match="float32"):
        render_gauss_newton_sweep(vol, src.double(), dirs, tgt, S)
    with pytest.raises(DiffusError, match="target"):
        render_gauss_newton_sweep(vol, src, dirs, tgt[:, :, 1:], S)
    with pytest.raises(DiffusError, match="target"):
        render_gauss_newton_sweep(vol, src, dirs, tgt, S, start=3)
    with pytest.raises(DiffusError, match="pivot"):
        render_gauss_newton_sweep(vol, src, dirs, tgt, S, pivot=torch.zeros(3))
    with pytest.raises(DiffusError, match="pivot"):
        render_gauss_newton_sweep(vol, src, dirs, tgt, S, pivot=torch.zeros((1, 3), dtype=torch.float64))
    med, hint = torch.zeros((P, 3)), torch.zeros((P, 3))
    with pytest.raises(ValueError, match="probe"):
        register_sweep(vol, tgt, src, med, hint, 1.0, R, S, probe="phased")
    with pytest.raises(ValueError, match="radius"):
        register_sweep(vol, tgt, src, med, hint, 1.0, R, S, radius=3.0)
    with pytest.raises(ValueError, match="width"):
        register_sweep(vol, tgt, src, med, hint, 1.0, R, S, probe="linear")
    with pytest.raises(ValueError, match="float32"):
        register_sweep(vol, tgt, src.double(), med, hint, 1.0, R, S)
    with pytest.raises(ValueError, match="targets"):
        register_sweep(vol, tgt, src, med, hint, 1.0, R + 1, S)
    with pytest.raises(ValueError, match=r"\(P,3\)"):
        register_sweep(vol, tgt, src, med[:1], hint, 1.0, R, S)


@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()                       # nvcc cross-compiles without a GPU
    return _lib.load()


def test_sweep_struct_layout_matches_header(lib):
    from diffus_b200._lib import DiffusGaussNewtonSweepArgs
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef struct DiffusGaussNewtonSweepArgs \{(.*?)\} DiffusGaussNewtonSweepArgs;", text, flags=re.S).group(1)
    fields = [re.split(r"[\s\*]+", f.strip())[-1] for f in body.split(";") if f.strip()]
    assert fields == [f[0] for f in DiffusGaussNewtonSweepArgs._fields_]


def test_sweep_argument_validation_without_a_device(lib):
    from diffus_b200._lib import DiffusGaussNewtonSweepArgs
    g = DiffusGaussNewtonSweepArgs()
    assert lib.diffus_render_gauss_newton_sweep(None, None) == -1
    assert lib.diffus_render_gauss_newton_sweep_workspace_bytes(None) == 0
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -1        # NULL volume
    a = g.fwd
    a.volume.data = 0x1000
    a.volume.dim[0] = a.volume.dim[1] = a.volume.dim[2] = 8
    a.sources = a.directions = 0x1000
    a.n_poses, a.n_rays, a.n_samples, a.sampler = 2, 4, 16, 1
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -1        # NULL target / outputs
    g.target, g.loss, g.jtr = 0x1000, 0x2000, 0x3000
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -1        # NULL jtj
    g.jtj = 0x4000
    a.sampler = 0
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -5        # nearest: no pose derivative
    a.sampler, a.pose_dtype = 1, 1
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -5        # float64 poses
    a.pose_dtype = 3
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -3        # unknown pose dtype
    a.pose_dtype = 0
    need = lib.diffus_render_gauss_newton_sweep_workspace_bytes(C.byref(g))
    assert need >= 2 * 4 * 32 * 4
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -4        # no workspace
    g.pivot = 0x6000
    assert lib.diffus_render_gauss_newton_sweep_workspace_bytes(C.byref(g)) < need   # no room for the mean of the origins
    g.pivot = None
    a.start = 3
    assert lib.diffus_render_gauss_newton_sweep_workspace_bytes(C.byref(g)) > need   # median, ties and its tangent
    g.workspace, g.workspace_bytes = 0x5000, need
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -4        # too small for start > 0
    a.start = 15
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -2        # start > S-2
    a.start, a.n_rays = 0, 0
    assert lib.diffus_render_gauss_newton_sweep(C.byref(g), None) == -2        # no rays
