"""GPU: coarse-to-fine pose recovery (``recover_poses_coarse_to_fine``): its one-level case is ``recover_poses``, and no level
compares losses across volumes."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

N, P, R, S, ALPHA, ANGLE = 64, 32, 32, 96, 5e-3, math.radians(60.0)


def dev():
    return torch.device("cuda:0")


def sharp_scene(vox, deg):
    """The MRI-shaped phantom (sharp tissue boundaries, 2 % voxel noise) at 64^3 on the geometry of
    test_gpu_gauss_newton.py's Levenberg-Marquardt test; start poses a twist of `vox` voxels and `deg` degrees off."""
    from diffus_b200 import PreparedVolume, fan_directions, render_frames
    from diffus_b200.phantoms import intensity_to_impedance, mri_phantom, pose_sweep
    from diffus_b200.pose_recovery import apply_fan_twist
    vol = PreparedVolume(intensity_to_impedance(mri_phantom(N)).to(dev()), "texture")
    src, _, med, hint = pose_sweep(P, n_rays=R, n=N, seed=8, return_params=True)
    src, med, hint = src.to(dev()), med.to(dev()), hint.to(dev())
    with torch.no_grad():
        targets = render_frames(vol, src, fan_directions(med, hint, ANGLE, R), S, ALPHA, sampler="trilinear")
    g = torch.Generator().manual_seed(0)
    u = torch.randn((P, 6), generator=g)
    u[:, :3] = u[:, :3] / u[:, :3].norm(dim=-1, keepdim=True) * vox
    u[:, 3:] = u[:, 3:] / u[:, 3:].norm(dim=-1, keepdim=True) * math.radians(deg)
    return vol, targets, (src, med, hint), apply_fan_twist(src, med, hint, u.to(dev()))


def test_one_sharp_level_is_recover_poses():
    from diffus_b200 import recover_poses, recover_poses_coarse_to_fine
    vol, targets, _, start = sharp_scene(1.0, 1.0)
    a, ha = recover_poses(vol, targets, *start, ANGLE, R, S, ALPHA, iterations=4)
    b, hb = recover_poses_coarse_to_fine(vol, targets, *start, ANGLE, R, S, ALPHA, sigmas=(0.0,), iterations=4)
    assert len(hb) == 1 and torch.equal(hb[0], ha)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_each_level_starts_from_its_own_volumes_loss():
    """Every level's history is non-increasing, and its first row is the previous level's final poses evaluated on THIS
    level's volume -- never a loss carried over from another volume."""
    from diffus_b200 import (PreparedVolume, fan_directions, recover_poses_coarse_to_fine, render_gauss_newton,
                             smooth_volume)
    vol, targets, _, start = sharp_scene(2.0, 2.0)
    sigmas, iters = (3.0, 1.5, 0.0), (4, 3, 2)
    poses, hist = recover_poses_coarse_to_fine(vol, targets, *start, ANGLE, R, S, ALPHA, sigmas=sigmas, iterations=iters)
    assert [tuple(h.shape) for h in hist] == [(k + 1, P) for k in iters]
    for h in hist:
        assert (h[1:] <= h[:-1]).all(), "the accept / reject rule never lets a pose's loss grow within a level"
    for lvl in range(len(sigmas) - 1):
        (s, m, h), _ = recover_poses_coarse_to_fine(vol, targets, *start, ANGLE, R, S, ALPHA, sigmas=sigmas[:lvl + 1],
                                                     iterations=iters[:lvl + 1])
        nxt = sigmas[lvl + 1]
        level = vol if nxt == 0.0 else PreparedVolume(smooth_volume(vol, nxt), "texture")
        loss, _, _ = render_gauss_newton(level, s, fan_directions(m, h, ANGLE, R), targets, S, ALPHA)
        assert torch.equal(hist[lvl + 1][0], loss), lvl
        assert not torch.equal(hist[lvl + 1][0], hist[lvl][-1])              # the volumes differ, so do the losses
    assert all(torch.equal(x, y) for x, y in zip(poses, recover_poses_coarse_to_fine(
        vol, targets, *start, ANGLE, R, S, ALPHA, sigmas=sigmas, iterations=iters)[0]))

