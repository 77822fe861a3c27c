"""Pose recovery by Levenberg-Marquardt on the Gauss-Newton systems of :func:`render_gauss_newton`.

A pose update is the rigid twist ``xi = (v, w)`` about the current pose, rotating about the source:
``p_k(xi) = (s + v) + k Rot(w) d_i``.  :func:`apply_pose_twist` applies it to explicit sources / directions and
:func:`apply_fan_twist` to the pose parameters of a fan (source, median direction, in-plane hint), which the fan generator
turns back into the rotated fan.  The functions are plain torch and run on any device (the test oracle differentiates them on
the CPU).
"""
from __future__ import annotations

import math
import numbers

import torch

from .renderer import PreparedVolume, smooth_volume


def _rotate(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Rodrigues rotation of the vectors ``x`` (..., 3) by the rotation vectors ``w`` (broadcast against ``x``), smooth at
    ``w = 0`` (series below 1e-4 rad), so forward- and reverse-mode derivatives there are exact."""
    w = w.expand_as(x)
    th2 = (w * w).sum(-1, keepdim=True)
    small = th2 < 1e-8
    th2s = torch.where(small, torch.ones_like(th2), th2)
    th = torch.sqrt(th2s)
    a = torch.where(small, 1.0 - th2 / 6.0, torch.sin(th) / th)
    b = torch.where(small, 0.5 - th2 / 24.0, (1.0 - torch.cos(th)) / th2s)
    wx = torch.linalg.cross(w, x, dim=-1)
    return x + a * wx + b * torch.linalg.cross(w, wx, dim=-1)


def apply_pose_twist(sources: torch.Tensor, directions: torch.Tensor, delta: torch.Tensor):
    """``(sources + v, Rot(w) directions)`` for ``delta`` (P,6) = (v, w): sources (P,3), directions (P,R,3) or a shared (R,3)
    fan, which becomes (P,R,3)."""
    v, w = delta[..., :3], delta[..., 3:]
    dirs = directions if directions.dim() == 3 else directions.unsqueeze(0).expand(sources.shape[0], -1, -1)
    return sources + v, _rotate(dirs, w.unsqueeze(-2))


def apply_fan_twist(sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, delta: torch.Tensor):
    """The same twist on fan parameters: ``(sources + v, Rot(w) median, Rot(w) hint)``, all (P,3).  The fan of the rotated
    parameters is the rotated fan (:func:`diffus_b200.fan_directions` is rotation-equivariant)."""
    v, w = delta[..., :3], delta[..., 3:]
    return sources + v, _rotate(median, w), _rotate(hint, w)


def fan_frame_angle(median_a, hint_a, median_b, hint_b) -> torch.Tensor:
    """Angle (radians, per pose) of the rotation between the orthonormal frames (m^, u^, m^ x u^) of two fans."""
    def frame(m, h):
        m = m.double() / m.double().norm(dim=-1, keepdim=True)
        u = h.double() - (h.double() * m).sum(-1, keepdim=True) * m
        u = u / u.norm(dim=-1, keepdim=True)
        return torch.stack([m, u, torch.linalg.cross(m, u, dim=-1)], dim=-1)
    r = frame(median_a, hint_a) @ frame(median_b, hint_b).transpose(-1, -2)
    c = ((r.diagonal(dim1=-2, dim2=-1).sum(-1) - 1.0) / 2.0).clamp(-1.0, 1.0)
    return torch.arccos(c)


def recover_poses(volume, targets: torch.Tensor, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor,
                  opening_angle: float, n_rays: int, num_samples: int, attenuation_coeff: float = 0.5, start=0,
                  iterations: int = 10, damping: float = 1e-3):
    """Levenberg-Marquardt pose recovery of a batch of fans against their target frames.

    Each pose solves ``(JtJ + lam diag(JtJ) + eps I) delta = -Jtr`` (float64, Marquardt scaling), renders the candidate
    pose's Gauss-Newton system, and keeps the candidate only if its own loss went down (``lam`` shrinks) -- else it stays put
    and ``lam`` grows.  Every pose's loss therefore never increases.  One iteration is one CUDA-graph replay
    (:class:`diffus_b200.graphs.GraphedFanGaussNewtonStep`); nothing leaves the device until the loop ends.

    ``targets`` (P,R,S-start), ``sources`` / ``median`` / ``hint`` (P,3) float32 start poses.  Returns
    ``((sources, median, hint), history)`` with ``history`` the (iterations + 1, P) loss ``sum (frame - target)^2`` of each
    pose before the first and after every iteration.
    """
    from .graphs import GraphedFanGaussNewtonStep
    step = GraphedFanGaussNewtonStep(volume, targets, n_rays, num_samples, opening_angle, attenuation_coeff, start)
    step.reset(sources, median, hint, damping)
    vol = volume.volume if isinstance(volume, PreparedVolume) else volume
    history = torch.empty((iterations + 1, step.P), dtype=torch.float32, device=vol.device)
    history[0].copy_(step.loss)
    for i in range(iterations):
        step()
        history[i + 1].copy_(step.loss)
    return (step.sources.clone(), step.median.clone(), step.hint.clone()), history


def _schedule(sigmas, iterations):
    """Validated ``(sigmas, iterations)`` lists of one coarse-to-fine schedule (host only)."""
    sig = [float(s) for s in sigmas]
    if not sig or not all(math.isfinite(s) and s >= 0.0 for s in sig):
        raise ValueError(f"sigmas must be a non-empty sequence of finite values >= 0, got {tuple(sigmas)!r}")
    its = [iterations] * len(sig) if isinstance(iterations, numbers.Integral) else list(iterations)
    if len(its) != len(sig):
        raise ValueError(f"iterations must be an int or one per level ({len(sig)}), got {len(its)}")
    if not all(isinstance(k, numbers.Integral) and not isinstance(k, bool) and k >= 0 for k in its):
        raise ValueError(f"iterations must be non-negative ints, got {its!r}")
    return sig, [int(k) for k in its]


def recover_poses_coarse_to_fine(volume, targets: torch.Tensor, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor,
                                 opening_angle: float, n_rays: int, num_samples: int, attenuation_coeff: float = 0.5, start=0, *,
                                 sigmas=(4.0, 2.0, 1.0, 0.0), iterations=10, damping: float = 1e-3, layout=None):
    """Levenberg-Marquardt pose recovery from a blurred volume to the sharp one (a Gaussian scale space).

    On a volume with sharp tissue boundaries the frame depends on the pose through one-voxel gradient cells, so a Gauss-Newton
    step is only valid within about a voxel.  Level l renders from ``smooth_volume(volume, sigmas[l])`` instead, where the
    basin of the true pose is about sigma wide, and starts from the previous level's poses; the target frames stay as they
    are.  A sigma of 0 uses ``volume`` as given.  Each level is :func:`recover_poses` with ``iterations`` (an int, or one per
    level) and a fresh ``damping``; its first history row is the incoming poses' loss on that level's own volume, so no
    accept / reject compares losses across volumes.  ``layout`` of the blurred levels' :class:`PreparedVolume` defaults to the
    caller's layout, else ``'texture'``; each level's copy is released before the next is built.

    Returns ``((sources, median, hint), histories)``: one (iterations_l + 1, P) loss history per level.
    """
    sig, its = _schedule(sigmas, iterations)
    if layout is None:
        layout = volume.layout if isinstance(volume, PreparedVolume) else "texture"
    base = volume.volume if isinstance(volume, PreparedVolume) else volume
    poses, histories = (sources, median, hint), []
    for sigma, k in zip(sig, its):
        if sigma == 0.0:
            level = volume
        else:
            with torch.no_grad():
                level = PreparedVolume(smooth_volume(base, sigma), layout)
        poses, hist = recover_poses(level, targets, *poses, opening_angle, n_rays, num_samples, attenuation_coeff, start,
                                    iterations=k, damping=damping)
        histories.append(hist)
        if level is not volume:
            level.close()
        del level
    return poses, histories
