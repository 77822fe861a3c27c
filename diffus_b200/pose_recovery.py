"""Pose recovery by Levenberg-Marquardt on the Gauss-Newton systems of :func:`render_gauss_newton`.

A pose update is the rigid twist ``xi = (v, w)`` about the current pose, rotating about the source:
``p_k(xi) = (s + v) + k Rot(w) d_i``.  :func:`apply_pose_twist` applies it to explicit sources / directions and
:func:`apply_fan_twist` to the pose parameters of a fan (source, median direction, in-plane hint), which the fan generator
turns back into the rotated fan.  Array probes (one origin per ray, :func:`diffus_b200.probe_rays`) turn about their PIVOT
``c``, the float64 mean of a pose's origins: ``p_k(xi) = c + v + Rot(w) (s_i - c + k d_i)``; :func:`apply_pose_twist` takes their
(P,R,3) origins and :func:`apply_probe_twist` their parameters.  The functions are plain torch and run on any device (the test
oracle differentiates them on the CPU).

A tracked sweep knows the relative poses of its frames; what is unknown is one rigid transform ``x' = R x + t`` between the
tracker and the volume.  :func:`register_sweep` fits it by Levenberg-Marquardt on ONE Gauss-Newton system of all frames
(:func:`diffus_b200.render_gauss_newton_sweep`), with the twist taken about the image of the start sweep's origin centroid
(:func:`compose_sweep_twist`, :func:`apply_rigid_transform`).
"""
from __future__ import annotations

import math
import numbers

import torch

from .renderer import PreparedVolume, _resolve_start, smooth_volume


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


def probe_pivot(origins: torch.Tensor) -> torch.Tensor:
    """The pivot of array-probe poses: the float64 mean of each pose's (P,R,3) origins -> (P,3) float64."""
    return origins.to(torch.float64).mean(-2)


def apply_pose_twist(sources: torch.Tensor, directions: torch.Tensor, delta: torch.Tensor):
    """``(sources + v, Rot(w) directions)`` for ``delta`` (P,6) = (v, w): sources (P,3), directions (P,R,3) or a shared (R,3)
    fan, which becomes (P,R,3).  Per-ray sources (P,R,3) turn about their pivot ``c`` (:func:`probe_pivot`):
    ``c + v + Rot(w) (s_i - c)``, evaluated in float64 and returned in the sources' dtype."""
    v, w = delta[..., :3], delta[..., 3:]
    dirs = directions if directions.dim() == 3 else directions.unsqueeze(0).expand(sources.shape[0], -1, -1)
    if sources.dim() == 3:
        c = probe_pivot(sources).unsqueeze(-2)
        s = c + v.unsqueeze(-2).to(torch.float64) + _rotate(sources.to(torch.float64) - c, w.unsqueeze(-2).to(torch.float64))
        return s.to(sources.dtype), _rotate(dirs, w.unsqueeze(-2))
    return sources + v, _rotate(dirs, w.unsqueeze(-2))


def apply_fan_twist(sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, delta: torch.Tensor):
    """The same twist on fan parameters: ``(sources + v, Rot(w) median, Rot(w) hint)``, all (P,3).  The fan of the rotated
    parameters is the rotated fan (:func:`diffus_b200.fan_directions` is rotation-equivariant)."""
    v, w = delta[..., :3], delta[..., 3:]
    return sources + v, _rotate(median, w), _rotate(hint, w)


def apply_probe_twist(centre: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, delta: torch.Tensor, pivot: torch.Tensor):
    """The twist about ``pivot`` (P,3) on array-probe parameters: ``(pivot + v + Rot(w) (centre - pivot), Rot(w) median,
    Rot(w) hint)``.  The rays of the twisted parameters are the twisted rays (:func:`diffus_b200.probe_rays` places the origins
    rigidly in the frame of median and hint), so with the pivot of the current origins this is :func:`apply_pose_twist` on
    them.  The centre is formed in float64 and returned in its own dtype."""
    v, w = delta[..., :3], delta[..., 3:]
    c = pivot.to(torch.float64)
    centre2 = (c + v.to(torch.float64) + _rotate(centre.to(torch.float64) - c, w.to(torch.float64))).to(centre.dtype)
    return centre2, _rotate(median, w), _rotate(hint, w)


def rotation_matrix(w: torch.Tensor) -> torch.Tensor:
    """``Rot(w)`` (3,3) of one rotation vector ``w`` (3,), by :func:`_rotate` on the unit vectors (elementwise only, so it records
    into a CUDA graph)."""
    eye = torch.eye(3, dtype=w.dtype, device=w.device)
    return _rotate(eye, w.reshape(1, 3)).transpose(0, 1)


def _mat_vec(m: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """``m @ x`` for a (3,3) matrix and (..., 3) vectors, elementwise (no library GEMM inside the graphed step)."""
    return (m * x.unsqueeze(-2)).sum(-1)


def compose_sweep_twist(rot: torch.Tensor, trans: torch.Tensor, delta: torch.Tensor, pivot: torch.Tensor):
    """The transform ``x -> c + v + Rot(w) (R x + t - c)`` of the twist ``delta`` (6,) = (v, w) about ``pivot`` c (3,) after
    ``x -> R x + t``: returns ``(Rot(w) R, c + v + Rot(w) (t - c))``, in the dtype of ``rot``."""
    delta = delta.to(rot.dtype)
    c = pivot.to(rot.dtype)
    w = rotation_matrix(delta[3:])
    return (w.unsqueeze(-1) * rot.unsqueeze(0)).sum(1), c + delta[:3] + _mat_vec(w, trans - c)


def apply_rigid_transform(rot: torch.Tensor, trans: torch.Tensor, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor):
    """``(R s + t, R m, R h)`` on pose parameters (P,3) each, in the dtype of ``rot``: the points move, the two orientation
    vectors turn."""
    f = rot.dtype
    return _mat_vec(rot, sources.to(f)) + trans, _mat_vec(rot, median.to(f)), _mat_vec(rot, hint.to(f))


PROBES = ("sector", "convex", "linear")


def probe_keywords(probe: str, radius, width):
    """Validated ``(probe, radius, width)`` of the pose-recovery drivers (host only): ``'sector'`` takes neither keyword,
    ``'convex'`` a finite radius >= 0 and ``'linear'`` a finite width > 0."""
    if probe not in PROBES:
        raise ValueError(f"probe must be one of {PROBES}, got {probe!r}")
    if probe == "sector":
        if radius not in (None, 0, 0.0) or width is not None:
            raise ValueError("radius and width only apply to probe='convex' and probe='linear'")
        return probe, 0.0, None
    if probe == "convex":
        if width is not None:
            raise ValueError("a convex probe takes radius, not width")
        rho = 0.0 if radius is None else float(radius)
        if not (math.isfinite(rho) and rho >= 0.0):
            raise ValueError(f"a convex probe needs a finite radius >= 0, got {radius!r}")
        return probe, rho, None
    if radius not in (None, 0, 0.0):
        raise ValueError("a linear probe takes width, not radius")
    if width is None or not (math.isfinite(float(width)) and float(width) > 0.0):
        raise ValueError(f"a linear probe needs a finite width > 0, got {width!r}")
    return probe, 0.0, float(width)


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
                  iterations: int = 10, damping: float = 1e-3, *, probe: str = "sector", radius=None, width=None):
    """Levenberg-Marquardt pose recovery of a batch of fans against their target frames.

    Each pose solves ``(JtJ + lam diag(JtJ) + eps I) delta = -Jtr`` (float64, Marquardt scaling), renders the candidate
    pose's Gauss-Newton system, and keeps the candidate only if its own loss went down (``lam`` shrinks) -- else it stays put
    and ``lam`` grows.  Every pose's loss therefore never increases.  One iteration is one CUDA-graph replay
    (:class:`diffus_b200.graphs.GraphedFanGaussNewtonStep`); nothing leaves the device until the loop ends.

    ``targets`` (P,R,S-start), ``sources`` / ``median`` / ``hint`` (P,3) float32 start poses.  Returns
    ``((sources, median, hint), history)`` with ``history`` the (iterations + 1, P) loss ``sum (frame - target)^2`` of each
    pose before the first and after every iteration.

    ``probe='convex'`` (``radius``) or ``'linear'`` (``width``; ``opening_angle`` is then unused) recovers array probes
    instead: ``sources`` are their centres and the rays come from :func:`diffus_b200.probe_rays`; the twist turns each probe
    about its pivot (:func:`apply_probe_twist`).  The default ``'sector'`` is the point-source fan.
    """
    probe, radius, width = probe_keywords(probe, radius, width)
    from .graphs import GraphedFanGaussNewtonStep
    step = GraphedFanGaussNewtonStep(volume, targets, n_rays, num_samples, opening_angle, attenuation_coeff, start, probe=probe,
                                     radius=radius, width=width)
    step.reset(sources, median, hint, damping)
    history = torch.empty((iterations + 1, step.P), dtype=torch.float32, device=step.loss.device)
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
                                 sigmas=(4.0, 2.0, 1.0, 0.0), iterations=10, damping: float = 1e-3, layout=None,
                                 probe: str = "sector", radius=None, width=None):
    """Levenberg-Marquardt pose recovery from a blurred volume to the sharp one (a Gaussian scale space).

    On a volume with sharp tissue boundaries the frame depends on the pose through one-voxel gradient cells, so a Gauss-Newton
    step is only valid within about a voxel.  Level l renders from ``smooth_volume(volume, sigmas[l])`` instead, where the
    basin of the true pose is about sigma wide, and starts from the previous level's poses; the target frames stay as they
    are.  A sigma of 0 uses ``volume`` as given.  Each level is :func:`recover_poses` with ``iterations`` (an int, or one per
    level) and a fresh ``damping``; its first history row is the incoming poses' loss on that level's own volume, so no
    accept / reject compares losses across volumes.  ``layout`` of the blurred levels' :class:`PreparedVolume` defaults to the
    caller's layout, else ``'texture'``; each level's copy is released before the next is built.

    ``probe``, ``radius`` and ``width`` select the probe as in :func:`recover_poses`.

    Returns ``((sources, median, hint), histories)``: one (iterations_l + 1, P) loss history per level.
    """
    sig, its = _schedule(sigmas, iterations)
    probe, radius, width = probe_keywords(probe, radius, width)
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
                                    iterations=k, damping=damping, probe=probe, radius=radius, width=width)
        histories.append(hist)
        if level is not volume:
            level.close()
        del level
    return poses, histories


def register_sweep(volume, targets: torch.Tensor, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor,
                   opening_angle: float, n_rays: int, num_samples: int, attenuation_coeff: float = 0.5, start=0,
                   iterations: int = 10, damping: float = 1e-3, *, probe: str = "sector", radius=None, width=None):
    """Levenberg-Marquardt registration of a whole tracked sweep: ONE rigid transform for every frame.

    The relative poses of the frames (``sources``, ``median``, ``hint``, (P,3) float32: the start sweep) are kept; the transform
    ``x' = R x + t`` applied to all of them is fitted to the target frames ``targets`` (P, n_rays, S-start).  Each iteration solves
    ``(JtJ + lam diag(JtJ) + eps I) delta = -Jtr`` (float64, Marquardt scaling) on the sweep's one system
    (:func:`diffus_b200.render_gauss_newton_sweep`), with the twist about the image of the start sweep's origin centroid under
    the current transform; composes the candidate transform in float64 (:func:`compose_sweep_twist`); applies it to the START
    poses in float64, rounded to float32 once (:func:`apply_rigid_transform`: no rounding accumulates from step to step); renders
    the candidate's system and keeps it only if the total loss went down (``lam`` shrinks), else stays and raises ``lam``.  One
    iteration is one CUDA-graph replay (:class:`diffus_b200.graphs.GraphedSweepGaussNewtonStep`).

    ``probe``, ``radius`` and ``width`` select the probe as in :func:`recover_poses`.  Returns ``((R (3,3), t (3,)),
    (sources, median, hint), history)``: the float64 transform mapping the start sweep onto the registered one, the registered
    poses, and the float64 (iterations + 1,) total loss ``sum (frame - target)^2`` before the first and after every iteration.
    """
    probe, radius, width = probe_keywords(probe, radius, width)
    poses = (sources, median, hint)
    if any(not isinstance(x, torch.Tensor) or x.dim() != 2 or x.shape[-1] != 3 or x.shape[0] != sources.shape[0] for x in poses):
        raise ValueError("sources, median and hint must all be (P,3) tensors")
    if any(x.dtype != torch.float32 for x in poses):
        raise ValueError("register_sweep takes float32 poses (the transform itself is float64)")
    want = (sources.shape[0], int(n_rays), int(num_samples) - _resolve_start(start, num_samples))
    if tuple(targets.shape) != want:
        raise ValueError(f"targets must be {want} (poses, rays, samples after the crop), got {tuple(targets.shape)}")
    from .graphs import GraphedSweepGaussNewtonStep
    step = GraphedSweepGaussNewtonStep(volume, targets, n_rays, num_samples, opening_angle, attenuation_coeff, start, probe=probe,
                                       radius=radius, width=width)
    step.reset(sources, median, hint, damping)
    history = torch.empty((iterations + 1,), dtype=torch.float64, device=step.loss.device)
    history[0].copy_(step.loss)
    for i in range(iterations):
        step()
        history[i + 1].copy_(step.loss)
    return (step.rot.clone(), step.trans.clone()), (step.sources.clone(), step.median.clone(), step.hint.clone()), history
