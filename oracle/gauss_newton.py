"""Gauss-Newton system of each pose's frame residual w.r.t. a rigid twist of the pose.  TEST INFRASTRUCTURE ONLY.

Built on :mod:`oracle.port` without restating the kernel's formulas: the Jacobian is taken by torch forward-mode autograd
through the port's ``plot_beam_frame`` (trilinear sampler, ``src/renderer.py:201-275``) of the pose moved by
``diffus_b200.pose_recovery.apply_pose_twist``.  Runs in the dtype of the volume (fp64 for the reference value, fp32 to measure
the algorithm's own float32 drift).
"""
from __future__ import annotations

import torch

from . import port


def pose_gauss_newton(volume, sources, directions, target, num_samples, attenuation_coeff=0.5, start=0):
    """Gauss-Newton system of each pose's frame residual w.r.t. a rigid twist ``xi = (v, w)`` of the pose, in the dtype of
    ``volume``: ``J = d frame / d xi`` at ``xi = 0`` by torch forward-mode autograd through :func:`oracle.port.plot_beam_frame`
    (``sampler='trilinear'``, ``src/renderer.py:201-275``) of the pose moved by ``diffus_b200.pose_recovery.apply_pose_twist``;
    ``res = frame - target``.  Returns ``loss (P,) = sum res^2``, ``JtJ (P,6,6)``, ``Jtr (P,6)`` and the frames (P,R,S-start)."""
    import torch.autograd.forward_ad as fwAD
    from diffus_b200.pose_recovery import apply_pose_twist
    dt = volume.dtype
    eye = torch.eye(6, dtype=dt)
    losses, jtjs, jtrs, frames = [], [], [], []
    for p in range(sources.shape[0]):
        src = sources[p:p + 1].to(dt)
        dirs = (directions[p] if directions.dim() == 3 else directions).to(dt).unsqueeze(0)
        cols = []
        for j in range(6):
            with fwAD.dual_level():
                xi = fwAD.make_dual(torch.zeros((1, 6), dtype=dt), eye[j:j + 1])
                s2, d2 = apply_pose_twist(src, dirs, xi)
                f = port.plot_beam_frame(volume, s2[0], d2[0], num_samples, attenuation_coeff, start=start, sampler="trilinear")[3]
                f, t = fwAD.unpack_dual(f)
            cols.append(t.reshape(-1))
        J = torch.stack(cols, dim=-1)
        res = f.reshape(-1) - target[p].reshape(-1).to(f.dtype)
        losses.append((res * res).sum())
        jtjs.append(J.T @ J)
        jtrs.append(J.T @ res)
        frames.append(f)
    return torch.stack(losses), torch.stack(jtjs), torch.stack(jtrs), torch.stack(frames)

