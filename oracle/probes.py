"""Linear and convex array probes in float64.  TEST INFRASTRUCTURE ONLY.

A restatement of ``diffus_probe_rays`` (``include/diffus_b200.h``) from pose parameters (centre, median, hint), each (P,3):
``m^ = median / |median|``, ``u^`` = the hint made orthogonal to ``m^`` and normalised, ray parameters spread over
``[-x/2, x/2]`` as ``lo + i * step`` with the last one pinned to ``x/2`` (numpy.linspace's rule, also the fans').

* convex (opening angle, radius rho): ``d_i = cos a_i m^ + sin a_i u^``, ``origin_i = centre + rho d_i``;
* linear (width w): ``d_i = m^``, ``origin_i = centre + t_i u^``.

Differentiable with torch autograd; returns float64 (P,R,3) origins and directions.

Rendering from one origin per ray: :func:`ray_points`, :func:`plot_beam_frame` and :func:`pose_gauss_newton` are
:mod:`oracle.port`'s ``ray_points`` / ``plot_beam_frame`` and :mod:`oracle.gauss_newton`'s ``pose_gauss_newton`` with (R,3)
origins in place of the one source -- the same samplers, reflection, median rule, echo and attenuation, taken from the port.
"""
from __future__ import annotations

import torch

from . import port


def frame(median: torch.Tensor, hint: torch.Tensor):
    m = median.double()
    m = m / m.norm(dim=-1, keepdim=True)
    h = hint.double()
    u = h - (h * m).sum(-1, keepdim=True) * m
    return m, u / u.norm(dim=-1, keepdim=True)


def spread(extent: float, n: int) -> torch.Tensor:
    lo, hi = -extent / 2, extent / 2
    if n == 1:
        return torch.tensor([lo], dtype=torch.float64)
    step = (hi - lo) / (n - 1)
    t = torch.arange(n, dtype=torch.float64) * step + lo
    t[-1] = hi
    return t


def convex_rays(centre, median, hint, opening_angle: float, n_rays: int, radius: float):
    m, u = frame(median, hint)
    a = spread(opening_angle, n_rays).view(1, -1, 1)
    d = torch.cos(a) * m.unsqueeze(1) + torch.sin(a) * u.unsqueeze(1)
    return centre.double().unsqueeze(1) + radius * d, d


def linear_rays(centre, median, hint, width: float, n_rays: int):
    m, u = frame(median, hint)
    t = spread(width, n_rays).view(1, -1, 1)
    o = centre.double().unsqueeze(1) + t * u.unsqueeze(1)
    return o, m.unsqueeze(1).expand(-1, n_rays, -1)


def probe_rays(kind: str, centre, median, hint, n_rays: int, opening_angle=None, radius: float = 0.0, width=None):
    if kind == "convex":
        return convex_rays(centre, median, hint, opening_angle, n_rays, radius)
    if kind == "linear":
        return linear_rays(centre, median, hint, width, n_rays)
    raise ValueError(kind)


def ray_points(origins: torch.Tensor, directions: torch.Tensor, num_samples: int) -> torch.Tensor:
    """``points[r, k] = origins[r] + k * directions[r]``: :func:`oracle.port.ray_points` (float32 steps, separate roundings,
    torch promotion) with one origin per ray."""
    steps = torch.arange(0, num_samples, dtype=torch.float32).view(1, -1, 1)
    return origins.unsqueeze(1) + steps * directions.unsqueeze(1)


def plot_beam_frame(volume, origins, directions, num_samples, attenuation_coeff=0.5, start=0, sampler="nearest"):
    """:func:`oracle.port.plot_beam_frame` (closed-form echo) for (R,3) ``origins``, one per ray of ``directions`` (R,3)."""
    pts = ray_points(origins, directions, num_samples)
    if sampler == "nearest":
        x, y, z, imp = port.sample_nearest(volume, pts)
    elif sampler == "trilinear":
        x, y, z, imp = port.sample_trilinear(volume, pts)
    else:
        raise ValueError(sampler)
    r = port.reflection_coeff(imp[:, :-1], imp[:, 1:])
    start = port.resolve_start(start, num_samples)
    if start > 0:
        r = r[:, start:]
        med = r[:, 0].median()
        r = torch.cat([med.expand(r.shape[0], 1), r[:, 1:]], dim=1)
    echo = port.echo_closed_form(r)
    att = torch.exp(-attenuation_coeff * torch.arange(echo.shape[1]).float())
    return x[:, start:], y[:, start:], z[:, start:], echo * att[None, :]


def pose_gauss_newton(volume, origins, directions, target, num_samples, attenuation_coeff=0.5, start=0):
    """:func:`oracle.gauss_newton.pose_gauss_newton` for (P,R,3) origins: ``J = d frame / d xi`` at ``xi = 0`` by forward-mode
    autograd through :func:`plot_beam_frame` (trilinear) of the rays moved by ``diffus_b200.pose_recovery.apply_pose_twist``,
    which turns per-ray origins about their pivot.  Returns ``loss (P,)``, ``JtJ (P,6,6)``, ``Jtr (P,6)`` and the frames."""
    import torch.autograd.forward_ad as fwAD
    from diffus_b200.pose_recovery import apply_pose_twist
    dt = volume.dtype
    eye = torch.eye(6, dtype=dt)
    losses, jtjs, jtrs, frames = [], [], [], []
    for p in range(origins.shape[0]):
        org = origins[p:p + 1].to(dt)
        dirs = (directions[p] if directions.dim() == 3 else directions).to(dt).unsqueeze(0)
        cols = []
        for j in range(6):
            with fwAD.dual_level():
                xi = fwAD.make_dual(torch.zeros((1, 6), dtype=dt), eye[j:j + 1])
                o2, d2 = apply_pose_twist(org, dirs, xi)
                f = plot_beam_frame(volume, o2[0], d2[0], num_samples, attenuation_coeff, start=start, sampler="trilinear")[3]
                f, t = fwAD.unpack_dual(f)
            cols.append(t.reshape(-1))
        J = torch.stack(cols, dim=-1)
        res = f.reshape(-1) - target[p].reshape(-1).to(f.dtype)
        losses.append((res * res).sum())
        jtjs.append(J.T @ J)
        jtrs.append(J.T @ res)
        frames.append(f)
    return torch.stack(losses), torch.stack(jtjs), torch.stack(jtrs), torch.stack(frames)
