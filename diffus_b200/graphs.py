"""CUDA-graph capture of the fused pose-recovery step.

One 128 x 512 frame is ~20 us of device work but ~250 us of PyTorch eager bookkeeping (autograd engine, tensor
allocation, ctypes argument packing).  A pose-recovery loop calls the same step thousands of times with the
same shapes, so the step is captured once -- the C ABI never allocates or synchronises, which is what makes it
capturable -- and replayed with new poses written into static buffers.
"""
from __future__ import annotations

import torch

from . import ops
from ._lib import SAMPLER_TRILINEAR
from .renderer import _resolve_start, _sampler_id, _target, _unwrap


def _capture(dev, step, prime=None):
    """Run ``prime`` and then ``step`` twice on a side stream (lazy module loads, kernel attributes, library handles), then
    capture ``step`` into a CUDA graph.  Returns the graph and what the captured ``step`` returned."""
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        if prime is not None:
            prime()
        for _ in range(2):
            step()
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    return graph, out


def _ray_fn(probe: str, opening_angle, radius, width, n_rays: int):
    """``(rays, args)``: ``rays(poses)`` gives the (origins, directions) of (3,P,3) pose parameters [sources | median | hint]
    -- a sector fan's origins are its (P,3) sources, an array probe has one origin per ray (P,R,3) -- and ``args`` the
    ``(kind id, angle, radius, width)`` of an array probe for ``ops.probe_rays_*`` (None for a sector fan)."""
    if probe == "sector":
        return (lambda poses: (poses[0], ops.fan_directions_fwd(poses[1], poses[2], opening_angle, n_rays))), None
    args = ops.probe_args(probe, opening_angle, radius, width)
    kid, angle, rho, wid = args
    return (lambda poses: ops.probe_rays_fwd(kid, poses[0], poses[1], poses[2], n_rays, angle, rho, wid)), args


class GraphedPoseStep:
    """``loss, grad_sources, grad_directions = step(sources, directions)`` for fixed shapes, volume and targets.

    Equivalent to ``render_mse_loss(volume, sources, directions, targets, ...)`` + ``backward()``; outputs are
    static tensors that the next call overwrites.
    """

    def __init__(self, volume, targets: torch.Tensor, n_rays: int, num_samples: int, attenuation_coeff: float = 0.5,
                 start=0, sampler: str = "trilinear", shared_directions: bool = False):
        vol, bricks = _unwrap(volume)
        dev = vol.device
        tgt = _target(targets)
        P = tgt.shape[0]
        self.sources = torch.zeros((P, 3), dtype=torch.float32, device=dev)
        self.directions = torch.zeros((n_rays, 3) if shared_directions else (P, n_rays, 3), dtype=torch.float32, device=dev)
        self.directions[..., 1] = 1.0
        args = (vol, bricks, list(vol.shape), self.sources, self.directions, tgt, int(num_samples),
                _resolve_start(start, num_samples), float(attenuation_coeff), _sampler_id(sampler), False, False,
                _sampler_id(sampler) == SAMPLER_TRILINEAR, False)
        self.graph, (self.loss, _, _, self.grad_sources, self.grad_directions) = _capture(dev, lambda: ops.render_mse_impl(*args))
        self._keep = args

    def __call__(self, sources: torch.Tensor, directions: torch.Tensor):
        self.sources.copy_(sources.reshape(self.sources.shape), non_blocking=True)
        self.directions.copy_(directions.reshape(self.directions.shape), non_blocking=True)
        self.graph.replay()
        gd = self.grad_directions if self.directions.dim() == 3 else self.grad_directions.sum(0)
        return self.loss[0], self.grad_sources, gd


class GraphedFanPoseStep:
    """The same step driven by pose PARAMETERS: ``loss, g_sources, g_median, g_hint = step(sources, median, hint)``.

    The fans are generated on the device (``ops.fan_directions``) and the gradient w.r.t. the (P,R,3) directions is
    folded back onto the two (P,3) orientation vectors inside the graph, so a step moves 9 floats per pose in each
    direction instead of 3 + 3R.  Outputs are static tensors that the next call overwrites.

    ``probe='convex'`` (``radius``) or ``'linear'`` (``width``): array probes, whose ``sources`` are the probe centres.  The
    graph then generates the per-ray origins and directions (``ops.probe_rays_fwd``), runs the fused step with one origin per
    ray and folds the (P,R,3) gradients back onto centre, median and hint (``ops.probe_rays_bwd``).
    """

    def __init__(self, volume, targets: torch.Tensor, n_rays: int, num_samples: int, opening_angle: float,
                 attenuation_coeff: float = 0.5, start=0, *, probe: str = "sector", radius=None, width=None):
        from .pose_recovery import probe_keywords
        probe, radius, width = probe_keywords(probe, radius, width)
        rays, probe_args = _ray_fn(probe, opening_angle, radius, width, n_rays)
        vol, bricks = _unwrap(volume)
        dev = vol.device
        tgt = targets.to(torch.float32).contiguous()
        P = tgt.shape[0]
        # one static input block (3, P, 3) = [sources | median | hint] and one static output block
        # [g_sources | g_median | g_hint | loss]: a step is one H2D copy, one graph launch, one D2H copy
        self.poses = torch.zeros((3, P, 3), dtype=torch.float32, device=dev)
        self.sources, self.median, self.hint = self.poses[0], self.poses[1], self.poses[2]
        self.median[:, 1] = 1.0
        self.hint[:, 0] = 1.0
        self.out = torch.zeros((9 * P + 1,), dtype=torch.float32, device=dev)
        start_i = _resolve_start(start, num_samples)

        # every result is written straight into its slice of the static output block: the graph is five kernels (fans, fused
        # step, two reductions, fan backward) with no copy kernels behind them
        o_gs, o_gm, o_gh, o_loss = self.out[:3 * P], self.out[3 * P:6 * P], self.out[6 * P:9 * P], self.out[9 * P:]

        def step():
            org, dirs = rays(self.poses)
            _, _, _, go, gd = ops.render_mse_impl(vol, bricks, list(vol.shape), org, dirs, tgt, int(num_samples), start_i,
                                                  float(attenuation_coeff), SAMPLER_TRILINEAR, False, False, True, False,
                                                  loss_out=o_loss, grad_sources_out=None if probe_args else o_gs)
            if probe_args:
                ops.probe_rays_bwd(probe_args[0], self.sources, self.median, self.hint, go, gd, n_rays, *probe_args[1:],
                                   grad_centre_out=o_gs, grad_median_out=o_gm, grad_hint_out=o_gh)
            else:
                ops.fan_directions_bwd(self.median, self.hint, gd, opening_angle, n_rays, grad_median_out=o_gm, grad_hint_out=o_gh)

        self.graph, _ = _capture(dev, step)
        self.P = P
        self.loss = self.out[9 * P]
        self.grad_sources = self.out[:3 * P].view(P, 3)
        self.grad_median = self.out[3 * P:6 * P].view(P, 3)
        self.grad_hint = self.out[6 * P:9 * P].view(P, 3)
        self._keep = (vol, bricks, tgt)

    def __call__(self, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor):
        self.sources.copy_(sources, non_blocking=True)
        self.median.copy_(median, non_blocking=True)
        self.hint.copy_(hint, non_blocking=True)
        self.graph.replay()
        return self.loss, self.grad_sources, self.grad_median, self.grad_hint

    def packed(self, poses: torch.Tensor) -> torch.Tensor:
        """One copy in, one launch: ``poses`` is (3, P, 3) = [sources | median | hint] (e.g. pinned host memory); returns the
        static output block ``[g_sources (P,3) | g_median (P,3) | g_hint (P,3) | loss]`` as one (9P + 1) tensor."""
        self.poses.copy_(poses, non_blocking=True)
        self.graph.replay()
        return self.out


def _solve_spd6(a: torch.Tensor, b: torch.Tensor):
    """Batched Cholesky solve of (P,n,n) symmetric positive definite systems with elementwise tensor operations only, so that
    it records into a CUDA graph (torch.linalg's batched factorisations invalidated the capture on the B200 with torch 2.11).
    Returns ``(x (P,n), ok (P,))``; ``ok`` is False where a pivot was not positive."""
    n = a.shape[-1]
    L = torch.zeros_like(a)
    ok = torch.ones(a.shape[:-2], dtype=torch.bool, device=a.device)
    for j in range(n):
        col = a[:, j:, j] - (L[:, j:, :j] * L[:, j:j + 1, :j]).sum(-1)
        piv = col[:, 0]
        ok = ok & (piv > 0)
        d = torch.sqrt(piv.clamp_min(1e-300))
        L[:, j:, j] = col / d[:, None]
    y = torch.zeros_like(b)
    for i in range(n):
        y[:, i] = (b[:, i] - (L[:, i, :i] * y[:, :i]).sum(-1)) / L[:, i, i]
    x = torch.zeros_like(b)
    for i in reversed(range(n)):
        x[:, i] = (y[:, i] - (L[:, i + 1:, i] * x[:, i + 1:]).sum(-1)) / L[:, i, i]
    return x, ok


class _LevenbergMarquardt:
    """The Marquardt-damped solve and the accept / reject of the graphed Gauss-Newton steps, on the static ``jtj``, ``jtr``,
    ``loss``, ``lam`` and candidate ``c_loss`` of a subclass."""

    LAM_DOWN, LAM_UP, LAM_MIN, LAM_MAX = 1.0 / 3.0, 4.0, 1e-9, 1e9

    def _delta(self, jtj: torch.Tensor, jtr: torch.Tensor) -> torch.Tensor:
        """The float64 step of the batched systems (P,6,6), (P,6): ``(JtJ + lam diag(JtJ) + eps I) delta = -Jtr``; zero where the
        damped system is not positive definite or the step is not finite."""
        a = jtj.double()
        d = a.diagonal(dim1=-2, dim2=-1)
        eps = 1e-12 * d.amax(-1, keepdim=True) + 1e-30
        a = a + torch.diag_embed(self.lam[:, None] * d + eps)
        delta, ok = _solve_spd6(a, -jtr.double())
        ok = ok & torch.isfinite(delta).all(-1)
        return torch.where(ok[:, None], delta, torch.zeros_like(delta))

    def _accept(self, *pairs) -> None:
        """Where the candidate's loss went down, copy each ``(candidate, state[, pose dim])`` over the state and shrink ``lam``;
        else keep the state and grow ``lam``.  (NaN: rejected.)  ``pose dim``: the dimension of the state that runs over the
        poses of the (P,) loss, 0 if not given."""
        acc = self.c_loss < self.loss
        for cand, cur, *dim in pairs:
            d = dim[0] if dim else 0
            mask = acc.reshape((1,) * d + acc.shape + (1,) * (cur.dim() - d - acc.dim()))
            cur.copy_(torch.where(mask, cand, cur))
        self.lam.copy_(torch.where(acc, self.lam * self.LAM_DOWN, self.lam * self.LAM_UP).clamp(self.LAM_MIN, self.LAM_MAX))


class GraphedFanGaussNewtonStep(_LevenbergMarquardt):
    """One Levenberg-Marquardt iteration of fan pose recovery as one CUDA-graph replay (see ``pose_recovery.recover_poses``).

    Static state on the device: the current poses (``sources``, ``median``, ``hint``, (P,3) each), their loss (P,), JtJ
    (P,6,6) and Jtr (P,6), and the damping ``lam`` (P,).  A replay solves the damped system of every pose in float64, applies
    the twist to the fan parameters, generates the candidate fans, renders their Gauss-Newton systems
    (``ops.render_gauss_newton_impl``) and accepts or rejects each pose on its own loss.  Call :meth:`reset` before the first
    replay.

    ``probe='convex'`` (``radius``) or ``'linear'`` (``width``): array probes with ``sources`` their centres.  The systems are
    rendered from the rays of ``ops.probe_rays_fwd`` with one origin per ray, and the step is applied to the parameters by
    ``apply_probe_twist`` about the pivot of the current origins -- the point the kernel's twist turns about.
    """

    def __init__(self, volume, targets: torch.Tensor, n_rays: int, num_samples: int, opening_angle: float,
                 attenuation_coeff: float = 0.5, start=0, *, probe: str = "sector", radius=None, width=None):
        from .pose_recovery import apply_fan_twist, apply_probe_twist, probe_keywords, probe_pivot
        probe, radius, width = probe_keywords(probe, radius, width)
        rays, array = _ray_fn(probe, opening_angle, radius, width, n_rays)
        vol, bricks = _unwrap(volume)
        dev = vol.device
        tgt = targets.to(torch.float32).contiguous()
        P = tgt.shape[0]
        start_i = _resolve_start(start, num_samples)
        self.P = P
        self.poses = torch.zeros((3, P, 3), dtype=torch.float32, device=dev)       # [sources | median | hint]
        self.sources, self.median, self.hint = self.poses[0], self.poses[1], self.poses[2]
        self.median[:, 1] = 1.0
        self.hint[:, 0] = 1.0
        self.cand = torch.zeros_like(self.poses)
        self.loss = torch.zeros((P,), dtype=torch.float32, device=dev)
        self.jtj = torch.zeros((P, 6, 6), dtype=torch.float32, device=dev)
        self.jtr = torch.zeros((P, 6), dtype=torch.float32, device=dev)
        self.c_loss, self.c_jtj, self.c_jtr = torch.zeros_like(self.loss), torch.zeros_like(self.jtj), torch.zeros_like(self.jtr)
        self.lam = torch.ones((P,), dtype=torch.float64, device=dev)

        def system(poses, loss, jtj, jtr):
            src, dirs = rays(poses)
            ops.render_gauss_newton_impl(vol, bricks, list(vol.shape), src, dirs, tgt, int(num_samples), start_i,
                                         float(attenuation_coeff), loss_out=loss, jtj_out=jtj, jtr_out=jtr)

        def step():
            delta = self._delta(self.jtj, self.jtr).float()
            if array:
                s, m, h = apply_probe_twist(self.sources, self.median, self.hint, delta, probe_pivot(rays(self.poses)[0]))
            else:
                s, m, h = apply_fan_twist(self.sources, self.median, self.hint, delta)
            self.cand[0].copy_(s)
            self.cand[1].copy_(m)
            self.cand[2].copy_(h)
            system(self.cand, self.c_loss, self.c_jtj, self.c_jtr)
            self._accept((self.cand, self.poses, 1), (self.c_loss, self.loss), (self.c_jtj, self.jtj), (self.c_jtr, self.jtr))

        self._system = system
        self.graph, _ = _capture(dev, step, lambda: system(self.poses, self.loss, self.jtj, self.jtr))
        self._keep = (vol, bricks, tgt)

    def reset(self, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, damping: float = 1e-3) -> None:
        """Start poses (P,3 each) and the initial damping; evaluates their Gauss-Newton systems (eagerly, on the device)."""
        self.sources.copy_(sources, non_blocking=True)
        self.median.copy_(median, non_blocking=True)
        self.hint.copy_(hint, non_blocking=True)
        self.lam.fill_(float(damping))
        self._system(self.poses, self.loss, self.jtj, self.jtr)

    def __call__(self) -> torch.Tensor:
        """One iteration; returns the static (P,) loss after it."""
        self.graph.replay()
        return self.loss


class GraphedSweepGaussNewtonStep(_LevenbergMarquardt):
    """One Levenberg-Marquardt iteration of tracked-sweep registration as one CUDA-graph replay (see
    ``pose_recovery.register_sweep``).

    Static state on the device: the start poses in float64 (``start``, (3,P,3)), their origin centroid ``c0``, the current
    transform (``rot`` (3,3), ``trans`` (3,), float64), its ``pivot = rot c0 + trans``, the current poses (``sources``,
    ``median``, ``hint``: the transform applied to the start poses, rounded once to float32), the sweep's float64 loss (), JtJ
    (6,6) and Jtr (6,), and the damping ``lam``.  A replay solves the damped 6x6 system (``_solve_spd6`` with a batch of one),
    composes the candidate transform with the twist about the pivot, applies it to the start poses, renders the candidate's
    sweep system (``ops.render_gauss_newton_sweep_impl``, about the candidate's pivot) and accepts or rejects it on the total
    loss.  Call :meth:`reset` before the first replay.  ``probe``, ``radius`` and ``width`` as for
    :class:`GraphedFanGaussNewtonStep`.
    """

    def __init__(self, volume, targets: torch.Tensor, n_rays: int, num_samples: int, opening_angle: float,
                 attenuation_coeff: float = 0.5, start=0, *, probe: str = "sector", radius=None, width=None):
        from .pose_recovery import apply_rigid_transform, compose_sweep_twist, probe_keywords
        probe, radius, width = probe_keywords(probe, radius, width)
        rays, array = _ray_fn(probe, opening_angle, radius, width, n_rays)
        vol, bricks = _unwrap(volume)
        dev = vol.device
        tgt = targets.to(torch.float32).contiguous()
        P = tgt.shape[0]
        start_i = _resolve_start(start, num_samples)
        f64 = dict(dtype=torch.float64, device=dev)
        self.P = P
        self.start = torch.zeros((3, P, 3), **f64)                                  # [sources | median | hint] of the start
        self.start[1, :, 1] = 1.0
        self.start[2, :, 0] = 1.0
        self.c0 = torch.zeros((3,), **f64)
        self.poses = self.start.float()
        self.sources, self.median, self.hint = self.poses[0], self.poses[1], self.poses[2]
        self.cand = torch.zeros_like(self.poses)
        self.rot, self.trans, self.pivot = torch.eye(3, **f64), torch.zeros((3,), **f64), torch.zeros((3,), **f64)
        self.loss, self.jtj, self.jtr = torch.zeros((), **f64), torch.zeros((6, 6), **f64), torch.zeros((6,), **f64)
        self.c_rot, self.c_trans, self.c_pivot = torch.zeros_like(self.rot), torch.zeros_like(self.trans), torch.zeros_like(self.pivot)
        self.c_loss, self.c_jtj, self.c_jtr = torch.zeros_like(self.loss), torch.zeros_like(self.jtj), torch.zeros_like(self.jtr)
        self.lam = torch.ones((1,), **f64)

        def system(poses, pivot, loss, jtj, jtr):
            src, dirs = rays(poses)
            ops.render_gauss_newton_sweep_impl(vol, bricks, list(vol.shape), src, dirs, tgt, int(num_samples), start_i,
                                               float(attenuation_coeff), pivot, loss_out=loss, jtj_out=jtj, jtr_out=jtr)

        def step():
            delta = self._delta(self.jtj.unsqueeze(0), self.jtr.unsqueeze(0))[0]
            r, t = compose_sweep_twist(self.rot, self.trans, delta, self.pivot)
            self.c_rot.copy_(r)
            self.c_trans.copy_(t)
            self.c_pivot.copy_((self.c_rot * self.c0).sum(-1) + self.c_trans)
            s, m, h = apply_rigid_transform(self.c_rot, self.c_trans, self.start[0], self.start[1], self.start[2])
            self.cand[0].copy_(s)
            self.cand[1].copy_(m)
            self.cand[2].copy_(h)
            system(self.cand, self.c_pivot, self.c_loss, self.c_jtj, self.c_jtr)
            self._accept((self.cand, self.poses), (self.c_rot, self.rot), (self.c_trans, self.trans), (self.c_pivot, self.pivot),
                         (self.c_loss, self.loss), (self.c_jtj, self.jtj), (self.c_jtr, self.jtr))

        def centroid(poses):
            """The float64 mean of all P*R ray origins of ``poses`` (a sector fan's R rays share its source)."""
            return (rays(poses)[0] if array else poses[0]).reshape(-1, 3).double().mean(0)

        self._system, self._centroid = system, centroid
        self.graph, _ = _capture(dev, step, lambda: system(self.poses, self.pivot, self.loss, self.jtj, self.jtr))
        self._keep = (vol, bricks, tgt)

    def reset(self, sources: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, damping: float = 1e-3) -> None:
        """The start sweep (P,3 each), the identity transform and the initial damping; evaluates the start's system (eagerly, on
        the device) about the start's origin centroid."""
        for i, x in enumerate((sources, median, hint)):
            self.start[i].copy_(x, non_blocking=True)
            self.poses[i].copy_(x, non_blocking=True)
        self.rot.copy_(torch.eye(3, dtype=torch.float64))
        self.trans.zero_()
        self.c0.copy_(self._centroid(self.poses))
        self.pivot.copy_(self.c0)
        self.lam.fill_(float(damping))
        self._system(self.poses, self.pivot, self.loss, self.jtj, self.jtr)

    def __call__(self) -> torch.Tensor:
        """One iteration; returns the static float64 () total loss after it."""
        self.graph.replay()
        return self.loss
