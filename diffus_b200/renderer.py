"""Drop-in for the reference's renderer hot path (``src/renderer.py`` of gduguey/DiffUS).

Same names, argument meaning, return conventions and error behaviour as the reference for
``UltrasoundRenderer`` (``src/renderer.py:18-275``), ``compute_echo_traces`` (``:439``),
``propagate_full_rays_batched`` (``:412``) and ``custom_nearest_sampler`` (``:741``), with
keyword-only extensions (``sampler=``, ``return_indices=``) and a batched entry point
(:func:`render_frames`) that adds a leading pose dimension.  Numbers come from the sm_100a
kernels behind ``include/diffus_b200.h``; inputs must live on a CUDA device.

Deliberate differences from the reference (all documented in DESIGN.md):

* no ``print`` calls, no matplotlib visualiser (the reference's ``visualize=True`` default
  crashes on grad-requiring volumes, ``src/renderer.py:783``);
* the ``start > 0`` median replacement is out of place, so autograd works (the
  reference's in-place write at ``:243-244`` raises under autograd);
* ``artifacts=True`` (numpy/scipy, unseeded random, CPU only; ``:264-273``) is out of scope
  and raises ``NotImplementedError``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import ops
from ._lib import SAMPLER_NEAREST, SAMPLER_TRILINEAR, DiffusError

_SAMPLERS = {"nearest": SAMPLER_NEAREST, "prop": SAMPLER_NEAREST, "trilinear": SAMPLER_TRILINEAR}


def _sampler_id(sampler) -> int:
    try:
        return _SAMPLERS[sampler]
    except KeyError:
        raise ValueError(f"unknown sampler {sampler!r}; expected 'nearest' or 'trilinear'") from None


def _canon_pose(source: torch.Tensor, directions: torch.Tensor, device) -> Tuple[torch.Tensor, torch.Tensor, bool]:
    """Apply torch's promotion rules for ``source + steps * directions`` (``src/renderer.py:124``).

    ``steps`` is float32.  The product has dtype promote(float32, directions); the sum
    promote(product, source).  Returns float32 tensors, or float64 tensors plus a flag
    telling the kernel that the product must be rounded to float32 first.
    """
    source = torch.as_tensor(source, device=device)
    directions = torch.as_tensor(directions, device=device)
    dir_f64 = directions.dtype == torch.float64
    src_f64 = source.dtype == torch.float64
    if dir_f64 or src_f64:
        return source.to(torch.float64), directions.to(torch.float64), (not dir_f64)
    return source.to(torch.float32), directions.to(torch.float32), False


class PreparedVolume:
    """A volume plus a device-side packed copy laid out for the gathers.

    ``layout='brick'``: 4x4x2-voxel 128-byte bricks, one float per voxel -- a ray's gathers touch ~3x fewer
    cache lines per load instruction than in the torch layout.  ``layout='quad'``: one float4 per voxel holding
    the voxel and its three +p1 / +p2 neighbours, so a trilinear cell is two 16-byte loads instead of eight
    4-byte ones (4x the memory; faster only while the copy stays L2-resident).  ``'auto'`` picks ``'quad'`` up
    to 40 MiB of packed data (about 136^3 voxels) and ``'brick'`` above.  ``layout='texture'``: a layered 2-D CUDA
    array behind a texture object -- a trilinear cell is two ``tld4`` texel gathers with the address arithmetic and the
    border clamp done by the texture unit, at 1x the memory.  Building the copy costs one pass over the volume, so it pays for
    pose sweeps, not for a single frame.  Gradients still flow to ``volume`` (the LINEAR tensor).
    """

    QUAD_AUTO_MAX_BYTES = 40 << 20      # measured: once the float4 copy outgrows L2 (256^3 = 256 MiB) its random DRAM sectors lose to the L2-resident bricks

    def __init__(self, volume: torch.Tensor, layout: str = "auto"):
        if volume.dim() != 3:
            raise ValueError("volume must be (D,H,W)")
        if layout not in ("auto", "brick", "quad", "texture"):
            raise ValueError("layout must be 'auto', 'brick', 'quad' or 'texture'")
        if layout == "auto":
            layout = "quad" if volume.numel() * 16 <= self.QUAD_AUTO_MAX_BYTES else "brick"
        if volume.dtype != torch.float32 or not volume.is_contiguous():
            # a converted copy would silently go stale when the caller updates their own tensor in place
            raise ValueError("PreparedVolume needs a contiguous float32 volume (it watches the tensor for in-place updates)")
        self.layout = layout
        self.volume = volume
        self.shape = tuple(volume.shape)
        self._texture = None
        self.refresh()

    def close(self) -> None:
        """Release the packed copy now; the next use rebuilds it.  The TEXTURE layout's CUDA array lives outside torch's
        allocator and stays allocated until closed, so a caller that builds prepared volumes in a loop closes each one."""
        if self._texture is not None:
            self._texture.close()
            self._texture = None
        self._bricks, self._version = None, None

    def refresh(self) -> "PreparedVolume":
        """Rebuild the packed copy (done automatically when the volume tensor was modified in place)."""
        if self.layout == "texture":
            if self._texture is None:
                self._texture = ops.VolumeTexture(self.volume)
            else:
                self._texture.update(self.volume)
            self._bricks = self._texture.token
        else:
            self._bricks = ops.to_quads(self.volume) if self.layout == "quad" else ops.to_bricks(self.volume)
        self._version = self.volume._version
        return self

    @property
    def bricks(self) -> torch.Tensor:
        if self.volume._version != self._version:
            self.refresh()
        return self._bricks


def _unwrap(volume) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """``(volume, packed copy or None)`` of a tensor or a :class:`PreparedVolume`, the volume as a contiguous float32 tensor.
    Not detached: autograd still reaches the caller's tensor."""
    bricks = None
    if isinstance(volume, PreparedVolume):
        bricks, volume = volume.bricks, volume.volume
    return (volume if volume.dtype == torch.float32 else volume.float()).contiguous(), bricks


def _target(target: torch.Tensor) -> torch.Tensor:
    """Target frames as a contiguous float32 (P,R,S-start) tensor; one (R,S-start) frame is a batch of one."""
    tgt = target.to(torch.float32).contiguous()
    return tgt.unsqueeze(0) if tgt.dim() == 2 else tgt


def render_frames(volume, sources: torch.Tensor, directions: torch.Tensor, num_samples: int,
                  attenuation_coeff: float = 0.5, start=0, *, sampler: str = "nearest") -> torch.Tensor:
    """Batched ``plot_beam_frame``: (P,3) sources, (P,R,3) or (R,3) directions -> (P,R,S-start) frames.  Float32 sources
    of shape (P,R,3) give every ray its own origin (linear and convex array probes, :func:`diffus_b200.probe_rays`).

    Differentiable w.r.t. ``volume`` and, with ``sampler='trilinear'``, w.r.t. ``sources``
    and ``directions``.  ``volume`` is a (D,H,W) CUDA tensor or a :class:`PreparedVolume`.
    """
    vol32, bricks = _unwrap(volume)
    if vol32.dim() != 3:
        raise ValueError("volume must be (D,H,W)")
    sid = _sampler_id(sampler)
    src, dirs, product_f32 = _canon_pose(sources, directions, vol32.device)
    if src.dim() == 1:
        src = src.unsqueeze(0)
    start_i = _resolve_start(start, num_samples)
    need_grad = torch.is_grad_enabled() and (vol32.requires_grad or src.requires_grad or dirs.requires_grad)
    if need_grad:
        return ops.RenderFunction.apply(vol32, bricks, list(vol32.shape), src.contiguous(), dirs.contiguous(), int(num_samples),
                                        int(start_i), float(attenuation_coeff), sid, product_f32)
    frame, _ = ops.render_fwd_impl(vol32, bricks, list(vol32.shape), src.contiguous(), dirs.contiguous(), int(num_samples),
                                   int(start_i), float(attenuation_coeff), sid, product_f32, False)
    return frame


def render_mse_loss(volume, sources: torch.Tensor, directions: torch.Tensor, target: torch.Tensor,
                    num_samples: int, attenuation_coeff: float = 0.5, start=0, *, sampler: str = "trilinear",
                    return_frame: bool = False):
    """``mse_loss(render_frames(...), target)`` as ONE fused forward + loss + backward pass.

    The step every pose-recovery / MLP-training loop of the reference runs (render, compare
    with the real frames, back-propagate): the kernel gathers each sample once, evaluates
    the frame, the loss and the reverse scan in shared memory, and hands autograd the
    finished gradients.  Returns the scalar loss (differentiable w.r.t. ``volume`` and, for
    the trilinear sampler, ``sources`` / ``directions``), plus the frames if asked.  Per-ray sources (P,R,3) get (P,R,3)
    gradients.
    """
    vol32, bricks = _unwrap(volume)
    sid = _sampler_id(sampler)
    src, dirs, product_f32 = _canon_pose(sources, directions, vol32.device)
    if src.dim() == 1:
        src = src.unsqueeze(0)
    start_i = _resolve_start(start, num_samples)
    loss, frame = ops.RenderMSELoss.apply(vol32, bricks, list(vol32.shape), src.contiguous(), dirs.contiguous(), _target(target),
                                          int(num_samples), int(start_i), float(attenuation_coeff), sid, product_f32,
                                          bool(return_frame))
    return (loss, frame) if return_frame else loss


def render_gauss_newton(volume, sources: torch.Tensor, directions: torch.Tensor, target: torch.Tensor, num_samples: int,
                        attenuation_coeff: float = 0.5, start=0, *, sampler: str = "trilinear"):
    """Gauss-Newton system of every pose's frame residual in one forward-mode render pass.

    A pose update is the twist ``xi = (v, w)``: ``sources + v`` and the directions rotated by ``Rot(w)`` about the source
    (:func:`diffus_b200.pose_recovery.apply_pose_twist`).  With ``res = frame - target`` and ``J = d frame / d xi`` at
    ``xi = 0``, returns per pose ``loss (P,) = sum res^2``, ``JtJ (P,6,6) = J^T J`` and ``Jtr (P,6) = J^T res``.  ``2 Jtr / n``
    is the gradient of :func:`render_mse_loss` (mean over n elements) in twist coordinates.  Per-ray sources (P,R,3) (array
    probes) turn about the pose's pivot, the float64 mean of its origins (:func:`diffus_b200.pose_recovery.apply_pose_twist`).
    ``sources`` (P,3) or (P,R,3) and
    ``directions`` (P,R,3) or (R,3) are float32 (float64 poses are not supported); ``volume`` is a (D,H,W) CUDA tensor or a
    :class:`PreparedVolume`.  Only the trilinear sampler has a pose derivative.  The outputs are NOT differentiable: they
    are what a Gauss-Newton / Levenberg-Marquardt step consumes (:func:`diffus_b200.pose_recovery.recover_poses`).
    """
    if _sampler_id(sampler) != SAMPLER_TRILINEAR:
        raise DiffusError("render_gauss_newton needs sampler='trilinear' (the nearest sampler has no pose derivative)")
    vol32, bricks = _unwrap(volume)
    src = torch.as_tensor(sources, device=vol32.device)
    dirs = torch.as_tensor(directions, device=vol32.device)
    if src.dtype != torch.float32 or dirs.dtype != torch.float32:
        raise DiffusError("render_gauss_newton takes float32 sources and directions")
    if src.dim() == 1:
        src = src.unsqueeze(0)
    return ops.render_gauss_newton_impl(vol32.detach(), bricks, list(vol32.shape), src.detach().contiguous(), dirs.detach().contiguous(),
                                        _target(target.detach()), int(num_samples), _resolve_start(start, num_samples),
                                        float(attenuation_coeff))


def render_gauss_newton_sweep(volume, sources: torch.Tensor, directions: torch.Tensor, target: torch.Tensor, num_samples: int,
                              attenuation_coeff: float = 0.5, start=0, *, pivot=None):
    """Gauss-Newton system of a whole tracked sweep: ONE rigid twist ``xi = (v, w)`` about ONE pivot ``c`` moves every pose,
    ``p_k = c + v + Rot(w) (s_i - c + k d_i)`` with ``s_i`` the pose's source or, for per-ray sources (P,R,3), the ray's own
    origin.  With ``res = frame - target`` over all P poses and ``J = d frame / d xi`` at ``xi = 0``, returns float64
    ``loss () = sum res^2``, ``JtJ (6,6) = J^T J`` and ``Jtr (6,) = J^T res``; ``2 Jtr / n`` is the gradient of
    :func:`render_mse_loss` (mean over n elements) w.r.t. the shared twist.  It equals ``sum_p A_p^T JtJ_p A_p`` and
    ``sum_p A_p^T Jtr_p`` of :func:`render_gauss_newton` with ``A_p = [[I, -[c_p - c]x], [0, I]]``, ``c_p`` the point pose p
    turns about there.

    ``pivot`` is a (3,) float64 tensor on the volume's device, or None for the float64 mean of all ray origins.  Sources and
    directions are as for :func:`render_gauss_newton` (float32, trilinear sampler).  The outputs are not differentiable: they are
    what :func:`diffus_b200.pose_recovery.register_sweep` consumes.
    """
    vol32, bricks = _unwrap(volume)
    src = torch.as_tensor(sources, device=vol32.device)
    dirs = torch.as_tensor(directions, device=vol32.device)
    if src.dtype != torch.float32 or dirs.dtype != torch.float32:
        raise DiffusError("render_gauss_newton_sweep takes float32 sources and directions")
    if src.dim() == 1:
        src = src.unsqueeze(0)
    if pivot is not None:
        pivot = torch.as_tensor(pivot)
        if tuple(pivot.shape) != (3,) or pivot.dtype != torch.float64:
            raise DiffusError(f"pivot must be a float64 (3,) tensor, got {pivot.dtype} {tuple(pivot.shape)}")
        pivot = pivot.to(vol32.device).contiguous()
    tgt = _target(target.detach())
    start_i = _resolve_start(start, num_samples)
    want = (src.shape[0], dirs.shape[-2], int(num_samples) - start_i)
    if tuple(tgt.shape) != want:
        raise DiffusError(f"target must be {want} (poses, rays, samples after the crop), got {tuple(tgt.shape)}")
    return ops.render_gauss_newton_sweep_impl(vol32.detach(), bricks, list(vol32.shape), src.detach().contiguous(),
                                              dirs.detach().contiguous(), tgt, int(num_samples), start_i,
                                              float(attenuation_coeff), pivot)


def smooth_volume(volume, sigma: float, truncate: float = 4.0) -> torch.Tensor:
    """Isotropic Gaussian smoothing of a (D,H,W) volume on the device: ``scipy.ndimage.gaussian_filter(volume, sigma,
    mode='nearest', truncate=truncate)`` computed in float32, radius ``int(truncate * sigma + 0.5)`` <= 64.  Beyond a face the
    edge voxel repeats (the renderer's border rule).  ``sigma = 0`` returns an exact copy.

    ``volume`` is a CUDA tensor or a :class:`PreparedVolume` (its ``volume`` is smoothed); returns a new float32 tensor.  Not
    differentiable: a volume that requires grad, with grad enabled, raises rather than being silently detached.
    """
    vol = volume.volume if isinstance(volume, PreparedVolume) else volume
    if torch.is_grad_enabled() and vol.requires_grad:
        raise DiffusError("smooth_volume is not differentiable; call it under torch.no_grad() or on a detached volume")
    return ops.gaussian_blur_volume(vol, sigma, truncate)


def _resolve_start(start, num_samples: int) -> int:
    """``src/renderer.py:237-240``: a float start is a fraction of ``num_samples``."""
    if type(start) is float:
        start = int(start * num_samples)
    if type(start) is int:
        start = max(0, start)
    return int(start)


class UltrasoundRenderer:
    def __init__(self, num_samples: int, attenuation_coeff: float = 0.5):
        """
        num_samples: how many points to sample along each ray
        attenuation_coeff: controls exponential decay of echoes with depth
        """
        self.num_samples = num_samples
        self.attenuation_coeff = attenuation_coeff

    @staticmethod
    def compute_reflection_coeff(Z1: torch.Tensor, Z2: torch.Tensor) -> torch.Tensor:
        """Signed amplitude reflection coefficient ``(Z2 - Z1) / (Z1 + Z2)`` (reference ``:27-33``).

        A public elementwise helper; inside the renderer this is fused into the march kernel.
        """
        return (Z2 - Z1) / (Z1 + Z2)

    @staticmethod
    def trace_ray(volume: torch.Tensor, source: torch.Tensor, directions: torch.Tensor, num_samples: int,
                  start: int = 0, *, sampler: str = "nearest"):
        """Sample the volume along rays (reference ``:89-180``): returns ``x, y, z, values``.

        ``x, y, z`` are int64 (R, num_samples) clamped nearest-voxel indices and ``values``
        the (R, num_samples) impedances.  ``start`` is accepted for signature parity; as in
        the reference it only affected the debug plot.
        """
        vol32, bricks = _unwrap(volume)
        if directions.ndim == 1:
            directions = directions.unsqueeze(0)
        src, dirs, product_f32 = _canon_pose(source, directions, vol32.device)
        src = src.reshape(1, 3).contiguous()
        dirs = dirs.contiguous()
        dims = list(vol32.shape)
        x, y, z = ops.ray_indices(dims, src, dirs, int(num_samples), 0, product_f32)
        if torch.is_grad_enabled() and (vol32.requires_grad or src.requires_grad or dirs.requires_grad):
            values = ops.TraceValuesFunction.apply(vol32, bricks, dims, src, dirs, int(num_samples), _sampler_id(sampler),
                                                   product_f32)
        else:
            values = ops.trace_values(vol32, bricks, dims, src, dirs, int(num_samples), _sampler_id(sampler), product_f32)
        return x[0], y[0], z[0], values[0]

    def simulate_rays(self, volume: torch.Tensor, source: torch.Tensor, directions: torch.Tensor,
                      num_samples: int = 0, MRI: bool = False, start=0, *, sampler: str = "nearest"):
        """Reflection coefficients along each ray (reference ``:35-71``).

        Returns ``x, y, z, R`` with ``R`` of shape (n_rays, num_samples-1), squeezed to 1-D for
        a single ray as in the reference; ``MRI=True`` returns the sampled values ``Z1`` instead.
        """
        if num_samples == 0:
            num_samples = self.num_samples
        x, y, z, impedances = self.trace_ray(volume=volume, source=source, directions=directions,
                                             num_samples=num_samples, start=start, sampler=sampler)
        if impedances.ndim == 1:
            impedances = impedances.unsqueeze(0)
        Z1 = impedances[:, :-1]
        Z2 = impedances[:, 1:]
        R = self.compute_reflection_coeff(Z1, Z2)
        if MRI:
            return Z1
        return x, y, z, R.squeeze(0)

    def plot_beam_frame(self, volume: torch.Tensor, source: torch.Tensor, directions: torch.Tensor,
                        angle: float = 45.0, plot: bool = True, artifacts: bool = False, ax=None, cmap=None,
                        std_radial: float = 0.01, std_local: float = 0.15, max_sigma: float = 4.0,
                        alpha: float = 5, start: float = 0, *, sampler: str = "nearest",
                        return_indices: bool = True, **kwargs):
        """Simulate the rays of one probe pose and return the B-mode fan frame (reference ``:201-275``).

        Args as in the reference: ``volume`` (D,H,W) impedance, ``source`` (3,), ``directions``
        (n_rays,3) unit vectors; ``angle``, ``plot``, ``ax``, ``cmap`` never affected the
        numbers and are ignored; ``start`` (int, or float fraction of ``num_samples``) crops the
        near field and replaces the first kept reflection coefficient by its median over rays.

        Returns ``(x[:, start:], y[:, start:], z[:, start:], frame)``; with
        ``return_indices=False`` the three index tensors are ``None`` (they are 6x the size of
        the frame and only feed plotting / splatting).
        """
        if artifacts:
            raise NotImplementedError(
                "artifacts=True (numpy/scipy speckle, blur, sharpen; unseeded, CPU-only, non-differentiable in the "
                "reference, src/renderer.py:264-273) is outside the B200 hot path")
        vol = volume.volume if isinstance(volume, PreparedVolume) else volume
        directions = torch.as_tensor(directions, device=vol.device)
        if directions.ndim != 2 or directions.shape[0] < 2:
            # the reference squeezes a single ray to 1-D and then fails to unpack (B, N) (:71, :425)
            raise ValueError("plot_beam_frame needs directions of shape (n_rays, 3) with n_rays >= 2")
        start_i = _resolve_start(start, self.num_samples)
        frame = render_frames(volume, torch.as_tensor(source, device=vol.device).reshape(1, 3), directions,
                              self.num_samples, self.attenuation_coeff, start_i, sampler=sampler)[0]
        if not return_indices:
            return None, None, None, frame
        src, dirs, product_f32 = _canon_pose(source, directions, vol.device)
        x, y, z = ops.ray_indices(list(vol.shape), src.reshape(1, 3).contiguous(), dirs.contiguous(),
                                  int(self.num_samples), start_i, product_f32)
        return x[0], y[0], z[0], frame


def compute_echo_traces(refLR: torch.Tensor, spacing: float = 1.0, c: float = 1.54e3):
    """Echo line per ray from reflection coefficients (reference ``src/renderer.py:439-457``).

    ``refLR`` (B, N) -> ``(echo (B, N+1), delays_us (N+1,))`` with ``echo = [0, d0^(1..N)]``,
    ``d0^(k)`` the surface return of the first ``k`` interfaces; differentiable in ``refLR``.
    The scan kernels compute in float32: a float64 (or half) ``refLR`` is evaluated in float32 and the result cast back to its
    dtype, so float64 inputs do NOT buy float64 accuracy here (the reference's float64 run differs from this by ~1e-7 of peak).
    """
    if refLR.dim() != 2:
        B, N = refLR.shape      # same ValueError as the reference's unpacking (:425)
    echo = ops.echo_fwd(refLR) if refLR.shape[1] > 0 else refLR.new_zeros((refLR.shape[0], 1))
    echo = echo.to(refLR.dtype) if refLR.dtype in (torch.float64, torch.float16, torch.bfloat16) else echo
    delays_us = 2 * spacing * torch.arange(refLR.shape[1] + 1, device=refLR.device) / c
    return echo, delays_us


def gaussian_pulse(length: int, sigma: float):
    """1-D Gaussian pulse normalised to peak 1 (reference ``src/renderer.py:481-496``); host numpy, like the reference."""
    import numpy as np
    t = np.linspace(-length // 2, length // 2, length)
    pulse = np.exp(-0.5 * (t / sigma) ** 2)
    return pulse / pulse.max()


def compute_gaussian_pulse(refLR: torch.Tensor, spacing: float = 1.0, c: float = 1.54e3, length: int = 10, sigma: int = 1,
                           pulse=None) -> torch.Tensor:
    """Echo traces convolved with a Gaussian pulse (reference ``src/renderer.py:459-479``).

    Off the hot path (the call is commented out on HEAD, ``:250``): the echo line comes from the scan kernel and the short
    1-D convolution from ``conv1d_rows_kernel`` (differentiable in ``refLR``; the pulse is a constant, as in the reference,
    where it is a numpy array).  ``pulse``: optional (1, 1, L) tensor like the reference's.
    """
    echo_signals, _ = compute_echo_traces(refLR, spacing, c)
    if pulse is None:
        pulse = torch.tensor(gaussian_pulse(length=length, sigma=sigma), dtype=echo_signals.dtype, device=echo_signals.device)
    else:
        if pulse.requires_grad:
            raise NotImplementedError("compute_gaussian_pulse is differentiable in refLR only (the reference's pulse is a numpy constant)")
        length = pulse.shape[-1]
    return ops.Conv1dRows.apply(echo_signals, pulse.reshape(-1), int(length) // 2)


def propagate_full_rays_batched(refLR: torch.Tensor) -> torch.Tensor:
    """Cumulative surface return per truncation depth (reference ``src/renderer.py:412-436``)."""
    echo, _ = compute_echo_traces(refLR)
    return torch.cumsum(echo, dim=1)


def differentiable_splat(x, y, z, intensities, H=256, W=256, sigma=2.0):
    """Splat ray samples onto the 2-D plane of highest coordinate variance (reference ``src/renderer.py:694-737``).

    Same recipe as the reference -- axes of largest variance, round + clamp to pixels, non-accumulating write
    (for duplicate pixels the last sample wins), Gaussian blur of image and hit mask, ratio, transposed -- with
    the axis choice made on the device (no ``.item()`` syncs).  Differentiable w.r.t. ``intensities``.
    """
    return ops.SplatFunction.apply(x, y, z, intensities, int(H), int(W), float(sigma))


def rotate_around_apex(x, z, apex, median):
    """Rotate fan points so that the median direction maps onto [0, 1] (reference ``src/renderer.py:655-692``).

    Same arithmetic as the reference (which shifts x by the hard-wired 128, not by the apex).  The rotation angle is
    formed from ``median`` in float32 with the reference's own torch expression (three scalars, on the host); the
    element-wise part is ONE kernel with the reference's rounding order, feeding :func:`differentiable_splat`.
    """
    median_vec = torch.as_tensor(median, dtype=torch.float32).detach().cpu()
    median_vec = median_vec / median_vec.norm()
    angle = torch.atan2(median_vec[0], median_vec[1])
    cos_a, sin_a = float(torch.cos(angle)), float(torch.sin(angle))
    apex = torch.as_tensor(apex, dtype=torch.float32).detach().cpu()
    return ops.rotate_apex(x, z, cos_a, sin_a, 128.0, float(apex[0]), float(apex[1]))


def custom_nearest_sampler(Z: torch.Tensor, points: torch.Tensor, visualize: bool = False, sampler: str = "prop",
                           start: int = 100):
    """Volume lookup at explicit points (reference ``src/renderer.py:741-819``).

    ``points`` (B, S, 3) in voxel coordinates -> ``x, y, z`` int64 (B, S) clamped nearest indices and values (B, S).
    ``sampler='prop'`` (the reference's default) is the nearest lookup; ``'trilinear'`` the notebook-era one.
    ``visualize`` and ``start`` only drove the reference's matplotlib debug plot and are ignored.  The renderer
    itself never materialises ``points`` (ray setup is fused into the march kernels).
    """
    if points.dim() != 3 or points.shape[-1] != 3:
        raise ValueError("points must be (batch, samples, 3)")
    return ops.sample_points(Z, points, _sampler_id(sampler))
