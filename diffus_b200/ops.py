"""torch.library custom ops over the C ABI (``libdiffus_b200.so``), with autograd.

PyTorch is plumbing here: it owns device memory and streams and carries autograd; every
number is produced by the hand-written kernels behind ``include/diffus_b200.h``.  All ops
require CUDA tensors and raise otherwise -- there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Tuple

import torch

from . import _lib
from ._lib import (LAYOUT_BRICK, LAYOUT_LINEAR, LAYOUT_QUAD, LAYOUT_TEXTURE, MLP_NPARAMS, POSE_F32, POSE_F32_PER_RAY, POSE_F64,
                   PROBE_CONVEX, PROBE_LINEAR, SAMPLER_NEAREST,
                   SAMPLER_TRILINEAR, DiffusRenderArgs, DiffusRenderBwdArgs)

SEG = 512  # PREFIX_STRIDE of csrc/common.cuh: the forward saves a 2x2 prefix every SEG columns


def launch_count() -> int:
    """Kernels this process has enqueued through the library (bench.py reports it as gpu_launches)."""
    return _lib.load().diffus_launch_count()


def _require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.DiffusError(
                "diffus_b200 ops run only on CUDA tensors (sm_100a kernels); there is no CPU fallback")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise _lib.DiffusError(f"tensors on different devices: {dev} vs {t.device}")
    return dev


try:                                        # the raw handle of torch's current stream without building a Stream object
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:                      # pragma: no cover
    _raw_stream = None


def _stream(dev: torch.device) -> C.c_void_p:
    if _raw_stream is not None:
        return C.c_void_p(_raw_stream(dev.index if dev.index is not None else torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


class _on_device:
    """``with torch.cuda.device(dev)`` only when ``dev`` is not already current (the context manager costs ~4 us per call)."""
    __slots__ = ("ctx",)

    def __init__(self, dev: torch.device):
        idx = dev.index
        self.ctx = None if idx is None or idx == torch.cuda.current_device() else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            return self.ctx.__exit__(*exc)
        return False


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _nseg(sout: int) -> int:
    return (sout + SEG - 1) // SEG


# TEXTURE layout: the CUDA array + texture object live outside torch's allocator.  The ops receive a one-element int64
# CUDA tensor as ``bricks`` (the token); this registry maps the token's address to the texture object it stands for.
_TEXTURES = {}


class VolumeTexture:
    """A read-only copy of a (D,H,W) float32 volume in a layered 2-D CUDA array behind a texture object."""

    def __init__(self, volume: torch.Tensor):
        dev = _require_cuda(volume)
        lib = _lib.load()
        v = volume.detach().contiguous().float()
        self.dims = tuple(v.shape)
        self.device = dev
        tex, arr = C.c_uint64(0), C.c_uint64(0)
        with _on_device(dev):
            _lib.check(lib.diffus_volume_texture_create(v.data_ptr(), C.byref((C.c_int32 * 3)(*self.dims)), C.byref(tex),
                                                        C.byref(arr), _stream(dev)), "diffus_volume_texture_create")
            self.token = torch.zeros((1,), dtype=torch.int64, device=dev)
        self.texture, self.array = tex.value, arr.value
        _TEXTURES[self.token.data_ptr()] = self

    def update(self, volume: torch.Tensor) -> None:
        v = volume.detach().contiguous().float()
        if tuple(v.shape) != self.dims:
            raise _lib.DiffusError("volume shape changed; build a new VolumeTexture")
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().diffus_volume_texture_update(self.array, v.data_ptr(), C.byref((C.c_int32 * 3)(*self.dims)),
                                                                _stream(self.device)), "diffus_volume_texture_update")

    def close(self) -> None:
        if self.texture:
            _TEXTURES.pop(self.token.data_ptr(), None)
            try:
                with torch.cuda.device(self.device):
                    torch.cuda.current_stream(self.device).synchronize()     # no launch may still read the array
                    _lib.load().diffus_volume_texture_destroy(self.texture, self.array)
            finally:
                self.texture = self.array = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _texture_of(bricks: torch.Tensor) -> "VolumeTexture":
    try:
        return _TEXTURES[bricks.data_ptr()]
    except KeyError:
        raise _lib.DiffusError("int64 `bricks` tensor is not the token of a live VolumeTexture") from None


def _packed_layout(bricks: Optional[torch.Tensor]) -> int:
    """Layout of the packed copy handed to the ops as ``bricks``: none -> LINEAR, 1-D float -> BRICK, (n, 4) -> QUAD,
    int64 token -> TEXTURE."""
    if bricks is None or bricks.numel() == 0:
        return LAYOUT_LINEAR
    if bricks.dtype == torch.int64:
        return LAYOUT_TEXTURE
    return LAYOUT_QUAD if bricks.dim() == 2 else LAYOUT_BRICK


def _grad_volume_shape(bricks: Optional[torch.Tensor], dims) -> Tuple[int, ...]:
    """The gradient has the gathered layout (LINEAR / BRICK); a QUAD volume scatters into a BRICK buffer."""
    layout = _packed_layout(bricks)
    if layout == LAYOUT_LINEAR:
        return tuple(dims)
    if layout == LAYOUT_BRICK:
        return (bricks.numel(),)
    return (_lib.load().diffus_brick_elems(C.byref((C.c_int32 * 3)(*dims))),)


def _zero_grad_volume(bricks: Optional[torch.Tensor], dims, dev) -> torch.Tensor:
    """The zero-filled buffer d loss / d volume is accumulated into, in the layout of :func:`_grad_volume_shape`."""
    return torch.zeros(_grad_volume_shape(bricks, dims), dtype=torch.float32, device=dev)


def _linear_grad_volume(gvol: torch.Tensor, bricks: Optional[torch.Tensor], dims) -> torch.Tensor:
    """The gradient of a packed volume comes back in bricks: convert it to the (D,H,W) layout of the volume tensor."""
    return from_bricks(gvol, dims) if bricks is not None and bricks.numel() > 0 else gvol


def _pose_grad(need_pose: bool, sampler: int) -> bool:
    """Only the trilinear sampler has a pose derivative."""
    return bool(need_pose) and sampler == SAMPLER_TRILINEAR


def _check_target(target: torch.Tensor, P: int, R: int, sout: int) -> None:
    if tuple(target.shape) != (P, R, sout) or target.dtype != torch.float32 or not target.is_contiguous():
        raise _lib.DiffusError(f"target must be contiguous float32 {(P, R, sout)}")


def _workspace(args, nbytes: int, dev) -> torch.Tensor:
    """Scratch of ``nbytes`` (from the entry point's ``*_workspace_bytes``) set in ``args``; the caller keeps the tensor alive
    until the call is enqueued."""
    ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=dev)
    args.workspace, args.workspace_bytes = ws.data_ptr(), nbytes
    return ws


def _fill_render_args(a: DiffusRenderArgs, volume, bricks, dims, sources, directions, n_samples, start, alpha,
                      sampler, product_f32):
    layout = _packed_layout(bricks)
    if layout == LAYOUT_TEXTURE:
        a.volume.data = _texture_of(bricks).texture          # the 64-bit texture object travels in the pointer field
    else:
        a.volume.data = (volume if layout == LAYOUT_LINEAR else bricks).data_ptr()
    a.volume.dim[0], a.volume.dim[1], a.volume.dim[2] = dims
    a.volume.layout = layout
    a.sources = sources.data_ptr()
    a.directions = directions.data_ptr()
    a.pose_dtype = _pose_tag(sources, directions)
    a.product_f32 = int(product_f32)
    P = sources.shape[0]
    R = directions.shape[-2]
    a.n_poses, a.n_rays = P, R
    a.dir_pose_stride = R * 3 if directions.dim() == 3 else 0     # (R,3): one fan shared by all poses
    a.n_samples, a.start, a.sampler, a.attenuation = n_samples, start, sampler, alpha
    return P, R


def _pose_tag(sources, directions) -> int:
    """(P,3) sources: one source per pose; (P,R,3): one origin per ray (array probes, float32 only)."""
    if sources.dim() == 3:
        if sources.dtype != torch.float32:
            raise _lib.DiffusError("per-ray sources (P,R,3) must be float32: there is no float64 per-ray form")
        if sources.shape[1] != directions.shape[-2] or sources.shape[2] != 3 or not sources.is_contiguous():
            raise _lib.DiffusError("per-ray sources must be contiguous (P,R,3) with R the rays of the directions")
        return POSE_F32_PER_RAY
    return POSE_F64 if sources.dtype == torch.float64 else POSE_F32


def _check_inputs(volume, bricks, dims, sources, directions):
    if volume.dtype != torch.float32 or not volume.is_contiguous():
        raise _lib.DiffusError("volume must be a contiguous float32 tensor")
    if sources.dtype not in (torch.float32, torch.float64) or sources.dtype != directions.dtype:
        raise _lib.DiffusError("sources/directions must both be float32 or both float64")
    if sources.dim() not in (2, 3) or sources.shape[-1] != 3 or not sources.is_contiguous():
        raise _lib.DiffusError("sources must be contiguous (P,3), or (P,R,3) for one origin per ray")
    _pose_tag(sources, directions)
    if directions.shape[-1] != 3 or directions.dim() not in (2, 3) or not directions.is_contiguous():
        raise _lib.DiffusError("directions must be contiguous (R,3) or (P,R,3)")
    if directions.dim() == 3 and directions.shape[0] != sources.shape[0]:
        raise _lib.DiffusError("directions (P,R,3) must have one fan per source")
    if len(dims) != 3:
        raise _lib.DiffusError("dims must have three entries")


# ---------------------------------------------------------------------------------------
# render
# ---------------------------------------------------------------------------------------
def render_fwd_impl(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
               directions: torch.Tensor, n_samples: int, start: int, alpha: float, sampler: int,
               product_f32: bool, save_prefix: bool, prefix_only: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """``prefix_only``: only the 512-column transfer-matrix prefixes are wanted (the fused backward of long rays):
    no frame is formed or written and the last segment is not walked."""
    dev = _require_cuda(volume, bricks, sources, directions)
    _check_inputs(volume, bricks, dims, sources, directions)
    lib = _lib.load()
    a = DiffusRenderArgs()
    with _on_device(dev):
        P, R = _fill_render_args(a, volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler,
                                 product_f32)
        sout = n_samples - start
        nseg = _nseg(sout)
        prefix_only = prefix_only and save_prefix and nseg > 1
        frame = torch.empty((0,) if prefix_only else (P, R, max(sout, 0)), dtype=torch.float32, device=dev)
        prefix = torch.empty((P, R, nseg - 1, 4) if (save_prefix and nseg > 1) else (0,), dtype=torch.float32,
                             device=dev)         # (a fresh tensor even when empty: outputs of a custom op must not be shared)
        a.frame = frame.data_ptr() if frame.numel() else None
        a.seg_prefix = _ptr(prefix)
        wbytes = lib.diffus_render_workspace_bytes(C.byref(a)) if start > 0 else 0      # only the median needs scratch
        ws = _workspace(a, wbytes, dev) if wbytes else None
        _lib.check(lib.diffus_render_forward(C.byref(a), _stream(dev)), "diffus_render_forward")
    return frame, prefix


@torch.library.custom_op("diffus::render_fwd", mutates_args=())
def render_fwd(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
               directions: torch.Tensor, n_samples: int, start: int, alpha: float, sampler: int,
               product_f32: bool, save_prefix: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    return render_fwd_impl(volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32, save_prefix)


@render_fwd.register_fake
def _(volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32, save_prefix):
    P, R = sources.shape[0], directions.shape[-2]
    sout = n_samples - start
    nseg = _nseg(sout)
    frame = volume.new_empty((P, R, sout), dtype=torch.float32)
    prefix = volume.new_empty((P, R, nseg - 1, 4) if (save_prefix and nseg > 1) else (0,), dtype=torch.float32)
    return frame, prefix


def render_bwd_impl(grad_frame: torch.Tensor, volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int],
               sources: torch.Tensor, directions: torch.Tensor, prefix: torch.Tensor, n_samples: int, start: int,
               alpha: float, sampler: int, product_f32: bool, need_volume: bool,
               need_pose: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    dev = _require_cuda(grad_frame, volume, bricks, sources, directions)
    _check_inputs(volume, bricks, dims, sources, directions)
    lib = _lib.load()
    b = DiffusRenderBwdArgs()
    with _on_device(dev):
        P, R = _fill_render_args(b.fwd, volume, bricks, dims, sources, directions, n_samples, start, alpha,
                                 sampler, product_f32)
        grad_frame = grad_frame.contiguous().float()
        need_pose = _pose_grad(need_pose, sampler)
        gvol = _zero_grad_volume(bricks, dims, dev) if need_volume else torch.empty((0,), dtype=torch.float32, device=dev)
        gsrc = torch.empty(tuple(sources.shape) if need_pose else (0,), dtype=torch.float32, device=dev)
        gdir = torch.empty((P, R, 3) if need_pose else (0,), dtype=torch.float32, device=dev)
        b.fwd.seg_prefix = _ptr(prefix)
        b.grad_frame = grad_frame.data_ptr()
        b.grad_volume, b.grad_sources, b.grad_directions = _ptr(gvol), _ptr(gsrc), _ptr(gdir)
        b.target, b.loss, b.fwd.frame = None, None, None
        ws = _workspace(b, lib.diffus_render_bwd_workspace_bytes(C.byref(b)), dev)
        b.fwd.workspace, b.fwd.workspace_bytes = None, 0
        _lib.check(lib.diffus_render_backward(C.byref(b), _stream(dev)), "diffus_render_backward")
        if need_volume:
            gvol = _linear_grad_volume(gvol, bricks, dims)
    return gvol, gsrc, gdir


@torch.library.custom_op("diffus::render_bwd", mutates_args=())
def render_bwd(grad_frame: torch.Tensor, volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int],
               sources: torch.Tensor, directions: torch.Tensor, prefix: torch.Tensor, n_samples: int, start: int,
               alpha: float, sampler: int, product_f32: bool, need_volume: bool,
               need_pose: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return render_bwd_impl(grad_frame, volume, bricks, dims, sources, directions, prefix, n_samples, start, alpha, sampler, product_f32, need_volume, need_pose)


@render_bwd.register_fake
def _(grad_frame, volume, bricks, dims, sources, directions, prefix, n_samples, start, alpha, sampler, product_f32,
      need_volume, need_pose):
    P, R = sources.shape[0], directions.shape[-2]
    need_pose = _pose_grad(need_pose, sampler)
    gvol = volume.new_empty(tuple(dims) if need_volume else (0,), dtype=torch.float32)
    gsrc = volume.new_empty(tuple(sources.shape) if need_pose else (0,), dtype=torch.float32)
    gdir = volume.new_empty((P, R, 3) if need_pose else (0,), dtype=torch.float32)
    return gvol, gsrc, gdir


def _render_setup(ctx, inputs, output):
    (volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32, save_prefix) = inputs
    ctx.save_for_backward(volume, bricks if bricks is not None else volume.new_empty(0), sources, directions,
                          output[1])
    ctx.has_bricks = bricks is not None
    ctx.meta = (list(dims), n_samples, start, alpha, sampler, product_f32, save_prefix)


def _pose_grads(ctx, need_pose, gs, gd, src_dtype, dir_dtype, dir_dim, scale=None):
    """d/d sources and d/d directions (inputs 3 and 4) in their dtypes, or None where not requested: the (P,R,3) direction
    gradient of a fan shared by all poses (R,3) is summed over the poses; ``scale`` multiplies both before the cast."""
    gsrc = gdir = None
    if need_pose and ctx.needs_input_grad[3]:
        gsrc = (gs if scale is None else gs * scale).to(src_dtype)
    if need_pose and ctx.needs_input_grad[4]:
        d = gd if dir_dim == 3 else gd.sum(0)
        gdir = (d if scale is None else d * scale).to(dir_dtype)
    return gsrc, gdir


def _render_grads(ctx, grad_frame, bwd):
    """The backward of a render: ``(d volume, None, None, d sources, d directions)`` through ``bwd`` (the registered op or its
    impl) from what :func:`_render_setup` saved."""
    volume, bricks, sources, directions, prefix = ctx.saved_tensors
    dims, n_samples, start, alpha, sampler, product_f32, save_prefix = ctx.meta
    need_volume = ctx.needs_input_grad[0]
    need_pose = _pose_grad(ctx.needs_input_grad[3] or ctx.needs_input_grad[4], sampler)
    if _nseg(n_samples - start) > 1 and not save_prefix:
        raise _lib.DiffusError("render_fwd was called with save_prefix=False but a gradient was requested")
    if not (need_volume or need_pose):
        return None, None, None, None, None
    gv, gs, gd = bwd(grad_frame, volume, bricks if ctx.has_bricks else None, dims, sources, directions, prefix, n_samples,
                     start, alpha, sampler, product_f32, need_volume, need_pose)
    gsrc, gdir = _pose_grads(ctx, need_pose, gs, gd, sources.dtype, directions.dtype, directions.dim())
    return gv if need_volume else None, None, None, gsrc, gdir


def _render_backward(ctx, grad_frame, grad_prefix):
    return _render_grads(ctx, grad_frame, render_bwd) + (None,) * 6


torch.library.register_autograd("diffus::render_fwd", _render_backward, setup_context=_render_setup)


class RenderFunction(torch.autograd.Function):
    """Eager-mode autograd wrapper of render_fwd/render_bwd that skips the dispatcher (the registered
    ``diffus::render_fwd`` op carries the same autograd for torch.compile / fake-tensor users)."""

    @staticmethod
    def forward(ctx, volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32):
        out = render_fwd_impl(volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32, True)
        _render_setup(ctx, (volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler, product_f32, True), out)
        return out[0]

    @staticmethod
    def backward(ctx, grad_frame):
        return _render_grads(ctx, grad_frame, render_bwd_impl) + (None,) * 5


# ---------------------------------------------------------------------------------------
# fused forward + MSE loss + backward: one gather pass per pose-recovery / training step
# ---------------------------------------------------------------------------------------
def render_mse_impl(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
               directions: torch.Tensor, target: torch.Tensor, n_samples: int, start: int, alpha: float,
               sampler: int, product_f32: bool, need_volume: bool, need_pose: bool,
               want_frame: bool, keep_brick_grad: bool = False, n_total: Optional[int] = None,
               grad_volume_out: Optional[torch.Tensor] = None, loss_out: Optional[torch.Tensor] = None,
               grad_sources_out: Optional[torch.Tensor] = None
               ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """loss = mean((frame - target)^2) with d loss/d volume, d loss/d sources, d loss/d directions.

    Returns ``(loss (1,), frame or empty, grad_volume or empty, grad_sources or empty,
    grad_directions (P,R,3) or empty)``.  For rays of at most 512 columns, and for rays of 513..2048 columns
    with a pose gradient only (one CTA per ray, one 512-column pass per warp), this is ONE kernel
    launch (+ one launch for the two small reductions); other long rays first run the forward kernel for the
    512-column segment prefixes.

    ``n_total``: number of frame elements of the GLOBAL batch when this call renders one rank's shard of it -- loss and
    gradients are then this shard's share of the global mean, so that a SUM all-reduce over ranks gives exactly the
    single-process result even for ragged shards.  ``grad_volume_out`` (a zero-filled buffer in the gradient layout) and
    ``loss_out`` (1 float) let a training loop hand in persistent buffers instead of fresh allocations; ``grad_sources_out``
    (3P floats, 3PR for per-ray sources) likewise for d loss / d sources (a slice of a CUDA graph's static output block).
    """
    dev = _require_cuda(volume, bricks, sources, directions, target)
    _check_inputs(volume, bricks, dims, sources, directions)
    lib = _lib.load()
    b = DiffusRenderBwdArgs()
    with _on_device(dev):
        P, R = _fill_render_args(b.fwd, volume, bricks, dims, sources, directions, n_samples, start, alpha,
                                 sampler, product_f32)
        sout = n_samples - start
        _check_target(target, P, R, sout)
        need_pose = _pose_grad(need_pose, sampler)
        n = P * R * sout if n_total is None else int(n_total)
        def empty():                      # outputs of a custom op must not alias each other
            return torch.empty((0,), dtype=torch.float32, device=dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev) if loss_out is None else loss_out
        frame = torch.empty((P, R, sout), dtype=torch.float32, device=dev) if want_frame else empty()
        if need_volume and grad_volume_out is not None:
            gshape = _grad_volume_shape(bricks, dims)
            if tuple(grad_volume_out.shape) != tuple(gshape) or grad_volume_out.dtype != torch.float32:
                raise _lib.DiffusError(f"grad_volume_out must be float32 {tuple(gshape)}")
            gvol = grad_volume_out
        else:
            gvol = _zero_grad_volume(bricks, dims, dev) if need_volume else empty()
        gsrc = _out_buffer(grad_sources_out, tuple(sources.shape), dev, "grad_sources_out") if need_pose else empty()
        gdir = torch.empty((P, R, 3), dtype=torch.float32, device=dev) if need_pose else empty()
        b.grad_frame = None
        b.grad_volume, b.grad_sources, b.grad_directions = _ptr(gvol), _ptr(gsrc), _ptr(gdir)
        # rays longer than 512 columns: the 512-column prefixes come from a prefix-only run of the forward kernel -- unless
        # the library walks the passes of a ray in one CTA (513..2048 columns, pose gradient only) and forms them itself
        prefix = None
        need_prefix = _lib.check_count(lib.diffus_render_bwd_needs_prefix(C.byref(b)), "diffus_render_bwd_needs_prefix")
        if need_prefix:
            _, prefix = render_fwd_impl(volume, bricks, dims, sources, directions, n_samples, start, alpha, sampler,
                                        product_f32, True, prefix_only=True)
        b.fwd.frame = _ptr(frame)
        b.fwd.seg_prefix = _ptr(prefix)
        b.target, b.grad_scale, b.loss_scale, b.loss = target.data_ptr(), 2.0 / n, 1.0 / n, loss.data_ptr()
        ws = _workspace(b, lib.diffus_render_bwd_workspace_bytes(C.byref(b)), dev)
        _lib.check(lib.diffus_render_backward(C.byref(b), _stream(dev)), "diffus_render_backward (fused MSE)")
        if need_volume and not keep_brick_grad:
            gvol = _linear_grad_volume(gvol, bricks, dims)
    return loss, frame, gvol, gsrc, gdir


@torch.library.custom_op("diffus::render_mse", mutates_args=())
def render_mse(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
               directions: torch.Tensor, target: torch.Tensor, n_samples: int, start: int, alpha: float,
               sampler: int, product_f32: bool, need_volume: bool, need_pose: bool,
               want_frame: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return render_mse_impl(volume, bricks, dims, sources, directions, target, n_samples, start, alpha, sampler, product_f32, need_volume, need_pose, want_frame)


@render_mse.register_fake
def _(volume, bricks, dims, sources, directions, target, n_samples, start, alpha, sampler, product_f32, need_volume,
      need_pose, want_frame):
    P, R = sources.shape[0], directions.shape[-2]
    need_pose = _pose_grad(need_pose, sampler)
    def e():
        return volume.new_empty((0,), dtype=torch.float32)
    return (volume.new_empty((1,), dtype=torch.float32),
            volume.new_empty((P, R, n_samples - start), dtype=torch.float32) if want_frame else e(),
            volume.new_empty(tuple(dims), dtype=torch.float32) if need_volume else e(),
            volume.new_empty(tuple(sources.shape), dtype=torch.float32) if need_pose else e(),
            volume.new_empty((P, R, 3), dtype=torch.float32) if need_pose else e())


class RenderMSELoss(torch.autograd.Function):
    """Autograd wrapper of the fused step: the gradients are produced in the forward call."""

    @staticmethod
    def forward(ctx, volume, bricks, dims, sources, directions, target, n_samples, start, alpha, sampler,
                product_f32, want_frame):
        need_volume = ctx.needs_input_grad[0]
        need_pose = _pose_grad(ctx.needs_input_grad[3] or ctx.needs_input_grad[4], sampler)
        loss, frame, gvol, gsrc, gdir = render_mse_impl(volume.detach(), bricks, dims, sources.detach(),
                                                        directions.detach(), target, n_samples, start, alpha, sampler,
                                                        product_f32, need_volume, need_pose, want_frame)
        ctx.save_for_backward(gvol, gsrc, gdir)
        ctx.flags = (need_volume, need_pose, sources.dtype, directions.dtype, directions.dim())
        ctx.mark_non_differentiable(frame)
        return loss.reshape(()), frame

    @staticmethod
    def backward(ctx, gloss, gframe):
        gvol, gsrc, gdir = ctx.saved_tensors
        need_volume, need_pose, sdt, ddt, ddim = ctx.flags
        out_v = gvol * gloss if need_volume and ctx.needs_input_grad[0] else None
        out_s, out_d = _pose_grads(ctx, need_pose, gsrc, gdir, sdt, ddt, ddim, scale=gloss)
        return out_v, None, None, out_s, out_d, None, None, None, None, None, None, None


# ---------------------------------------------------------------------------------------
# Gauss-Newton system of each pose: one forward-mode render pass
# ---------------------------------------------------------------------------------------
def render_gauss_newton_impl(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
                             directions: torch.Tensor, target: torch.Tensor, n_samples: int, start: int, alpha: float,
                             loss_out: Optional[torch.Tensor] = None, jtj_out: Optional[torch.Tensor] = None,
                             jtr_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Per pose p, with res = frame - target and J = d frame / d xi for a rigid twist xi = (v, w) of the pose about its source
    (per-ray sources (P,R,3): about the pose's pivot, the float64 mean of its origins):
    ``loss[p] = sum res^2``, ``JtJ[p] = J^T J`` (6x6), ``Jtr[p] = J^T res`` (6).  Trilinear sampler, float32 poses.

    Two launches (+ two for the median when ``start > 0``).  ``*_out``: caller-provided output buffers (static tensors of a
    CUDA graph), else fresh tensors."""
    dev = _require_cuda(volume, bricks, sources, directions, target)
    _check_inputs(volume, bricks, dims, sources, directions)
    lib = _lib.load()
    g = _lib.DiffusGaussNewtonArgs()
    with _on_device(dev):
        P, R = _fill_render_args(g.fwd, volume, bricks, dims, sources, directions, n_samples, start, alpha, SAMPLER_TRILINEAR,
                                 False)
        _check_target(target, P, R, n_samples - start)
        loss = _out_buffer(loss_out, (P,), dev, "loss_out")
        jtj = _out_buffer(jtj_out, (P, 6, 6), dev, "jtj_out")
        jtr = _out_buffer(jtr_out, (P, 6), dev, "jtr_out")
        g.target, g.loss, g.jtr, g.jtj = target.data_ptr(), loss.data_ptr(), jtr.data_ptr(), jtj.data_ptr()
        ws = _workspace(g, lib.diffus_render_gauss_newton_workspace_bytes(C.byref(g)), dev)
        _lib.check(lib.diffus_render_gauss_newton(C.byref(g), _stream(dev)), "diffus_render_gauss_newton")
    return loss.view(P), jtj.view(P, 6, 6), jtr.view(P, 6)


def render_gauss_newton_sweep_impl(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
                                   directions: torch.Tensor, target: torch.Tensor, n_samples: int, start: int, alpha: float,
                                   pivot: Optional[torch.Tensor] = None, loss_out: Optional[torch.Tensor] = None,
                                   jtj_out: Optional[torch.Tensor] = None,
                                   jtr_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """ONE system for all poses of a tracked sweep, with res = frame - target and J = d frame / d xi for one rigid twist
    xi = (v, w) about ``pivot`` c shared by every pose: ``p_k = c + v + Rot(w) (s_i - c + k d_i)`` (s_i the pose's source or the
    ray's own origin).  Returns float64 ``loss () = sum res^2``, ``JtJ (6,6)``, ``Jtr (6,)`` over all P x R x (S-start) elements.
    ``pivot``: a (3,) float64 CUDA tensor (read on the device, so a graph replay sees its current value), or None for the mean of
    all ray origins.  Trilinear sampler, float32 poses.

    Four launches (+ two for the pivot when none is given, + two for the median when ``start > 0``).  ``*_out``: caller-provided
    float64 output buffers (static tensors of a CUDA graph), else fresh tensors."""
    dev = _require_cuda(volume, bricks, sources, directions, target)
    _check_inputs(volume, bricks, dims, sources, directions)
    if pivot is not None and (tuple(pivot.shape) != (3,) or pivot.dtype != torch.float64 or not pivot.is_contiguous()
                              or pivot.device != dev):
        raise _lib.DiffusError(f"pivot must be a contiguous float64 (3,) tensor on {dev}")
    lib = _lib.load()
    g = _lib.DiffusGaussNewtonSweepArgs()
    with _on_device(dev):
        P, R = _fill_render_args(g.fwd, volume, bricks, dims, sources, directions, n_samples, start, alpha, SAMPLER_TRILINEAR,
                                 False)
        _check_target(target, P, R, n_samples - start)
        loss = _out_buffer(loss_out, (), dev, "loss_out", torch.float64)
        jtj = _out_buffer(jtj_out, (6, 6), dev, "jtj_out", torch.float64)
        jtr = _out_buffer(jtr_out, (6,), dev, "jtr_out", torch.float64)
        g.target, g.loss, g.jtr, g.jtj = target.data_ptr(), loss.data_ptr(), jtr.data_ptr(), jtj.data_ptr()
        g.pivot = None if pivot is None else pivot.data_ptr()
        ws = _workspace(g, lib.diffus_render_gauss_newton_sweep_workspace_bytes(C.byref(g)), dev)
        _lib.check(lib.diffus_render_gauss_newton_sweep(C.byref(g), _stream(dev)), "diffus_render_gauss_newton_sweep")
    return loss.view(()), jtj.view(6, 6), jtr.view(6)


@torch.library.custom_op("diffus::render_gn", mutates_args=())
def render_gn(volume: torch.Tensor, bricks: Optional[torch.Tensor], dims: List[int], sources: torch.Tensor,
              directions: torch.Tensor, target: torch.Tensor, n_samples: int, start: int,
              alpha: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return render_gauss_newton_impl(volume, bricks, dims, sources, directions, target, n_samples, start, alpha)


@render_gn.register_fake
def _(volume, bricks, dims, sources, directions, target, n_samples, start, alpha):
    P = sources.shape[0]
    return (volume.new_empty((P,), dtype=torch.float32), volume.new_empty((P, 6, 6), dtype=torch.float32),
            volume.new_empty((P, 6), dtype=torch.float32))


# ---------------------------------------------------------------------------------------
# indices / raw values
# ---------------------------------------------------------------------------------------
def ray_indices(dims, sources, directions, n_samples, start, product_f32=False):
    """int64 (P,R,S-start) nearest-voxel indices x, y, z (reference ``src/renderer.py:754-756``)."""
    dev = _require_cuda(sources, directions)
    lib = _lib.load()
    a = DiffusRenderArgs()
    with _on_device(dev):
        dummy = torch.empty((1,), dtype=torch.float32, device=dev)
        P, R = _fill_render_args(a, dummy, None, dims, sources, directions, n_samples, start, 0.0, SAMPLER_NEAREST,
                                 product_f32)
        out = torch.empty((3, P, R, n_samples - start), dtype=torch.int64, device=dev)
        _lib.check(lib.diffus_ray_indices(C.byref(a), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                          _stream(dev)), "diffus_ray_indices")
    return out[0], out[1], out[2]


def trace_values(volume, bricks, dims, sources, directions, n_samples, sampler, product_f32=False):
    """float32 (P,R,S) impedances along the rays (reference ``trace_ray``'s values)."""
    dev = _require_cuda(volume, bricks, sources, directions)
    _check_inputs(volume, bricks, dims, sources, directions)
    lib = _lib.load()
    a = DiffusRenderArgs()
    with _on_device(dev):
        P, R = _fill_render_args(a, volume, bricks, dims, sources, directions, n_samples, 0, 0.0, sampler, product_f32)
        out = torch.empty((P, R, n_samples), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_trace_values(C.byref(a), out.data_ptr(), _stream(dev)), "diffus_trace_values")
    return out


def sample_points(volume: torch.Tensor, points: torch.Tensor, sampler: int):
    """Values and clamped nearest indices at explicit points (..., 3); volume (D,H,W) float32 CUDA."""
    dev = _require_cuda(volume, points)
    lib = _lib.load()
    v = volume.detach().float().contiguous()
    pts = points.detach().float().reshape(-1, 3).contiguous()
    n = pts.shape[0]
    vol = _lib.DiffusVolume()
    vol.data = v.data_ptr()
    vol.dim[0], vol.dim[1], vol.dim[2] = v.shape
    vol.layout = LAYOUT_LINEAR
    with _on_device(dev):
        val = torch.empty((n,), dtype=torch.float32, device=dev)
        idx = torch.empty((3, n), dtype=torch.int64, device=dev)
        if n:
            _lib.check(lib.diffus_sample_points(C.byref(vol), pts.data_ptr(), n, sampler, val.data_ptr(), idx[0].data_ptr(),
                                                idx[1].data_ptr(), idx[2].data_ptr(), _stream(dev)), "diffus_sample_points")
    shape = points.shape[:-1]
    return idx[0].reshape(shape), idx[1].reshape(shape), idx[2].reshape(shape), val.reshape(shape)


def trace_values_bwd(grad_values, volume, bricks, dims, sources, directions, n_samples, sampler, product_f32,
                     need_volume, need_pose):
    dev = _require_cuda(grad_values, volume, bricks, sources, directions)
    lib = _lib.load()
    a = DiffusRenderArgs()
    with _on_device(dev):
        P, R = _fill_render_args(a, volume, bricks, dims, sources, directions, n_samples, 0, 0.0, sampler, product_f32)
        need_pose = _pose_grad(need_pose, sampler)
        g = grad_values.contiguous().float()
        gvol = _zero_grad_volume(bricks, dims, dev) if need_volume else None
        gsrc = torch.empty(tuple(sources.shape), dtype=torch.float32, device=dev) if need_pose else None
        gdir = torch.empty((P, R, 3), dtype=torch.float32, device=dev) if need_pose else None
        ws = torch.empty((max(P * R * 12 + 256, 256),), dtype=torch.uint8, device=dev)
        _lib.check(lib.diffus_trace_values_backward(C.byref(a), g.data_ptr(), _ptr(gvol), _ptr(gsrc), _ptr(gdir),
                                                    ws.data_ptr(), ws.numel(), _stream(dev)),
                   "diffus_trace_values_backward")
        if need_volume:
            gvol = _linear_grad_volume(gvol, bricks, dims)
    return gvol, gsrc, gdir


class TraceValuesFunction(torch.autograd.Function):
    """Sampled impedances along rays, differentiable like the reference's sampler."""

    @staticmethod
    def forward(ctx, volume, bricks, dims, sources, directions, n_samples, sampler, product_f32):
        ctx.save_for_backward(volume, sources, directions)
        ctx.bricks = bricks
        ctx.meta = (list(dims), n_samples, sampler, product_f32)
        return trace_values(volume, bricks, dims, sources, directions, n_samples, sampler, product_f32)

    @staticmethod
    def backward(ctx, grad):
        volume, sources, directions = ctx.saved_tensors
        dims, n_samples, sampler, product_f32 = ctx.meta
        need_volume = ctx.needs_input_grad[0]
        need_pose = _pose_grad(ctx.needs_input_grad[3] or ctx.needs_input_grad[4], sampler)
        gvol = gsrc = gdir = None
        if need_volume or need_pose:
            gvol, gs, gd = trace_values_bwd(grad, volume, ctx.bricks, dims, sources, directions, n_samples, sampler,
                                            product_f32, need_volume, need_pose)
            gsrc, gdir = _pose_grads(ctx, need_pose, gs, gd, sources.dtype, directions.dtype, directions.dim())
        return gvol, None, None, gsrc, gdir, None, None, None


# ---------------------------------------------------------------------------------------
# echo traces on explicit reflection coefficients
# ---------------------------------------------------------------------------------------
def echo_fwd_impl(refl: torch.Tensor) -> torch.Tensor:
    dev = _require_cuda(refl)
    lib = _lib.load()
    r = refl.contiguous().float()
    B, N = r.shape
    with _on_device(dev):
        out = torch.empty((B, N + 1), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_echo_forward(r.data_ptr(), B, N, out.data_ptr(), _stream(dev)), "diffus_echo_forward")
    return out


@torch.library.custom_op("diffus::echo_fwd", mutates_args=())
def echo_fwd(refl: torch.Tensor) -> torch.Tensor:
    return echo_fwd_impl(refl)


@echo_fwd.register_fake
def _(refl):
    return refl.new_empty((refl.shape[0], refl.shape[1] + 1), dtype=torch.float32)


def echo_bwd_impl(refl: torch.Tensor, grad_echo: torch.Tensor) -> torch.Tensor:
    dev = _require_cuda(refl, grad_echo)
    lib = _lib.load()
    r = refl.contiguous().float()
    g = grad_echo.contiguous().float()
    B, N = r.shape
    with _on_device(dev):
        out = torch.empty((B, N), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_echo_backward(r.data_ptr(), g.data_ptr(), B, N, out.data_ptr(), _stream(dev)),
                   "diffus_echo_backward")
    return out


@torch.library.custom_op("diffus::echo_bwd", mutates_args=())
def echo_bwd(refl: torch.Tensor, grad_echo: torch.Tensor) -> torch.Tensor:
    return echo_bwd_impl(refl, grad_echo)


@echo_bwd.register_fake
def _(refl, grad_echo):
    return refl.new_empty(refl.shape, dtype=torch.float32)


def _echo_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])


def _echo_backward(ctx, grad):
    (refl,) = ctx.saved_tensors
    return echo_bwd(refl, grad).to(refl.dtype)


torch.library.register_autograd("diffus::echo_fwd", _echo_backward, setup_context=_echo_setup)


# ---------------------------------------------------------------------------------------
# fans, bricks
# ---------------------------------------------------------------------------------------
def cone_directions(median: torch.Tensor, opening_angle: float, n_rays: int) -> torch.Tensor:
    """(P,2+) median directions -> (P,R,3) float32 fans in the z=0 plane, on the device."""
    dev = _require_cuda(median)
    lib = _lib.load()
    m = median[..., :2].to(torch.float64).contiguous()
    P = m.shape[0]
    with _on_device(dev):
        out = torch.empty((P, n_rays, 3), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_cone_directions(m.data_ptr(), P, n_rays, float(opening_angle), out.data_ptr(),
                                              _stream(dev)), "diffus_cone_directions")
    return out


def fan_directions_fwd(median: torch.Tensor, hint: torch.Tensor, opening_angle: float, n_rays: int) -> torch.Tensor:
    dev = _require_cuda(median, hint)
    lib = _lib.load()
    m, h = median.detach().float().contiguous(), hint.detach().float().contiguous()
    if m.dim() != 2 or m.shape[1] != 3 or h.shape != m.shape:
        raise _lib.DiffusError("median and hint must both be (P,3)")
    P = m.shape[0]
    with _on_device(dev):
        out = torch.empty((P, n_rays, 3), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_fan_directions(m.data_ptr(), h.data_ptr(), P, n_rays, float(opening_angle), out.data_ptr(),
                                             _stream(dev)), "diffus_fan_directions")
    return out


def _out_buffer(out: Optional[torch.Tensor], shape, dev, what: str, dtype=torch.float32) -> torch.Tensor:
    """A caller-provided contiguous output of the right size and dtype (e.g. a slice of a static block inside a CUDA graph), or a
    fresh tensor."""
    if out is None:
        return torch.empty(shape, dtype=dtype, device=dev)
    n = 1
    for d in shape:
        n *= d
    if out.dtype != dtype or not out.is_contiguous() or out.numel() != n or out.device != dev:
        raise _lib.DiffusError(f"{what} must be a contiguous {str(dtype).replace('torch.', '')} CUDA tensor of {n} elements on {dev}")
    return out


def fan_directions_bwd(median: torch.Tensor, hint: torch.Tensor, grad_dirs: torch.Tensor, opening_angle: float,
                       n_rays: int, grad_median_out: Optional[torch.Tensor] = None,
                       grad_hint_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    dev = _require_cuda(median, hint, grad_dirs)
    lib = _lib.load()
    m, h = median.detach().float().contiguous(), hint.detach().float().contiguous()
    g = grad_dirs.float().contiguous()
    P = m.shape[0]
    with _on_device(dev):
        gm = _out_buffer(grad_median_out, (P, 3), dev, "grad_median_out")
        gh = _out_buffer(grad_hint_out, (P, 3), dev, "grad_hint_out")
        _lib.check(lib.diffus_fan_directions_backward(m.data_ptr(), h.data_ptr(), g.data_ptr(), P, n_rays, float(opening_angle),
                                                      gm.data_ptr(), gh.data_ptr(), _stream(dev)),
                   "diffus_fan_directions_backward")
    return gm, gh


class FanDirectionsFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, median, hint, opening_angle, n_rays):
        ctx.save_for_backward(median, hint)
        ctx.angle, ctx.n_rays = float(opening_angle), int(n_rays)
        return fan_directions_fwd(median, hint, opening_angle, n_rays)

    @staticmethod
    def backward(ctx, grad):
        median, hint = ctx.saved_tensors
        gm, gh = fan_directions_bwd(median, hint, grad, ctx.angle, ctx.n_rays)
        return gm.to(median.dtype), gh.to(hint.dtype), None, None


def fan_directions(median: torch.Tensor, normal_hint: torch.Tensor, opening_angle: float, n_rays: int) -> torch.Tensor:
    """Fans of a batch of poses from their parameters, on the device and differentiable: (P,3) median directions and
    (P,3) in-plane hints -> (P,R,3) float32 unit directions ``cos(a) m^ + sin(a) u^`` -- ``generate_cone_directions``
    (reference ``src/cone.py:242-259``) generalised from the z = 0 plane to the plane spanned by median and hint."""
    return FanDirectionsFunction.apply(median, normal_hint, opening_angle, n_rays)


_PROBE_KINDS = {"convex": PROBE_CONVEX, "linear": PROBE_LINEAR}


def probe_kind(kind: str) -> int:
    try:
        return _PROBE_KINDS[kind]
    except KeyError:
        raise ValueError(f"unknown probe kind {kind!r}; expected 'convex' or 'linear'") from None


def _probe_params(median, hint):
    m, h = median.detach().float().contiguous(), hint.detach().float().contiguous()
    if m.dim() != 2 or m.shape[1] != 3 or h.shape != m.shape:
        raise _lib.DiffusError("centre, median and hint must all be (P,3)")
    return m, h


def probe_rays_fwd(kind: int, centre: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, n_rays: int, opening_angle: float,
                   radius: float, width: float, origins_out: Optional[torch.Tensor] = None,
                   directions_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(P,R,3) origins and directions of convex / linear array probes (``include/diffus_b200.h``: ``diffus_probe_rays``)."""
    dev = _require_cuda(centre, median, hint)
    lib = _lib.load()
    m, h = _probe_params(median, hint)
    c = centre.detach().float().contiguous()
    if c.shape != m.shape:
        raise _lib.DiffusError("centre, median and hint must all be (P,3)")
    P = m.shape[0]
    with _on_device(dev):
        o = _out_buffer(origins_out, (P, n_rays, 3), dev, "origins_out")
        d = _out_buffer(directions_out, (P, n_rays, 3), dev, "directions_out")
        _lib.check(lib.diffus_probe_rays(kind, c.data_ptr(), m.data_ptr(), h.data_ptr(), P, n_rays, float(opening_angle),
                                         float(radius), float(width), o.data_ptr(), d.data_ptr(), _stream(dev)),
                   "diffus_probe_rays")
    return o.view(P, n_rays, 3), d.view(P, n_rays, 3)


def probe_rays_bwd(kind: int, centre: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, grad_origins: torch.Tensor,
                   grad_directions: torch.Tensor, n_rays: int, opening_angle: float, radius: float, width: float,
                   grad_centre_out: Optional[torch.Tensor] = None, grad_median_out: Optional[torch.Tensor] = None,
                   grad_hint_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    dev = _require_cuda(centre, median, hint, grad_origins, grad_directions)
    lib = _lib.load()
    m, h = _probe_params(median, hint)
    c = centre.detach().float().contiguous()
    P = m.shape[0]
    go, gd = grad_origins.float().contiguous(), grad_directions.float().contiguous()
    if go.numel() != P * n_rays * 3 or gd.numel() != P * n_rays * 3:
        raise _lib.DiffusError(f"grad_origins and grad_directions must be {(P, n_rays, 3)}")
    with _on_device(dev):
        gc = _out_buffer(grad_centre_out, (P, 3), dev, "grad_centre_out")
        gm = _out_buffer(grad_median_out, (P, 3), dev, "grad_median_out")
        gh = _out_buffer(grad_hint_out, (P, 3), dev, "grad_hint_out")
        _lib.check(lib.diffus_probe_rays_backward(kind, c.data_ptr(), m.data_ptr(), h.data_ptr(), go.data_ptr(), gd.data_ptr(), P,
                                                  n_rays, float(opening_angle), float(radius), float(width), gc.data_ptr(),
                                                  gm.data_ptr(), gh.data_ptr(), _stream(dev)), "diffus_probe_rays_backward")
    return gc, gm, gh


class ProbeRaysFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, kind, centre, median, hint, n_rays, opening_angle, radius, width):
        ctx.save_for_backward(centre, median, hint)
        ctx.args = (int(kind), int(n_rays), float(opening_angle), float(radius), float(width))
        return probe_rays_fwd(kind, centre, median, hint, n_rays, opening_angle, radius, width)

    @staticmethod
    def backward(ctx, g_origins, g_dirs):
        centre, median, hint = ctx.saved_tensors
        kind, n_rays, angle, radius, width = ctx.args
        if g_origins is None:
            g_origins = torch.zeros((centre.shape[0], n_rays, 3), dtype=torch.float32, device=centre.device)
        if g_dirs is None:
            g_dirs = torch.zeros((centre.shape[0], n_rays, 3), dtype=torch.float32, device=centre.device)
        gc, gm, gh = probe_rays_bwd(kind, centre, median, hint, g_origins, g_dirs, n_rays, angle, radius, width)
        return None, gc.to(centre.dtype), gm.to(median.dtype), gh.to(hint.dtype), None, None, None, None


def probe_args(kind: str, opening_angle, radius, width) -> Tuple[int, float, float, float]:
    """Host-side check of the keywords of one probe kind -> ``(kind id, opening_angle, radius, width)`` for the kernels."""
    kid = probe_kind(kind)
    if kid == PROBE_CONVEX:
        if opening_angle is None:
            raise ValueError("a convex probe needs opening_angle")
        if not (math.isfinite(float(radius)) and float(radius) >= 0.0):
            raise ValueError(f"a convex probe needs a finite radius >= 0, got {radius!r}")
        return kid, float(opening_angle), float(radius), 0.0
    if width is None or not (math.isfinite(float(width)) and float(width) > 0.0):
        raise ValueError(f"a linear probe needs a finite width > 0, got {width!r}")
    return kid, 0.0, 0.0, float(width)


def probe_rays(kind: str, centre: torch.Tensor, median: torch.Tensor, hint: torch.Tensor, n_rays: int, *, opening_angle=None,
               radius: float = 0.0, width=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Rays of linear and convex array probes from their pose parameters, on the device and differentiable.

    ``centre``, ``median`` and ``hint`` are (P,3); ``m^ = median / |median|`` and ``u^`` is the hint made orthogonal to it and
    normalised (as in :func:`fan_directions`).  Returns ``(origins, directions)``, both (P,R,3) float32, to be rendered with
    the origins as per-ray ``sources``:

    * ``'convex'`` (``opening_angle``, ``radius`` rho >= 0): ray i leaves ``centre + rho d_i`` along ``d_i = cos a_i m^ +
      sin a_i u^``, ``a = linspace(-angle/2, angle/2, R)``.  With rho = 0 it is the sector probe of :func:`fan_directions`.
    * ``'linear'`` (``width`` w > 0): ray i leaves ``centre + t_i u^`` along ``m^``, ``t = linspace(-w/2, w/2, R)``.
    """
    kid, angle, rho, w = probe_args(kind, opening_angle, radius, width)
    return ProbeRaysFunction.apply(kid, centre, median, hint, int(n_rays), angle, rho, w)


def gather_probe(buffer_mib: int = 64, reads_per_thread: int = 64, n_threads: int = 148 * 8 * 256, repeats: int = 5,
                 device: Optional[torch.device] = None) -> dict:
    """Roofline probe (SURVEY 8d): random 32-byte-sector reads over a ``buffer_mib`` MiB buffer, timed with CUDA events.

    64 MiB (a 256^3 float32 volume) stays in L2 and gives the L2 -> SM random-sector rate the gather-bound march
    competes with; a buffer well above L2 (126 MB) gives the HBM random-sector rate.  Returns sectors/s and GB/s
    (32 bytes per sector).
    """
    dev = device or torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    with _on_device(dev):
        n = buffer_mib * (1 << 20) // 4
        buf = torch.ones((n,), dtype=torch.float32, device=dev)
        sink = torch.empty((n_threads,), dtype=torch.float32, device=dev)

        def launch(seed):
            _lib.check(lib.diffus_gather_probe(buf.data_ptr(), n, reads_per_thread, n_threads, seed, sink.data_ptr(),
                                               _stream(dev)), "diffus_gather_probe")
        for w in range(3):
            launch(w)                                     # warm-up: the buffer settles in L2 if it fits
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(repeats):
            launch(100 + r)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / repeats
        if abs(float(sink[0]) - reads_per_thread) > 0.5:
            raise _lib.DiffusError("gather probe returned a wrong sum")
    sectors = n_threads * reads_per_thread
    return {"buffer_mib": buffer_mib, "sectors_per_launch": sectors, "ms": ms, "sectors_per_s": sectors / (ms * 1e-3),
            "gb_per_s": sectors * 32 / (ms * 1e-3) / 1e9}


def to_bricks(volume: torch.Tensor) -> torch.Tensor:
    """LINEAR (D,H,W) float32 -> 1-D brick buffer (4x4x2 voxels per 128-byte line)."""
    dev = _require_cuda(volume)
    lib = _lib.load()
    v = volume.detach().contiguous().float()
    dim = (C.c_int32 * 3)(*v.shape)
    with _on_device(dev):
        out = torch.empty((lib.diffus_brick_elems(C.byref(dim)),), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_volume_to_bricks(v.data_ptr(), C.byref(dim), out.data_ptr(), _stream(dev)),
                   "diffus_volume_to_bricks")
    return out


def to_quads(volume: torch.Tensor) -> torch.Tensor:
    """LINEAR (D,H,W) float32 -> (n, 4) quad buffer: each voxel with its +p1, +p2, +p1+p2 neighbours (2x2x2 per 128 B)."""
    dev = _require_cuda(volume)
    lib = _lib.load()
    v = volume.detach().contiguous().float()
    dim = (C.c_int32 * 3)(*v.shape)
    with _on_device(dev):
        out = torch.empty((lib.diffus_quad_elems(C.byref(dim)) // 4, 4), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_volume_to_quads(v.data_ptr(), C.byref(dim), out.data_ptr(), _stream(dev)),
                   "diffus_volume_to_quads")
    return out


def gaussian_blur_volume(volume: torch.Tensor, sigma: float, truncate: float = 4.0) -> torch.Tensor:
    """``scipy.ndimage.gaussian_filter(volume, sigma, mode='nearest', truncate=truncate)`` of a (D,H,W) CUDA volume, computed in
    float32 (three separable passes); a new (D,H,W) float32 tensor.  Not differentiable."""
    dev = _require_cuda(volume)
    if volume.dim() != 3:
        raise _lib.DiffusError("volume must be (D,H,W)")
    v = volume.detach().contiguous().float()
    dim = (C.c_int32 * 3)(*v.shape)
    with _on_device(dev):
        out = torch.empty_like(v)
        scratch = torch.empty_like(v)
        _lib.check(_lib.load().diffus_volume_gaussian_blur(v.data_ptr(), C.byref(dim), float(sigma), float(truncate), out.data_ptr(),
                                                           scratch.data_ptr(), _stream(dev)), "diffus_volume_gaussian_blur")
    return out


def from_bricks(bricks: torch.Tensor, dims) -> torch.Tensor:
    dev = _require_cuda(bricks)
    lib = _lib.load()
    dim = (C.c_int32 * 3)(*dims)
    with _on_device(dev):
        out = torch.empty(tuple(dims), dtype=torch.float32, device=dev)
        _lib.check(lib.diffus_bricks_to_volume(bricks.data_ptr(), C.byref(dim), out.data_ptr(), _stream(dev)),
                   "diffus_bricks_to_volume")
    return out


# ---------------------------------------------------------------------------------------
# scan conversion (differentiable_splat)
# ---------------------------------------------------------------------------------------
def _splat_call(fwd: bool, coords, val, H, W, sigma, grad_out=None):
    dev = _require_cuda(*coords, val, grad_out)
    lib = _lib.load()
    c = [t.reshape(-1).to(torch.float32).contiguous() for t in coords]
    v = val.reshape(-1).to(torch.float32).contiguous()
    n = v.numel()
    with _on_device(dev):
        wbytes = lib.diffus_splat_workspace_bytes(H, W)
        ws = torch.empty((wbytes,), dtype=torch.uint8, device=dev)
        if fwd:
            out = torch.empty((W, H), dtype=torch.float32, device=dev)
            _lib.check(lib.diffus_splat_forward(c[0].data_ptr(), c[1].data_ptr(), c[2].data_ptr(), v.data_ptr(), n, H, W,
                                                float(sigma), out.data_ptr(), ws.data_ptr(), wbytes, _stream(dev)),
                       "diffus_splat_forward")
        else:
            g = grad_out.to(torch.float32).contiguous()
            out = torch.empty((n,), dtype=torch.float32, device=dev)
            _lib.check(lib.diffus_splat_backward(c[0].data_ptr(), c[1].data_ptr(), c[2].data_ptr(), v.data_ptr(), n, H, W,
                                                 float(sigma), g.data_ptr(), out.data_ptr(), ws.data_ptr(), wbytes,
                                                 _stream(dev)), "diffus_splat_backward")
    return out


class SplatFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, z, intensities, H, W, sigma):
        ctx.save_for_backward(x, y, z, intensities)
        ctx.meta = (H, W, sigma)
        return _splat_call(True, (x, y, z), intensities, H, W, sigma)

    @staticmethod
    def backward(ctx, grad):
        x, y, z, val = ctx.saved_tensors
        H, W, sigma = ctx.meta
        g = _splat_call(False, (x, y, z), val, H, W, sigma, grad).reshape(val.shape).to(val.dtype)
        return None, None, None, g, None, None, None


# ---------------------------------------------------------------------------------------
# MLP
# ---------------------------------------------------------------------------------------
MLP_PATH_AUTO, MLP_PATH_CUDA_CORES, MLP_PATH_PIECEWISE = 0, 1, 3
_MLP_PATH = MLP_PATH_AUTO      # tests and benchmarks pin a path through mlp_path(); AUTO = the piecewise-linear table for volumes


class mlp_path:
    """Context manager pinning the MLP forward and weight gradient to the CUDA-core kernels or the piecewise-linear
    table (default: automatic)."""

    def __init__(self, path: int):
        self.path = path

    def __enter__(self):
        global _MLP_PATH
        self.saved, _MLP_PATH = _MLP_PATH, self.path

    def __exit__(self, *exc):
        global _MLP_PATH
        _MLP_PATH = self.saved


def mlp_fwd_impl(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], out_scale: float,
            fill: float) -> torch.Tensor:
    dev = _require_cuda(params, x, mask)
    lib = _lib.load()
    if params.numel() != MLP_NPARAMS:
        raise _lib.DiffusError(f"params must hold {MLP_NPARAMS} floats")
    p = params.contiguous().float()
    xc = x.contiguous().float()
    m = None if mask is None else mask.contiguous().to(torch.uint8)
    with _on_device(dev):
        out = torch.empty(x.shape, dtype=torch.float32, device=dev)
        if xc.numel():
            _lib.check(lib.diffus_mlp_forward_ex(p.data_ptr(), xc.data_ptr(), _ptr(m), xc.numel(), out_scale, fill,
                                                 out.data_ptr(), _MLP_PATH, _stream(dev)), "diffus_mlp_forward")
    return out


@torch.library.custom_op("diffus::mlp_fwd", mutates_args=())
def mlp_fwd(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], out_scale: float,
            fill: float) -> torch.Tensor:
    return mlp_fwd_impl(params, x, mask, out_scale, fill)


@mlp_fwd.register_fake
def _(params, x, mask, out_scale, fill):
    return x.new_empty(x.shape, dtype=torch.float32)


def mlp_bwd_impl(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], grad_out: torch.Tensor,
            out_scale: float, grad_params_out: Optional[torch.Tensor] = None,
            workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``grad_params_out`` (>= 1153 floats, ACCUMULATED into) and ``workspace`` let a training loop reuse persistent buffers:
    the weight gradient then lands directly in the flat buffer that is all-reduced."""
    dev = _require_cuda(params, x, mask, grad_out)
    lib = _lib.load()
    p = params.contiguous().float()
    xc = x.contiguous().float()
    g = grad_out.contiguous().float()
    m = None if mask is None else mask.contiguous().to(torch.uint8)
    with _on_device(dev):
        gp = torch.zeros((MLP_NPARAMS,), dtype=torch.float32, device=dev) if grad_params_out is None else grad_params_out
        n = xc.numel()
        if n:
            wbytes = lib.diffus_mlp_bwd_workspace_bytes(n)
            ws = workspace if workspace is not None and workspace.numel() >= wbytes else \
                torch.empty((wbytes,), dtype=torch.uint8, device=dev)
            _lib.check(lib.diffus_mlp_backward_ex(p.data_ptr(), xc.data_ptr(), _ptr(m), g.data_ptr(), n, out_scale,
                                                  gp.data_ptr(), ws.data_ptr(), wbytes, _MLP_PATH, _stream(dev)),
                       "diffus_mlp_backward")
    return gp


@torch.library.custom_op("diffus::mlp_bwd", mutates_args=())
def mlp_bwd(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], grad_out: torch.Tensor,
            out_scale: float) -> torch.Tensor:
    return mlp_bwd_impl(params, x, mask, grad_out, out_scale)


@mlp_bwd.register_fake
def _(params, x, mask, grad_out, out_scale):
    return params.new_empty((MLP_NPARAMS,), dtype=torch.float32)


def _mlp_setup(ctx, inputs, output):
    params, x, mask, out_scale, fill = inputs
    ctx.save_for_backward(params, x, mask if mask is not None else x.new_empty(0))
    ctx.has_mask = mask is not None
    ctx.out_scale = out_scale


def mlp_input_grad_impl(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], grad_out: torch.Tensor,
                        out_scale: float) -> torch.Tensor:
    dev = _require_cuda(params, x, mask, grad_out)
    p, xc, g = params.contiguous().float(), x.contiguous().float(), grad_out.contiguous().float()
    m = None if mask is None else mask.contiguous().to(torch.uint8)
    with _on_device(dev):
        gx = torch.empty(x.shape, dtype=torch.float32, device=dev)
        if xc.numel():
            _lib.check(_lib.load().diffus_mlp_input_grad(p.data_ptr(), xc.data_ptr(), _ptr(m), g.data_ptr(), xc.numel(), out_scale,
                                                         gx.data_ptr(), _stream(dev)), "diffus_mlp_input_grad")
    return gx


@torch.library.custom_op("diffus::mlp_input_grad", mutates_args=())
def mlp_input_grad(params: torch.Tensor, x: torch.Tensor, mask: Optional[torch.Tensor], grad_out: torch.Tensor,
                   out_scale: float) -> torch.Tensor:
    return mlp_input_grad_impl(params, x, mask, grad_out, out_scale)


@mlp_input_grad.register_fake
def _(params, x, mask, grad_out, out_scale):
    return x.new_empty(x.shape, dtype=torch.float32)


def _mlp_backward(ctx, grad):
    params, x, mask = ctx.saved_tensors
    gp = gx = None
    m = mask if ctx.has_mask else None
    if ctx.needs_input_grad[0]:
        gp = mlp_bwd(params, x, m, grad, ctx.out_scale).to(params.dtype)
    if ctx.needs_input_grad[1]:                    # the input gradient nn.Sequential gives the reference's callers
        gx = mlp_input_grad(params, x, m, grad, ctx.out_scale).to(x.dtype)
    return gp, gx, None, None, None


torch.library.register_autograd("diffus::mlp_fwd", _mlp_backward, setup_context=_mlp_setup)


# ---------------------------------------------------------------------------------------
# training-loop pieces: Adam, volume slices, rotate_around_apex, log compression, image losses
# ---------------------------------------------------------------------------------------
def adam_step(params: torch.Tensor, grads: torch.Tensor, state: torch.Tensor, lr: float, betas=(0.9, 0.999), eps: float = 1e-8,
              weight_decay: float = 0.0, grad_scale: float = 1.0) -> None:
    """One ``torch.optim.Adam`` step on a flat float32 parameter vector, in place, one launch.

    ``state`` is ``[exp_avg | exp_avg_sq | step]`` (2n + 1 floats, zero before the first step)."""
    dev = _require_cuda(params, grads, state)
    n = params.numel()
    if grads.numel() < n or state.numel() != 2 * n + 1 or params.dtype != torch.float32 or grads.dtype != torch.float32 \
            or state.dtype != torch.float32 or not (params.is_contiguous() and grads.is_contiguous() and state.is_contiguous()):
        raise _lib.DiffusError("adam_step needs contiguous float32 params (n), grads (>= n) and state (2n + 1)")
    with _on_device(dev):
        _lib.check(_lib.load().diffus_adam_step(params.data_ptr(), grads.data_ptr(), state.data_ptr(), n, lr, betas[0], betas[1], eps,
                                                weight_decay, grad_scale, _stream(dev)), "diffus_adam_step")


class Conv1dRows(torch.autograd.Function):
    """``F.conv1d(x.unsqueeze(1), w[None, None], padding=pad).squeeze(1)`` on (rows, n) float32 CUDA rows (the PSF step of
    ``compute_gaussian_pulse``, reference ``src/renderer.py:476``); differentiable w.r.t. the rows."""

    @staticmethod
    def forward(ctx, x, w, pad):
        dev = _require_cuda(x, w)
        xc, wc = x.detach().contiguous().float(), w.detach().contiguous().float().reshape(-1)
        rows, n_in, taps = xc.shape[0], xc.shape[1], wc.numel()
        n_out = n_in + 2 * pad - taps + 1
        with _on_device(dev):
            out = torch.empty((rows, max(n_out, 0)), dtype=torch.float32, device=dev)
            _lib.check(_lib.load().diffus_conv1d_rows_forward(xc.data_ptr(), rows, n_in, wc.data_ptr(), taps, pad, out.data_ptr(),
                                                              _stream(dev)), "diffus_conv1d_rows_forward")
        ctx.save_for_backward(wc)
        ctx.meta = (rows, n_in, taps, pad, x.dtype)
        return out.to(x.dtype)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        (wc,) = ctx.saved_tensors
        rows, n_in, taps, pad, dt = ctx.meta
        dev = gout.device
        g = gout.contiguous().float()
        with _on_device(dev):
            gin = torch.empty((rows, n_in), dtype=torch.float32, device=dev)
            _lib.check(_lib.load().diffus_conv1d_rows_backward(g.data_ptr(), rows, n_in, wc.data_ptr(), taps, pad, gin.data_ptr(),
                                                               _stream(dev)), "diffus_conv1d_rows_backward")
        return gin.to(dt), None, None


def volume_slice(volume: torch.Tensor, dims, layout: int, axis: int, index: int, slice_: Optional[torch.Tensor] = None,
                 scatter: bool = False) -> torch.Tensor:
    """Copy one slice out of (``scatter=False``) or into (``scatter=True``) a LINEAR / BRICK volume buffer."""
    dev = _require_cuda(volume, slice_)
    rest = [d for a, d in enumerate(dims) if a != axis]
    with _on_device(dev):
        if slice_ is None:
            slice_ = torch.empty(rest, dtype=torch.float32, device=dev)
        elif slice_.numel() != rest[0] * rest[1] or slice_.dtype != torch.float32 or not slice_.is_contiguous():
            raise _lib.DiffusError(f"slice must be contiguous float32 {tuple(rest)}")
        _lib.check(_lib.load().diffus_volume_slice(volume.data_ptr(), C.byref((C.c_int32 * 3)(*dims)), layout, axis, index,
                                                   slice_.data_ptr(), int(scatter), _stream(dev)), "diffus_volume_slice")
    return slice_


class SliceInsertFunction(torch.autograd.Function):
    """``out = volume.clone(); out[..., index (along axis) ...] = slice`` with gradients to both (LINEAR layout)."""

    @staticmethod
    def forward(ctx, volume, slice_, axis, index):
        out = volume.detach().clone()
        volume_slice(out, list(out.shape), LAYOUT_LINEAR, axis, index, slice_.detach().contiguous().float(), scatter=True)
        ctx.meta = (axis, index)
        return out

    @staticmethod
    def backward(ctx, grad):
        axis, index = ctx.meta
        g = grad.contiguous().float()
        gs = volume_slice(g, list(g.shape), LAYOUT_LINEAR, axis, index) if ctx.needs_input_grad[1] else None
        gv = None
        if ctx.needs_input_grad[0]:                  # the inserted slice replaced the volume's own values: no gradient there
            gv = g.clone()
            rest = [d for a, d in enumerate(g.shape) if a != axis]
            volume_slice(gv, list(gv.shape), LAYOUT_LINEAR, axis, index, torch.zeros(rest, dtype=torch.float32, device=g.device),
                         scatter=True)
        return gv, gs, None, None


def rotate_apex(x: torch.Tensor, z: torch.Tensor, cos_a: float, sin_a: float, shift: float, apex0: float, apex1: float):
    dev = _require_cuda(x, z)
    xf, zf = x.to(torch.float32).contiguous(), z.to(torch.float32).contiguous()
    with _on_device(dev):
        xr, zr = torch.empty_like(xf), torch.empty_like(zf)
        if xf.numel():
            _lib.check(_lib.load().diffus_rotate_around_apex(xf.data_ptr(), zf.data_ptr(), xf.numel(), cos_a, sin_a, shift, apex0, apex1,
                                                             xr.data_ptr(), zr.data_ptr(), _stream(dev)), "diffus_rotate_around_apex")
    return xr, zr


class LogCompressFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img):
        dev = _require_cuda(img)
        x = img.detach().contiguous().float()
        with _on_device(dev):
            out = torch.empty_like(x)
            _lib.check(_lib.load().diffus_log_compress_forward(x.data_ptr(), x.numel(), out.data_ptr(), None, _stream(dev)),
                       "diffus_log_compress_forward")
        ctx.save_for_backward(x)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        (x,) = ctx.saved_tensors
        g = grad.contiguous().float()
        with torch.cuda.device(x.device):
            gx = torch.empty_like(x)
            _lib.check(_lib.load().diffus_log_compress_backward(x.data_ptr(), g.data_ptr(), x.numel(), gx.data_ptr(), _stream(x.device)),
                       "diffus_log_compress_backward")
        return gx


def rf_to_bmode(profiles: torch.Tensor, hilbert_kernel: torch.Tensor) -> torch.Tensor:
    dev = _require_cuda(profiles, hilbert_kernel)
    rf = profiles.detach().contiguous().float()
    if rf.dim() != 2 or hilbert_kernel.numel() != rf.shape[1]:
        raise _lib.DiffusError("profiles must be (n_rays, n_samples) and the Hilbert kernel n_samples long")
    with _on_device(dev):
        out = torch.empty_like(rf)
        ws = torch.empty((4,), dtype=torch.uint8, device=dev)
        _lib.check(_lib.load().diffus_rf_to_bmode(rf.data_ptr(), rf.shape[0], rf.shape[1], hilbert_kernel.contiguous().float().data_ptr(),
                                                  out.data_ptr(), ws.data_ptr(), 4, _stream(dev)), "diffus_rf_to_bmode")
    return out


class MaskedMSEEdgeFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, synth, real, mask, edge_weight):
        dev = _require_cuda(synth, real, mask)
        if synth.dim() != 2 or real.shape != synth.shape or mask.shape != synth.shape:
            raise _lib.DiffusError("synth, real and mask must be (H, W) images of one shape")
        a, b = synth.detach().contiguous().float(), real.detach().contiguous().float()
        m = mask.contiguous().to(torch.uint8)
        H, W = a.shape
        with _on_device(dev):
            stats = torch.empty((3,), dtype=torch.float32, device=dev)
            _lib.check(_lib.load().diffus_masked_mse_edge_forward(a.data_ptr(), b.data_ptr(), m.data_ptr(), H, W, edge_weight,
                                                                  stats.data_ptr(), _stream(dev)), "diffus_masked_mse_edge_forward")
        ctx.save_for_backward(a, b, m, stats)
        ctx.edge_weight = edge_weight
        return stats[0].clone()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        a, b, m, stats = ctx.saved_tensors
        H, W = a.shape
        g = grad.reshape(1).contiguous().float()
        with torch.cuda.device(a.device):
            ga = torch.empty_like(a)
            _lib.check(_lib.load().diffus_masked_mse_edge_backward(a.data_ptr(), b.data_ptr(), m.data_ptr(), H, W, ctx.edge_weight,
                                                                   stats.data_ptr(), g.data_ptr(), ga.data_ptr(), _stream(a.device)),
                       "diffus_masked_mse_edge_backward")
        return ga, None, None, None


class SSIMLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, synth, real, normalize, ksize, sigma, k1, k2):
        dev = _require_cuda(synth, real)
        if synth.dim() != 2 or real.shape != synth.shape:
            raise _lib.DiffusError("synth and real must be (H, W) images of one shape")
        a, b = synth.detach().contiguous().float(), real.detach().contiguous().float()
        H, W = a.shape
        lib = _lib.load()
        wbytes = lib.diffus_ssim_workspace_bytes(H, W, ksize)
        if wbytes <= 0:
            raise _lib.DiffusError(f"SSIM window {ksize} does not fit a {H} x {W} image (or exceeds 33)")
        with _on_device(dev):
            ws = torch.empty((wbytes,), dtype=torch.uint8, device=dev)
            loss = torch.empty((1,), dtype=torch.float32, device=dev)
            _lib.check(lib.diffus_ssim_loss_forward(a.data_ptr(), b.data_ptr(), H, W, ksize, sigma, k1, k2, int(normalize), loss.data_ptr(),
                                                    ws.data_ptr(), wbytes, _stream(dev)), "diffus_ssim_loss_forward")
        ctx.save_for_backward(a, b, ws)
        ctx.meta = (int(normalize), ksize, sigma)
        return loss.reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        a, b, ws = ctx.saved_tensors
        normalize, ksize, sigma = ctx.meta
        H, W = a.shape
        g = grad.reshape(1).contiguous().float()
        with torch.cuda.device(a.device):
            ga = torch.empty_like(a)
            _lib.check(_lib.load().diffus_ssim_loss_backward(a.data_ptr(), b.data_ptr(), H, W, ksize, sigma, normalize, g.data_ptr(),
                                                             ga.data_ptr(), ws.data_ptr(), ws.numel(), _stream(a.device)),
                       "diffus_ssim_loss_backward")
        return ga, None, None, None, None, None, None
