"""MRI -> impedance MLP training fused with rendering (BASELINE config 4; reference notebooks
``[DEMO] Train MRI to Impedance MLP*.ipynb``, ``ImpedanceLearner.training_forward`` + ``train_step``).

One step, everything in the brick layout the gathers use (no layout conversions inside the step):

    Z_bricks  = out_scale * MLP(mri_bricks)           piecewise-linear table, written once
    loss, dZ  = fused render + MSE + backward          dZ scattered with red.add into brick-local lines
    dWeights  = MLP backward from (mri_bricks, dZ)     atomic-free block partials, fixed-order reduction
    all-reduce of the 1 153 weight gradients (+ shared-pose gradients) across ranks, one flat buffer
"""
from __future__ import annotations

from typing import Optional

import torch

from . import distributed as dist_utils
from . import ops
from ._lib import SAMPLER_TRILINEAR
from .impedance import ImpedanceEstimator, pack_params
from .renderer import _canon_pose, _resolve_start, _sampler_id


class TrainingVolume:
    """An MRI volume (and optional mask) copied once into the brick layout of the gathers."""

    def __init__(self, mri: torch.Tensor, mask: Optional[torch.Tensor] = None):
        if mri.dim() != 3:
            raise ValueError("mri must be (D,H,W)")
        self.dims = list(mri.shape)
        self.mri_bricks = ops.to_bricks(mri.float())
        self.mask_bricks = None if mask is None else (ops.to_bricks(mask.float()) > 0.5).to(torch.uint8)


class _MLPRenderMSE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, params, tv, sources, directions, targets, n_samples, start, alpha, sampler, product_f32,
                out_scale, fill):
        z_bricks = ops.mlp_fwd_impl(params.detach(), tv.mri_bricks, tv.mask_bricks, out_scale, fill)
        need_pose = (ctx.needs_input_grad[2] or ctx.needs_input_grad[3]) and sampler == SAMPLER_TRILINEAR
        loss, _, gz, gsrc, gdir = ops.render_mse_impl(z_bricks, z_bricks, tv.dims, sources.detach(), directions.detach(),
                                                      targets, n_samples, start, alpha, sampler, product_f32,
                                                      ctx.needs_input_grad[0], need_pose, False, keep_brick_grad=True)
        ctx.save_for_backward(params, gz, gsrc, gdir)
        ctx.tv, ctx.out_scale = tv, out_scale
        ctx.flags = (need_pose, sources.dtype, directions.dtype, directions.dim())
        return loss.reshape(())

    @staticmethod
    def backward(ctx, gloss):
        params, gz, gsrc, gdir = ctx.saved_tensors
        need_pose, sdt, ddt, ddim = ctx.flags
        gp = gs = gd = None
        if ctx.needs_input_grad[0]:
            gp = ops.mlp_bwd_impl(params.detach(), ctx.tv.mri_bricks, ctx.tv.mask_bricks, gz, ctx.out_scale) * gloss
        if need_pose and ctx.needs_input_grad[2]:
            gs = (gsrc * gloss).to(sdt)
        if need_pose and ctx.needs_input_grad[3]:
            gd = ((gdir if ddim == 3 else gdir.sum(0)) * gloss).to(ddt)
        return gp, None, gs, gd, None, None, None, None, None, None, None, None


def mlp_render_mse_loss(model: ImpedanceEstimator, mri, sources: torch.Tensor, directions: torch.Tensor,
                        targets: torch.Tensor, num_samples: int, attenuation_coeff: float = 0.5, start=0, *,
                        sampler: str = "trilinear", out_scale: float = 1.0, mask: Optional[torch.Tensor] = None,
                        fill: float = 400.0) -> torch.Tensor:
    """MSE between frames rendered from ``out_scale * MLP(mri)`` and ``targets``.

    Differentiable in the MLP weights and (trilinear) the poses.  ``mri`` is a (D,H,W) CUDA tensor or a
    :class:`TrainingVolume` prepared once (saves the per-step brick copy of the input).
    """
    tv = mri if isinstance(mri, TrainingVolume) else TrainingVolume(mri, mask)
    src, dirs, product_f32 = _canon_pose(sources, directions, tv.mri_bricks.device)
    if src.dim() == 1:
        src = src.unsqueeze(0)
    tgt = targets.to(torch.float32).contiguous()
    if tgt.dim() == 2:
        tgt = tgt.unsqueeze(0)
    return _MLPRenderMSE.apply(pack_params(model), tv, src.contiguous(), dirs.contiguous(), tgt, int(num_samples),
                               _resolve_start(start, num_samples), float(attenuation_coeff), _sampler_id(sampler),
                               product_f32, float(out_scale), float(fill))


def train_step(model: ImpedanceEstimator, optimizer: torch.optim.Optimizer, mri, sources: torch.Tensor,
               directions: torch.Tensor, targets: torch.Tensor, num_samples: int, attenuation_coeff: float = 0.5,
               start=0, **kw) -> torch.Tensor:
    """zero_grad -> fused loss -> backward -> all-reduce of the weight gradients -> optimizer.step(), through autograd and
    a ``torch.optim`` optimiser (any optimiser, any extra loss terms).  Each rank's loss is the mean over ITS poses, so
    the gradients are weighted by the rank's share of the global batch before the SUM all-reduce: the update equals the
    single-process one for ragged shards too.  :class:`FusedTrainer` is the same step without autograd or torch.optim."""
    optimizer.zero_grad(set_to_none=True)
    loss = mlp_render_mse_loss(model, mri, sources, directions, targets, num_samples, attenuation_coeff, start, **kw)
    loss.backward()
    n_local = float(targets.numel())
    share = dist_utils.global_share(n_local, targets.device)
    dist_utils.allreduce_module_grads(model, weight=share)
    optimizer.step()
    return loss.detach()


class FusedTrainer:
    """The MLP -> render -> MSE training step of BASELINE config 4 with nothing but this library's kernels and one NCCL call.

    Persistent state, allocated once: the 1 153 weights as ONE flat float32 vector (the module's parameters become views of
    it, so ``model.state_dict()`` stays the reference's), one flat all-reduce buffer ``[weight gradients | loss]`` that the
    MLP backward and the fused render kernel write into directly (no ``cat`` / ``copy_`` round trip), the Adam moments and
    step counter, the impedance bricks and their gradient bricks.  One :meth:`step`:

        Z bricks = out_scale * MLP(mri bricks)                       piecewise-linear table kernel
        loss, dZ = fused render + MSE + backward                     loss and gradients pre-scaled by 1 / global elements
        dW      += MLP backward(mri bricks, dZ)                      into the flat buffer
        all-reduce(SUM) of the flat buffer over ranks                4.6 KB, one NCCL launch
        Adam                                                         one launch (torch.optim.Adam's arithmetic)

    ``slice_index`` switches to ``ImpedanceLearner.training_forward``'s slice mode (GPU notebook cell 16): the volume is
    the MRI itself except slice ``[:, :, k]``, which is ``MLP(mri[:, :, k])`` -- the MLP runs on that slice only.
    """

    def __init__(self, model: ImpedanceEstimator, mri: torch.Tensor, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, *, sampler: str = "trilinear", out_scale: float = 1.0,
                 slice_index: Optional[int] = None, gather: str = "auto"):
        """``gather='texture'`` (full-volume mode): the MLP writes the impedance volume in torch order, it is copied into a
        layered CUDA array each step (one device-to-device copy of the volume) and the march gathers it with ``tld4``; the
        gradient still lands in bricks, which is the order the MLP backward reads the MRI in."""
        from ._lib import LAYOUT_BRICK, MLP_NPARAMS
        if gather not in ("auto", "brick", "texture"):
            raise ValueError("gather must be 'auto', 'brick' or 'texture'")
        if gather == "auto":      # measured on config 4 (4096 frames): trilinear 5.99 (brick) vs 5.62 ms (texture), nearest 2.97 vs 3.08 ms
            gather = "texture" if (sampler == "trilinear" and slice_index is None) else "brick"
        if gather == "texture" and slice_index is not None:
            raise ValueError("gather='texture' is for the full-volume mode")
        self.gather = gather
        if mri.dim() != 3 or not mri.is_cuda:
            raise ValueError("mri must be a (D,H,W) CUDA tensor")
        dev = mri.device
        self.model, self.dims, self.device = model, list(mri.shape), dev
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.sampler, self.out_scale, self.slice_index = _sampler_id(sampler), float(out_scale), slice_index
        self._layout_brick = LAYOUT_BRICK
        # flat parameters; the module's tensors become views of them
        self.params = pack_params(model).detach().to(dev, torch.float32).contiguous().clone()
        off = 0
        for prm in (model.model[0].weight, model.model[0].bias, model.model[2].weight, model.model[2].bias,
                    model.model[4].weight, model.model[4].bias):
            n = prm.numel()
            prm.data = self.params[off:off + n].view(prm.shape)
            off += n
        self.n = MLP_NPARAMS
        self.flat = torch.zeros((self.n + 1,), dtype=torch.float32, device=dev)          # [dW | loss]: the all-reduce buffer
        self.grads, self.loss = self.flat[:self.n], self.flat[self.n:]
        self.state = torch.zeros((2 * self.n + 1,), dtype=torch.float32, device=dev)     # Adam moments + step
        mri32 = mri.detach().float().contiguous()
        self.mri_bricks = ops.to_bricks(mri32)
        self.grad_bricks = torch.zeros_like(self.mri_bricks)
        self.texture = None
        if slice_index is None:
            self.x = self.mri_bricks
            self.z_bricks = torch.empty_like(self.mri_bricks)
            if gather == "texture":
                self.x_linear = mri32
        else:
            self.x = mri32[:, :, slice_index].contiguous()                               # (D, H) slice the MLP sees
            self.z_bricks = self.mri_bricks.clone()                                      # the rest of the volume never changes
            self.grad_slice = torch.empty_like(self.x)
        wbytes = _mlp_ws_bytes(self.x.numel())
        self.mlp_ws = torch.empty((wbytes,), dtype=torch.uint8, device=dev)

    def forward_volume(self) -> torch.Tensor:
        """The impedance volume of the current weights as :meth:`step` renders it: bricks, or with ``gather='texture'`` the
        (D,H,W) tensor whose copy sits in the CUDA array."""
        if self.gather == "texture":
            self.z_linear = ops.mlp_fwd_impl(self.params, self.x_linear, None, self.out_scale, 0.0)
            if self.texture is None:
                self.texture = ops.VolumeTexture(self.z_linear)
            else:
                self.texture.update(self.z_linear)
            return self.z_linear
        if self.slice_index is None:
            z = ops.mlp_fwd_impl(self.params, self.x, None, self.out_scale, 0.0)
            self.z_bricks = z
        else:
            zs = ops.mlp_fwd_impl(self.params, self.x.reshape(-1), None, self.out_scale, 0.0).reshape(self.x.shape)
            ops.volume_slice(self.z_bricks, self.dims, self._layout_brick, 2, self.slice_index, zs, scatter=True)
        return self.z_bricks

    def step(self, sources: torch.Tensor, directions: torch.Tensor, targets: torch.Tensor, num_samples: int,
             attenuation_coeff: float = 0.5, start=0, n_total: Optional[int] = None) -> torch.Tensor:
        """One training step on this rank's pose shard; returns the GLOBAL mean loss (a device scalar, after the all-reduce).
        ``n_total``: frame elements of the global batch (default: ``world_size`` x this shard)."""
        rank, world = dist_utils.world()
        tgt = targets if targets.dtype == torch.float32 and targets.is_contiguous() else targets.float().contiguous()
        if n_total is None:
            n_total = tgt.numel() * world
        self.flat.zero_()
        self.grad_bricks.zero_()
        z = self.forward_volume()
        packed = self.texture.token if self.gather == "texture" else z
        ops.render_mse_impl(z, packed, self.dims, sources, directions, tgt, int(num_samples), _resolve_start(start, num_samples),
                            float(attenuation_coeff), self.sampler, False, True, False, False, keep_brick_grad=True,
                            n_total=n_total, grad_volume_out=self.grad_bricks, loss_out=self.loss)
        if self.slice_index is None:
            gz = self.grad_bricks
        else:
            gz = ops.volume_slice(self.grad_bricks, self.dims, self._layout_brick, 2, self.slice_index, self.grad_slice)
        ops.mlp_bwd_impl(self.params, self.x.reshape(-1), None, gz.reshape(-1), self.out_scale, grad_params_out=self.grads,
                         workspace=self.mlp_ws)
        if world > 1:
            torch.distributed.all_reduce(self.flat)                                       # SUM: shards are pre-scaled by 1 / n_total
        ops.adam_step(self.params, self.grads, self.state, self.lr, self.betas, self.eps, self.weight_decay)
        return self.loss[0]


def _mlp_ws_bytes(n: int) -> int:
    from . import _lib
    return int(_lib.load().diffus_mlp_bwd_workspace_bytes(int(n)))


def training_forward(model: ImpedanceEstimator, renderer, x: torch.Tensor, source: torch.Tensor, directions: torch.Tensor,
                     angle: float = 45.0, start=0, *, slice_idx: Optional[int] = None, sampler: str = "nearest",
                     return_indices: bool = True):
    """``ImpedanceLearner.training_forward`` of the reference's training notebooks, differentiable in the MLP weights.

    ``slice_idx=None``: ``Z_vol = mlp(x)`` over the whole volume (``[DEMO] Train MRI to Impedance MLP.ipynb`` cell 19).
    ``slice_idx=k``: ``Z_vol = x.clone(); Z_vol[:, :, k] = mlp(x[:, :, k])`` (the GPU notebook's cell 16: the fan lies in
    that slice).  Then ``renderer.plot_beam_frame(volume=Z_vol, source, directions, angle, plot=False, artifacts=False,
    start)``; returns its ``(x, y, z, intensities)``.
    """
    x = x.float()
    if slice_idx is None:
        z_vol = model.impedance_volume(x)
    else:
        xs = x[:, :, slice_idx].contiguous()
        z_slice = ops.mlp_fwd(pack_params(model), xs.reshape(-1), None, 1.0, 0.0).reshape(xs.shape)
        z_vol = ops.SliceInsertFunction.apply(x, z_slice, 2, int(slice_idx))
    return renderer.plot_beam_frame(volume=z_vol, source=source, directions=directions, angle=angle, plot=False,
                                    artifacts=False, start=start, sampler=sampler, return_indices=return_indices)
