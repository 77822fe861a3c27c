"""MRI preprocessing helpers -- drop-ins for ``create_brain_mask`` and ``zscore_normalize`` (reference ``src/utils.py:12-39``).

The reference runs these on the CPU with scipy before ``compute_impedance_volume``; here they are small device
kernels (threshold + 6-neighbour morphology, masked mean / std), so a whole MRI -> impedance volume stays on the GPU.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, ops


def create_brain_mask(volume: torch.Tensor, threshold=50, iterations: int = 2) -> torch.Tensor:
    """``volume > threshold`` cleaned by ``iterations`` binary dilations then erosions (bool tensor, same device)."""
    dev = ops._require_cuda(volume)
    lib = _lib.load()
    v = volume.float().contiguous()
    dim = (C.c_int32 * 3)(*v.shape)
    with torch.cuda.device(dev):
        mask = torch.empty(v.shape, dtype=torch.uint8, device=dev)
        scratch = torch.empty(v.shape, dtype=torch.uint8, device=dev)
        _lib.check(lib.diffus_brain_mask(v.data_ptr(), C.byref(dim), float(threshold), int(iterations), mask.data_ptr(),
                                         scratch.data_ptr(), ops._stream(dev)), "diffus_brain_mask")
    return mask.bool()


def zscore_normalize(volume: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """``(volume - mean) / (std + 1e-8)`` with mean and (unbiased) std over the voxels where ``mask > 0``."""
    dev = ops._require_cuda(volume, mask)
    lib = _lib.load()
    v = volume.float().contiguous()
    m = (mask > 0).to(torch.uint8).contiguous()
    with torch.cuda.device(dev):
        out = torch.empty_like(v)
        ws = torch.empty((64,), dtype=torch.uint8, device=dev)
        _lib.check(lib.diffus_masked_zscore(v.data_ptr(), m.data_ptr(), v.numel(), out.data_ptr(), ws.data_ptr(), 64,
                                            ops._stream(dev)), "diffus_masked_zscore")
    return out
