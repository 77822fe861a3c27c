"""Gaussian smoothing of a volume in float64: the reference for ``diffus_volume_gaussian_blur``.  TEST INFRASTRUCTURE ONLY.

``scipy.ndimage.gaussian_filter`` with ``mode='nearest'`` (the edge voxel repeats beyond a face, the renderer's border rule).
"""
from __future__ import annotations

import numpy as np


def gaussian_radius(sigma: float, truncate: float = 4.0) -> int:
    """scipy's radius of the truncated kernel: ``int(truncate * sigma + 0.5)``."""
    return int(float(truncate) * float(sigma) + 0.5)


def gaussian_weights(sigma: float, truncate: float = 4.0) -> np.ndarray:
    """The 2r+1 float64 weights scipy correlates with: ``exp(-x^2 / (2 sigma^2))`` over x = -r..r, normalised to sum 1."""
    r = gaussian_radius(sigma, truncate)
    x = np.arange(-r, r + 1)
    phi = np.exp(-0.5 / (float(sigma) ** 2) * x ** 2)
    return phi / phi.sum()


def gaussian_blur(volume, sigma: float, truncate: float = 4.0) -> np.ndarray:
    """``scipy.ndimage.gaussian_filter(volume, sigma, mode='nearest', truncate=truncate)`` in float64."""
    from scipy.ndimage import gaussian_filter
    return gaussian_filter(np.asarray(volume, dtype=np.float64), float(sigma), mode="nearest", truncate=float(truncate))
