"""CPU restatement of the DiffUS B-mode renderer hot path.  TEST INFRASTRUCTURE ONLY.

Every function cites the reference file:line (relative to the reference repo root) whose
arithmetic it restates.  Written against torch so it runs in fp32 or fp64 and gives
gradients through autograd; nothing here is imported by the product package.

Pinned by: ``tests/golden/*.npz`` (outputs of the real reference, made by
``oracle/make_golden.py``) and, when ``/root/reference`` is importable, live comparison in
``tests/test_oracle_vs_reference.py``.
"""
from __future__ import annotations

import math

import numpy as np
import torch

# ----------------------------------------------------------------------------------------
# geometry  (src/cone.py:242-259)
# ----------------------------------------------------------------------------------------


def generate_cone_directions(direction_mri_world, opening_angle, n_rays) -> torch.Tensor:
    """Fan of unit directions in the z=0 plane around a median direction.

    Follows ``src/cone.py:242-259``: normalise the first two components ``d``;
    ``ortho = (-d_y, d_x)``; ``a = linspace(-theta/2, theta/2, n)`` in float64;
    ``v = cos(a) d + sin(a) ortho``; rows ``[v_x, v_y, 0]`` cast to float32.
    """
    d = np.asarray(direction_mri_world, dtype=np.float64)[:2]
    d = d / np.linalg.norm(d)
    ortho = np.array([-d[1], d[0]])
    a = np.linspace(-opening_angle / 2, opening_angle / 2, n_rays)
    v = np.cos(a)[:, None] * d[None, :] + np.sin(a)[:, None] * ortho[None, :]
    out = np.zeros((n_rays, 3), dtype=np.float64)
    out[:, :2] = v
    return torch.tensor(out, dtype=torch.float32)


# ----------------------------------------------------------------------------------------
# ray points and samplers  (src/renderer.py:119-124, :741-759)
# ----------------------------------------------------------------------------------------


def ray_points(source: torch.Tensor, directions: torch.Tensor, num_samples: int) -> torch.Tensor:
    """``points[r, k] = source + k * directions[r]`` (``src/renderer.py:119-124``).

    ``steps`` is a float32 arange; the product and the sum are separate roundings and the
    result dtype follows torch promotion (fp64 directions/source give fp64 points).
    """
    if directions.ndim == 1:
        directions = directions.unsqueeze(0)
    steps = torch.arange(0, num_samples, dtype=torch.float32).view(1, -1, 1)
    return source + steps * directions.unsqueeze(1)


def nearest_indices(shape, points: torch.Tensor):
    """Round-half-even, clamp to the volume (``src/renderer.py:751-756``)."""
    D, H, W = shape
    p = points.float()
    x = torch.clamp(p[..., 0].round().long(), 0, D - 1)
    y = torch.clamp(p[..., 1].round().long(), 0, H - 1)
    z = torch.clamp(p[..., 2].round().long(), 0, W - 1)
    return x, y, z


def sample_nearest(volume: torch.Tensor, points: torch.Tensor):
    """``Z[x, y, z]`` at the nearest voxel with border clamp (``src/renderer.py:754-759``)."""
    x, y, z = nearest_indices(volume.shape, points)
    return x, y, z, volume[x, y, z]


def sample_trilinear(volume: torch.Tensor, points: torch.Tensor):
    """Border-clamped trilinear interpolation at continuous index coordinates.

    Restates what ``F.grid_sample(mode='bilinear', padding_mode='border',
    align_corners=True)`` computes for the reference's notebook-era sampler
    (``notebooks/[DEPR] fxiafixing_voxel_plot.ipynb`` cell 29; the same grid construction
    survives at ``src/renderer.py:802-815``): each coordinate is clamped to
    ``[0, size-1]`` first, ``i0 = floor``, weights ``(1-f, f)``, the ``+1`` corner clamped.
    The derivative w.r.t. a coordinate is exactly zero when ``p <= 0`` or ``p >= size-1``
    (ATen's ``clip_coordinates_set_grad``), which the ``where`` below reproduces.
    """
    D, H, W = volume.shape
    pts = points.to(volume.dtype)
    x, y, z = nearest_indices(volume.shape, points)
    idx0, idx1, frac = [], [], []
    for a, n in enumerate((D, H, W)):
        p = pts[..., a]
        inside = (p > 0) & (p < n - 1)
        pc = torch.where(inside, p, p.detach().clamp(0, n - 1))
        i0 = pc.detach().floor()
        f = pc - i0
        i0 = i0.long().clamp(0, n - 1)
        i1 = (i0 + 1).clamp(max=n - 1)
        idx0.append(i0)
        idx1.append(i1)
        frac.append(f)
    val = 0
    for cx in (0, 1):
        wx = frac[0] if cx else 1 - frac[0]
        ix = idx1[0] if cx else idx0[0]
        for cy in (0, 1):
            wy = frac[1] if cy else 1 - frac[1]
            iy = idx1[1] if cy else idx0[1]
            for cz in (0, 1):
                wz = frac[2] if cz else 1 - frac[2]
                iz = idx1[2] if cz else idx0[2]
                val = val + volume[ix, iy, iz] * (wx * wy * wz)
    return x, y, z, val


# ----------------------------------------------------------------------------------------
# reflection and propagation  (src/renderer.py:27-33, :367-457)
# ----------------------------------------------------------------------------------------


def reflection_coeff(Z1: torch.Tensor, Z2: torch.Tensor) -> torch.Tensor:
    """Signed amplitude coefficient ``(Z2 - Z1) / (Z1 + Z2)`` (``src/renderer.py:33``)."""
    return (Z2 - Z1) / (Z1 + Z2)


def _layered_system(r: torch.Tensor):
    """The ``2(n+1) x 2(n+1)`` system of ``src/renderer.py:384-405`` for ``n`` interfaces.

    Unknowns ``[g0, d0, g1, d1, ..., gn, dn]`` (right- and left-going amplitudes);
    ``g0 = 1``; ``dn = 0``; per interface i:
    ``g_{i+1} = (1 + r_i) g_i + r_i d_{i+1}`` and ``d_i = r_i g_i + (1 - r_i) d_{i+1}``.
    """
    B, n = r.shape
    size = 2 * (n + 1)
    A = torch.zeros((B, size, size), dtype=r.dtype)
    b = torch.zeros((B, size), dtype=r.dtype)
    b[:, 0] = 1
    A[:, 0, 0] = 1
    A[:, -1, -1] = 1
    if n:
        i = torch.arange(n)
        g, d, gn, dn = 2 * i, 2 * i + 1, 2 * i + 2, 2 * i + 3
        A[:, gn, g] = -(1 + r)
        A[:, gn, dn] = -r
        A[:, gn, gn] = 1
        A[:, d, g] = -r
        A[:, d, dn] = -(1 - r)
        A[:, d, d] = 1
    return A, b


def surface_return_dense(r: torch.Tensor) -> torch.Tensor:
    """``d0`` of the truncated stacks, literally as the reference computes it.

    For every truncation depth ``k = 0..N`` solve the dense system of the first ``k``
    interfaces and keep ``d0`` (``src/renderer.py:407-408, :428-431``); NaNs become 0.
    O(N^4) flops per ray -- this IS the reference's cost.
    """
    B, N = r.shape
    cols = []
    for k in range(N + 1):
        A, b = _layered_system(r[:, :k])
        w = torch.nan_to_num(torch.linalg.solve(A, b), nan=0.0)
        cols.append(w[:, 1])
    return torch.stack(cols, dim=1)


def echo_dense_solve(r: torch.Tensor) -> torch.Tensor:
    """Echo line of ``compute_echo_traces`` (``src/renderer.py:434-435, :453-454``).

    The reference cumulative-sums ``d0`` over depth, then takes the first difference and
    left-pads a zero, i.e. ``echo = [0, d0^(1), ..., d0^(N)]`` up to the rounding of the
    cumsum round trip (kept here so fp32 runs reproduce the reference's own noise).
    """
    d0 = torch.cumsum(surface_return_dense(r), dim=1)
    return torch.nn.functional.pad(d0[:, 1:] - d0[:, :-1], (1, 0))


def echo_closed_form(r: torch.Tensor) -> torch.Tensor:
    """Same echo line as :func:`echo_dense_solve` in O(N) per ray.

    ``echo[k] = P_k[0,1] / P_k[1,1]`` with ``P_k = prod_{i<k} [[1-2 r_i^2, r_i], [-r_i, 1]]``
    and ``echo[0] = 0`` -- eliminating the interior unknowns of the system at
    ``src/renderer.py:393-405`` gives exactly this 2x2 transfer-matrix product.  NaN rule
    of ``src/renderer.py:408``: once a NaN coefficient is included every later entry is 0.
    Verified against the dense form and the live reference in the tests.
    """
    B, N = r.shape
    one = torch.ones(B, dtype=r.dtype)
    zero = torch.zeros(B, dtype=r.dtype)
    p00, p01, p10, p11 = one, zero, zero, one
    out = [zero]
    for k in range(N):
        rk = r[:, k]
        a = 1 - 2 * rk * rk
        p00, p01, p10, p11 = p00 * a - p01 * rk, p00 * rk + p01, p10 * a - p11 * rk, p10 * rk + p11
        out.append(torch.nan_to_num(p01 / p11, nan=0.0))
    return torch.stack(out, dim=1)


def delays_us(n: int, spacing: float = 1.0, c: float = 1.54e3) -> torch.Tensor:
    """Second return value of ``compute_echo_traces`` (``src/renderer.py:455``)."""
    return 2 * spacing * torch.arange(n) / c


# ----------------------------------------------------------------------------------------
# the path itself  (src/renderer.py:35-71, :201-275)
# ----------------------------------------------------------------------------------------


def resolve_start(start, num_samples: int) -> int:
    """``src/renderer.py:237-240``: a float start is a fraction of ``num_samples``."""
    if type(start) is float:
        start = int(start * num_samples)
    if type(start) is int:
        start = max(0, start)
    return start


def plot_beam_frame(volume, source, directions, num_samples, attenuation_coeff=0.5, start=0,
                    sampler="nearest", propagation="closed_form"):
    """``UltrasoundRenderer.plot_beam_frame`` with ``artifacts=False`` (``src/renderer.py:201-275``).

    sample (``:228`` -> ``:57`` -> ``:178``) -> reflection (``:65-68``) -> start crop and
    the median-over-rays replacement of column 0 (``:241-244``, restated out of place so
    autograd works) -> echo line (``:251``) -> ``* exp(-alpha k)`` with k restarting at 0
    after the crop (``:256-259``) -> ``(x[:, start:], y[:, start:], z[:, start:], frame)``.
    """
    pts = ray_points(source, directions, num_samples)
    if sampler == "nearest":
        x, y, z, imp = sample_nearest(volume, pts)
    elif sampler == "trilinear":
        x, y, z, imp = sample_trilinear(volume, pts)
    else:
        raise ValueError(sampler)
    r = reflection_coeff(imp[:, :-1], imp[:, 1:])
    start = resolve_start(start, num_samples)
    if start > 0:
        r = r[:, start:]
        med = r[:, 0].median()
        r = torch.cat([med.expand(r.shape[0], 1), r[:, 1:]], dim=1)
    if propagation == "closed_form":
        echo = echo_closed_form(r)
    elif propagation == "dense":
        echo = echo_dense_solve(r)
    else:
        raise ValueError(propagation)
    depths = torch.arange(echo.shape[1]).float()
    att = torch.exp(-attenuation_coeff * depths)
    frame = echo * att[None, :]          # fp32 attenuation, promoted if the echo is fp64
    return x[:, start:], y[:, start:], z[:, start:], frame


# ----------------------------------------------------------------------------------------
# MRI -> impedance MLP  (src/impedance.py:6-17)
# ----------------------------------------------------------------------------------------


def mlp_forward(x, w1, b1, w2, b2, w3, b3):
    """``Linear(1,32)-ReLU-Linear(32,32)-ReLU-Linear(32,1)`` (``src/impedance.py:10-17``).

    ``x`` (M, 1); weights in ``nn.Linear`` layout (out, in).
    """
    h1 = torch.relu(x @ w1.t() + b1)
    h2 = torch.relu(h1 @ w2.t() + b2)
    return h2 @ w3.t() + b3


def mlp_piecewise_table(w1, b1, w2, b2, w3, b3):
    """The same network (``src/impedance.py:10-17``) as the piecewise-linear function of its scalar input that it is --
    the restatement the CUDA path ``DIFFUS_MLP_PATH_PIECEWISE`` evaluates (csrc/mlp_pwl_kernels.cu), checked here against
    :func:`mlp_forward`.  Returns ``(breakpoints (B,), P (B+1,), Q (B+1,), midpoints (B+1,))`` in float64 with
    ``mlp(x) = P[r] x + Q[r]`` for ``r = searchsorted(breakpoints, x, side='right')``.

    Layer-1 units switch at ``-b1_i / w1_i``; between two such points the layer-1 mask is fixed, every layer-2 pre-activation
    is affine in x and switches at most once.  Masks are taken at the midpoint of each region."""
    import numpy as np
    w1 = np.asarray(w1, dtype=np.float64).reshape(-1)
    b1 = np.asarray(b1, dtype=np.float64).reshape(-1)
    w2 = np.asarray(w2, dtype=np.float64)
    b2 = np.asarray(b2, dtype=np.float64).reshape(-1)
    w3 = np.asarray(w3, dtype=np.float64).reshape(-1)
    b3 = float(np.asarray(b3, dtype=np.float64).reshape(-1)[0])

    def mid(a, b):
        if np.isinf(a) and np.isinf(b):
            return 0.0
        if np.isinf(a):
            return b - 1.0 - abs(b)
        if np.isinf(b):
            return a + 1.0 + abs(a)
        return 0.5 * (a + b)

    def affine(xm):
        m1 = (w1 * xm + b1) > 0
        return m1, w2 @ (m1 * w1), w2 @ (m1 * b1) + b2

    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(w1 != 0, -b1 / w1, np.inf)
    first = np.sort(t[np.isfinite(t)])
    edges = np.concatenate([[-np.inf], first, [np.inf]])
    bps = list(first)
    for a, b in zip(edges[:-1], edges[1:]):
        if not a < b:
            continue
        _, p, q = affine(mid(a, b))
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.where(p != 0, -q / p, np.inf)
        bps += [v for v in r if a < v < b]
    bps = np.sort(np.asarray(bps, dtype=np.float64))
    edges = np.concatenate([[-np.inf], bps, [np.inf]])
    P, Q, xm = [], [], []
    for a, b in zip(edges[:-1], edges[1:]):
        x0 = mid(a, b)
        _, p, q = affine(x0)
        m2 = (p * x0 + q) > 0
        P.append(float(w3 @ (m2 * p)))
        Q.append(float(w3 @ (m2 * q)) + b3)
        xm.append(x0)
    return bps, np.asarray(P), np.asarray(Q), np.asarray(xm)


def mlp_piecewise_grads(x, g, w1, b1, w2, b2, w3, b3):
    """d/d(parameters) of ``sum_v g_v mlp(x_v)`` from two moments per region, ``G0 = sum g`` and ``G1 = sum g x`` (inside a
    region the Jacobian of the network w.r.t. its parameters is affine in x).  Returns the gradients in ``nn.Linear`` layout."""
    import numpy as np
    bps, _, _, xm = mlp_piecewise_table(w1, b1, w2, b2, w3, b3)
    w1 = np.asarray(w1, dtype=np.float64).reshape(-1)
    b1 = np.asarray(b1, dtype=np.float64).reshape(-1)
    w2 = np.asarray(w2, dtype=np.float64)
    b2 = np.asarray(b2, dtype=np.float64).reshape(-1)
    w3 = np.asarray(w3, dtype=np.float64).reshape(-1)
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    g = np.asarray(g, dtype=np.float64).reshape(-1)
    r = np.searchsorted(bps, x, side="right")
    G0 = np.bincount(r, weights=g, minlength=len(xm))
    G1 = np.bincount(r, weights=g * x, minlength=len(xm))
    gw1, gb1, gw2, gb2, gw3, gb3 = np.zeros(32), np.zeros(32), np.zeros((32, 32)), np.zeros(32), np.zeros(32), 0.0
    for k, x0 in enumerate(xm):
        if G0[k] == 0 and G1[k] == 0:
            continue
        m1 = (w1 * x0 + b1) > 0
        p, q = w2 @ (m1 * w1), w2 @ (m1 * b1) + b2
        m2 = (p * x0 + q) > 0
        u = m1 * (w2.T @ (m2 * w3))                            # d out / d h1 under both masks
        gw1 += u * G1[k]
        gb1 += u * G0[k]
        gw2 += np.outer(m2 * w3, m1 * (w1 * G1[k] + b1 * G0[k]))
        gb2 += m2 * w3 * G0[k]
        gw3 += m2 * (p * G1[k] + q * G0[k])
        gb3 += G0[k]
    return gw1.reshape(32, 1), gb1, gw2, gb2, gw3.reshape(1, 32), np.asarray([gb3])


# ----------------------------------------------------------------------------------------
# MRI preprocessing  (src/utils.py:12-39, src/impedance.py:39-54)  -- SURVEY row f4
# ----------------------------------------------------------------------------------------


def create_brain_mask(volume: torch.Tensor, threshold=50, iterations: int = 2) -> torch.Tensor:
    """``volume > threshold`` then 2 binary dilations and 2 erosions (``src/utils.py:12-21``).

    scipy's defaults restated with shifts: the structuring element is the 6-neighbour cross and everything
    outside the volume counts as 0 (so erosion eats one layer per pass at the border).
    """
    import torch.nn.functional as F
    m = volume > threshold

    def neighbours(x):
        p = F.pad(x, (1, 1, 1, 1, 1, 1), value=False)
        return [p[2:, 1:-1, 1:-1], p[:-2, 1:-1, 1:-1], p[1:-1, 2:, 1:-1], p[1:-1, :-2, 1:-1], p[1:-1, 1:-1, 2:], p[1:-1, 1:-1, :-2]]

    for _ in range(iterations):
        for nb in neighbours(m):
            m = m | nb
    for _ in range(iterations):
        nbs = neighbours(m)
        for nb in nbs:
            m = m & nb
    return m


def zscore_normalize(volume: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """``(volume - mean) / (std + 1e-8)`` over the masked voxels, unbiased std (``src/utils.py:23-39``)."""
    volume = volume.float()
    inside = volume[mask > 0]
    return (volume - inside.mean()) / (inside.std() + 1e-8)


def compute_impedance_volume(volume, params, threshold=50):
    """``ImpedanceEstimator.compute_impedance_volume`` (``src/impedance.py:39-54``): MLP x 1e6 inside the mask, 400 outside."""
    mask = create_brain_mask(volume, threshold)
    vn = zscore_normalize(volume, mask)
    z = mlp_forward(vn[mask].unsqueeze(1), *params).squeeze() * 1e6
    out = torch.full_like(volume, 400.0)
    out[mask] = z
    return out


# ----------------------------------------------------------------------------------------
# scan conversion  (src/renderer.py:694-737)  -- SURVEY row f1
# ----------------------------------------------------------------------------------------


def splat(x, y, z, intensities, H=256, W=256, sigma=2.0, last_wins=True, dtype=torch.float32):
    """``differentiable_splat`` (``src/renderer.py:694-737``).

    Pick the two axes of largest coordinate variance (descending); round+clamp to pixels;
    NON-accumulating indexed write of intensities and ones; blur both with a normalised
    separable Gaussian of size ``int(6 sigma) | 1``; divide; return transposed.

    Duplicate pixels: ``index_put_(accumulate=False)`` leaves WHICH write survives undefined
    (torch 2.11's CPU kernel is parallel: measured here, the first and the last duplicate
    both win, depending on thread chunking).  ``last_wins=True`` pins the sequential
    reading -- the sample with the highest flat index survives -- while keeping torch's
    backward, in which every duplicate receives its pixel's gradient.

    ``dtype`` is the precision of the image arithmetic (scatter, blur, ratio): float32 as in the reference, float64 for a
    reference value.  The pixel indices are rounded from float32 coordinates either way, as in the reference.
    """
    import torch.nn.functional as F
    coords = [x, y, z]
    variances = [c.float().var().item() for c in coords]
    a0, a1 = sorted(range(3), key=lambda i: -variances[i])[:2]
    c0 = coords[a0].to(torch.float32)
    c1 = coords[a1].to(torch.float32)
    val = intensities.to(dtype)
    img = torch.zeros((1, 1, H, W), dtype=dtype)
    wgt = torch.zeros_like(img)
    i0 = torch.clamp(c0.round().long(), 0, W - 1)
    i1 = torch.clamp(c1.round().long(), 0, H - 1)
    if last_wins:
        flat = (i1 * W + i0).reshape(-1)
        order = torch.arange(flat.numel())
        winner = torch.full((H * W,), -1, dtype=torch.long).scatter_reduce(0, flat, order, "amax", include_self=True)
        vflat = val.reshape(-1)
        val = (vflat + (vflat.detach()[winner[flat]] - vflat.detach())).reshape(val.shape)   # value of the winner, own gradient
    img[0, 0, i1, i0] += val
    wgt[0, 0, i1, i0] += 1
    size = int(6 * sigma) | 1
    t = (torch.arange(size) - size // 2).to(dtype)
    k1 = torch.exp(-0.5 * (t / sigma) ** 2)
    k1 = k1 / k1.sum()
    k2 = (k1[:, None] @ k1[None, :])[None, None]
    bi = F.conv2d(img, k2, padding=size // 2)
    bw = F.conv2d(wgt, k2, padding=size // 2)
    return (bi / (bw + 1e-8))[0, 0].T


def flops_dense_per_ray(n_interfaces: int) -> float:
    """Rough LU flop count of the reference's per-depth solves, for reporting only."""
    return sum(2.0 / 3.0 * (2 * (k + 1)) ** 3 for k in range(n_interfaces + 1))


__all__ = [n for n in dir() if not n.startswith("_") and n not in ("math", "np", "torch", "annotations")]


# ----------------------------------------------------------------------------------------
# training-loop pieces  -- SURVEY row f3 / f1 epilogue
# ----------------------------------------------------------------------------------------


def rotate_around_apex(x, z, apex, median):
    """``src/renderer.py:655-692``: shift x by the hard-wired 128, rotate by atan2(m_x, m_y) of the normalised median with a
    2 x 2 matrix product over the stacked 1-D coordinate arrays, add the apex."""
    x_shifted = x - 128
    z_shifted = z
    median_vec = torch.as_tensor(median, dtype=torch.float32)
    median_vec = median_vec / median_vec.norm()
    angle = torch.atan2(median_vec[0], median_vec[1])
    cos_a, sin_a = torch.cos(angle), torch.sin(angle)
    rot = torch.tensor([[cos_a, -sin_a], [sin_a, cos_a]])
    rotated = rot @ torch.stack((x_shifted, z_shifted), dim=0)
    return rotated[0] + apex[0], rotated[1] + apex[1]


def masked_mse_edge_loss(a, b, mask, edge_weight=0.5):
    """``UltrasoundSynthesisModel.loss`` + ``gradient_loss`` of ``notebooks/[DEMO] Train MRI to Impedance MLP.ipynb`` cell 19:
    ``mse(a[mask], b[mask]) + 0.5 * l1(|a[:,1:] - a[:,:-1]|[mask[:,1:]], |b[:,1:] - b[:,:-1]|[mask[:,1:]])``."""
    import torch.nn.functional as F
    main = F.mse_loss(a[mask], b[mask])
    a_grad = torch.abs(a[:, 1:] - a[:, :-1])
    b_grad = torch.abs(b[:, 1:] - b[:, :-1])
    return main + edge_weight * F.l1_loss(a_grad[mask[:, 1:]], b_grad[mask[:, 1:]])


def ssim_piq(x, y, kernel_size=11, kernel_sigma=1.5, k1=0.01, k2=0.03):
    """``piq.ssim(x, y, data_range=1.0)`` for single-channel (H, W) images below 384 pixels (no down-sampling).

    piq is a dependency of the reference's GPU training notebook (cell 16) that is neither vendored by the reference nor
    installed here, so this is a restatement of its published algorithm (piq 0.8 ``ssim`` / ``_ssim_per_channel`` /
    ``gaussian_filter``; Wang et al. 2004) and NOT pinned by running piq: window = outer product of
    ``exp(-(i - (K-1)/2)^2 / (2 sigma^2))`` normalised to sum 1; VALID filtering (no padding); ``mu_x, mu_y``;
    ``sigma_xx = E[x^2] - mu_x^2`` etc.; ``cs = (2 sigma_xy + c2) / (sigma_xx + sigma_yy + c2)``;
    ``ss = (2 mu_x mu_y + c1) / (mu_x^2 + mu_y^2 + c1) * cs``; mean over the map; ``c1 = k1^2, c2 = k2^2`` at data_range 1.
    """
    import torch.nn.functional as F
    coords = torch.arange(kernel_size, dtype=x.dtype) - (kernel_size - 1) / 2.0
    g = coords ** 2
    g = (-(g.unsqueeze(0) + g.unsqueeze(1)) / (2 * kernel_sigma ** 2)).exp()
    kernel = (g / g.sum())[None, None]
    X, Y = x[None, None], y[None, None]
    c1, c2 = k1 ** 2, k2 ** 2
    mu_x, mu_y = F.conv2d(X, kernel), F.conv2d(Y, kernel)
    mu_xx, mu_yy, mu_xy = mu_x ** 2, mu_y ** 2, mu_x * mu_y
    sigma_xx = F.conv2d(X ** 2, kernel) - mu_xx
    sigma_yy = F.conv2d(Y ** 2, kernel) - mu_yy
    sigma_xy = F.conv2d(X * Y, kernel) - mu_xy
    cs = (2.0 * sigma_xy + c2) / (sigma_xx + sigma_yy + c2)
    ss = (2.0 * mu_xy + c1) / (mu_xx + mu_yy + c1) * cs
    return ss.mean()


def ssim_loss(synth, real, normalize=True, **kw):
    """``UltrasoundSynthesisModel.loss`` of ``notebooks/[DEMO] Train MRI to Impedance MLP - GPU.ipynb`` cell 16:
    ``synth = (synth - min) / (max - min + 1e-8)``; ``1 - piq.ssim(synth, real, data_range=1.0)``."""
    if normalize:
        synth = (synth - synth.min()) / (synth.max() - synth.min() + 1e-8)
    return 1 - ssim_piq(synth, real, **kw)


def process_rf_to_bmode(profiles):
    """``notebooks/[DEMO] Renderer Alternatives.ipynb`` cell 14: ``log1p(|hilbert(rf, axis=1)|) / max``.

    ``scipy.signal.hilbert`` restated with numpy's FFT (its algorithm: ``ifft(fft(x) * h)`` with ``h = [1, 2, .., 2, 1, 0, ..]``
    for even and ``[1, 2, .., 2, 0, ..]`` for odd lengths); the fixture in tests/golden was made by the notebook's own cell
    with scipy."""
    rf = profiles.detach().cpu().numpy().astype(np.float64)
    n = rf.shape[1]
    h = np.zeros(n)
    if n % 2 == 0:
        h[0] = h[n // 2] = 1
        h[1:n // 2] = 2
    else:
        h[0] = 1
        h[1:(n + 1) // 2] = 2
    analytic = np.fft.ifft(np.fft.fft(rf, axis=1) * h[None, :], axis=1)
    bmode = np.log1p(np.abs(analytic))
    return bmode / np.max(bmode)


def log_compress(img):
    """The log-compression step alone, differentiable: ``log1p(|img|) / max(log1p(|img|))``."""
    b = torch.log1p(img.abs())
    return b / b.max()


def adam_steps(params, grads, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
    """``torch.optim.Adam`` (the optimiser of ``src/impedance.py:26-35`` and of the training notebooks) applied to one flat
    parameter vector for the given sequence of gradients; returns the parameter vector after every step."""
    p = torch.nn.Parameter(params.clone())
    opt = torch.optim.Adam([p], lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
    out = []
    for g in grads:
        p.grad = g.clone()
        opt.step()
        out.append(p.detach().clone())
    return out


__all__ = [n for n in dir() if not n.startswith("_") and n not in ("math", "np", "torch", "annotations")]
