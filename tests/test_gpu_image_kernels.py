"""GPU: the image-space, preprocessing and training-loop kernels against float64 references (or exact equality, for copies
and masks) at the shapes where their tiles, grid-stride loops and single-CTA reductions reach an edge.

Kernel edges exercised here:
  * SSIM: 16 x 16 output tiles with a (16 + K - 1)^2 halo, K up to 33, a (H - K + 1) x (W - K + 1) valid map; a single-CTA
    min / max whose gradient is split evenly over ties;
  * masked MSE + edge: a single-CTA forward; a backward grid-stride loop capped at 148 x 4 CTAs with a right-neighbour term;
  * log compression: single-CTA max and tie count;
  * RF -> B-mode: one CTA per line, the shared-memory opt-in above 48 KB (6 145 samples and more), a frame max over CTAs;
  * conv1d rows: a grid-stride loop capped at 148 x 8 CTAs, negative flipped padding in the backward;
  * volume slice, brain mask, z-score: grid-stride loops capped at 148 x 8 / 148 x 16 CTAs, brick addressing.
Every random input is seeded."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import NOISE_FACTOR, assert_frame_close, assert_grad_close, oracle_grads

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def gen(seed):
    return torch.Generator().manual_seed(seed)


def assert_scalar_close(got, want, what, rtol, noise=0.0):
    """|got - want| <= max(rtol |want|, NOISE_FACTOR x the float32 noise of the reference); NaN never passes."""
    want = float(want)
    scale = max(abs(want), 1e-30)
    assert_frame_close(np.array([float(got)]), np.array([want]), what, atol=max(rtol, NOISE_FACTOR * noise / scale), rtol=0.0)


# ---------------------------------------------------------------------------------------------------------------------
# 1 - SSIM
# ---------------------------------------------------------------------------------------------------------------------
def _ssim_shapes(K):
    return [(K, K),                    # a 1 x 1 map
            (K + 1, K + 15),           # a 2 x 16 map: one tile wide, exactly
            (K + 14, K + 16),          # 15 x 17
            (K + 15, K + 30),          # 16 x 31
            (K + 32, K + 31),          # 33 x 32
            (K + 70, K),               # tall and thin: 71 x 1
            (K, K + 100)]              # short and wide: 1 x 101


SSIM_CASES = [(K, sigma, H, W) for K, sigma in ((1, 0.5), (3, 0.8), (7, 1.0), (11, 1.5), (33, 5.0)) for H, W in _ssim_shapes(K)]
SSIM_CASES += [(11, 1.5, 383, 200), (33, 4.0, 200, 383)]        # below piq's 384 down-sampling limit


def _ssim_check(synth, real, normalize, what, **kw):
    from diffus_b200.losses import ssim_loss
    from oracle import port
    fn = lambda s_: (lambda l_: (l_, l_))(port.ssim_loss(s_, real.to(s_.dtype), normalize=normalize, **kw))
    (gw,), noise, want = oracle_grads(fn, synth)
    loss32 = port.ssim_loss(synth.float(), real.float(), normalize=normalize, **kw).item()
    sd = synth.float().to(dev()).requires_grad_(True)
    got = ssim_loss(sd, real.float().to(dev()), normalize=normalize, **kw)
    got.backward()
    # the local variances E[x^2] - mu^2 cancel: the port's own float32 run sets the floor of both tolerances (see
    # test_gpu_training.py::test_ssim_loss_matches_port).  A one-pixel window (K = 1) has exactly zero variance in piq; the
    # kernel forms E[x^2] - mu^2 with one FMA, which leaves the rounding error of x * x (<= 2^-24 x^2) against c2 = 9e-4:
    # up to 7e-5 of each window's SSIM, magnified by 1 / (1 - SSIM) in the loss.  Rounding the product instead zeroes the
    # variance but makes the backward's 1 / c2 terms cancel inexactly (20x the gradient error), so K = 1 gets 5e-4 on the loss.
    rtol = 5e-4 if kw.get("kernel_size") == 1 else 2e-5
    assert_scalar_close(got.item(), want.item(), f"{what}: loss", rtol=rtol, noise=abs(loss32 - want.item()))
    assert_grad_close(sd.grad.cpu().numpy(), gw.numpy(), f"{what}: d loss / d synth", noise=noise[0])
    return sd, got


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("K,sigma,H,W", SSIM_CASES)
def test_ssim_matches_port_at_tile_and_window_edges(K, sigma, H, W, normalize):
    g = gen(1000 * K + H + 7 * W)
    real = torch.rand((H, W), generator=g, dtype=torch.float64)
    synth = 0.7 * real + 0.3 * torch.rand((H, W), generator=g, dtype=torch.float64)
    if normalize:
        synth = 3.0 * synth - 1.0
    _ssim_check(synth, real, normalize, f"ssim K={K} {H}x{W}", kernel_size=K, kernel_sigma=sigma)


@pytest.mark.parametrize("k1,k2", [(0.05, 0.1), (0.001, 0.3)])
def test_ssim_non_default_constants(k1, k2):
    g = gen(11)
    real = torch.rand((40, 53), generator=g, dtype=torch.float64)
    synth = 0.5 * real + 0.5 * torch.rand((40, 53), generator=g, dtype=torch.float64)
    _ssim_check(synth, real, True, f"ssim k1={k1} k2={k2}", kernel_size=7, kernel_sigma=1.2, k1=k1, k2=k2)


@pytest.mark.parametrize("normalize", [True, False])
def test_ssim_ties_at_the_minimum_and_the_maximum(normalize):
    """Minima and maxima tied across different 16 x 16 tiles: the normalisation's gradient is split evenly over them."""
    g = gen(12)
    real = torch.rand((70, 90), generator=g, dtype=torch.float64)
    synth = 0.2 + 0.6 * torch.rand((70, 90), generator=g, dtype=torch.float64)
    for r, c in ((0, 0), (35, 47), (69, 89)):
        synth[r, c] = 0.0
    for r, c in ((0, 89), (17, 3), (69, 0), (50, 60)):
        synth[r, c] = 1.0
    _ssim_check(synth, real, normalize, "ssim with tied extrema")


def test_ssim_constant_synth():
    """max - min = 0: the 1e-8 of the normalisation decides the result, and every pixel is both the minimum and the maximum."""
    real = torch.rand((37, 45), generator=gen(13), dtype=torch.float64)
    _ssim_check(torch.full((37, 45), 0.3, dtype=torch.float64), real, True, "ssim of a constant image", kernel_size=7)


def test_ssim_is_bit_identical_on_repeat():
    from diffus_b200.losses import ssim_loss
    g = gen(14)
    real = torch.rand((120, 97), generator=g).to(dev())
    synth = torch.rand((120, 97), generator=g).to(dev())
    out = []
    for _ in range(2):
        s = synth.clone().requires_grad_(True)
        loss = ssim_loss(s, real, kernel_size=11)
        loss.backward()
        out.append((loss.detach().clone(), s.grad.clone()))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


# ---------------------------------------------------------------------------------------------------------------------
# masked MSE + edge
# ---------------------------------------------------------------------------------------------------------------------
MSE_SHAPES = [(1, 1), (1, 37), (29, 1), (13, 37), (37, 13), (700, 901)]      # 700 x 901 > 1024 x 148 x 4 pixels
MSE_MASKS = ["all", "random", "pixel", "column0", "checkerboard", "last_column", "empty"]


def _mask(kind, H, W, g):
    m = torch.zeros((H, W), dtype=torch.bool)
    if kind == "all":
        m[:] = True
    elif kind == "random":
        m = torch.rand((H, W), generator=g) > 0.35
    elif kind == "pixel":
        m[H // 2, W // 2] = True
    elif kind == "column0":
        m[:, 0] = True                                  # no edge term: N2 = 0
    elif kind == "checkerboard":
        m = (torch.arange(H)[:, None] + torch.arange(W)[None, :]) % 2 == 0     # no right neighbour is in the mask
    elif kind == "last_column":
        m[:, -1] = True
    return m


def _dyadic(shape, g):
    """Values on a 1/16 grid: every difference and |difference| is exact in float32, so ties |da| = |db| and da = 0 (where
    torch's sign is 0) are met exactly as often as in float64."""
    return torch.randint(-48, 49, shape, generator=g).double() / 16


def _mse_check(a, b, m, edge_weight, what):
    from diffus_b200.losses import masked_mse_edge_loss
    from oracle import port
    a64 = a.clone().requires_grad_(True)
    want = port.masked_mse_edge_loss(a64, b, m, edge_weight)
    gl = 1.7
    (gw,) = torch.autograd.grad(gl * want, a64)
    ad = a.float().to(dev()).requires_grad_(True)
    got = masked_mse_edge_loss(ad, b.float().to(dev()), m.to(dev()), edge_weight)
    (gl * got).backward()
    if torch.isnan(want):                                # an empty mask or an empty edge set: torch's mean of nothing
        assert torch.isnan(got).item(), f"{what}: loss {got.item()} where torch's is NaN"
    else:
        assert_scalar_close(got.item(), want.item(), f"{what}: loss", rtol=1e-6)
    assert_grad_close(ad.grad.cpu().numpy(), gw.numpy(), f"{what}: d loss / d synth")


@pytest.mark.parametrize("kind", MSE_MASKS)
@pytest.mark.parametrize("H,W", MSE_SHAPES)
def test_masked_mse_edge_matches_port(H, W, kind):
    g = gen(H * 1000 + W + MSE_MASKS.index(kind))
    a, b = _dyadic((H, W), g), _dyadic((H, W), g)
    _mse_check(a, b, _mask(kind, H, W, g), 0.5, f"masked mse {H}x{W} {kind}")


@pytest.mark.parametrize("edge_weight", [0.0, 1.75, -0.3])
def test_masked_mse_edge_weight(edge_weight):
    g = gen(21)
    a, b = _dyadic((31, 45), g), _dyadic((31, 45), g)
    _mse_check(a, b, _mask("random", 31, 45, g), edge_weight, f"masked mse, edge weight {edge_weight}")


def test_masked_mse_edge_sign_ties():
    """|da| = |db| everywhere (b = 3 - a), and runs of equal columns (da = 0): every edge term is at a kink of |.|."""
    g = gen(22)
    a = _dyadic((23, 41), g)
    a[:, 10:20] = a[:, 10:11]
    b = 3.0 - a
    b[5] = a[5]                                          # one row with da = db
    _mse_check(a, b, _mask("random", 23, 41, g), 0.5, "masked mse at sign ties")


# ---------------------------------------------------------------------------------------------------------------------
# log compression
# ---------------------------------------------------------------------------------------------------------------------
def _log_input(n, seed):
    x = 3.0 * torch.randn(n, generator=gen(seed), dtype=torch.float64).float().double()
    x[1::7] = 0.0                                        # exact zeros: d|x|/dx = 0 there
    top = 20.0
    x[0] = top
    if n > 2:
        x[n // 2] = -top                                 # a negative element carries the maximum |x|
        x[n - 1] = top                                   # ... tied with others in different warps
    if n > 600:
        x[517] = top
    return x


@pytest.mark.parametrize("n", [1, 31, 1023, 1024, 1025, 70001, 300000])
def test_log_compress_matches_port(n):
    from diffus_b200.losses import log_compress
    from oracle import port
    x = _log_input(n, n)
    w = torch.randn(n, generator=gen(n + 1), dtype=torch.float64)
    x64 = x.clone().requires_grad_(True)
    want = port.log_compress(x64)
    (gw,) = torch.autograd.grad((want * w).sum(), x64)
    outs = []
    for _ in range(2):
        xd = x.float().to(dev()).requires_grad_(True)
        got = log_compress(xd)
        (got * w.float().to(dev())).sum().backward()
        outs.append((got.detach(), xd.grad))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), "not bit-identical on repeat"
    assert_frame_close(outs[0][0].cpu().numpy(), want.detach().numpy(), f"log_compress n={n}", atol=1e-7, rtol=1e-5)
    assert_grad_close(outs[0][1].cpu().numpy(), gw.numpy(), f"d log_compress / dx, n={n}")


# ---------------------------------------------------------------------------------------------------------------------
# RF -> B-mode
# ---------------------------------------------------------------------------------------------------------------------
def _bmode_float32(rf32, g32):
    """The kernel's algorithm -- the circular convolution with Im(ifft(h)), |.|, log1p, / max -- evaluated in float32 on the
    host (float32 BLAS sums): how far a float32 evaluation of it drifts from the float64 FFT reference."""
    from numpy.lib.stride_tricks import sliding_window_view
    S = rf32.shape[1]
    windows = sliding_window_view(np.concatenate([g32, g32])[::-1], S)     # windows[S - 1 - n][m] = g[(n - m) mod S]
    acc = np.empty_like(rf32)
    for n0 in range(0, S, 1024):
        rows = S - 1 - np.arange(n0, min(S, n0 + 1024))
        acc[:, n0:n0 + len(rows)] = rf32 @ np.ascontiguousarray(windows[rows]).T
    b = np.log1p(np.sqrt(rf32 * rf32 + acc * acc))
    return b / b.max()


RF_CASES = [(S, 3) for S in (1, 2, 3, 255, 256, 257, 1024, 6144, 6145)] + [(28000, 1), (28000, 2)]
RF_CASES += [(S, rays) for S in (256, 257) for rays in (1, 128, 1000)] + [(6145, 128)]


@pytest.mark.parametrize("S,rays", RF_CASES)
def test_rf_to_bmode_matches_port(S, rays):
    """6 145 samples is the first line length over 48 KB of shared memory (a line and its kernel); 28 000 is the ABI limit."""
    from diffus_b200.losses import hilbert_kernel, process_rf_to_bmode
    from oracle import port
    rf = (0.05 * torch.randn((rays, S), generator=gen(S + rays))).float()
    if rays > 1:
        rf[0] *= 3.0
        rf[-1] = rf[0]                                   # the frame maximum tied between the first and the last CTA
    want = port.process_rf_to_bmode(rf)
    noise = float(np.abs(_bmode_float32(rf.numpy(), hilbert_kernel(S).numpy()) - want).max())
    got = process_rf_to_bmode(rf.to(dev())).cpu().numpy()
    # each output sums S products in float32; the tolerance is the float32 drift of the same convolution (8x), >= 1e-6
    assert_frame_close(got, want, f"rf -> b-mode S={S} rays={rays}", atol=max(NOISE_FACTOR * noise, 1e-6), rtol=1e-5)
    if rays > 1:
        assert got[0].max() == got[-1].max() == 1.0


# ---------------------------------------------------------------------------------------------------------------------
# conv1d rows (compute_gaussian_pulse)
# ---------------------------------------------------------------------------------------------------------------------
def _conv_cases():
    out = []
    for taps in (1, 2, 10, 127, 128):
        for pad in sorted({0, taps // 2, taps - 1, taps + 3}):
            for n_in in (300, taps - 1):                 # taps - 1: a row shorter than the kernel
                if n_in >= 1 and n_in + 2 * pad - taps + 1 >= 1:
                    out.append((3, n_in, taps, pad))
    return out + [(700, 500, 127, 63), (620, 501, 10, 13)]          # rows x n_out > 148 x 8 x 256: the grid-stride loop wraps


@pytest.mark.parametrize("rows,n_in,taps,pad", _conv_cases())
def test_conv1d_rows_matches_torch(rows, n_in, taps, pad):
    """pad > taps - 1 makes the backward's flipped padding taps - 1 - pad negative."""
    from diffus_b200 import ops
    g = gen(rows + n_in + 1000 * taps + pad)
    x = torch.randn((rows, n_in), generator=g, dtype=torch.float64).float().double()
    w = torch.randn(taps, generator=g, dtype=torch.float64).float().double()
    n_out = n_in + 2 * pad - taps + 1
    gout = torch.randn((rows, n_out), generator=g, dtype=torch.float64)
    fn = lambda x_: (lambda y_: ((y_ * gout.to(y_.dtype)).sum(), y_))(F.conv1d(x_.unsqueeze(1), w.to(x_.dtype)[None, None],
                                                                                padding=pad).squeeze(1))
    (gw,), noise, want = oracle_grads(fn, x)
    xd = x.float().to(dev()).requires_grad_(True)
    got = ops.Conv1dRows.apply(xd, w.float().to(dev()), pad)
    assert got.shape == (rows, n_out)
    (got * gout.float().to(dev())).sum().backward()
    assert_frame_close(got.detach().cpu().numpy(), want.detach().numpy(), f"conv1d rows taps={taps} pad={pad} n_in={n_in}")
    assert_grad_close(xd.grad.cpu().numpy(), gw.numpy(), f"conv1d rows d/dx taps={taps} pad={pad} n_in={n_in}", noise=noise[0])


# ---------------------------------------------------------------------------------------------------------------------
# volume slice (LINEAR / BRICK)
# ---------------------------------------------------------------------------------------------------------------------
SLICE_DIMS = [(5, 7, 3), (1, 6, 9), (6, 1, 5), (7, 5, 1), (9, 13, 10)]


def _brick_offsets(dims):
    """Float offset of every voxel in the 4 x 4 x 2 brick buffer (csrc/common.cuh axis_x / axis_y / axis_z), on the host."""
    D, H, W = dims
    nbj, nbk = (H + 3) // 4, (W + 1) // 2
    sy, sx = nbk * 32, nbj * nbk * 32
    i, j, k = np.meshgrid(np.arange(D), np.arange(H), np.arange(W), indexing="ij")
    return (i >> 2) * sx + (i & 3) * 8 + (j >> 2) * sy + (j & 3) * 2 + (k >> 1) * 32 + (k & 1)


@pytest.mark.parametrize("where", ["first", "middle", "last"])
@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("layout", ["linear", "brick"])
@pytest.mark.parametrize("dims", SLICE_DIMS)
def test_volume_slice_gather_and_scatter(dims, layout, axis, where):
    from diffus_b200 import ops
    index = {"first": 0, "middle": dims[axis] // 2, "last": dims[axis] - 1}[where]
    g = gen(sum(d * 10 ** i for i, d in enumerate(dims)) + axis)
    vol = torch.randn(dims, generator=g)
    rest = [d for a, d in enumerate(dims) if a != axis]
    new = torch.randn(rest, generator=g)
    lay = ops.LAYOUT_BRICK if layout == "brick" else ops.LAYOUT_LINEAR
    buf = ops.to_bricks(vol.to(dev())) if layout == "brick" else vol.to(dev()).clone()
    got = ops.volume_slice(buf, list(dims), lay, axis, index)
    assert torch.equal(got.cpu(), vol.select(axis, index)), "gather"
    before = buf.cpu().view(torch.int32).reshape(-1).clone()             # bits: padding voxels of the brick buffer are arbitrary
    ops.volume_slice(buf, list(dims), lay, axis, index, new.to(dev()).contiguous(), scatter=True)
    want = vol.clone()
    want.select(axis, index).copy_(new)
    after = buf.cpu().view(torch.int32).reshape(-1)
    if layout == "brick":
        assert torch.equal(ops.from_bricks(buf, list(dims)).cpu(), want), "scatter"
        offs = torch.from_numpy(_brick_offsets(dims))
        sel = offs.select(axis, index).reshape(-1)
        assert torch.equal(after[sel], new.reshape(-1).view(torch.int32)), "scatter through the brick addressing"
    else:
        assert torch.equal(buf.cpu(), want), "scatter"
        sel = torch.arange(vol.numel()).reshape(dims).select(axis, index).reshape(-1)
    untouched = torch.ones(after.numel(), dtype=torch.bool)
    untouched[sel] = False
    assert torch.equal(after[untouched], before[untouched]), "a voxel outside the slice changed"


@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("dims", [(5, 7, 3), (1, 6, 9), (7, 5, 1)])
def test_slice_insert_gradients(dims, axis):
    from diffus_b200.ops import SliceInsertFunction
    g = gen(sum(dims) + axis)
    index = dims[axis] - 1
    vol = torch.randn(dims, generator=g)
    sl = torch.randn([d for a, d in enumerate(dims) if a != axis], generator=g)
    w = torch.randn(dims, generator=g)
    v_ref, s_ref = vol.clone().requires_grad_(True), sl.clone().requires_grad_(True)
    out_ref = v_ref.clone()
    out_ref.select(axis, index).copy_(s_ref)
    (out_ref * w).sum().backward()
    vd, sd = vol.to(dev()).requires_grad_(True), sl.to(dev()).requires_grad_(True)
    out = SliceInsertFunction.apply(vd, sd, axis, index)
    (out * w.to(dev())).sum().backward()
    assert torch.equal(out.detach().cpu(), out_ref.detach())
    assert torch.equal(vd.grad.cpu(), v_ref.grad) and torch.equal(sd.grad.cpu(), s_ref.grad)


# ---------------------------------------------------------------------------------------------------------------------
# Adam
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 1023, 1024, 1025, 65536])
def test_adam_matches_torch_optim_over_200_steps(n):
    """Weight decay, a gradient scale and 200 steps (the bias corrections of late steps), against torch.optim.Adam in float32."""
    from diffus_b200 import ops
    from oracle import port
    steps, lr, betas, eps, wd = 200, 3e-3, (0.9, 0.99), 1e-8, 0.05
    scale = torch.tensor(0.37, dtype=torch.float32)
    g = gen(n)
    p0 = torch.randn(n, generator=g)
    grads = torch.randn((steps, n), generator=g) * torch.rand((1, n), generator=g) * 3
    want = torch.stack(port.adam_steps(p0, [gr * scale for gr in grads], lr=lr, betas=betas, eps=eps, weight_decay=wd))
    p = p0.to(dev())
    state = torch.zeros((2 * n + 1,), device=dev())
    gd = grads.to(dev())
    hist = []
    for s in range(steps):
        ops.adam_step(p, gd[s], state, lr, betas=betas, eps=eps, weight_decay=wd, grad_scale=float(scale))
        hist.append(p.clone())
    got = torch.stack(hist).cpu()
    peak = float(want.abs().max())
    assert_frame_close(got.numpy(), want.numpy(), f"adam n={n}, every step", atol=2e-7 / peak, rtol=2e-6)
    assert state[-1].item() == steps


# ---------------------------------------------------------------------------------------------------------------------
# brain mask and z-score
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("iterations", [0, 1, 2, 5])
@pytest.mark.parametrize("dims", [(1, 17, 23), (19, 1, 13), (11, 9, 1), (1, 1, 6), (21, 18, 25), (96, 96, 72)])
def test_brain_mask_equals_port(dims, iterations):
    """Integer volumes put many voxels exactly on the threshold (the rule is >); 96 x 96 x 72 > 148 x 16 x 256 voxels."""
    from diffus_b200.utils import create_brain_mask
    from oracle import port
    vol = torch.randint(0, 101, dims, generator=gen(sum(dims) + iterations)).float()
    vol[tuple(d // 2 for d in dims)] = 50.0
    want = port.create_brain_mask(vol, 50, iterations=iterations)
    got = create_brain_mask(vol.to(dev()), 50, iterations=iterations)
    assert torch.equal(got.cpu(), want)


def _zscore_case(kind):
    g = gen(len(kind))
    if kind == "large":
        vol = 100.0 * torch.rand((96, 96, 72), generator=g)
        return vol, vol > 30.0
    vol = 50.0 + 10.0 * torch.randn((13, 17, 11), generator=g)
    mask = torch.zeros(vol.shape, dtype=torch.bool)
    if kind == "two":
        mask[0, 0, 0] = mask[12, 16, 10] = True
    elif kind == "one":
        mask[6, 8, 5] = True
    elif kind.startswith("bright"):                       # mean / std = 1e3 or 1e4
        vol = float(kind[len("bright"):]) + torch.randn(vol.shape, generator=g)
        mask = torch.rand(vol.shape, generator=g) > 0.3
    return vol, mask


@pytest.mark.parametrize("kind", ["two", "one", "empty", "large", "bright1000", "bright10000"])
def test_zscore_matches_float64(kind):
    from diffus_b200.utils import zscore_normalize
    vol, mask = _zscore_case(kind)
    v = vol.double()
    inside = v[mask]
    want = ((v - inside.mean()) / (inside.std() + 1e-8)).numpy()
    got = zscore_normalize(vol.to(dev()), mask.to(dev())).cpu().numpy()
    if kind in ("one", "empty"):                          # torch: the std of one value (and the mean of none) is NaN
        assert np.isnan(want).all() and np.isnan(got).all()
        return
    # float64 statistics and one rounding of the output: 1e-6
    assert_frame_close(got, want, f"zscore {kind}", atol=1e-6, rtol=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
# splat
# ---------------------------------------------------------------------------------------------------------------------
SPLAT_CASES = [(1, 40, 2000, 2.0), (40, 1, 2000, 2.0), (23, 57, 3000, 2.0), (1, 40, 2000, 10.4), (23, 57, 3000, 10.4),
               (20, 30, 70000, 1.0)]                     # sigma 10.4: the 63-pixel window; 70 000 samples on 600 pixels


@pytest.mark.parametrize("H,W,n,sigma", SPLAT_CASES)
def test_splat_matches_port(H, W, n, sigma):
    from diffus_b200 import differentiable_splat
    from oracle import port
    g = gen(H * 100 + W + n)
    # coordinates outside the image clamp to its border; x has the largest variance (the image's width), then y, then z
    cx = torch.rand(n, generator=g) * (max(H, W) + 30) - 10
    cy = torch.rand(n, generator=g) * (H + 20) - 10
    cz = torch.rand(n, generator=g) * 2.0
    v = torch.randn(n, generator=g)
    w = torch.randn((W, H), generator=g)
    # the port's image arithmetic in float64 (the reference value) and in float32 (the drift the 1e-4 may be widened by): the
    # gradient of a pixel sums up to 63 x 63 window weights of random-signed upstream gradients
    fn = lambda v_: (lambda img_: ((img_ * w.to(v_.dtype)).sum(), img_))(port.splat(cx, cy, cz, v_, H=H, W=W, sigma=sigma,
                                                                                        dtype=v_.dtype))
    (gw,), noise, want = oracle_grads(fn, v)
    vd = v.to(dev()).requires_grad_(True)
    got = differentiable_splat(cx.to(dev()), cy.to(dev()), cz.to(dev()), vd, H=H, W=W, sigma=sigma)
    assert got.shape == (W, H)
    (got * w.to(dev())).sum().backward()
    peak = float(want.detach().abs().max())
    assert_frame_close(got.detach().cpu().numpy(), want.detach().numpy(), f"splat {H}x{W} n={n} sigma={sigma}",
                       atol=2e-6 / peak, rtol=2e-5)
    assert_grad_close(vd.grad.cpu().numpy(), gw.numpy(), f"splat d/dintensities {H}x{W} n={n} sigma={sigma}", noise=noise[0])
