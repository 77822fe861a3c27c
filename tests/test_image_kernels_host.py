"""CPU: the float64 oracles that tests/test_gpu_image_kernels.py trusts, pinned by independent implementations (scipy, explicit
loops), and the host-side argument checks of the image-space, preprocessing and training-loop entry points of the C ABI.

Every call in the ABI tests passes fake pointers only to calls whose host checks reject them: nothing reaches a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import port

E_NULL, E_SHAPE, E_ENUM, E_WORKSPACE, E_UNSUPPORTED = -1, -2, -3, -4, -5
P = 0x1000                                           # a fake device pointer: never dereferenced, every call below is rejected


# ---------------------------------------------------------------------------------------------------------------------
# the oracles
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2, 3, 64, 255, 256, 257, 1025])
def test_rf_to_bmode_oracle_matches_scipy_hilbert(S):
    from scipy.signal import hilbert
    rf = torch.randn((5, S), generator=torch.Generator().manual_seed(S), dtype=torch.float64)
    b = np.log1p(np.abs(hilbert(rf.numpy(), axis=1)))
    np.testing.assert_allclose(port.process_rf_to_bmode(rf), b / b.max(), rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("dims", [(1, 9, 7), (6, 1, 11), (5, 8, 1), (1, 1, 13), (9, 10, 7), (12, 5, 16)])
@pytest.mark.parametrize("iterations", [1, 2, 5])
def test_brain_mask_oracle_matches_scipy_morphology(dims, iterations):
    from scipy import ndimage
    vol = torch.randint(0, 101, dims, generator=torch.Generator().manual_seed(sum(dims) + iterations)).float()
    m = vol.numpy() > 50                                 # voxels equal to the threshold are outside (the rule is >)
    m = ndimage.binary_dilation(m, iterations=iterations, border_value=0)
    m = ndimage.binary_erosion(m, iterations=iterations, border_value=0)
    np.testing.assert_array_equal(port.create_brain_mask(vol, 50, iterations=iterations).numpy(), m)
    # iterations=0: scipy reads 0 as "until nothing changes"; the port (and the reference's loop) does no pass at all
    np.testing.assert_array_equal(port.create_brain_mask(vol, 50, iterations=0).numpy(), vol.numpy() > 50)


@pytest.mark.parametrize("K,sigma,shape", [(1, 1.0, (4, 6)), (3, 0.5, (7, 5)), (7, 1.5, (9, 12)), (11, 1.5, (13, 11)),
                                           (5, 5.0, (5, 5))])
def test_ssim_oracle_matches_a_loop_over_windows(K, sigma, shape):
    gen = torch.Generator().manual_seed(K)
    x = torch.rand(shape, generator=gen, dtype=torch.float64)
    y = torch.rand(shape, generator=gen, dtype=torch.float64)
    k1, k2 = 0.02, 0.05
    c = np.arange(K) - (K - 1) / 2
    w = np.exp(-(c[:, None] ** 2 + c[None, :] ** 2) / (2 * sigma ** 2))
    w /= w.sum()
    X, Y = x.numpy(), y.numpy()
    vals = []
    for r in range(shape[0] - K + 1):
        for q in range(shape[1] - K + 1):
            px, py = X[r:r + K, q:q + K], Y[r:r + K, q:q + K]
            mx, my = (w * px).sum(), (w * py).sum()
            vx, vy, cxy = (w * px * px).sum() - mx * mx, (w * py * py).sum() - my * my, (w * px * py).sum() - mx * my
            vals.append((2 * mx * my + k1 ** 2) * (2 * cxy + k2 ** 2) / ((mx * mx + my * my + k1 ** 2) * (vx + vy + k2 ** 2)))
    got = port.ssim_piq(x, y, kernel_size=K, kernel_sigma=sigma, k1=k1, k2=k2).item()
    assert abs(got - np.mean(vals)) <= 1e-12


@pytest.mark.parametrize("edge_weight", [0.5, 1.75])
def test_masked_mse_edge_oracle_matches_a_pixel_sum(edge_weight):
    gen = torch.Generator().manual_seed(3)
    a = torch.randint(-8, 9, (7, 9), generator=gen).double() / 4        # ties |da| = |db| and da = 0 occur
    b = torch.randint(-8, 9, (7, 9), generator=gen).double() / 4
    mask = torch.rand((7, 9), generator=gen) > 0.4
    s1 = n1 = s2 = n2 = 0.0
    for i in range(7):
        for j in range(9):
            if not mask[i, j]:
                continue
            s1 += float(a[i, j] - b[i, j]) ** 2
            n1 += 1
            if j >= 1:
                s2 += abs(abs(float(a[i, j] - a[i, j - 1])) - abs(float(b[i, j] - b[i, j - 1])))
                n2 += 1
    want = s1 / n1 + edge_weight * s2 / n2
    assert abs(port.masked_mse_edge_loss(a, b, mask, edge_weight).item() - want) <= 1e-12 * want


# ---------------------------------------------------------------------------------------------------------------------
# host-side argument checks
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()                       # nvcc cross-compiles without a GPU
    return _lib.load()


def test_ssim_arguments_are_checked_on_the_host(lib):
    assert lib.diffus_ssim_workspace_bytes(32, 32, 11) > 0
    assert lib.diffus_ssim_workspace_bytes(32, 32, 35) == 0                    # K > 33
    assert lib.diffus_ssim_workspace_bytes(8, 32, 11) == 0                     # K > H
    assert lib.diffus_ssim_workspace_bytes(32, 8, 11) == 0                     # K > W
    big = 1 << 30

    def fwd(H, W, K, sigma=1.5, ws=P, nbytes=big, loss=P):
        return lib.diffus_ssim_loss_forward(P, P, H, W, K, sigma, 0.01, 0.03, 1, loss, ws, nbytes, None)

    def bwd(H, W, K, sigma=1.5, ws=P, nbytes=big):
        return lib.diffus_ssim_loss_backward(P, P, H, W, K, sigma, 1, P, P, ws, nbytes, None)

    for call in (fwd, bwd):
        assert call(32, 32, 10) == E_UNSUPPORTED                                # even window
        assert call(64, 64, 35) == E_UNSUPPORTED                                # K > 33
        assert call(8, 64, 11) == E_SHAPE                                       # K > H
        assert call(64, 8, 11) == E_SHAPE                                       # K > W
        assert call(32, 32, 0) == E_SHAPE
        assert call(32, 32, 11, sigma=0.0) == E_SHAPE
        assert call(32, 32, 11, sigma=float("nan")) == E_SHAPE
        need = lib.diffus_ssim_workspace_bytes(32, 32, 11)
        assert call(32, 32, 11, nbytes=need - 1) == E_WORKSPACE                # a short workspace
        assert call(32, 32, 11, ws=None) == E_WORKSPACE
    assert fwd(32, 32, 11, loss=None) == E_NULL
    assert lib.diffus_ssim_loss_backward(P, P, 32, 32, 11, 1.5, 1, None, P, P, big, None) == E_NULL


def test_rf_to_bmode_arguments_are_checked_on_the_host(lib):
    assert lib.diffus_rf_to_bmode(P, 4, 28001, P, P, P, 4, None) == E_UNSUPPORTED    # a line and its kernel must fit shared memory
    assert lib.diffus_rf_to_bmode(P, 4, 28000, P, P, P, 3, None) == E_WORKSPACE     # 28 000 passes the size check ...
    assert lib.diffus_rf_to_bmode(P, 4, 28000, P, P, None, 4, None) == E_WORKSPACE   # ... and needs the 4-byte workspace
    assert lib.diffus_rf_to_bmode(P, 0, 16, P, P, P, 4, None) == E_SHAPE
    assert lib.diffus_rf_to_bmode(P, 4, 0, P, P, P, 4, None) == E_SHAPE
    assert lib.diffus_rf_to_bmode(P, 4, 16, None, P, P, 4, None) == E_NULL


def test_adam_arguments_are_checked_on_the_host(lib):
    assert lib.diffus_adam_step(P, P, P, 65537, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None) == E_UNSUPPORTED   # one CTA
    assert lib.diffus_adam_step(P, P, P, 0, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None) == E_SHAPE
    assert lib.diffus_adam_step(P, None, P, 16, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None) == E_NULL


def test_volume_slice_arguments_are_checked_on_the_host(lib):
    dim = (C.c_int32 * 3)(5, 6, 7)
    for axis, index in ((3, 0), (-1, 0), (0, 5), (1, 6), (2, 7), (2, -1)):
        assert lib.diffus_volume_slice(P, C.byref(dim), 0, axis, index, P, 0, None) == E_SHAPE, (axis, index)
    for layout in (2, 3, -1, 7):                                                # QUAD and TEXTURE have no slice kernel
        assert lib.diffus_volume_slice(P, C.byref(dim), layout, 0, 0, P, 1, None) == E_ENUM, layout
    zero = (C.c_int32 * 3)(5, 0, 7)
    assert lib.diffus_volume_slice(P, C.byref(zero), 0, 0, 0, P, 0, None) == E_SHAPE
    assert lib.diffus_volume_slice(P, C.byref(dim), 0, 0, 0, None, 0, None) == E_NULL


def test_conv1d_rows_arguments_are_checked_on_the_host(lib):
    for call in (lib.diffus_conv1d_rows_forward, lib.diffus_conv1d_rows_backward):
        assert call(P, 4, 300, P, 129, 0, P, None) == E_UNSUPPORTED          # taps > 128
        assert call(P, 4, 5, P, 9, 0, P, None) == E_SHAPE                    # n_out = 5 - 9 + 1 < 1
        assert call(P, 4, 5, P, 9, 1, P, None) == E_SHAPE                    # n_out = 0
        assert call(P, 4, 60, P, 9, -1, P, None) == E_SHAPE                  # negative padding
        assert call(P, 0, 60, P, 9, 4, P, None) == E_SHAPE
        assert call(P, 4, 60, P, 0, 4, P, None) == E_SHAPE
        assert call(P, 4, 60, None, 9, 4, P, None) == E_NULL


def test_brain_mask_and_zscore_arguments_are_checked_on_the_host(lib):
    dim = (C.c_int32 * 3)(4, 5, 6)
    assert lib.diffus_brain_mask(P, C.byref(dim), 50.0, 65, P, P, None) == E_SHAPE     # iterations > 64
    assert lib.diffus_brain_mask(P, C.byref(dim), 50.0, -1, P, P, None) == E_SHAPE
    flat = (C.c_int32 * 3)(4, 0, 6)
    assert lib.diffus_brain_mask(P, C.byref(flat), 50.0, 2, P, P, None) == E_SHAPE
    assert lib.diffus_brain_mask(P, C.byref(dim), 50.0, 2, P, None, None) == E_NULL
    assert lib.diffus_masked_zscore(P, P, 120, P, P, 63, None) == E_WORKSPACE          # a short workspace
    assert lib.diffus_masked_zscore(P, P, 120, P, None, 64, None) == E_WORKSPACE
    assert lib.diffus_masked_zscore(P, P, 0, P, P, 64, None) == E_SHAPE
    assert lib.diffus_masked_zscore(P, None, 120, P, P, 64, None) == E_NULL


def test_masked_mse_log_compress_and_splat_arguments_are_checked_on_the_host(lib):
    for H, W in ((0, 8), (8, 0), (-1, 8)):
        assert lib.diffus_masked_mse_edge_forward(P, P, P, H, W, 0.5, P, None) == E_SHAPE
        assert lib.diffus_masked_mse_edge_backward(P, P, P, H, W, 0.5, P, P, P, None) == E_SHAPE
    assert lib.diffus_masked_mse_edge_forward(P, P, None, 8, 8, 0.5, P, None) == E_NULL
    assert lib.diffus_log_compress_forward(P, 0, P, None, None) == E_SHAPE
    assert lib.diffus_log_compress_backward(P, P, 0, P, None) == E_SHAPE
    nbytes = lib.diffus_splat_workspace_bytes(8, 8)
    assert nbytes > 0 and lib.diffus_splat_workspace_bytes(0, 8) == 0
    assert lib.diffus_splat_forward(P, P, P, P, 16, 8, 8, 10.7, P, P, nbytes, None) == E_UNSUPPORTED   # window 65 > 63
    assert lib.diffus_splat_forward(P, P, P, P, 16, 8, 8, 1.0, P, P, nbytes - 1, None) == E_WORKSPACE
    assert lib.diffus_splat_backward(P, P, P, P, 16, 8, 8, 0.0, P, P, P, nbytes, None) == E_SHAPE
