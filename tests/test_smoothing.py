"""CPU: the float64 smoothing oracle, the C-ABI argument checks of ``diffus_volume_gaussian_blur`` and the schedule checks of
``recover_poses_coarse_to_fine`` -- all before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch


def test_oracle_is_gaussian_filter1d_along_each_axis():
    from scipy.ndimage import gaussian_filter1d
    from oracle import smoothing
    g = np.random.default_rng(0)
    v = g.standard_normal((9, 6, 11))
    for sigma, truncate in ((0.7, 4.0), (2.0, 3.0), (5.0, 4.0)):            # 5.0: the radius exceeds every dimension
        want = v
        for axis in range(3):
            want = gaussian_filter1d(want, sigma, axis=axis, mode="nearest", truncate=truncate)
        np.testing.assert_allclose(smoothing.gaussian_blur(v, sigma, truncate), want, rtol=1e-13, atol=1e-13)


def test_oracle_weights_sum_to_one_with_scipys_radius():
    from oracle import smoothing
    for sigma, truncate, r in ((1.0, 4.0, 4), (2.5, 4.0, 10), (0.3, 4.0, 1), (0.1, 4.0, 0), (6.0, 4.0, 24), (1.0, 2.6, 3),
                               (16.0, 4.0, 64)):
        w = smoothing.gaussian_weights(sigma, truncate)
        assert smoothing.gaussian_radius(sigma, truncate) == r == int(truncate * sigma + 0.5)
        assert w.shape == (2 * r + 1,)
        assert abs(w.sum() - 1.0) < 1e-15
        np.testing.assert_array_equal(w, w[::-1])


@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()                       # nvcc cross-compiles without a GPU
    return _lib.load()


def test_gaussian_blur_argument_validation_without_a_device(lib):
    dim = (C.c_int32 * 3)(8, 9, 10)
    n = 8 * 9 * 10 * 4                                              # bytes per buffer
    src, dst, scr = 0x100000, 0x200000, 0x300000                    # fake, non-overlapping device addresses
    blur = lib.diffus_volume_gaussian_blur
    assert blur(None, C.byref(dim), 1.0, 4.0, dst, scr, None) == -1
    assert blur(src, None, 1.0, 4.0, dst, scr, None) == -1
    assert blur(src, C.byref(dim), 1.0, 4.0, None, scr, None) == -1
    assert blur(src, C.byref(dim), 1.0, 4.0, dst, None, None) == -1
    for bad in ((0, 9, 10), (8, -1, 10), (8, 9, 0)):
        assert blur(src, C.byref((C.c_int32 * 3)(*bad)), 1.0, 4.0, dst, scr, None) == -2
    for sigma, truncate in ((-0.5, 4.0), (float("nan"), 4.0), (float("inf"), 4.0), (1.0, 0.0), (1.0, -4.0), (1.0, float("nan")),
                            (1.0, float("inf"))):
        assert blur(src, C.byref(dim), sigma, truncate, dst, scr, None) == -2, (sigma, truncate)
    assert blur(src, C.byref(dim), 1.0, 4.0, src, scr, None) == -2                   # dst is src
    assert blur(src, C.byref(dim), 1.0, 4.0, dst, dst, None) == -2                   # scratch is dst
    assert blur(src, C.byref(dim), 1.0, 4.0, src + n - 4, scr, None) == -2           # dst overlaps src's last voxel
    assert blur(src, C.byref(dim), 1.0, 4.0, dst, src - n + 4, None) == -2           # scratch overlaps src's first voxel
    assert blur(src, C.byref(dim), 16.2, 4.0, dst, scr, None) == -5                  # r = int(65.3) > 64
    assert blur(src, C.byref(dim), 1.0, 1e30, dst, scr, None) == -5
    assert lib.diffus_error_string(-5) not in (b"ok", b"unknown error")


def test_coarse_to_fine_rejects_bad_schedules_before_touching_a_device():
    from diffus_b200 import recover_poses_coarse_to_fine
    z = torch.zeros((2, 3))
    t = torch.zeros((2, 4, 8))

    def run(**kw):
        recover_poses_coarse_to_fine(torch.zeros((4, 4, 4)), t, z, z, z, 1.0, 4, 8, **kw)
    for sigmas in ((), [], (2.0, -1.0), (float("nan"),), (1.0, float("inf"))):
        with pytest.raises(ValueError, match="sigmas"):
            run(sigmas=sigmas)
    for iterations in ((5, 5), [3, 3, 3, 3, 3], (5, -1, 2, 1), (5, 2.5, 1, 1), -2, True):
        with pytest.raises(ValueError, match="iterations"):
            run(iterations=iterations)
