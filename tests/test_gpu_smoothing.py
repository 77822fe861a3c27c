"""GPU: ``smooth_volume`` (``diffus_volume_gaussian_blur``) against the float64 scipy oracle, its copy and determinism rules,
and its output as the volume of every render layout."""
import numpy as np
import pytest
import torch

from conftest import assert_frame_close

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _blur_error(vol, sigma, truncate=4.0):
    """max |kernel - oracle| / max |oracle| with the oracle run on the float32 values of the arguments the kernel receives."""
    from diffus_b200 import smooth_volume
    from oracle import smoothing
    got = smooth_volume(vol.to(dev()), sigma, truncate).cpu().numpy()
    want = smoothing.gaussian_blur(vol.numpy(), float(np.float32(sigma)), float(np.float32(truncate)))
    assert got.shape == want.shape and got.dtype == np.float32
    return float(np.abs(got - want).max() / np.abs(want).max())


@pytest.mark.parametrize("shape", [(1, 1, 1), (5, 7, 3), (37, 41, 29), (64, 64, 64)])
@pytest.mark.parametrize("sigma", [0.3, 1.0, 2.5, 6.0])
def test_blur_matches_scipy(shape, sigma):
    g = torch.Generator().manual_seed(sum(shape) + int(10 * sigma))
    vol = 1.0 + torch.rand(shape, generator=g)                      # impedance-like: positive, about one value
    err = _blur_error(vol, sigma)
    print(f"{shape} sigma={sigma}: max |err| / max |ref| = {err:.2e}")
    assert err <= 2e-6


def test_blur_radius_beyond_the_dimensions_repeats_the_edge_voxels():
    """r = 40 against dimensions of 3..50: the clamped index repeats an edge voxel up to 40 times per side."""
    g = torch.Generator().manual_seed(5)
    vol = 1.0 + torch.rand((3, 50, 17), generator=g)
    err = _blur_error(vol, 10.0)
    print(f"r=40 over (3,50,17): {err:.2e}")
    assert err <= 2e-6


def test_blur_of_the_mri_phantom_at_full_size():
    from diffus_b200.phantoms import intensity_to_impedance, mri_phantom
    err = _blur_error(intensity_to_impedance(mri_phantom(256, "t1", seed=0)), 4.0)
    print(f"256^3 MRI phantom sigma=4: {err:.2e}")
    assert err <= 2e-6


def test_sigma_zero_is_the_input_and_two_calls_are_bit_identical():
    from diffus_b200 import PreparedVolume, smooth_volume
    g = torch.Generator().manual_seed(1)
    vol = torch.randn((33, 20, 47), generator=g).to(dev())
    vol[3, 4, 5] = float("nan")
    vol[0, 0, 0] = -0.0
    same = smooth_volume(vol, 0.0)
    assert same.data_ptr() != vol.data_ptr()
    assert torch.equal(same.view(torch.int32), vol.view(torch.int32))          # bit-equal, NaN and -0 included
    assert torch.equal(smooth_volume(PreparedVolume(vol.nan_to_num(), "brick"), 0.0), vol.nan_to_num())
    ok = vol.nan_to_num()
    for sigma in (0.8, 3.0, 16.0):
        a, b = smooth_volume(ok, sigma), smooth_volume(ok, sigma)
        assert torch.equal(a, b), sigma


def test_not_differentiable_raises_instead_of_detaching():
    from diffus_b200 import smooth_volume
    from diffus_b200._lib import DiffusError
    vol = torch.rand((8, 8, 8), device=dev()).requires_grad_(True)
    with pytest.raises(DiffusError, match="not differentiable"):
        smooth_volume(vol, 1.0)
    with torch.no_grad():
        assert smooth_volume(vol, 1.0).shape == (8, 8, 8)
    with pytest.raises(DiffusError, match="code -5"):
        smooth_volume(vol.detach(), 20.0)                                        # r = 80 > 64
    with pytest.raises(DiffusError, match="no CPU fallback"):
        smooth_volume(vol.detach().cpu(), 1.0)


@pytest.mark.parametrize("layout", ["brick", "quad", "texture", "auto"])
def test_blurred_volume_feeds_every_layout_and_renders(layout):
    from diffus_b200 import PreparedVolume, render_frames, smooth_volume
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n = 48
    blurred = smooth_volume(layered_phantom(n, seed=3).to(dev()), 1.5)
    sources, dirs = pose_sweep(4, n_rays=16, n=n, seed=2)
    sources, dirs = sources.to(dev()), dirs.to(dev())
    want = render_frames(blurred, sources, dirs, 80, 1e-3, sampler="trilinear")
    pv = PreparedVolume(blurred, layout)
    got = render_frames(pv, sources, dirs, 80, 1e-3, sampler="trilinear")
    assert torch.isfinite(got).all() and float(got.abs().max()) > 0
    assert_frame_close(got.cpu().numpy(), want.cpu().numpy(), f"{layout} vs linear")
    pv.close()
    torch.testing.assert_close(render_frames(pv, sources, dirs, 80, 1e-3, sampler="trilinear"), got, rtol=0, atol=0)
