"""GPU: ``ops.launch_count()`` (the library's own count of the kernels it enqueued) against the kernels of the ``diffus``
namespace that torch.profiler records for the same call, over the dispatch paths whose launch numbers differ: each sampler
and layout, the start > 0 median, per-ray sources, long rays with and without the prefix pre-pass, the two-stage loss sum
of more than 2^18 rays, the Gauss-Newton systems with and without a given pivot, and the radius-0 blur (a copy, no kernel)."""
import pytest
import torch

from diffus_b200 import PreparedVolume, ops
from diffus_b200._lib import SAMPLER_NEAREST, SAMPLER_TRILINEAR

pytestmark = pytest.mark.gpu

N = 24


def _volume():
    g = torch.Generator().manual_seed(0)
    return (1.0 + torch.rand((N, N, N), generator=g)).cuda()


def _rays(P, R, step=0.5, per_ray=False):
    g = torch.Generator().manual_seed(1)
    src = torch.tensor([N * 0.5, N * 0.5, 1.0]).repeat(P, 1)
    d = torch.tensor([0.0, 0.0, 1.0]) + 0.2 * torch.randn((P, R, 3), generator=g)
    dirs = d / d.norm(dim=-1, keepdim=True) * step
    if per_ray:
        src = src[:, None, :] + 0.3 * torch.randn((P, R, 3), generator=g)
    return src.cuda().contiguous(), dirs.cuda().contiguous()


def _launches(fn):
    """(library count, profiled diffus kernels) of one call."""
    torch.cuda.synchronize()
    n0 = ops.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    n = ops.launch_count() - n0
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "diffus" in e.name]
    return n, len(names)


def _prepared(vol, layout):
    return (vol, None) if layout == "linear" else (vol, PreparedVolume(vol, layout).bricks)


def _mse(vol, bricks, src, dirs, S, start, need_volume, need_pose):
    P, R = src.shape[0], dirs.shape[-2]
    tgt = torch.zeros((P, R, S - start), device="cuda")
    return lambda: ops.render_mse_impl(vol, bricks, [N] * 3, src, dirs, tgt, S, start, 0.5, SAMPLER_TRILINEAR, False,
                                       need_volume, need_pose, False)


@pytest.mark.parametrize("layout", ["linear", "brick", "quad", "texture"])
@pytest.mark.parametrize("sampler", [SAMPLER_NEAREST, SAMPLER_TRILINEAR])
@pytest.mark.parametrize("start", [0, 3])
def test_render_forward_and_backward(layout, sampler, start):
    vol, bricks = _prepared(_volume(), layout)
    src, dirs = _rays(4, 32)
    S = 40

    def fwd_bwd():
        frame, prefix = ops.render_fwd_impl(vol, bricks, [N] * 3, src, dirs, S, start, 0.5, sampler, False, True)
        ops.render_bwd_impl(torch.ones_like(frame), vol, bricks, [N] * 3, src, dirs, prefix, S, start, 0.5, sampler, False,
                            True, True)
    n, k = _launches(fwd_bwd)
    assert n == k > 0


@pytest.mark.parametrize("per_ray", [False, True])
@pytest.mark.parametrize("start", [0, 3])
def test_fused_step_and_trace(per_ray, start):
    vol = _volume()
    src, dirs = _rays(4, 32, per_ray=per_ray)
    for need_volume, need_pose in ((True, True), (False, True), (True, False), (False, False)):
        n, k = _launches(_mse(vol, None, src, dirs, 40, start, need_volume, need_pose))
        assert n == k > 0, (need_volume, need_pose)

    def trace():
        ops.trace_values_bwd(torch.ones((4, 32, 40), device="cuda"), vol, None, [N] * 3, src, dirs, 40, SAMPLER_TRILINEAR,
                             False, True, True)
    n, k = _launches(trace)
    assert n == k > 0


@pytest.mark.parametrize("need_volume", [False, True])
def test_long_rays_with_and_without_the_prefix_pass(need_volume):
    vol = _volume()
    src, dirs = _rays(2, 8, step=0.02)
    S = 1500                                   # three 512-column passes: the pose-only gradient needs no pre-pass
    fn = _mse(vol, None, src, dirs, S, 0, need_volume, True)
    n, k = _launches(fn)
    assert n == k > 0


@pytest.mark.parametrize("need_pose", [False, True])
def test_two_stage_loss_sum_beyond_2_18_rays(need_pose):
    vol = _volume()
    src, dirs = _rays(2100, 128, step=2.0)     # 268 800 rays
    n, k = _launches(_mse(vol, None, src, dirs, 6, 0, False, need_pose))
    assert n == k == (4 if need_pose else 3)


@pytest.mark.parametrize("per_ray", [False, True])
@pytest.mark.parametrize("start", [0, 3])
def test_gauss_newton_systems(per_ray, start):
    vol = _volume()
    src, dirs = _rays(4, 32, per_ray=per_ray)
    tgt = torch.zeros((4, 32, 40 - start), device="cuda")
    n, k = _launches(lambda: ops.render_gauss_newton_impl(vol, None, [N] * 3, src, dirs, tgt, 40, start, 0.5))
    assert n == k > 0
    for pivot in (None, torch.zeros((3,), dtype=torch.float64, device="cuda")):
        n, k = _launches(lambda: ops.render_gauss_newton_sweep_impl(vol, None, [N] * 3, src, dirs, tgt, 40, start, 0.5, pivot))
        assert n == k > 0


@pytest.mark.parametrize("sigma", [0.0, 0.1, 1.0])
def test_gaussian_blur(sigma):
    vol = _volume()
    n, k = _launches(lambda: ops.gaussian_blur_volume(vol, sigma))
    assert n == k == (3 if sigma >= 0.125 else 0)


def test_texture_create_and_update_launch_no_kernel():
    vol = _volume()
    tex = None

    def create():
        nonlocal tex
        tex = ops.VolumeTexture(vol)
    assert _launches(create) == (0, 0)
    assert _launches(lambda: tex.update(vol)) == (0, 0)
    tex.close()
