"""GPU parity: the CUDA path (through the Python drop-in -> torch.library -> C ABI) against the
golden fixtures produced by the unmodified reference, and against the CPU oracle on seeded
inputs.  Tolerances (tests/conftest.py, north_star): frames |a-b| <= 1e-4 peak + 1e-5 |b|;
gradients 1e-4 relative element-wise above 1e-3 of the largest entry; indices bit-exact."""
import math

import numpy as np
import pytest
import torch

from conftest import GRAD_RTOL, NOISE_FACTOR, assert_frame_close, assert_grad_close, oracle_grads

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


NEAREST_CASES = ["a0", "a7", "afrac", "b0", "b5", "c0", "d0"]


def _start(g, name):
    s = float(g[f"{name}_start"])
    return s if bool(g[f"{name}_start_is_float"]) else int(s)


@pytest.mark.parametrize("name", NEAREST_CASES)
def test_plot_beam_frame_nearest_golden(golden_frames, name):
    from diffus_b200 import UltrasoundRenderer
    g = golden_frames
    vol = torch.tensor(g[f"{name}_volume"], device=dev())
    src = torch.tensor(g[f"{name}_source"], device=dev())
    dirs = torch.tensor(g[f"{name}_dirs"], device=dev())
    ren = UltrasoundRenderer(int(g[f"{name}_S"]), float(g[f"{name}_alpha"]))
    x, y, z, frame = ren.plot_beam_frame(volume=vol, source=src, directions=dirs, plot=False, artifacts=False,
                                         start=_start(g, name))
    assert frame.dtype == torch.float32 and x.dtype == torch.int64
    np.testing.assert_array_equal(x.cpu().numpy(), g[f"{name}_x"])
    np.testing.assert_array_equal(y.cpu().numpy(), g[f"{name}_y"])
    np.testing.assert_array_equal(z.cpu().numpy(), g[f"{name}_z"])
    assert_frame_close(frame.cpu().numpy(), g[f"{name}_frame64"], name)
    # the reference's own fp32 run is within the same tolerance of its fp64 run
    assert_frame_close(g[f"{name}_frame32"], g[f"{name}_frame64"], name + " (reference fp32 vs fp64)")


@pytest.mark.parametrize("name", ["a0", "b0", "d0"])
def test_simulate_rays_golden(golden_frames, name):
    from diffus_b200 import UltrasoundRenderer
    g = golden_frames
    vol = torch.tensor(g[f"{name}_volume"], device=dev())
    src = torch.tensor(g[f"{name}_source"], device=dev())
    dirs = torch.tensor(g[f"{name}_dirs"], device=dev())
    ren = UltrasoundRenderer(int(g[f"{name}_S"]), float(g[f"{name}_alpha"]))
    x, y, z, R = ren.simulate_rays(vol, src, dirs)
    np.testing.assert_allclose(R.cpu().numpy(), g[f"{name}_refl"], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_simulate_rays_is_differentiable_like_the_reference(sampler):
    """simulate_rays / trace_ray outputs carry gradients to the volume (and the pose for trilinear), SURVEY 3.2."""
    from diffus_b200 import PreparedVolume, UltrasoundRenderer
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    from oracle import port
    vol = layered_phantom(20, seed=7)
    sources, dirs = pose_sweep(1, n_rays=5, n=20, seed=1)
    src, d = sources[0], dirs[0]
    S = 30
    w = torch.randn((5, S - 1), generator=torch.Generator().manual_seed(0), dtype=torch.float64)

    def oracle(v_, s_, d_):
        imp = (port.sample_nearest if sampler == "nearest" else port.sample_trilinear)(v_, port.ray_points(s_, d_, S))[3]
        R_ = port.reflection_coeff(imp[:, :-1], imp[:, 1:])
        return (R_ * w.to(R_.dtype)).sum(), R_
    want, noise, R64 = oracle_grads(oracle, vol, src, d)
    for prepared in (False, True):
        v = vol.to(dev()).requires_grad_(True)
        s = src.to(dev()).requires_grad_(True)
        dd = d.to(dev()).requires_grad_(True)
        ren = UltrasoundRenderer(S, 1e-3)
        x, y, z, R = ren.simulate_rays(PreparedVolume(v) if prepared else v, s, dd, sampler=sampler)
        np.testing.assert_allclose(R.detach().cpu().numpy(), R64.detach().numpy(), rtol=1e-4, atol=1e-7)
        (R * w.float().to(dev())).sum().backward()
        assert_grad_close(v.grad.cpu().numpy(), want[0].numpy(), "d R / d volume", noise=noise[0])
        if sampler == "trilinear":
            assert_grad_close(s.grad.cpu().numpy(), want[1].numpy(), "d R / d source", noise=noise[1])
            assert_grad_close(dd.grad.cpu().numpy(), want[2].numpy(), "d R / d directions", noise=noise[2])
        else:
            assert s.grad is None


@pytest.mark.parametrize("name", NEAREST_CASES)
def test_packed_layouts_match_linear(golden_frames, name):
    """BRICK, QUAD and TEXTURE copies hold the same voxels and the kernels do the same arithmetic on them: bit-equal frames."""
    from diffus_b200 import PreparedVolume, render_frames
    g = golden_frames
    vol = torch.tensor(g[f"{name}_volume"], device=dev())
    src = torch.tensor(g[f"{name}_source"], device=dev()).float().reshape(1, 3)
    dirs = torch.tensor(g[f"{name}_dirs"], device=dev())
    S, alpha = int(g[f"{name}_S"]), float(g[f"{name}_alpha"])
    for sampler in ("nearest", "trilinear"):
        a = render_frames(vol, src, dirs, S, alpha, _start(g, name), sampler=sampler)
        for layout in ("brick", "quad", "texture"):
            b = render_frames(PreparedVolume(vol, layout), src, dirs, S, alpha, _start(g, name), sampler=sampler)
            assert torch.equal(a, b), f"{name} {sampler}: {layout} layout changes the result"


@pytest.mark.parametrize("name", ["t0", "t1", "t2"])
def test_trilinear_forward_and_gradients_golden(golden_tri, name):
    from diffus_b200 import UltrasoundRenderer
    g = golden_tri
    vol = torch.tensor(g[f"{name}_volume"], device=dev(), requires_grad=True)
    src = torch.tensor(g[f"{name}_source"], device=dev(), requires_grad=True)
    dirs = torch.tensor(g[f"{name}_dirs"], device=dev(), requires_grad=True)
    ren = UltrasoundRenderer(int(g[f"{name}_S"]), float(g[f"{name}_alpha"]))
    x, y, z, frame = ren.plot_beam_frame(volume=vol, source=src, directions=dirs, plot=False, sampler="trilinear")
    assert_frame_close(frame.detach().cpu().numpy(), g[f"{name}_frame64"], name)
    np.testing.assert_array_equal(x.cpu().numpy(), g[f"{name}_x"])
    w = torch.tensor(g[f"{name}_w"], device=dev(), dtype=torch.float32)
    (frame * w).sum().backward()
    # the reference-made gradients are the target; the port in both precisions supplies the fp32 noise of the same arithmetic
    from oracle import port
    w64, S, alpha = torch.tensor(g[f"{name}_w"]), int(g[f"{name}_S"]), float(g[f"{name}_alpha"])
    _, noise, _ = oracle_grads(lambda v_, s_, d_: (port.plot_beam_frame(v_, s_, d_, S, alpha, sampler="trilinear")[3] * w64.to(v_.dtype)).sum(),
                               torch.tensor(g[f"{name}_volume"]), torch.tensor(g[f"{name}_source"]), torch.tensor(g[f"{name}_dirs"]))
    assert_grad_close(vol.grad.cpu().numpy(), g[f"{name}_grad_volume"], name + " d/dvolume", noise=noise[0])
    assert_grad_close(src.grad.cpu().numpy(), g[f"{name}_grad_source"], name + " d/dsource", noise=noise[1])
    assert_grad_close(dirs.grad.cpu().numpy(), g[f"{name}_grad_dirs"], name + " d/ddirections", noise=noise[2])


def test_nearest_volume_gradient_golden(golden_tri):
    from diffus_b200 import UltrasoundRenderer
    g = golden_tri
    vol = torch.tensor(g["t0_volume"], device=dev(), requires_grad=True)
    src = torch.tensor(g["t0_source"], device=dev(), requires_grad=True)
    dirs = torch.tensor(g["t0_dirs"], device=dev())
    ren = UltrasoundRenderer(36, 1e-3)
    _, _, _, frame = ren.plot_beam_frame(volume=vol, source=src, directions=dirs, plot=False)
    assert_frame_close(frame.detach().cpu().numpy(), g["n0_frame64"], "n0")
    w = torch.tensor(g["n0_w"], device=dev(), dtype=torch.float32)
    (frame * w).sum().backward()
    assert_grad_close(vol.grad.cpu().numpy(), g["n0_grad_volume"], "n0 d/dvolume")
    assert src.grad is None          # HEAD: round().long() cuts the graph (SURVEY 3.2)


def test_gradient_of_a_ray_with_a_zero_over_zero_interface_is_finite():
    """Z1 + Z2 = 0 on one ray (the NaN rule of src/renderer.py:408): the reference's autograd returns NaN for that ray's
    coefficients (0 * NaN inside the solve's backward); here the whole ray contributes ZERO gradient -- finite, and the
    other rays keep theirs (DESIGN.md section 5, deliberate deviations)."""
    from diffus_b200 import compute_echo_traces
    gen = torch.Generator().manual_seed(3)
    r = (torch.rand((4, 300), generator=gen) - 0.5) * 0.2
    r[2, 40] = float("nan")
    r[3, 100] = float("inf")
    w = torch.randn((4, 301), generator=gen)
    rd = r.to(dev()).requires_grad_(True)
    echo, _ = compute_echo_traces(rd)
    assert torch.isfinite(echo).all() and (echo[2, 41:] == 0).all()
    (echo * w.to(dev())).sum().backward()
    g = rd.grad.cpu()
    assert torch.isfinite(g).all()
    assert (g[2] == 0).all() and (g[3] == 0).all()
    clean = r[:2].double().requires_grad_(True)
    from oracle import port
    (port.echo_closed_form(clean) * w[:2].double()).sum().backward()
    assert_grad_close(g[:2].numpy(), clean.grad.numpy(), "rays without a singular interface")


@pytest.mark.parametrize("S,step", [(400, 0.09), (1100, 0.033), (2048, 0.017)])
def test_render_gradient_of_rays_through_a_zero_impedance_block_is_finite(S, step):
    """The same rule inside the fused render kernels (one-pass, and one CTA per ray for the multi-pass rays, whose warps hand
    each other prefixes and adjoint maps that are NaN from the singular interface on): a ray that crosses a block of exactly
    zero impedance (0 / 0 interfaces) renders zeros from there on and contributes a ZERO pose gradient; every other ray is
    bit-identical to the same render without the block."""
    from diffus_b200 import render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    n, P, R = 36, 2, 12
    clean = layered_phantom(n, seed=11)
    holed = clean.clone()
    holed[15:21, 15:21, 15:21] = 0.0
    g = torch.Generator().manual_seed(S)
    sources = torch.tensor([[2.0, 3.0, 2.5], [n - 3.0, 4.0, n * 0.5]])
    aim = torch.tensor([n * 0.5, n * 0.5, n * 0.5]) - sources
    d = aim[:, None, :] / aim.norm(dim=-1)[:, None, None] + 0.45 * torch.randn((P, R, 3), generator=g)
    dirs = d / d.norm(dim=-1, keepdim=True) * step
    out = {}
    for name, vol in (("clean", clean), ("holed", holed)):
        v = vol.to(dev())
        with torch.no_grad():
            target = render_frames(clean.to(dev()), sources.to(dev()) + 0.4, dirs.to(dev()), S, 8e-4, sampler="trilinear")
        s_ = sources.to(dev()).requires_grad_(True)
        d_ = dirs.to(dev()).requires_grad_(True)
        loss, frame = render_mse_loss(v, s_, d_, target, S, 8e-4, 0, sampler="trilinear", return_frame=True)
        loss.backward()
        out[name] = (frame.detach().cpu(), d_.grad.cpu(), s_.grad.cpu(), float(loss.detach()))
    fc, gc, _, _ = out["clean"]
    fh, gh, sh, lh = out["holed"]
    assert torch.isfinite(fh).all() and torch.isfinite(gh).all() and torch.isfinite(sh).all() and np.isfinite(lh)
    untouched = (fc == fh).all(dim=-1)                    # rays whose trilinear cells never reach the block
    singular = (fh[..., -1] == 0) & ~untouched            # rays that went through exact zeros: NaN rule, zeros to the end
    assert untouched.any() and singular.any(), (untouched.sum().item(), singular.sum().item())
    assert torch.equal(gh[untouched], gc[untouched])
    assert (gh[singular] == 0).all()
    assert (fh[singular][:, -8:] == 0).all()


def test_echo_traces_golden(golden_echo):
    from diffus_b200 import compute_echo_traces, propagate_full_rays_batched
    g = golden_echo
    for name in ("nan_lead", "total_reflection", "air_tissue_air", "doc_example"):
        r = torch.tensor(g[f"ka_{name}_r"], device=dev(), dtype=torch.float32)
        echo, delays = compute_echo_traces(r)
        assert_frame_close(echo.cpu().numpy(), g[f"ka_{name}_echo"], name)
    r = torch.tensor(g["phantom_r"], device=dev())
    echo, delays = compute_echo_traces(r)
    assert_frame_close(echo.cpu().numpy(), g["phantom_echo"], "phantom")
    np.testing.assert_allclose(delays.cpu().numpy(), g["phantom_delays"], rtol=1e-6)
    assert_frame_close(propagate_full_rays_batched(r).cpu().numpy(), g["phantom_cumulative"], "phantom cumulative")
    for name in ("rand_a", "rand_b", "rand_c"):
        r = torch.tensor(g[f"{name}_r"], device=dev(), dtype=torch.float32)
        echo, _ = compute_echo_traces(r)
        assert_frame_close(echo.cpu().numpy(), g[f"{name}_echo64"], name)
    from conftest import load_golden
    b = load_golden("echo_brain_phantom2d.npz")                   # the notebook's air / bone phantom, |r| up to 0.9995
    echo, _ = compute_echo_traces(torch.tensor(b["r"], device=dev()))
    assert_frame_close(echo.cpu().numpy(), b["echo64"], "brain phantom 2d")


@pytest.mark.parametrize("B,N", [(3, 1), (5, 31), (4, 512), (2, 513), (3, 1200), (2, 2047)])
def test_echo_forward_backward_vs_oracle(B, N):
    """Ragged lengths across the 512-column segment boundary; gradient vs fp64 autograd of the oracle."""
    from diffus_b200 import compute_echo_traces
    from oracle import port
    g = torch.Generator().manual_seed(N)
    # coefficients of a layered medium: piecewise-constant tissue impedances + 0.5 % texture
    layers = 1.4e6 + 0.3e6 * torch.rand((B, N // 40 + 2), generator=g, dtype=torch.float64)
    Z = layers.repeat_interleave(40, dim=1)[:, :N + 1] * (1 + 0.005 * torch.randn((B, N + 1), generator=g, dtype=torch.float64))
    r64 = port.reflection_coeff(Z[:, :-1], Z[:, 1:]).float().double()          # float32-representable coefficients
    w = torch.randn((B, N + 1), generator=g, dtype=torch.float64)

    def oracle(r_):
        e_ = port.echo_closed_form(r_)
        return (e_ * w.to(e_.dtype)).sum(), e_
    (g64,), noise, e64 = oracle_grads(oracle, r64)
    r = r64.detach().float().to(dev()).requires_grad_(True)
    e, _ = compute_echo_traces(r)
    assert_frame_close(e.detach().cpu().numpy(), e64.detach().numpy(), f"echo {B}x{N}")
    (e * w.float().to(dev())).sum().backward()
    assert_grad_close(r.grad.cpu().numpy(), g64.numpy(), f"d echo/d r {B}x{N}", noise=noise[0])


def _oracle_frames(vol, sources, dirs, S, alpha, start, sampler):
    from oracle import port
    out = []
    for p in range(sources.shape[0]):
        d = dirs[p] if dirs.dim() == 3 else dirs
        out.append(port.plot_beam_frame(vol, sources[p], d, S, alpha, start=start, sampler=sampler)[3])
    return torch.stack(out)


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("S,start", [(64, 0), (600, 0), (1100, 37), (130, 129 - 1)])
def test_batched_poses_vs_oracle(sampler, S, start):
    """Leading pose dimension, multi-segment rays, start crop; fwd + all gradients vs the fp64 oracle."""
    from diffus_b200 import render_frames
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n = 40
    vol = layered_phantom(n, seed=3)
    sources, dirs = pose_sweep(3, n_rays=6, n=n, seed=S)
    alpha = 2e-3
    g = torch.Generator().manual_seed(1)
    w = torch.randn((3, 6, S - start), generator=g, dtype=torch.float64)

    def oracle(v_, s_, d_):
        f_ = _oracle_frames(v_, s_, d_, S, alpha, start, sampler)
        return (f_ * w.to(f_.dtype)).sum(), f_
    want, noise, f64 = oracle_grads(oracle, vol, sources, dirs)
    v = vol.to(dev()).requires_grad_(True)
    s = sources.to(dev()).requires_grad_(True)
    d = dirs.to(dev()).requires_grad_(True)
    f = render_frames(v, s, d, S, alpha, start, sampler=sampler)
    assert_frame_close(f.detach().cpu().numpy(), f64.detach().numpy(), f"{sampler} S={S} start={start}")
    (f * w.float().to(dev())).sum().backward()
    # (S, start) = (130, 128): every ray has left the volume, the only column with a gradient is the median-replaced one and
    # its two contributions +-w / (2 Z) land on the SAME clamped voxel: the reference gradient is exactly zero by cancellation,
    # so the check is against the size of one cancelling term instead of against max |reference| = 0
    term = float(w.abs().max() / (2.0 * vol.min())) if float(want[0].abs().max()) == 0.0 else 0.0
    assert_grad_close(v.grad.cpu().numpy(), want[0].numpy(), "d/dvolume", noise=max(noise[0], GRAD_RTOL * term / NOISE_FACTOR))
    if sampler == "trilinear":
        assert_grad_close(s.grad.cpu().numpy(), want[1].numpy(), "d/dsources", noise=noise[1])
        assert_grad_close(d.grad.cpu().numpy(), want[2].numpy(), "d/ddirections", noise=noise[2])
    else:
        assert s.grad is None and d.grad is None


@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
@pytest.mark.parametrize("S,start,prepared", [(96, 0, None), (700, 0, "quad"), (1300, 11, None), (513, 3, "brick"), (300, 0, "quad"),
                                              (512, 0, "texture"), (1100, 5, "texture")])
def test_fused_mse_step_matches_oracle_and_unfused(sampler, S, start, prepared):
    """render_mse_loss (one fused kernel) == mse_loss(render_frames) through autograd == fp64 oracle."""
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    n = 36
    vol = layered_phantom(n, seed=5)
    sources, dirs = pose_sweep(2, n_rays=5, n=n, seed=S + start)
    alpha = 1e-3
    with torch.no_grad():
        target = render_frames(vol.to(dev()), sources.to(dev()) + 0.7, dirs.to(dev()), S, alpha, start, sampler=sampler)
    tgt64 = target.cpu().double()

    def oracle(v_, s_, d_):
        f_ = _oracle_frames(v_, s_, d_, S, alpha, start, sampler)
        l_ = (f_ - tgt64.to(f_.dtype)).square().mean()
        return l_, l_
    want, noise, l64 = oracle_grads(oracle, vol, sources, dirs)
    noise = [3.0 * n for n in noise]

    def run(fused):
        v = vol.to(dev()).requires_grad_(True)
        s = sources.to(dev()).requires_grad_(True)
        d = dirs.to(dev()).requires_grad_(True)
        vv = PreparedVolume(v, prepared) if prepared else v
        if fused:
            loss, frame = render_mse_loss(vv, s, d, target, S, alpha, start, sampler=sampler, return_frame=True)
        else:
            frame = render_frames(vv, s, d, S, alpha, start, sampler=sampler)
            loss = torch.nn.functional.mse_loss(frame, target)
        (3.0 * loss).backward()
        return loss.detach(), frame.detach(), v.grad, s.grad, d.grad

    lf, ff, gvf, gsf, gdf = run(True)
    lu, fu, gvu, gsu, gdu = run(False)
    # same arithmetic, different scan tree (the backward walks 8-column chunks): agreement to rounding
    torch.testing.assert_close(ff, fu, rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(lf.item(), l64.item(), rtol=1e-4)
    np.testing.assert_allclose(lf.item(), lu.item(), rtol=1e-5)
    assert_grad_close(gvf.cpu().numpy(), 3.0 * want[0].numpy(), "fused d/dvolume", noise=noise[0])
    assert_grad_close(gvu.cpu().numpy(), 3.0 * want[0].numpy(), "unfused d/dvolume", noise=noise[0])
    if sampler == "trilinear":
        assert_grad_close(gsf.cpu().numpy(), 3.0 * want[1].numpy(), "fused d/dsources", noise=noise[1])
        assert_grad_close(gdf.cpu().numpy(), 3.0 * want[2].numpy(), "fused d/ddirections", noise=noise[2])
        assert_grad_close(gsu.cpu().numpy(), 3.0 * want[1].numpy(), "unfused d/dsources", noise=noise[1])
    else:
        assert gsf is None and gdf is None


@pytest.mark.parametrize("S,start,prepared,shared", [(2048, 0, None, False), (1537, 0, "texture", False), (1800, 37, "brick", True),
                                                     (2047, 0, "quad", False), (2053, 5, "texture", True), (1700, 0, None, False),
                                                     (513, 0, "texture", False), (1024, 0, None, True), (1100, 37, "brick", False),
                                                     (1536, 0, "quad", False), (1025, 1, "texture", False)])
def test_multi_pass_rays_one_cta_per_ray_vs_oracle(S, start, prepared, shared):
    """Rays of 513..2048 columns with pose gradients only (config 5's shape: 2048): one CTA walks the two to four 512-column
    passes of a ray together, one warp each (no forward pre-pass for the prefixes).  Fused MSE step and the autograd backward against the fp64 oracle
    (frame, loss, d/dsources, d/ddirections), and against the multi-pass kernel that the same call takes when the volume
    gradient is wanted too."""
    _pose_only_step_vs_oracle_and_volume_grad_kernel(S, start, prepared, shared, step=0.017)


@pytest.mark.parametrize("S,start,prepared,shared", [(512, 0, "texture", False), (512, 0, None, True), (129, 0, "brick", False),
                                                     (256, 0, "quad", False), (257, 1, "texture", False), (300, 37, None, False),
                                                     (385, 0, "texture", True), (540, 40, "brick", False), (128, 0, "texture", False)])
def test_one_pass_rays_pose_gradients_only_vs_oracle(S, start, prepared, shared):
    """Rays of at most 512 columns with pose gradients only (config 2 / 3's kernels: the one-pass forms, the single 512-column
    sweep above 256 columns), every layout, own and shared fans, start crops: the same checks as for the multi-pass rays."""
    _pose_only_step_vs_oracle_and_volume_grad_kernel(S, start, prepared, shared, step=0.07)


def _pose_only_step_vs_oracle_and_volume_grad_kernel(S, start, prepared, shared, step):
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom
    n, P, R = 36, 3, 5
    vol = layered_phantom(n, seed=7)
    g = torch.Generator().manual_seed(S + start)
    sources = torch.tensor([[3.0, 2.0, 4.0], [n * 0.5, n * 0.3, 1.5], [n - 3.5, n * 0.6, n - 4.0]])
    aim = torch.tensor([n * 0.5, n * 0.5, n * 0.5]) - sources
    d = aim[:, None, :] / aim.norm(dim=-1)[:, None, None] + 0.25 * torch.randn((P, R, 3), generator=g)
    dirs = d / d.norm(dim=-1, keepdim=True) * step            # sub-voxel steps: the samples cross the whole 36^3 volume
    if shared:
        dirs = dirs[0]
    alpha = 7e-4
    with torch.no_grad():
        target = render_frames(vol.to(dev()), sources.to(dev()) + 0.6, dirs.to(dev()), S, alpha, start, sampler="trilinear")
    tgt64 = target.cpu().double()

    def oracle(v_, s_, d_):
        f_ = _oracle_frames(v_, s_, d_, S, alpha, start, "trilinear")
        l_ = (f_ - tgt64.to(f_.dtype)).square().mean()
        return l_, (l_, f_)
    want, noise, (l64, f64) = oracle_grads(oracle, vol, sources, dirs)

    def run(fused, with_volume):
        v = vol.to(dev()).requires_grad_(with_volume)
        s = sources.to(dev()).requires_grad_(True)
        dd = dirs.to(dev()).requires_grad_(True)
        vv = PreparedVolume(v, prepared) if prepared else v
        if fused:
            loss, frame = render_mse_loss(vv, s, dd, target, S, alpha, start, sampler="trilinear", return_frame=True)
        else:
            frame = render_frames(vv, s, dd, S, alpha, start, sampler="trilinear")
            loss = torch.nn.functional.mse_loss(frame, target)
        loss.backward()
        return loss.detach(), frame.detach(), s.grad, dd.grad

    what = f"S={S} start={start} {prepared} shared={shared}"
    ref = run(True, True)                                   # pose + volume gradient: the multi-pass kernel
    for fused in (True, False):
        lf, ff, gs, gd = run(fused, False)                  # pose gradient only: one CTA per ray
        tag = f"{what} {'fused' if fused else 'autograd'}"
        assert_frame_close(ff.cpu().numpy(), f64.detach().numpy(), tag + " frame")
        np.testing.assert_allclose(lf.item(), l64.item(), rtol=1e-4)
        assert_grad_close(gs.cpu().numpy(), want[1].numpy(), tag + " d/dsources", noise=noise[1])
        assert_grad_close(gd.cpu().numpy(), want[2].numpy(), tag + " d/ddirections", noise=noise[2])
        # the two kernels differ only in the association order of the pass prefixes / adjoints
        torch.testing.assert_close(ff, ref[1], rtol=1e-5, atol=2e-6 * float(ff.abs().max()))
        np.testing.assert_allclose(lf.item(), ref[0].item(), rtol=1e-5)
        scale = float(ref[2].abs().max())
        torch.testing.assert_close(gs, ref[2], rtol=1e-3, atol=1e-4 * scale)
    # run to run identical (fixed-order sums across the four passes of a ray)
    a, b = run(True, False), run(True, False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("dims,R,S,start", [((1, 1, 1), 2, 2, 0), ((2, 3, 1), 3, 5, 3), ((5, 4, 7), 2, 33, 0),
                                             ((9, 9, 9), 37, 31, 29), ((6, 5, 4), 4, 513, 1), ((7, 3, 5), 3, 1025, 512)])
@pytest.mark.parametrize("sampler", ["nearest", "trilinear"])
def test_edge_shapes_vs_oracle(dims, R, S, start, sampler):
    """Degenerate volumes, two-sample rays, crops that leave two columns, rays that are one column over a pass boundary."""
    from diffus_b200 import render_frames, render_mse_loss
    g = torch.Generator().manual_seed(S + R)
    vol = 1.4e6 + 3e5 * torch.rand(dims, generator=g)
    src = torch.tensor([[0.3, 0.2, 0.1], [dims[0] * 0.5, dims[1] * 0.4, -1.5]])
    d = torch.randn((2, R, 3), generator=g)
    d = d / d.norm(dim=-1, keepdim=True) * 0.7                 # sub-voxel steps: long rays stay near the volume
    alpha = 1e-3
    def oracle(v_, s_, d_):
        f_ = _oracle_frames(v_, s_, d_, S, alpha, start, sampler)
        return f_.square().mean(), f_
    want, noise, f64 = oracle_grads(oracle, vol, src, d)
    tgt = torch.zeros_like(f64)
    v = vol.to(dev()).requires_grad_(True)
    s = src.to(dev()).requires_grad_(True)
    dd = d.to(dev()).requires_grad_(True)
    f = render_frames(v, s, dd, S, alpha, start, sampler=sampler)
    assert f.shape == (2, R, S - start)
    assert_frame_close(f.detach().cpu().numpy(), f64.detach().numpy(), f"{dims} R={R} S={S} start={start}")
    loss = render_mse_loss(v, s, dd, tgt.float().to(dev()), S, alpha, start, sampler=sampler)
    loss.backward()
    if want[0].abs().max() > 0:
        assert_grad_close(v.grad.cpu().numpy(), want[0].numpy(), "d/dvolume", noise=noise[0])
    if sampler == "trilinear" and want[1] is not None and want[1].abs().max() > 0:
        assert_grad_close(s.grad.cpu().numpy(), want[1].numpy(), "d/dsources", noise=noise[1])
        assert_grad_close(dd.grad.cpu().numpy(), want[2].numpy(), "d/ddirections", noise=noise[2])


@pytest.mark.parametrize("seed", range(24))
def test_randomised_configurations_vs_oracle(seed):
    """Seeded sweep over shapes, samplers, layouts, crops, pose dtypes and shared/own fans: frames, loss and every
    gradient against the fp64 oracle, through the fused and the unfused autograd paths."""
    import random
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    rnd = random.Random(seed)
    g = torch.Generator().manual_seed(1000 + seed)
    dims = (rnd.randint(3, 40), rnd.randint(3, 40), rnd.randint(3, 40))
    P, R = rnd.randint(1, 4), rnd.randint(2, 9)
    S = rnd.choice([2, 3, 17, 32, 33, 64, 100, 255, 256, 257, 511, 512, 513, 700, 1024, 1100])
    start = rnd.choice([0, 0, 0, 1, S // 3, max(S - 2, 0)]) if S > 3 else 0
    sampler = rnd.choice(["nearest", "trilinear"])
    u = rnd.random()
    prepared = None if u >= 0.5 else ("brick" if u < 0.15 else ("texture" if u < 0.33 else "quad"))
    shared = rnd.random() < 0.3
    pose64 = rnd.random() < 0.25
    alpha = rnd.choice([0.0, 1e-4, 1e-2, 0.5])
    base = 1.4e6 + 2e5 * torch.rand((max(dims[0] // 5, 1), max(dims[1] // 5, 1), max(dims[2] // 5, 1)), generator=g)
    vol = torch.nn.functional.interpolate(base[None, None], size=dims, mode="nearest")[0, 0].contiguous()
    vol = vol * (1 + 0.003 * torch.randn(dims, generator=g))
    centre = torch.tensor([d / 2.0 for d in dims])
    src = centre + (torch.rand((P, 3), generator=g) - 0.5) * torch.tensor(dims, dtype=torch.float32) * 1.2
    d = torch.randn((R, 3) if shared else (P, R, 3), generator=g)
    d = d / d.norm(dim=-1, keepdim=True) * min(1.0, 1.5 * max(dims) / S)        # keep long rays near the volume
    pdt = torch.float64 if pose64 else torch.float32
    with torch.no_grad():
        tgt = (_oracle_frames(vol.double(), src.to(pdt).double(), d.to(pdt).double(), S, alpha, start, sampler) * 0.5).float()

    def oracle(v_, s_, d_):
        # float64 poses are part of the case: only the volume (and a float32 pose) drops to float32 in the noise run
        if pose64:
            s_, d_ = s_.double(), d_.double()
        f_ = _oracle_frames(v_, s_, d_, S, alpha, start, sampler)
        l_ = (f_ - tgt.to(f_.dtype)).square().mean()
        return l_, (f_, l_)
    want, noise, (f64, l64) = oracle_grads(oracle, vol, src.to(pdt), d.to(pdt))
    what = f"seed {seed}: dims={dims} P={P} R={R} S={S} start={start} {sampler} prepared={prepared} shared={shared} pose64={pose64}"
    for fused in (True, False):
        v = vol.to(dev()).requires_grad_(True)
        s = src.to(pdt).to(dev()).requires_grad_(True)
        dd = d.to(pdt).to(dev()).requires_grad_(True)
        vv = PreparedVolume(v, prepared) if prepared else v
        if fused:
            loss, f = render_mse_loss(vv, s, dd, tgt.to(dev()), S, alpha, start, sampler=sampler, return_frame=True)
        else:
            f = render_frames(vv, s, dd, S, alpha, start, sampler=sampler)
            loss = torch.nn.functional.mse_loss(f, tgt.to(dev()))
        loss.backward()
        assert_frame_close(f.detach().cpu().numpy(), f64.detach().numpy(), what)
        np.testing.assert_allclose(loss.item(), l64.item(), rtol=1e-4, atol=1e-12, err_msg=what)
        if want[0].abs().max() > 0:
            assert_grad_close(v.grad.cpu().numpy(), want[0].numpy(), what + " d/dvolume", noise=noise[0])
        if sampler == "trilinear":
            if want[1].abs().max() > 0:
                assert_grad_close(s.grad.cpu().numpy(), want[1].numpy(), what + " d/dsources", noise=noise[1])
                assert_grad_close(dd.grad.cpu().numpy(), want[2].numpy(), what + " d/ddirections", noise=noise[2])
        else:
            assert s.grad is None and dd.grad is None


def test_shared_directions_and_float64_pose():
    from diffus_b200 import render_frames
    from diffus_b200.phantoms import layered_phantom
    from diffus_b200.cone import generate_cone_directions
    vol = layered_phantom(32, seed=1)
    dirs = generate_cone_directions([0.2, 1.0], 0.7, 5)
    sources = torch.tensor([[16.0, 0.5, 15.5], [10.25, 2.0, 20.0]])
    for sdt, ddt in ((torch.float64, torch.float32), (torch.float32, torch.float64), (torch.float64, torch.float64)):
        s64, d64 = sources.to(sdt), dirs.to(ddt)
        want = _oracle_frames(vol.double(), s64, d64, 48, 1e-3, 0, "nearest")
        got = render_frames(vol.to(dev()), s64.to(dev()), d64.to(dev()), 48, 1e-3, 0)
        assert_frame_close(got.cpu().numpy(), want.numpy(), f"pose dtypes {sdt},{ddt}")
    # shared fan, gradient summed over poses
    s = sources.to(dev()).requires_grad_(True)
    d = dirs.to(dev()).requires_grad_(True)
    f = render_frames(vol.to(dev()), s, d, 48, 1e-3, 0, sampler="trilinear")
    w = torch.randn(tuple(f.shape), generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    (gs, gd), noise, _ = oracle_grads(lambda s_, d_: (_oracle_frames(vol.to(s_.dtype), s_, d_, 48, 1e-3, 0, "trilinear") * w.to(s_.dtype)).sum(),
                                      sources, dirs)
    (f * w.float().to(dev())).sum().backward()
    assert_grad_close(s.grad.cpu().numpy(), gs.numpy(), "shared fan d/dsources", noise=noise[0])
    assert_grad_close(d.grad.cpu().numpy(), gd.numpy(), "shared fan d/ddirections", noise=noise[1])


def test_cone_directions_device_matches_host(golden_cone):
    from diffus_b200 import ops
    g = golden_cone
    for i in range(5):
        d = torch.tensor(g[f"cone{i}_d"][:2], device=dev()).reshape(1, 2)
        out = ops.cone_directions(d, float(g[f"cone{i}_angle"]), int(g[f"cone{i}_n"]))
        np.testing.assert_allclose(out[0].cpu().numpy(), g[f"cone{i}_dirs"], rtol=0, atol=1.2e-7)


def test_mlp_forward_backward_golden(golden_mlp):
    from diffus_b200 import ImpedanceEstimator
    g = golden_mlp
    model = ImpedanceEstimator(1)
    sd = {k[len("param_"):].replace("model_", "model.").replace("_weight", ".weight").replace("_bias", ".bias"): torch.tensor(v)
          for k, v in g.items() if k.startswith("param_")}
    model.load_state_dict(sd)
    model = model.to(dev())
    x = torch.tensor(g["x"], device=dev())
    y = model(x)
    np.testing.assert_allclose(y.detach().cpu().numpy(), g["y64"], rtol=1e-5, atol=1e-6)
    w = torch.tensor(g["w"], device=dev())
    (y * w).sum().backward()
    for name, p in model.named_parameters():
        want = g["grad_" + name.replace(".", "_")]
        assert_grad_close(p.grad.cpu().numpy(), want, name)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 257, 5000, 70001])
def test_mlp_forward_cuda_cores_and_piecewise_match_oracle(n):
    """The fp32 CUDA-core kernel and the piecewise-linear table vs the fp64 oracle."""
    from diffus_b200 import ImpedanceEstimator, ops
    from diffus_b200.impedance import pack_params
    from oracle import port
    torch.manual_seed(n)
    model = ImpedanceEstimator(1)
    x = torch.randn(n) * 2.0
    mask = torch.rand(n) > 0.2
    want = port.mlp_forward(x.double().reshape(-1, 1), *[p.detach().double() for p in model.parameters()]).reshape(-1) * 1e6
    want = torch.where(mask, want, torch.tensor(400.0, dtype=torch.float64))
    params = pack_params(model).detach().to(dev())
    with ops.mlp_path(ops.MLP_PATH_CUDA_CORES):
        cc = ops.mlp_fwd_impl(params, x.to(dev()), mask.to(dev()), 1e6, 400.0)
    with ops.mlp_path(ops.MLP_PATH_PIECEWISE):
        pw = ops.mlp_fwd_impl(params, x.to(dev()), mask.to(dev()), 1e6, 400.0)
        pw2 = ops.mlp_fwd_impl(params, x.to(dev()), None, 1.0, 0.0)
    np.testing.assert_allclose(cc.cpu().numpy(), want.numpy(), rtol=2e-5, atol=2.0)
    # the piecewise-linear table is built in float64: one float32 rounding of the exact value (+ one for the scale)
    np.testing.assert_allclose(pw.cpu().numpy(), want.numpy(), rtol=3e-7, atol=0.3)
    want2 = port.mlp_forward(x.double().reshape(-1, 1), *[p.detach().double() for p in model.parameters()]).reshape(-1)
    np.testing.assert_allclose(pw2.cpu().numpy(), want2.numpy(), rtol=2e-7, atol=2e-7)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 300, 5000, 70001])
def test_mlp_backward_cuda_cores_and_piecewise_match_oracle(n):
    """Weight gradient of the fp32 CUDA-core kernels and of the piecewise-linear table vs fp64 autograd of the oracle."""
    from diffus_b200 import ImpedanceEstimator, ops
    from diffus_b200.impedance import pack_params
    from oracle import port
    torch.manual_seed(100 + n)
    model = ImpedanceEstimator(1)
    x = torch.randn(n) * 2.0
    mask = torch.rand(n) > 0.2
    gup = torch.randn(n)
    if n > 1000:
        gup[200:700] = 0.0                                  # whole tiles without an upstream gradient are skipped

    def oracle(*prm):
        out = port.mlp_forward(x.to(prm[0].dtype).reshape(-1, 1), *prm).reshape(-1) * 3.0
        return (torch.where(mask, out, torch.zeros_like(out)) * gup.to(out.dtype)).sum()
    g64, noise, _ = oracle_grads(oracle, *[p.detach() for p in model.parameters()])
    want = torch.cat([g.reshape(-1) for g in g64]).numpy()
    params = pack_params(model).detach().to(dev())
    got = {}
    for name, path in (("cc", ops.MLP_PATH_CUDA_CORES), ("pwl", ops.MLP_PATH_PIECEWISE)):
        with ops.mlp_path(path):
            got[name] = ops.mlp_bwd_impl(params, x.to(dev()), mask.to(dev()), gup.to(dev()), 3.0).cpu().numpy()
            again = ops.mlp_bwd_impl(params, x.to(dev()), mask.to(dev()), gup.to(dev()), 3.0).cpu().numpy()
        np.testing.assert_array_equal(got[name], again)       # fixed-order reductions: run-to-run identical
        assert_grad_close(got[name], want, f"mlp weight gradient ({name})", noise=max(noise))


@pytest.mark.parametrize("n", [3, 4096 + 3, 50001])
def test_mlp_piecewise_path_falls_back_above_256_regions(n):
    """Weights with > 1000 linear pieces: the piecewise path must notice and evaluate the layers instead (forward inline,
    backward through the gated CUDA-core kernels); an unaligned view exercises the scalar loads."""
    from diffus_b200 import ops
    from oracle import port
    from test_oracle_golden import _zigzag_mlp
    prm = _zigzag_mlp()
    params = torch.cat([p.reshape(-1) for p in prm]).to(dev())
    gen = torch.Generator().manual_seed(n)
    x = torch.rand(n + 1, generator=gen) * 40.0 - 4.0
    gup = torch.randn(n + 1, generator=gen)
    xd, gd = x.to(dev())[1:], gup.to(dev())[1:]                  # 4-byte aligned only
    want = port.mlp_forward(x[1:].double().reshape(-1, 1), *[p.double() for p in prm]).reshape(-1)
    with ops.mlp_path(ops.MLP_PATH_PIECEWISE):
        got = ops.mlp_fwd_impl(params, xd, None, 1.0, 0.0)
        g1 = ops.mlp_bwd_impl(params, xd, None, gd, 1.0)
    with ops.mlp_path(ops.MLP_PATH_CUDA_CORES):
        g2 = ops.mlp_bwd_impl(params, xd, None, gd, 1.0)
    np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=2e-5, atol=2e-5 * float(want.abs().max()))
    np.testing.assert_array_equal(g1.cpu().numpy(), g2.cpu().numpy())     # the very same kernels ran


def test_mlp_piecewise_path_unaligned_and_tail():
    """Scalar-load path of the piecewise kernels (views that are not 16-byte aligned, n not a multiple of 4)."""
    from diffus_b200 import ImpedanceEstimator, ops
    from diffus_b200.impedance import pack_params
    from oracle import port
    torch.manual_seed(11)
    model = ImpedanceEstimator(1)
    n = 10007
    x, gup, mask = torch.randn(n + 1) * 2.0, torch.randn(n + 1), torch.rand(n + 1) > 0.3
    params = pack_params(model).detach().to(dev())
    prm = [p.detach().double() for p in model.parameters()]
    want = torch.where(mask[1:], port.mlp_forward(x[1:].double().reshape(-1, 1), *prm).reshape(-1) * 2.0, torch.tensor(-1.0, dtype=torch.float64))
    with ops.mlp_path(ops.MLP_PATH_PIECEWISE):
        got = ops.mlp_fwd_impl(params, x.to(dev())[1:], mask.to(dev())[1:], 2.0, -1.0)
        ga = ops.mlp_bwd_impl(params, x.to(dev())[1:], mask.to(dev())[1:], gup.to(dev())[1:], 2.0)
        gb = ops.mlp_bwd_impl(params, x[1:].clone().to(dev()), mask[1:].clone().to(dev()), gup[1:].clone().to(dev()), 2.0)
    np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=3e-7, atol=3e-7)
    assert_grad_close(ga.cpu().numpy(), gb.cpu().numpy(), "aligned vs unaligned piecewise backward")


@pytest.mark.parametrize("weights", ["default", "zigzag"])
def test_mlp_input_gradient_matches_autograd(weights):
    """d / d x through ImpedanceEstimator (the slope of the linear piece) vs float64 autograd of the layered oracle."""
    from diffus_b200 import ImpedanceEstimator, ops
    from diffus_b200.impedance import pack_params
    from oracle import port
    from test_oracle_golden import _zigzag_mlp
    torch.manual_seed(21)
    model = ImpedanceEstimator(1)
    prm = _zigzag_mlp() if weights == "zigzag" else [p.detach() for p in model.parameters()]
    n = 4099
    gen = torch.Generator().manual_seed(4)
    x = (torch.rand(n, generator=gen) * 40.0 - 4.0) if weights == "zigzag" else torch.randn(n, generator=gen) * 2.0
    gup, mask = torch.randn(n, generator=gen), torch.rand(n, generator=gen) > 0.25
    x64 = x.double().requires_grad_(True)
    out = port.mlp_forward(x64.reshape(-1, 1), *[p.double() for p in prm]).reshape(-1) * 3.0
    (torch.where(mask, out, torch.zeros_like(out)) * gup.double()).sum().backward()
    params = torch.cat([p.reshape(-1) for p in prm]).to(dev())
    got = ops.mlp_input_grad_impl(params, x.to(dev()), mask.to(dev()), gup.to(dev()), 3.0)
    # a sample within float32 rounding of a breakpoint may sit on the other piece: compare away from the kinks
    want = x64.grad.numpy()
    err = np.abs(got.cpu().numpy() - want)
    tol = 1e-5 * np.abs(want).max() + 1e-5 * np.abs(want)
    assert (err > tol).mean() < 2e-3, f"{(err > tol).sum()} of {n} input gradients off"
    if weights == "default":                       # and through autograd: the module's forward hands d/dx back
        m = model.to(dev())
        xd = x.to(dev()).reshape(-1, 1).requires_grad_(True)
        (m(xd).reshape(-1) * gup.to(dev())).sum().backward()
        x2 = x.double().requires_grad_(True)
        (port.mlp_forward(x2.reshape(-1, 1), *[p.double() for p in prm]).reshape(-1) * gup.double()).sum().backward()
        e2 = np.abs(xd.grad.reshape(-1).cpu().numpy() - x2.grad.numpy())
        assert (e2 > 1e-5 * np.abs(x2.grad.numpy()).max() + 1e-5 * np.abs(x2.grad.numpy())).mean() < 2e-3


def test_mlp_volume_masked_and_large():
    from diffus_b200 import ImpedanceEstimator
    from oracle import port
    torch.manual_seed(3)
    model = ImpedanceEstimator(1)
    vol = torch.randn(37, 29, 41)
    mask = torch.rand(37, 29, 41) > 0.3
    params = [p.detach().double() for p in model.parameters()]
    want = port.mlp_forward(vol.double().reshape(-1, 1), *params).reshape(vol.shape) * 1e6
    want = torch.where(mask, want, torch.tensor(400.0, dtype=torch.float64))
    m = model.to(dev())
    got = m.impedance_volume(vol.to(dev()), mask.to(dev()), out_scale=1e6, fill=400.0)
    np.testing.assert_allclose(got.detach().cpu().numpy(), want.numpy(), rtol=2e-5, atol=2.0)   # 2e-6 of the 1e6 scale
    # weight gradient through a sparse upstream gradient (most tiles skipped)
    gup = torch.zeros_like(vol)
    gup[5:9, 3:20, 7:30] = torch.randn(4, 17, 23)
    m.zero_grad()
    (m.impedance_volume(vol.to(dev()), mask.to(dev()), out_scale=2.0, fill=0.0) * gup.to(dev())).sum().backward()
    ref = ImpedanceEstimator(1).double()
    ref.load_state_dict({k: v.double().cpu() for k, v in model.state_dict().items()})
    out = ref.model(vol.double().reshape(-1, 1)).reshape(vol.shape) * 2.0
    (torch.where(mask, out, torch.zeros_like(out)) * gup.double()).sum().backward()
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert_grad_close(p.grad.cpu().numpy(), q.grad.numpy(), name)


def test_mlp_render_training_step_vs_oracle():
    """Config 4 in miniature: MLP -> volume -> frames -> MSE; weight and pose gradients vs fp64 autograd of the oracle."""
    from diffus_b200 import ImpedanceEstimator
    from diffus_b200.phantoms import mri_phantom, pose_sweep
    from diffus_b200.training import mlp_render_mse_loss, train_step
    from oracle import port
    n, S, alpha = 24, 40, 1e-3
    torch.manual_seed(5)
    model = ImpedanceEstimator(1)
    with torch.no_grad():                                  # keep the impedances positive and tissue-like
        model.model[4].bias.fill_(1.5)
        model.model[4].weight.mul_(0.3)
    mri = mri_phantom(n, "t2", seed=2) / 1000.0
    sources, dirs = pose_sweep(3, n_rays=5, n=n, seed=9)
    g = torch.Generator().manual_seed(3)
    targets = 0.01 * torch.randn((3, 5, S), generator=g)
    from oracle import port as _port

    def oracle(s_, *prm):
        Z_ = _port.mlp_forward(mri.to(s_.dtype).reshape(-1, 1), *prm).reshape(mri.shape) * 1e6
        f_ = _oracle_frames(Z_, s_, dirs.to(s_.dtype), S, alpha, 0, "trilinear")
        l_ = (f_ - targets.to(s_.dtype)).square().mean()
        return l_, l_
    g64, noise, l64 = oracle_grads(oracle, sources, *[p.detach() for p in model.parameters()])
    m = model.to(dev())
    s = sources.to(dev()).requires_grad_(True)
    from diffus_b200 import render_mse_loss
    from diffus_b200.training import TrainingVolume
    for mode in ("fused", "prepared", "unfused"):
        m.zero_grad()
        s.grad = None
        if mode == "unfused":         # plain composition: MLP op -> linear volume -> render op, through autograd
            Z = m.impedance_volume(mri.to(dev()), None, out_scale=1e6, fill=400.0)
            loss = render_mse_loss(Z, s, dirs.to(dev()), targets.to(dev()), S, alpha)
        else:
            vol_in = TrainingVolume(mri.to(dev())) if mode == "prepared" else mri.to(dev())
            loss = mlp_render_mse_loss(m, vol_in, s, dirs.to(dev()), targets.to(dev()), S, alpha, out_scale=1e6)
        loss.backward()
        np.testing.assert_allclose(loss.item(), l64.item(), rtol=1e-5)      # the frames' own relative tolerance
        for i, (name, p) in enumerate(m.named_parameters()):
            assert_grad_close(p.grad.cpu().numpy(), g64[1 + i].numpy(), f"d/d{name} ({mode})", noise=noise[1 + i])
        assert_grad_close(s.grad.cpu().numpy(), g64[0].numpy(), "d/dsources", noise=noise[0])
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    l0 = train_step(m, opt, mri.to(dev()), sources.to(dev()), dirs.to(dev()), targets.to(dev()), S, alpha, out_scale=1e6)
    for _ in range(10):
        l1 = train_step(m, opt, mri.to(dev()), sources.to(dev()), dirs.to(dev()), targets.to(dev()), S, alpha, out_scale=1e6)
    assert l1 < l0


def test_splat_golden_and_gradient(golden_splat):
    """differentiable_splat (row f1): golden images from the reference; duplicates: last sample wins; gradient vs oracle."""
    from diffus_b200 import differentiable_splat
    from oracle import port
    g = golden_splat
    x, y, z = (torch.tensor(g[k], device=dev()) for k in ("x", "y", "z"))
    val = torch.tensor(g["val"], device=dev())
    for sigma in (0.5, 1.0):
        img = differentiable_splat(x, y, z, val, H=64, W=64, sigma=sigma)
        assert img.shape == (64, 64)
        np.testing.assert_allclose(img.cpu().numpy(), g[f"img_sigma{sigma}"], rtol=1e-5, atol=1e-6)
    # float coordinates (after rotate_around_apex), many duplicate pixels, axis choice y-z, non-square image
    gen = torch.Generator().manual_seed(4)
    n = 5000
    cx = torch.full((n,), 7.25)
    cy = torch.rand(n, generator=gen) * 70 - 3
    cz = torch.rand(n, generator=gen) * 40 - 2
    v = torch.randn(n, generator=gen)
    v64 = v.clone().requires_grad_(True)
    want = port.splat(cx, cy, cz, v64, H=40, W=72, sigma=2.0)
    w = torch.randn(want.shape, generator=gen)
    (gw,) = torch.autograd.grad((want * w).sum(), v64)
    vd = v.to(dev()).requires_grad_(True)
    got = differentiable_splat(cx.to(dev()), cy.to(dev()), cz.to(dev()), vd, H=40, W=72, sigma=2.0)
    np.testing.assert_allclose(got.detach().cpu().numpy(), want.detach().numpy(), rtol=2e-5, atol=2e-6)
    (got * w.to(dev())).sum().backward()
    assert_grad_close(vd.grad.cpu().numpy(), gw.numpy(), "d splat / d intensities")
    # end to end with the renderer's own outputs, as every HEAD-era notebook does
    from diffus_b200 import UltrasoundRenderer
    from diffus_b200.phantoms import layered_phantom, config1_pose
    vol = layered_phantom(64, seed=1)
    src, dirs = config1_pose(64, 24)
    xi, yi, zi, frame = UltrasoundRenderer(80, 1e-3).plot_beam_frame(vol.to(dev()), src.to(dev()), dirs.to(dev()), plot=False)
    img = differentiable_splat(xi, yi, zi, frame, H=64, W=64, sigma=0.5)
    ref_img = port.splat(xi.cpu(), yi.cpu(), zi.cpu(), frame.cpu(), H=64, W=64, sigma=0.5)
    np.testing.assert_allclose(img.cpu().numpy(), ref_img.numpy(), rtol=2e-5, atol=2e-6)


def test_compute_impedance_volume_golden(golden_impvol):
    """Row f4: create_brain_mask + zscore_normalize + MLP x 1e6, against the reference's scipy/torch CPU pipeline."""
    from diffus_b200 import ImpedanceEstimator
    from diffus_b200.utils import create_brain_mask, zscore_normalize
    g = golden_impvol
    vol = torch.tensor(g["volume"], device=dev())
    mask = create_brain_mask(vol, 50)
    assert mask.dtype == torch.bool
    np.testing.assert_array_equal(mask.cpu().numpy(), g["mask"])
    vn = zscore_normalize(vol, mask)
    np.testing.assert_allclose(vn.cpu().numpy(), g["vol_norm"], rtol=2e-5, atol=2e-6)
    model = ImpedanceEstimator(1)
    model.load_state_dict({k[len("param_"):].replace("model_", "model.").replace("_weight", ".weight").replace("_bias", ".bias"):
                           torch.tensor(v) for k, v in g.items() if k.startswith("param_")})
    Z = ImpedanceEstimator.compute_impedance_volume(vol, model.to(dev()), threshold=50)
    np.testing.assert_allclose(Z.cpu().numpy(), g["Z"], rtol=5e-5, atol=5.0)
    assert (Z[~mask] == 400.0).all()


def test_compute_gaussian_pulse_vs_oracle():
    from diffus_b200 import compute_gaussian_pulse, gaussian_pulse
    from oracle import port
    g = torch.Generator().manual_seed(3)
    r = 0.01 * torch.randn((4, 60), generator=g)
    got = compute_gaussian_pulse(r.to(dev()), length=20, sigma=4)
    echo = port.echo_closed_form(r.double())
    pulse = torch.tensor(gaussian_pulse(20, 4), dtype=torch.float64)[None, None]
    want = torch.nn.functional.conv1d(echo.unsqueeze(1), pulse, padding=10).squeeze(1)
    assert got.shape == want.shape
    np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-4, atol=1e-6)
    # gradient through the convolution kernel and the echo scan, odd and even pulse lengths (even: the output is one longer)
    for length, sigma in ((20, 4), (9, 2), (1, 1)):
        w = torch.randn((4, 60 + 1 + 2 * (length // 2) - length + 1), generator=g, dtype=torch.float64)
        r64 = r.double().requires_grad_(True)
        pulse = torch.tensor(gaussian_pulse(length, sigma), dtype=torch.float64)[None, None]
        (torch.nn.functional.conv1d(port.echo_closed_form(r64).unsqueeze(1), pulse, padding=length // 2).squeeze(1) * w).sum().backward()
        rd = r.to(dev()).requires_grad_(True)
        out = compute_gaussian_pulse(rd, length=length, sigma=sigma)
        assert tuple(out.shape) == tuple(w.shape)
        (out * w.float().to(dev())).sum().backward()
        assert_grad_close(rd.grad.cpu().numpy(), r64.grad.numpy(), f"compute_gaussian_pulse d/drefLR (length {length})")


def test_custom_nearest_sampler_explicit_points():
    from diffus_b200 import custom_nearest_sampler
    from oracle import port
    g = torch.Generator().manual_seed(8)
    vol = torch.rand((9, 7, 11), generator=g)
    pts = torch.rand((4, 13, 3), generator=g) * torch.tensor([12.0, 10.0, 14.0]) - 2.0
    pts[0, 0] = torch.tensor([2.5, 3.5, 4.5])                     # round-half-even ties
    x, y, z, v = custom_nearest_sampler(vol.to(dev()), pts.to(dev()))
    xo, yo, zo, vo = port.sample_nearest(vol, pts)
    assert torch.equal(x.cpu(), xo) and torch.equal(y.cpu(), yo) and torch.equal(z.cpu(), zo)
    assert torch.equal(v.cpu(), vo)
    _, _, _, vt = custom_nearest_sampler(vol.to(dev()), pts.to(dev()), sampler="trilinear")
    np.testing.assert_allclose(vt.cpu().numpy(), port.sample_trilinear(vol.double(), pts.double())[3].numpy(), rtol=1e-5, atol=1e-6)


def test_train_model_runs_on_the_gpu():
    """ImpedanceEstimator.train_model (reference src/impedance.py:19-37) on a tissue table, through the MLP kernels."""
    from diffus_b200 import ImpedanceEstimator
    X = torch.tensor([[-1.2], [-0.3], [0.4], [1.5]], device=dev())
    y = torch.tensor([[1.38], [1.52], [1.60], [1.68]], device=dev())
    torch.manual_seed(0)
    model = ImpedanceEstimator.train_model(X, y, epochs=300, lr=1e-2)
    assert torch.nn.functional.mse_loss(model(X), y).item() < 1e-3


def test_full_size_properties_config1():
    """BASELINE config 1 at full size (256^3, 128 x 512): properties that need no oracle run."""
    from diffus_b200 import UltrasoundRenderer, PreparedVolume, render_frames
    from diffus_b200.phantoms import layered_phantom, config1_pose
    vol = layered_phantom(256, seed=0).to(dev())
    src, dirs = config1_pose(256, 128)
    src, dirs = src.to(dev()), dirs.to(dev())
    ren = UltrasoundRenderer(512, 1e-4)
    x, y, z, f = ren.plot_beam_frame(vol, src, dirs, plot=False)
    assert f.shape == (128, 512) and torch.isfinite(f).all()
    assert (f[:, 0] == 0).all()
    # rays are independent: rendering a subset of rays gives the same rows
    _, _, _, f2 = ren.plot_beam_frame(vol, src, dirs[40:50], plot=False)
    assert torch.equal(f2, f[40:50])
    # determinism and layout independence
    assert torch.equal(render_frames(PreparedVolume(vol), src, dirs, 512, 1e-4)[0], f)
    # the echo only depends on impedance ratios: scaling the volume leaves the frame unchanged (power of two: exact)
    _, _, _, f3 = ren.plot_beam_frame(vol * 4.0, src, dirs, plot=False)
    assert torch.equal(f3, f)
    # truncation: the first 200 columns do not depend on the samples behind them
    _, _, _, f4 = UltrasoundRenderer(200, 1e-4).plot_beam_frame(vol, src, dirs, plot=False)
    assert torch.equal(f4, f[:, :200])
    # homogeneous medium: no interface, no echo
    _, _, _, f5 = ren.plot_beam_frame(torch.full_like(vol, 1.5e6), src, dirs, plot=False)
    assert (f5 == 0).all()
    # attenuation factorises: frame(alpha) = frame(0) * exp(-alpha k)
    _, _, _, f0 = UltrasoundRenderer(512, 0.0).plot_beam_frame(vol, src, dirs, plot=False)
    k = torch.arange(512, device=dev(), dtype=torch.float32)
    torch.testing.assert_close(f, f0 * torch.exp(-1e-4 * k), rtol=2e-6, atol=1e-9)
    # value range measured on the reference for this configuration (SURVEY 8d): [-0.081, 0.067]
    assert -0.09 < f.min().item() < -0.07 and 0.06 < f.max().item() < 0.075


def test_full_size_pose_sweep_properties_config3():
    """BASELINE config 3 at full size (1024 poses x 128 x 512 on 256^3): oracle-free checks of the batched fused path."""
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    from diffus_b200.phantoms import intensity_to_impedance, mri_phantom, pose_sweep
    vol = intensity_to_impedance(mri_phantom(256, "t1", seed=0)).to(dev())
    src, dirs = pose_sweep(1024, 128, 256, seed=5)
    src, dirs = src.to(dev()), dirs.to(dev())
    pv = PreparedVolume(vol)
    frames = render_frames(pv, src, dirs, 512, 1e-4, sampler="trilinear")
    assert frames.shape == (1024, 128, 512) and torch.isfinite(frames).all()
    # poses are independent: any pose rendered alone gives the same frame, in either layout
    for p in (0, 17, 900, 1023):
        assert torch.equal(render_frames(pv, src[p:p + 1], dirs[p:p + 1], 512, 1e-4, sampler="trilinear")[0], frames[p])
        assert torch.equal(render_frames(vol, src[p:p + 1], dirs[p:p + 1], 512, 1e-4, sampler="trilinear")[0], frames[p])
    # fused step: loss equals the unfused loss; zero loss and zero gradients at the target
    with torch.no_grad():
        target = render_frames(pv, src + torch.tensor([1.5, 0.0, -1.0], device=dev()), dirs, 512, 1e-4, sampler="trilinear")
    s = src.clone().requires_grad_(True)
    d = dirs.clone().requires_grad_(True)
    loss = render_mse_loss(pv, s, d, target, 512, 1e-4)
    loss.backward()
    ref_loss = torch.nn.functional.mse_loss(frames, target)
    np.testing.assert_allclose(loss.item(), ref_loss.item(), rtol=1e-4)
    assert torch.isfinite(s.grad).all() and torch.isfinite(d.grad).all()
    l0 = render_mse_loss(pv, src, dirs, frames, 512, 1e-4)
    assert l0.item() < 1e-12
    # directional derivative along the gradient (sum over poses) vs a central finite difference of the loss
    gs = s.grad / s.grad.norm()
    eps = 2e-2
    lp = render_mse_loss(pv, src + eps * gs, dirs, target, 512, 1e-4).item()
    lm = render_mse_loss(pv, src - eps * gs, dirs, target, 512, 1e-4).item()
    fd, an = (lp - lm) / (2 * eps), (s.grad * gs).sum().item()
    assert abs(fd - an) <= 0.1 * abs(an) + 1e-12, (fd, an)


def test_full_size_stress_geometry_config5():
    """BASELINE config 5 geometry (512^3 volume, 512 rays x 2048 samples: four 512-column passes), a few poses."""
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    vol = layered_phantom(512, seed=0).to(dev())
    src, dirs = pose_sweep(6, 512, 512, seed=2)
    src, dirs = src.to(dev()), dirs.to(dev())
    pv = PreparedVolume(vol)
    f = render_frames(pv, src, dirs, 2048, 1e-4, sampler="trilinear")
    assert f.shape == (6, 512, 2048) and torch.isfinite(f).all()
    assert torch.equal(render_frames(vol, src[2:3], dirs[2:3, 100:140], 2048, 1e-4, sampler="trilinear")[0], f[2, 100:140])
    # truncation invariance across pass boundaries: a 1300-sample render equals the first 1300 columns
    assert torch.equal(render_frames(pv, src, dirs, 1300, 1e-4, sampler="trilinear"), f[:, :, :1300])
    target = f * 0.9
    s = src.clone().requires_grad_(True)
    loss, fr = render_mse_loss(pv, s, dirs, target, 2048, 1e-4, return_frame=True)
    loss.backward()
    torch.testing.assert_close(fr, f, rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(loss.item(), torch.nn.functional.mse_loss(f, target).item(), rtol=1e-4)
    assert torch.isfinite(s.grad).all() and s.grad.abs().max() > 0


def test_graphed_pose_step_matches_eager():
    from diffus_b200 import PreparedVolume, render_frames, render_mse_loss
    from diffus_b200.graphs import GraphedPoseStep
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    vol = layered_phantom(48, seed=2).to(dev())
    src, dirs = pose_sweep(3, 16, 48, seed=1)
    src, dirs = src.to(dev()), dirs.to(dev())
    with torch.no_grad():
        target = render_frames(vol, src + 0.8, dirs, 96, 1e-3, sampler="trilinear")
    step = GraphedPoseStep(PreparedVolume(vol), target, 16, 96, 1e-3)
    for shift in (0.0, 0.3, -0.5):                       # replay with new poses
        s = (src + shift).clone().requires_grad_(True)
        d = dirs.clone().requires_grad_(True)
        loss = render_mse_loss(PreparedVolume(vol), s, d, target, 96, 1e-3)
        loss.backward()
        gl, gs, gd = step(src + shift, dirs)
        assert torch.equal(gl, loss.detach()) and torch.equal(gs, s.grad) and torch.equal(gd, d.grad)


def test_no_cpu_fallback():
    from diffus_b200 import render_frames
    from diffus_b200._lib import DiffusError
    with pytest.raises(DiffusError):
        render_frames(torch.zeros(4, 4, 4), torch.zeros(1, 3), torch.zeros(2, 3), 8)


def test_prepared_volume_layouts_and_auto_choice():
    """'auto' takes the float4 QUAD copy only while it stays small against L2; every layout renders the same frame and
    the gradient w.r.t. a QUAD volume (scattered into a BRICK buffer) equals the LINEAR one."""
    from diffus_b200 import PreparedVolume, render_frames
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    vol = layered_phantom(40, seed=3).to(dev())
    assert PreparedVolume(vol).layout == "quad" and PreparedVolume(vol, "brick").layout == "brick"
    big = torch.zeros((160, 160, 160), device=dev())
    assert PreparedVolume(big).layout == "brick"                        # 62.5 MiB of float4 would not stay in L2
    with pytest.raises(ValueError):
        PreparedVolume(vol, "tiles")
    src, dirs = pose_sweep(3, n_rays=6, n=40, seed=4)
    src, dirs = src.to(dev()), dirs.to(dev())
    grads = {}
    for layout in (None, "brick", "quad", "texture"):
        v = vol.clone().requires_grad_(True)
        f = render_frames(PreparedVolume(v, layout) if layout else v, src, dirs, 90, 1e-3, 5, sampler="trilinear")
        f.square().sum().backward()
        grads[layout] = (f.detach(), v.grad)
    for layout in ("brick", "quad", "texture"):
        assert torch.equal(grads[layout][0], grads[None][0])
        torch.testing.assert_close(grads[layout][1], grads[None][1], rtol=1e-5, atol=1e-12)     # atomics: order varies


def test_gather_probe_reports_a_plausible_roof():
    """The roofline probe of bench.py: random 32-byte sectors out of L2 are several times faster than out of HBM."""
    from diffus_b200 import ops
    l2 = ops.gather_probe(32, reads_per_thread=32, repeats=2)
    hbm = ops.gather_probe(512, reads_per_thread=32, repeats=2)
    assert l2["sectors_per_s"] > 2.0 * hbm["sectors_per_s"] > 0
    assert 100 < hbm["gb_per_s"] < 8000 and l2["gb_per_s"] < 40000


def test_fan_directions_device_matches_host_and_autograd():
    """Fans from pose parameters (median, in-plane hint, aperture): device forward vs the float64 host construction, and
    the backward (d/d median, d/d hint through the normalisation and the Gram-Schmidt step) vs float64 autograd."""
    from diffus_b200 import fan_directions
    from diffus_b200 import phantoms
    g = torch.Generator().manual_seed(11)
    P, R, angle = 7, 33, 1.1
    median = torch.randn((P, 3), generator=g) * 3.0
    hint = torch.randn((P, 3), generator=g)
    want = phantoms.fan_directions(median, hint, angle, R)
    m = median.to(dev()).requires_grad_(True)
    h = hint.to(dev()).requires_grad_(True)
    got = fan_directions(m, h, angle, R)
    assert got.shape == (P, R, 3) and got.dtype == torch.float32
    np.testing.assert_allclose(got.detach().cpu().numpy(), want.numpy(), rtol=0, atol=2e-7)
    w = torch.randn((P, R, 3), generator=g)
    (got * w.to(dev())).sum().backward()
    m64 = median.double().requires_grad_(True)
    h64 = hint.double().requires_grad_(True)
    mh = m64 / m64.norm(dim=-1, keepdim=True)
    u = h64 - (h64 * mh).sum(-1, keepdim=True) * mh
    u = u / u.norm(dim=-1, keepdim=True)
    a = torch.linspace(-angle / 2, angle / 2, R, dtype=torch.float64)
    d64 = torch.cos(a).view(1, -1, 1) * mh.unsqueeze(1) + torch.sin(a).view(1, -1, 1) * u.unsqueeze(1)
    (d64 * w.double()).sum().backward()
    assert_grad_close(m.grad.cpu().numpy(), m64.grad.numpy(), "d/d median", rtol=1e-5)
    assert_grad_close(h.grad.cpu().numpy(), h64.grad.numpy(), "d/d hint", rtol=1e-5)
    one = fan_directions(m[:1], h[:1], angle, 1)                      # a single ray sits at -angle/2 like numpy.linspace
    np.testing.assert_allclose(one.detach().cpu().numpy()[0, 0], want.numpy()[0, 0], atol=2e-7)


def test_graphed_fan_pose_step_matches_eager():
    from diffus_b200 import PreparedVolume, fan_directions, render_frames, render_mse_loss
    from diffus_b200.graphs import GraphedFanPoseStep
    from diffus_b200.phantoms import layered_phantom, pose_sweep
    vol = layered_phantom(32, seed=1).to(dev())
    angle = math.radians(50.0)
    src, dirs, med, hint = pose_sweep(5, 16, 32, seed=3, opening_angle=angle, return_params=True)
    src, dirs, med, hint = src.to(dev()), dirs.to(dev()), med.to(dev()), hint.to(dev())
    pv = PreparedVolume(vol, "brick")
    with torch.no_grad():
        target = render_frames(pv, src + 0.6, dirs, 96, 1e-3, sampler="trilinear")
    step = GraphedFanPoseStep(pv, target, 16, 96, angle, 1e-3)
    for shift in (0.0, 0.3):
        s = (src + shift).clone().requires_grad_(True)
        m = med.clone().requires_grad_(True)
        h = hint.clone().requires_grad_(True)
        loss = render_mse_loss(pv, s, fan_directions(m, h, angle, 16), target, 96, 1e-3)
        loss.backward()
        gl, gs, gm, gh = step(s.detach(), m.detach(), h.detach())
        torch.cuda.synchronize()
        np.testing.assert_allclose(gl.item(), loss.item(), rtol=1e-6)
        torch.testing.assert_close(gs, s.grad, rtol=1e-5, atol=1e-12)
        torch.testing.assert_close(gm, m.grad, rtol=1e-5, atol=1e-12)
        torch.testing.assert_close(gh, h.grad, rtol=1e-5, atol=1e-12)
