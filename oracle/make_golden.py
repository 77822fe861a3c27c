"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference.  TEST INFRASTRUCTURE.

Run in the build container (``python -m oracle.make_golden``); needs ``/root/reference``.
Every output array in the fixtures is produced by the reference's own code
(``src/renderer.py``, ``src/cone.py``, ``src/impedance.py`` at the mounted commit, torch
2.11.0 CPU); inputs are seeded here and stored next to the outputs so the fixtures are
self-contained on machines without the reference.
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import reference_loader as RL  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _np(t):
    return t.detach().cpu().numpy()


def _volume(shape, seed, lo=1.3e6, hi=1.8e6):
    g = torch.Generator().manual_seed(seed)
    return (lo + (hi - lo) * torch.rand(shape, generator=g, dtype=torch.float32)).contiguous()


def _blocky_volume(shape, seed, block=4):
    """Piecewise-constant tissue blocks (so that |r| has realistic sparsity) + 1 % noise."""
    g = torch.Generator().manual_seed(seed)
    coarse = [max(1, math.ceil(s / block)) for s in shape]
    c = 1.3e6 + 0.5e6 * torch.rand(coarse, generator=g)
    v = c.repeat_interleave(block, 0).repeat_interleave(block, 1).repeat_interleave(block, 2)
    v = v[: shape[0], : shape[1], : shape[2]]
    v = v * (1 + 0.01 * torch.randn(v.shape, generator=g))
    return v.float().contiguous()


def echo_cases(ref):
    R = ref.renderer
    out = {}
    # known-answer impedance sequences (SURVEY.md appendix B): NaN rule, |r| = 1, air gaps
    seqs = {
        "nan_lead": [0, 0, 1.5, 1.6, 0, 0, 1.5, 1.7],
        "total_reflection": [1.5, 1.6, 0, 1.5, 1.7, 1.7],
        "air_tissue_air": [400, 400, 1.6e6, 1.65e6, 1.6e6, 400, 400, 1.6e6],
        "doc_example": [1, 2, 1.5],
    }
    for name, z in seqs.items():
        Z = torch.tensor([z], dtype=torch.float64)
        r = R.UltrasoundRenderer.compute_reflection_coeff(Z[:, :-1], Z[:, 1:])
        with RL.quiet():
            e, d = R.compute_echo_traces(r)
        out[f"ka_{name}_Z"] = _np(Z)
        out[f"ka_{name}_r"] = _np(r)
        out[f"ka_{name}_echo"] = _np(e)
    # hand-written phantom of notebooks/[DEMO] Modeling Choices.ipynb cell 6
    zt = torch.tensor([[1.71e6, 1.71e6, 1.71e6, 1.65e6, 1.65e6, 1.65e6, 1.69e6, 1.69e6, 1.65e6, 1.65e6],
                       [1.71e6, 1.71e6, 1.65e6, 1.65e6, 1.65e6, 1.65e6, 1.69e6, 1.65e6, 1.65e6, 1.65e6],
                       [1.71e6, 1.71e6, 1.71e6, 1.65e6, 1.65e6, 1.65e6, 1.65e6, 1.71e6, 1.71e6, 1.71e6],
                       [1.71e6, 1.71e6, 1.71e6, 1.71e6, 1.65e6, 1.65e6, 1.65e6, 1.65e6, 1.71e6, 1.71e6],
                       [1.71e6, 1.71e6, 1.71e6, 1.71e6, 1.65e6, 1.65e6, 1.65e6, 1.71e6, 1.71e6, 1.71e6]])
    rt = R.UltrasoundRenderer.compute_reflection_coeff(zt[:, 1:], zt[:, :-1])   # argument order as in the notebook
    with RL.quiet():
        e, d = R.compute_echo_traces(rt)
        cum = R.propagate_full_rays_batched(rt)
    out["phantom_Z"], out["phantom_r"], out["phantom_echo"] = _np(zt), _np(rt), _np(e)
    out["phantom_cumulative"], out["phantom_delays"] = _np(cum), _np(d)
    # random coefficients, fp64 and fp32, incl. a ragged (odd) length
    g = torch.Generator().manual_seed(1)
    for name, B, N, amp in (("rand_a", 8, 48, 0.4), ("rand_b", 5, 77, 0.1), ("rand_c", 3, 1, 0.9)):
        r64 = (torch.rand((B, N), generator=g, dtype=torch.float64) - 0.5) * 2 * amp
        with RL.quiet():
            e64, _ = R.compute_echo_traces(r64)
            e32, _ = R.compute_echo_traces(r64.float())
        out[f"{name}_r"], out[f"{name}_echo64"], out[f"{name}_echo32"] = _np(r64), _np(e64), _np(e32)
    np.savez_compressed(os.path.join(OUT, "echo_traces.npz"), **out)


def frame_cases(ref):
    R, C = ref.renderer, ref.cone
    out = {}
    cases = []
    # (name, volume, source, directions, S, alpha, start)
    vol_a = _blocky_volume((32, 28, 36), 2)
    dirs_a = C.generate_cone_directions([0.3, 1.0], math.radians(50), 12)
    src_a = torch.tensor([14.3, 1.7, 17.2])
    cases.append(("a0", vol_a, src_a, dirs_a, 40, 1e-3, 0))
    cases.append(("a7", vol_a, src_a, dirs_a, 40, 1e-3, 7))
    cases.append(("afrac", vol_a, src_a, dirs_a, 40, 1e-3, 0.25))
    # general 3-D directions and an integer source, as in notebooks/[DEMO] Modeling Choices.ipynb cell 18
    th = np.radians(np.linspace(-13, 13, 9))
    dirs_b = torch.tensor(np.stack([-np.cos(th), 0.3 * np.ones_like(th), np.sin(th)], 1), dtype=torch.float32)
    dirs_b = dirs_b / dirs_b.norm(dim=1, keepdim=True)
    src_b = torch.tensor([30, 10, 15])
    cases.append(("b0", vol_a, src_b, dirs_b, 33, 1e-4, 0))
    cases.append(("b5", vol_a, src_b, dirs_b, 33, 0.5, 5))
    # negated impedance volume (the notebook renders `-Z_vol`) with air pockets -> NaN rule
    vol_c = vol_a.clone()
    vol_c[10:14, 8:12, :] = 0.0
    cases.append(("c0", -vol_c, src_a, dirs_a, 40, 1e-3, 0))
    # layered phantom, the benchmark geometry scaled down to 48^3
    sys.path.insert(0, ROOT)
    from diffus_b200.phantoms import layered_phantom
    vol_d = layered_phantom(48, seed=0)
    dirs_d = C.generate_cone_directions([0.0, 1.0], math.radians(60), 16)
    src_d = torch.tensor([24.0, 0.0, 24.0])
    cases.append(("d0", vol_d, src_d, dirs_d, 96, 1e-4, 0))
    for name, vol, src, dirs, S, alpha, start in cases:
        ren = R.UltrasoundRenderer(S, alpha)
        with RL.quiet():
            x, y, z, f32 = ren.plot_beam_frame(volume=vol.clone(), source=src, directions=dirs,
                                               plot=False, artifacts=False, start=start)
            _, _, _, f64 = ren.plot_beam_frame(volume=vol.double(), source=src, directions=dirs.double(),
                                               plot=False, artifacts=False, start=start)
            xs, ys, zs, rs = ren.simulate_rays(vol.clone(), src, dirs, start=0)
        if name == "a0" or vol is not vol_a:         # the cases on vol_a share a0's copy (tests/conftest.py::golden_frames)
            out[f"{name}_volume"] = _np(vol)
        out[f"{name}_source"], out[f"{name}_dirs"] = _np(src), _np(dirs)
        out[f"{name}_S"], out[f"{name}_alpha"] = np.int64(S), np.float64(alpha)
        out[f"{name}_start"] = np.float64(start)
        out[f"{name}_start_is_float"] = np.bool_(type(start) is float)
        out[f"{name}_x"], out[f"{name}_y"], out[f"{name}_z"] = _np(x), _np(y), _np(z)
        out[f"{name}_frame32"], out[f"{name}_frame64"] = _np(f32), _np(f64)
        out[f"{name}_refl"] = _np(rs)
    np.savez_compressed(os.path.join(OUT, "frames_nearest.npz"), **out)


def trilinear_cases(ref):
    R, C = ref.renderer, ref.cone
    out = {}
    g = torch.Generator().manual_seed(5)
    vol = _blocky_volume((24, 20, 28), 3, block=3)
    fan = C.generate_cone_directions([0.2, 1.0], math.radians(40), 9)
    th = np.radians(np.linspace(-20, 20, 7))
    obl = torch.tensor(np.stack([np.sin(th), np.cos(th) * 0.9, 0.35 * np.ones_like(th)], 1), dtype=torch.float32)
    obl = obl / obl.norm(dim=1, keepdim=True)
    cases = [
        ("t0", vol, torch.tensor([11.3, 0.0, 13.6]), fan, 36, 1e-3),      # source ON the p1=0 face
        ("t1", vol, torch.tensor([4.4, 2.2, 3.3]), obl, 30, 1e-2),        # oblique 3-D fan leaving the volume
        ("t2", vol, torch.tensor([12.0, 3.0, 9.0]), obl, 24, 1e-3),       # integer-valued coordinates
    ]
    for name, v, src, dirs, S, alpha in cases:
        v64 = v.double().requires_grad_(True)
        s64 = src.double().requires_grad_(True)
        d64 = dirs.double().requires_grad_(True)
        ren = R.UltrasoundRenderer(S, alpha)
        with RL.trilinear_sampler_installed(ref), RL.quiet():
            x, y, z, f = ren.plot_beam_frame(volume=v64, source=s64, directions=d64, plot=False, start=0)
        w = torch.randn(f.shape, generator=g, dtype=torch.float64)
        gv, gs, gd = torch.autograd.grad((f * w).sum(), [v64, s64, d64])
        out[f"{name}_volume"], out[f"{name}_source"], out[f"{name}_dirs"] = _np(v), _np(src), _np(dirs)
        out[f"{name}_S"], out[f"{name}_alpha"] = np.int64(S), np.float64(alpha)
        out[f"{name}_frame64"], out[f"{name}_w"] = _np(f), _np(w)
        out[f"{name}_grad_volume"], out[f"{name}_grad_source"], out[f"{name}_grad_dirs"] = _np(gv), _np(gs), _np(gd)
        out[f"{name}_x"], out[f"{name}_y"], out[f"{name}_z"] = _np(x), _np(y), _np(z)
    # nearest sampler: gradient w.r.t. the volume only (HEAD's differentiable input)
    v64 = vol.double().requires_grad_(True)
    ren = R.UltrasoundRenderer(36, 1e-3)
    with RL.quiet():
        x, y, z, f = ren.plot_beam_frame(volume=v64, source=cases[0][2], directions=fan.double(), plot=False, start=0)
    w = torch.randn(f.shape, generator=g, dtype=torch.float64)
    (gv,) = torch.autograd.grad((f * w).sum(), [v64])
    out["n0_frame64"], out["n0_w"], out["n0_grad_volume"] = _np(f), _np(w), _np(gv)
    np.savez_compressed(os.path.join(OUT, "frames_trilinear_grad.npz"), **out)


def cone_cases(ref):
    C = ref.cone
    out = {}
    for i, (d, ang, n) in enumerate([([0.0, 1.0], math.radians(60), 128), ([0.3, 1.0, 5.0], 0.8, 7),
                                     ([-2.0, 0.5], math.radians(27), 150), ([1.0, 0.0], 1e-3, 2),
                                     ([0.6, -0.8], math.pi, 1)]):
        out[f"cone{i}_d"], out[f"cone{i}_angle"], out[f"cone{i}_n"] = np.array(d, dtype=np.float64), np.float64(ang), np.int64(n)
        out[f"cone{i}_dirs"] = _np(C.generate_cone_directions(d, ang, n))
    np.savez_compressed(os.path.join(OUT, "cone_directions.npz"), **out)


def mlp_cases(ref):
    I = ref.impedance
    out = {}
    torch.manual_seed(0)
    model = I.ImpedanceEstimator(1)
    sd = model.state_dict()
    for k, v in sd.items():
        out["param_" + k.replace(".", "_")] = _np(v)
    g = torch.Generator().manual_seed(7)
    x = (torch.randn((257, 1), generator=g) * 1.5)
    y = model(x)
    w = torch.randn(y.shape, generator=g)
    grads = torch.autograd.grad((y * w).sum(), list(model.parameters()))
    out["x"], out["y"], out["w"] = _np(x), _np(y), _np(w)
    for (k, _), gr in zip(model.named_parameters(), grads):
        out["grad_" + k.replace(".", "_")] = _np(gr)
    # fp64 twin for tight checks
    m64 = I.ImpedanceEstimator(1).double()
    m64.load_state_dict({k: v.double() for k, v in sd.items()})
    out["y64"] = _np(m64(x.double()))
    np.savez_compressed(os.path.join(OUT, "impedance_mlp.npz"), **out)


def splat_cases(ref):
    R = ref.renderer
    out = {}
    g = torch.Generator().manual_seed(9)
    S, n = 40, 12
    k = torch.arange(S).float()
    th = torch.linspace(-0.4, 0.4, n)
    x = torch.clamp((30 + k[None] * torch.sin(th)[:, None]).round().long(), 0, 63)
    y = torch.clamp((2 + k[None] * torch.cos(th)[:, None]).round().long(), 0, 63)
    z = torch.full_like(x, 17)
    val = torch.randn((n, S), generator=g)
    for sigma in (0.5, 1.0):
        with RL.quiet():
            img = R.differentiable_splat(x, y, z, val, H=64, W=64, sigma=sigma)
        out[f"img_sigma{sigma}"] = _np(img)
    out["x"], out["y"], out["z"], out["val"] = _np(x), _np(y), _np(z), _np(val)
    np.savez_compressed(os.path.join(OUT, "splat.npz"), **out)


def brain_phantom2d_cases(ref):
    """generate_brain_phantom_2d of notebooks/[DEMO] Modeling Choices.ipynb cell 5 (air 400, bone 7.8e6: |r| up to 0.9995)."""
    R = ref.renderer
    rows, cols = 20, 10
    brain, tumor, csf, bone, air = 1.60e6, 1.68e6, 1.50e6, 7.80e6, 0.0004e6
    ph = torch.full((rows, cols), air)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, rows), torch.linspace(-1, 1, cols), indexing="ij")
    brain_mask = (xx ** 2 / 0.8 ** 2 + yy ** 2 / 0.95 ** 2) <= 1.0
    ph[brain_mask] = brain
    csf_mask = (xx ** 2 / 0.88 ** 2 + yy ** 2 / 1.05 ** 2) <= 1.0
    ph[csf_mask & (~brain_mask)] = csf
    ph[(abs(xx) < 0.2) & (abs(yy) < 0.3) & brain_mask] = tumor
    last = torch.where(brain_mask.any(dim=1))[0][-1]
    ph[last, brain_mask[last]] = bone
    r = R.UltrasoundRenderer.compute_reflection_coeff(ph[:, 1:], ph[:, :-1])
    with RL.quiet():
        e32, _ = R.compute_echo_traces(r)
        e64, _ = R.compute_echo_traces(r.double())
    np.savez_compressed(os.path.join(OUT, "echo_brain_phantom2d.npz"), Z=_np(ph), r=_np(r), echo32=_np(e32), echo64=_np(e64))


def impedance_volume_cases(ref):
    I, U = ref.impedance, ref.utils
    sys.path.insert(0, ROOT)
    from diffus_b200.phantoms import mri_phantom
    out = {}
    vol = mri_phantom(24, "t1", seed=3)
    vol[2:4, 2:4, 2:4] = 900.0            # an isolated speck: closed by dilation/erosion or not, as scipy decides
    vol[0, 10:14, 10:14] = 900.0          # touches the border (erosion's border_value=0 matters)
    torch.manual_seed(0)
    model = I.ImpedanceEstimator(1)
    for k, v in model.state_dict().items():
        out["param_" + k.replace(".", "_")] = _np(v)
    mask = U.create_brain_mask(vol.numpy(), 50)
    out["volume"], out["mask"] = _np(vol), _np(mask)
    out["vol_norm"] = _np(U.zscore_normalize(vol, mask))
    out["Z"] = _np(I.ImpedanceEstimator.compute_impedance_volume(vol, model, threshold=50))
    np.savez_compressed(os.path.join(OUT, "impedance_volume.npz"), **out)


def _notebook_cell(name, index):
    import json
    with open(os.path.join(RL.REFERENCE_ROOT, "notebooks", name)) as f:
        return "".join(json.load(f)["cells"][index]["source"])


def training_loop_cases(ref):
    """Row f3 / f1-epilogue fixtures.  rotate_around_apex: the reference function.  masked MSE + edge loss and
    process_rf_to_bmode: the notebook cells' own source, executed (they are not importable modules).  Adam: torch.optim.Adam.
    SSIM: piq is absent, so those numbers come from oracle/port.py's restatement (flagged in the fixture)."""
    import torch.nn as nn
    import torch.nn.functional as F
    from oracle import port
    R = ref.renderer
    out = {}
    g = torch.Generator().manual_seed(31)
    # rotate_around_apex on index-like coordinates (the notebooks pass x.float(), z.float())
    x = torch.randint(0, 256, (480,), generator=g).float()          # 1-D, as HEAD's matrix product requires (:686-687)
    z = torch.randint(0, 256, (480,), generator=g).float()
    apex, median = [131.7, 20.25], [-0.3, -0.9]
    with RL.quiet():
        xr, zr = R.rotate_around_apex(x, z, apex=torch.tensor(apex), median=median)
    out["rot_x"], out["rot_z"], out["rot_apex"], out["rot_median"] = _np(x), _np(z), np.array(apex), np.array(median)
    out["rot_x_out"], out["rot_z_out"] = _np(xr), _np(zr)
    # the CPU notebook's loss, from its own cell source
    ns = {"torch": torch, "nn": nn, "F": F, "np": np, "device": "cpu", "UltrasoundRenderer": R.UltrasoundRenderer,
          "rotate_around_apex": R.rotate_around_apex, "differentiable_splat": R.differentiable_splat}
    exec(_notebook_cell("[DEMO] Train MRI to Impedance MLP.ipynb", 19), ns)
    usm = ns["UltrasoundSynthesisModel"].__new__(ns["UltrasoundSynthesisModel"])
    H, W = 37, 44
    real = torch.rand((H, W), generator=g, dtype=torch.float64)
    synth = (real + 0.2 * torch.randn((H, W), generator=g, dtype=torch.float64)).requires_grad_(True)
    mask = torch.rand((H, W), generator=g) > 0.35
    mask[:, 0] = True
    usm.us_real_norm, usm.mask = real, mask
    with RL.quiet():
        loss = usm.loss(synth)
    (gs,) = torch.autograd.grad(loss, synth)
    out["mse_edge_synth"], out["mse_edge_real"], out["mse_edge_mask"] = _np(synth), _np(real), _np(mask)
    out["mse_edge_loss"], out["mse_edge_grad"] = _np(loss), _np(gs)
    # process_rf_to_bmode from its notebook cell (scipy.signal.hilbert), even and odd line lengths
    ns2 = {}
    exec(_notebook_cell("[DEMO] Renderer Alternatives.ipynb", 14).split("def plot_bmode_image")[0], ns2)
    stubs = {k: sys.modules.pop(k) for k in ("jax", "jax.numpy") if k in sys.modules}     # scipy's array-API probe trips over the jax stub
    for name, shape in (("rf_even", (6, 64)), ("rf_odd", (5, 33))):
        rf = 0.05 * torch.randn(shape, generator=g)
        out[name], out[name + "_bmode"] = _np(rf), ns2["process_rf_to_bmode"](rf)
    sys.modules.update(stubs)
    # torch.optim.Adam on the 1 153 weights, lr 0.01 as in the GPU notebook
    p0 = torch.randn(1153, generator=g)
    grads = [torch.randn(1153, generator=g) * 10.0 ** (-i) for i in range(4)]
    steps = port.adam_steps(p0, grads, lr=0.01)
    out["adam_p0"], out["adam_grads"], out["adam_params"] = _np(p0), _np(torch.stack(grads)), _np(torch.stack(steps))
    steps_wd = port.adam_steps(p0, grads, lr=1e-3, betas=(0.8, 0.99), eps=1e-6, weight_decay=0.1)
    out["adam_params_wd"] = _np(torch.stack(steps_wd))
    # SSIM loss (port; piq absent): a splat-like image with an exact-zero background (ties at the minimum)
    H, W = 48, 40
    real = torch.rand((H, W), generator=g, dtype=torch.float64)
    synth = torch.zeros((H, W), dtype=torch.float64)
    synth[8:40, 5:33] = real[8:40, 5:33] * 3.0 + 0.3 * torch.randn((32, 28), generator=g, dtype=torch.float64)
    synth.requires_grad_(True)
    for tag, norm in (("ssim_norm", True), ("ssim_raw", False)):
        l = port.ssim_loss(synth, real, normalize=norm)
        (gs,) = torch.autograd.grad(l, synth)
        out[tag + "_loss"], out[tag + "_grad"] = _np(l), _np(gs)
    out["ssim_synth"], out["ssim_real"] = _np(synth), _np(real)
    out["ssim_made_by"] = np.array("oracle/port.py restatement of piq.ssim (piq is not installed; parity unpinned)")
    np.savez_compressed(os.path.join(OUT, "training_loop.npz"), **out)


def _volume_fingerprint(vol):
    """A few numbers that pin a seeded volume regenerated on another machine (the 64 MiB tensor is not stored)."""
    v = vol.double().reshape(-1)
    idx = torch.arange(0, v.numel(), 104729)          # a prime stride
    return np.array([v.sum().item(), v.square().sum().item(), (v[idx] * torch.arange(1, idx.numel() + 1)).sum().item()])


def config1_full_cases(ref):
    """BASELINE config 1 AT FULL SIZE from the real reference: layered 256^3 phantom, 128 rays x 512 samples, nearest,
    forward, fp32 and fp64 (about 75 s + 150 s on 8 cores).  The volume is regenerated from its seed by the tests
    (``layered_phantom(256, seed=0)``) and checked against the stored fingerprint."""
    R = ref.renderer
    sys.path.insert(0, ROOT)
    from diffus_b200.phantoms import config1_pose, layered_phantom
    vol = layered_phantom(256, seed=0)
    src, dirs = config1_pose(256, 128)
    ren = R.UltrasoundRenderer(512, 1e-4)
    with RL.quiet():
        x, y, z, f32 = ren.plot_beam_frame(volume=vol.clone(), source=src, directions=dirs, plot=False, artifacts=False, start=0)
        _, _, _, f64 = ren.plot_beam_frame(volume=vol.double(), source=src, directions=dirs.double(), plot=False,
                                           artifacts=False, start=0)
    out = {"volume_fingerprint": _volume_fingerprint(vol), "source": _np(src), "dirs": _np(dirs), "S": np.int64(512),
           "alpha": np.float64(1e-4), "frame32": _np(f32), "frame64": _np(f64),
           "x": _np(x).astype(np.int16), "y": _np(y).astype(np.int16), "z": _np(z).astype(np.int16)}
    np.savez_compressed(os.path.join(OUT, "config1_full.npz"), **out)


def config2_reduced_cases(ref):
    """BASELINE config 2's geometry from the real reference with its trilinear sampler installed: the same 256^3 phantom
    and 128-ray fan, the first 128 samples (torch autograd through the dense solves needs ~190 GB at 512), fp64:
    frame, d/dsource, d/ddirections and the non-zero part of d/dvolume of sum(frame * w)."""
    R = ref.renderer
    sys.path.insert(0, ROOT)
    from diffus_b200.phantoms import config1_pose, layered_phantom
    vol = layered_phantom(256, seed=0)
    src, dirs = config1_pose(256, 128)
    S = 128
    g = torch.Generator().manual_seed(22)
    v64 = vol.double().requires_grad_(True)
    s64 = src.double().requires_grad_(True)
    d64 = dirs.double().requires_grad_(True)
    ren = R.UltrasoundRenderer(S, 1e-4)
    with RL.trilinear_sampler_installed(ref), RL.quiet():
        x, y, z, f = ren.plot_beam_frame(volume=v64, source=s64, directions=d64, plot=False, start=0)
    w = torch.randn(f.shape, generator=g, dtype=torch.float32).double()      # float32-representable: the kernels get the same weights
    gv, gs, gd = torch.autograd.grad((f * w).sum(), [v64, s64, d64])
    nz = gv.reshape(-1).nonzero().reshape(-1)
    out = {"volume_fingerprint": _volume_fingerprint(vol), "source": _np(src), "dirs": _np(dirs), "S": np.int64(S),
           "alpha": np.float64(1e-4), "frame64": _np(f), "w": _np(w).astype(np.float32),
           "grad_source": _np(gs), "grad_dirs": _np(gd),
           "grad_volume_index": _np(nz).astype(np.int32), "grad_volume_value": _np(gv.reshape(-1)[nz]).astype(np.float32)}
    np.savez_compressed(os.path.join(OUT, "config2_reduced.npz"), **out)


def median_tie_cases(ref):
    """start > 0 with the near field OUTSIDE the volume: the border clamp makes the first kept coefficient exactly 0 on
    most rays, so the median over rays is a tie.  Forward from the real reference (its autograd raises here,
    src/renderer.py:243-244); the tie rule of the gradient is torch's ``median()`` backward (evenly distributed over the
    tied elements), recorded on a small vector."""
    R, C = ref.renderer, ref.cone
    out = {}
    vol = _blocky_volume((24, 24, 24), 11, block=3)
    dirs = C.generate_cone_directions([0.0, 1.0], math.radians(70), 15)
    src = torch.tensor([12.0, -9.0, 12.0])              # 9 voxels in front of the p1 = 0 face
    for name, start in (("tie4", 4), ("tie9", 9), ("tie12", 12)):
        ren = R.UltrasoundRenderer(40, 1e-3)
        with RL.quiet():
            x, y, z, f64 = ren.plot_beam_frame(volume=vol.double(), source=src, directions=dirs.double(), plot=False, start=start)
            xs, ys, zs, rs = ren.simulate_rays(vol.double(), src, dirs.double())
        out[f"{name}_start"], out[f"{name}_frame64"], out[f"{name}_x"] = np.int64(start), _np(f64), _np(x)
        out[f"{name}_first_refl"] = _np(rs[:, start])
    out["volume"], out["source"], out["dirs"] = _np(vol), _np(src), _np(dirs)
    t = torch.tensor([0.0, 0.0, 3.0, 1.0, -1.0, 0.0, 2.0, 5.0], dtype=torch.float64, requires_grad=True)
    t.median().backward()
    out["tie_rule_input"], out["tie_rule_grad"] = _np(t), _np(t.grad)
    np.savez_compressed(os.path.join(OUT, "median_ties.npz"), **out)


def main():
    ref = RL.load()
    if ref is None:
        raise SystemExit("reference tree not found at " + RL.REFERENCE_ROOT)
    os.makedirs(OUT, exist_ok=True)
    only = sys.argv[1:]
    fns = (echo_cases, frame_cases, trilinear_cases, cone_cases, mlp_cases, splat_cases, impedance_volume_cases, brain_phantom2d_cases,
           training_loop_cases, median_tie_cases, config2_reduced_cases, config1_full_cases)      # the last one takes ~4 minutes
    for fn in fns:
        if only and fn.__name__ not in only:
            continue
        fn(ref)
        print("wrote", fn.__name__)
    with open(os.path.join(OUT, "PROVENANCE.txt"), "w") as f:
        f.write("Generated by oracle/make_golden.py from the unmodified reference at /root/reference\n"
                f"torch {torch.__version__}, numpy {np.__version__}\n"
                "harness shims: stubbed matplotlib/nibabel imports, visualize=False, stdout swallowed\n")


if __name__ == "__main__":
    main()
