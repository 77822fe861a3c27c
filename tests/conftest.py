import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


@pytest.fixture(scope="session")
def golden_echo():
    return load_golden("echo_traces.npz")


@pytest.fixture(scope="session")
def golden_frames():
    g = load_golden("frames_nearest.npz")
    for name in ("a7", "afrac", "b0", "b5"):                # these cases render case a0's volume; the file stores it once
        g[f"{name}_volume"] = g["a0_volume"]
    return g


@pytest.fixture(scope="session")
def golden_tri():
    return load_golden("frames_trilinear_grad.npz")


@pytest.fixture(scope="session")
def golden_cone():
    return load_golden("cone_directions.npz")


@pytest.fixture(scope="session")
def golden_mlp():
    return load_golden("impedance_mlp.npz")


@pytest.fixture(scope="session")
def golden_impvol():
    return load_golden("impedance_volume.npz")


@pytest.fixture(scope="session")
def golden_splat():
    return load_golden("splat.npz")


# Tolerances of BASELINE.json north_star:
#   frames    <= 1e-5 relative / 1e-4 absolute ON NORMALISED INTENSITY: the absolute term is scaled by the peak of the
#             reference frame (a raw B-mode line peaks at ~0.08 for tissue, at 1e3 for resonating air gaps);
#   gradients <= 1e-4 relative vs (fp64) torch autograd, ELEMENT-WISE for every entry above GRAD_FLOOR of the largest
#             one; smaller entries (sums that cancel) are held to the same absolute error as an entry at the floor.
FRAME_RTOL, FRAME_ATOL = 1e-5, 1e-4
GRAD_RTOL, GRAD_FLOOR = 1e-4, 1e-3

# DIFFUS_TOL_REPORT=<file>: every check appends (test, what, achieved error / tolerance) -- how the margins in
# profiles/r2_parity_margins.md were obtained.  DIFFUS_TOL_CALIBRATE=1 additionally records instead of failing.
_REPORT = os.environ.get("DIFFUS_TOL_REPORT")
_CALIBRATE = os.environ.get("DIFFUS_TOL_CALIBRATE") == "1"


def _record(kind, what, ratio, detail):
    if _REPORT:
        import json
        test = os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0]
        with open(_REPORT, "a") as f:
            f.write(json.dumps({"test": test, "kind": kind, "what": what, "err_over_tol": ratio, **detail}) + "\n")


def assert_frame_close(got, want, what="", atol=FRAME_ATOL, rtol=FRAME_RTOL):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if got.size == 0:
        return
    peak = float(np.abs(want).max())
    err = np.abs(got - want)
    tol = atol * peak + rtol * np.abs(want) + 1e-30
    ratio = float((err / tol).max())
    _record("frame", what, ratio, {"max_err": float(err.max()), "peak": peak})
    if _CALIBRATE:
        return
    assert ratio <= 1.0, (f"{what}: max err {err.max():.3e} at {np.unravel_index((err / tol).argmax(), err.shape)}, "
                          f"{ratio:.2f} x the tolerance ({atol:g} x peak {peak:.3e} + {rtol:g} |ref|)")


NOISE_FACTOR = 8.0


def oracle_grads(fn, *tensors):
    """Gradients of the CPU oracle in float64 AND the float32 noise of the same arithmetic.

    ``fn(*tensors_in_dtype)`` returns ``loss`` or ``(loss, aux)``; the float tensors are cast to float64 (the reference
    value) and to float32 (how far the reference's OWN algorithm drifts in the precision the kernels and the reference's
    fp32 runs work in).  Returns ``(grads64, noise, aux64)`` with ``noise[i] = max |grad32_i - grad64_i|`` (0 for an unused
    input).  ``assert_grad_close(..., noise=noise[i])`` then holds the kernel to 1e-4 element-wise OR to NOISE_FACTOR x that
    drift, whichever is larger: sums over hundreds of samples that cancel (d/d directions = sum_k k zbar_k grad Z_k) cannot be
    reproduced to 1e-4 of a small entry by ANY float32 evaluation, the reference's included."""
    out = {}
    for dt in (torch.float64, torch.float32):
        ins = [t.detach().to(dt).requires_grad_(True) for t in tensors]
        res = fn(*ins)
        loss, aux = res if isinstance(res, tuple) else (res, None)
        grads = torch.autograd.grad(loss, ins, allow_unused=True)
        out[dt] = (grads, aux)
    g64, aux64 = out[torch.float64]
    g32, _ = out[torch.float32]
    noise = [0.0 if a is None else float((b.double() - a).abs().max()) for a, b in zip(g64, g32)]
    return g64, noise, aux64


def assert_grad_close(got, want, what="", rtol=GRAD_RTOL, floor=GRAD_FLOOR, noise=None, noise_factor=NOISE_FACTOR):
    """fp32 kernels vs fp64 autograd: |got - want| <= rtol |want| for every entry with |want| > floor * max|want|,
    and <= rtol * floor * max|want| for the entries below that.  ``noise`` (see :func:`oracle_grads`): the absolute error the
    reference algorithm itself makes in float32 on this input; entries are then allowed ``noise_factor * noise`` if that is larger."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if got.size == 0:
        return
    scale = max(float(np.abs(want).max()), 1e-20)
    err = np.abs(got - want)
    strict = rtol * np.maximum(np.abs(want), floor * scale)
    tol = strict if noise is None else np.maximum(strict, noise_factor * float(noise))
    ratio = float((err / tol).max())
    _record("grad", what, ratio, {"max_err_over_scale": float(err.max() / scale), "scale": scale,
                                  "strict_ratio": float((err / strict).max()),
                                  "err_over_noise": None if not noise else float(err.max() / float(noise))})
    if _CALIBRATE:
        return
    k = np.unravel_index((err / tol).argmax(), err.shape)
    assert ratio <= 1.0, (f"{what}: entry {k}: got {got[k]:.6e} want {want[k]:.6e} (|ref| max {scale:.3e}); "
                          f"{ratio:.2f} x the tolerance (rtol {rtol:g}, floor {floor:g}, fp32 noise of the oracle {noise})")
