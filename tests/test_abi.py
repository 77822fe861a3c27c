"""CPU: the C-ABI library loads, exports every symbol include/diffus_b200.h declares, and rejects bad
arguments with its documented error codes before touching a device (no compute calls here)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "diffus_b200.h")


@pytest.fixture(scope="module")
def lib():
    from diffus_b200 import _lib, build
    build.build()                       # nvcc cross-compiles without a GPU
    return _lib.load()


def header_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(diffus_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported_and_bound(lib):
    from diffus_b200 import _lib
    names = header_functions()
    assert len(names) >= 17
    assert sorted(_lib.SIGNATURES) == names, "ctypes binding and header disagree"
    for n in names:
        assert getattr(lib, n) is not None


def test_abi_version_and_error_strings(lib):
    from diffus_b200 import _lib
    assert lib.diffus_abi_version() == _lib.ABI_VERSION
    text = open(HEADER).read()
    assert int(re.search(r"#define DIFFUS_ABI_VERSION (\d+)", text).group(1)) == _lib.ABI_VERSION
    assert lib.diffus_error_string(0) == b"ok"
    for code in (-1, -2, -3, -4, -5):
        assert lib.diffus_error_string(code) not in (b"ok", b"unknown error")


def test_struct_layout_matches_header(lib):
    """Field order/size of the ctypes mirrors (a mismatch would silently corrupt arguments)."""
    from diffus_b200._lib import DiffusRenderArgs, DiffusRenderBwdArgs, DiffusVolume
    assert C.sizeof(DiffusVolume) == 24
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for struct, cls in (("DiffusRenderArgs", DiffusRenderArgs), ("DiffusRenderBwdArgs", DiffusRenderBwdArgs)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
        fields = [re.split(r"[\s\*]+", f.strip())[-1].split("[")[0] for f in body.split(";") if f.strip()]
        assert fields == [f[0] for f in cls._fields_], struct


def test_argument_validation_without_a_device(lib):
    from diffus_b200._lib import DiffusRenderArgs, DiffusRenderBwdArgs
    a = DiffusRenderArgs()
    assert lib.diffus_render_forward(None, None) == -1
    assert lib.diffus_render_forward(C.byref(a), None) == -1           # NULL volume
    a.volume.data = 0x1000
    a.volume.dim[0] = a.volume.dim[1] = a.volume.dim[2] = 8
    a.sources = a.directions = a.frame = 0x1000
    a.n_poses, a.n_rays, a.n_samples = 1, 4, 1
    assert lib.diffus_render_forward(C.byref(a), None) == -2           # S < 2
    a.n_samples = 16
    a.sampler = 7
    assert lib.diffus_render_forward(C.byref(a), None) == -3           # unknown sampler
    a.sampler = 0
    a.start = 15
    assert lib.diffus_render_forward(C.byref(a), None) == -2           # start > S-2
    a.start = 3
    assert lib.diffus_render_workspace_bytes(C.byref(a)) > 0
    assert lib.diffus_render_forward(C.byref(a), None) == -4           # start > 0 needs the workspace
    a.start = 0
    a.dir_pose_stride = 5
    assert lib.diffus_render_forward(C.byref(a), None) == -2           # stride must be 0 or R*3
    a.dir_pose_stride = 0
    a.volume.dim[0] = a.volume.dim[1] = a.volume.dim[2] = 2048
    assert lib.diffus_render_forward(C.byref(a), None) == -5           # > 2^31 voxels: 32-bit offsets
    b = DiffusRenderBwdArgs()
    assert lib.diffus_render_backward(C.byref(b), None) == -1
    # which backward calls want the forward's 512-column prefixes (a pure function of shapes / enums / requested outputs)
    assert lib.diffus_render_bwd_needs_prefix(None) == -1
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == -2                     # no shape yet
    b.fwd.n_poses, b.fwd.n_rays, b.fwd.n_samples, b.fwd.sampler = 2, 8, 512, 1
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 0                      # one pass
    b.fwd.n_samples = 2048
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 1                      # no gradient output named yet: multi-pass form
    b.grad_sources = 0x1000
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 0                      # pose gradient only: one CTA per ray
    b.fwd.n_samples, b.fwd.start = 600, 37
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 0                      # 563 columns: two passes, two warps
    b.fwd.n_samples, b.fwd.start = 2049, 0
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 1                      # five passes
    b.fwd.n_samples = 2048
    b.grad_volume = 0x1000
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 1                      # with the volume gradient
    b.grad_volume, b.fwd.pose_dtype = None, 1
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 1                      # float64 poses
    b.fwd.pose_dtype, b.fwd.sampler = 0, 0
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == 1                      # nearest sampler: no pose gradient
    b.fwd.sampler = 9
    assert lib.diffus_render_bwd_needs_prefix(C.byref(b)) == -3
    assert lib.diffus_echo_forward(None, 1, 1, None, None) == -1
    assert lib.diffus_echo_forward(0x1000, 0, 4, 0x1000, None) == -2
    assert lib.diffus_mlp_forward(None, None, None, 4, 1.0, 0.0, None, None) == -1
    assert lib.diffus_mlp_backward(0x1000, 0x1000, None, 0x1000, 64, 1.0, 0x1000, None, 0, None) == -4
    assert lib.diffus_mlp_bwd_workspace_bytes(1 << 20) > 0
    dim = (C.c_int32 * 3)(10, 9, 7)
    assert lib.diffus_brick_elems(C.byref(dim)) == 3 * 3 * 4 * 32
    assert lib.diffus_cone_directions(None, 1, 1, 0.5, None, None) == -1
    # packed layouts, fans from pose parameters, the roofline probe, the explicit MLP backward path
    assert lib.diffus_quad_elems(C.byref(dim)) == 5 * 5 * 4 * 8 * 4
    assert lib.diffus_volume_to_quads(0x1000, C.byref(dim), 0x1008, None) == -5     # float4 loads: 16-byte alignment
    assert lib.diffus_volume_to_quads(None, C.byref(dim), 0x1000, None) == -1
    a2 = DiffusRenderArgs()
    a2.volume.data, a2.volume.layout = 0x1008, 2                                   # QUAD volume not 16-byte aligned
    a2.volume.dim[0] = a2.volume.dim[1] = a2.volume.dim[2] = 8
    a2.sources = a2.directions = a2.frame = 0x1000
    a2.n_poses, a2.n_rays, a2.n_samples = 1, 4, 16
    assert lib.diffus_render_forward(C.byref(a2), None) == -5
    a2.volume.layout = 4
    assert lib.diffus_render_forward(C.byref(a2), None) == -3                      # unknown layout
    # TEXTURE layout: the only allocating entry points validate before touching the device
    t, arr = C.c_uint64(0), C.c_uint64(0)
    assert lib.diffus_volume_texture_create(None, C.byref(dim), C.byref(t), C.byref(arr), None) == -1
    big = (C.c_int32 * 3)(4096, 8, 8)
    assert lib.diffus_volume_texture_create(0x1000, C.byref(big), C.byref(t), C.byref(arr), None) == -5   # > 2048 layers
    assert lib.diffus_volume_texture_update(0, 0x1000, C.byref(dim), None) == -1
    a2.volume.layout = 3
    a2.volume.dim[0] = 4096
    assert lib.diffus_render_forward(C.byref(a2), None) == -5                      # more layers than a layered array holds
    a2.volume.dim[0] = 8
    a2.volume.layout, a2.frame, a2.seg_prefix = 0, None, None
    assert lib.diffus_render_forward(C.byref(a2), None) == -1                      # no frame and no prefix buffer
    assert lib.diffus_fan_directions(None, 0x1000, 1, 4, 0.5, 0x1000, None) == -1
    assert lib.diffus_fan_directions(0x1000, 0x1000, 0, 4, 0.5, 0x1000, None) == -2
    assert lib.diffus_fan_directions_backward(0x1000, 0x1000, 0x1000, 1, 4, 0.5, None, 0x1000, None) == -1
    assert lib.diffus_gather_probe(None, 1 << 20, 64, 256, 1, 0x1000, None) == -1
    assert lib.diffus_gather_probe(0x1000, 1 << 20, 60, 256, 1, 0x1000, None) == -2   # reads per thread: multiples of 8
    assert lib.diffus_mlp_backward_ex(0x1000, 0x1000, None, 0x1000, 64, 1.0, 0x1000, 0x1000, 1 << 20, 9, None) == -3
    assert lib.diffus_mlp_backward_ex(0x1000, 0x1000, None, 0x1000, 64, 1.0, 0x1000, 0x1000, 1 << 20, 2, None) == -3  # removed path
    assert lib.diffus_mlp_forward_ex(0x1000, 0x1000, None, 64, 1.0, 0.0, 0x1000, 2, None) == -3
    assert lib.diffus_mlp_backward_ex(0x1000, 0x1000, None, 0x1000, 64, 1.0, 0x1000, 0x1000, 16, 3, None) == -4   # piecewise path: workspace too small
    assert lib.diffus_mlp_input_grad(0x1000, None, None, 0x1000, 64, 1.0, 0x1000, None) == -1
    assert lib.diffus_conv1d_rows_forward(0x1000, 4, 60, None, 9, 4, 0x1000, None) == -1
    assert lib.diffus_conv1d_rows_forward(0x1000, 4, 60, 0x1000, 200, 100, 0x1000, None) == -5
    assert lib.diffus_conv1d_rows_backward(0x1000, 4, 3, 0x1000, 9, 0, 0x1000, None) == -2
    assert lib.diffus_mlp_input_grad(0x1000, 0x1000, None, 0x1000, 0, 1.0, 0x1000, None) == -2


def test_library_is_sm100a_native(lib):
    """The shipped binary carries sm_100a SASS (no PTX-JIT fallback needed on the B200 box)."""
    import shutil
    import subprocess
    from diffus_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
