"""GLF_DTYPE_F16 at the C ABI, host-only: fp16 is an I/O dtype of glf_desc, sized like fp32 input (a packed bf16 copy
of x is kept for backward), and refused by the fp32-exact arm.  No compute calls here."""
import ctypes as C

import pytest

import glfusion_b200
from glfusion_b200 import _lib as L


def _desc(**kw):
    d = L.GlfDesc()
    d.B, d.T, d.H, d.W, d.C, d.Ci = 2, 4, 28, 28, 256, 128
    d.mode, d.io_dtype, d.x_layout, d.dz_layout = L.MODE_DOT, L.DTYPE_BF16, L.LAYOUT_TOKEN, L.LAYOUT_TOKEN
    d.training, d.bn_layer = 1, 1
    d.eps_bn = d.eps_ln = 1e-5
    d.momentum = 0.1
    d.reserved[1] = 1
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _sizes(**kw):
    lib = glfusion_b200.load_library()
    s = L.GlfSizes()
    rc = lib.glf_tpavi_sizes(C.byref(_desc(**kw)), C.byref(s))
    return rc, s


def test_f16_enum_value():
    assert L.DTYPE_F16 == 2
    assert glfusion_b200.load_library().glf_version() == 100


@pytest.mark.parametrize("layout", [L.LAYOUT_TOKEN, L.LAYOUT_NCTHW])
def test_f16_sizes_keep_a_packed_bf16_copy_of_x(layout):
    rows = 2 * 4 * 28 * 28
    rc_b, sb = _sizes()
    rc_h, sh = _sizes(io_dtype=L.DTYPE_F16, x_layout=layout)
    rc_f, sf = _sizes(io_dtype=L.DTYPE_F32, x_layout=layout)
    assert rc_b == rc_h == rc_f == 0
    assert sh.saved_bytes >= sb.saved_bytes + rows * 256 * 2
    # the same blobs as fp32 input: x is converted to bf16 once, everything else is dtype independent
    assert (sh.saved_bytes, sh.ws_fwd_bytes, sh.ws_bwd_bytes) == (sf.saved_bytes, sf.ws_fwd_bytes, sf.ws_bwd_bytes)


def test_f32x3_with_f16_is_refused_naming_fp16():
    lib = glfusion_b200.load_library()
    rc, _ = _sizes(io_dtype=L.DTYPE_F16, precision=L.PRECISION_F32X3)
    assert rc < 0
    assert "fp16" in lib.glf_last_error().decode().lower()
    assert _sizes(io_dtype=L.DTYPE_F32, precision=L.PRECISION_F32X3)[0] == 0


@pytest.mark.parametrize("io", [3, 7, -1])
def test_unknown_io_dtype_still_fails(io):
    lib = glfusion_b200.load_library()
    rc, _ = _sizes(io_dtype=io)
    assert rc < 0
    assert "io_dtype" in lib.glf_last_error().decode().lower()


def test_fused_layernorm_z_dtype_field():
    """reserved[2] names the z / dz dtype of glf_fusion_ln_*: bf16 (0) or fp16; x_g / x_l stay bf16."""
    lib = glfusion_b200.load_library()
    kw = dict(reserved=(C.c_int32 * 4)(1, 1, 0, 0))
    assert lib.glf_fusion_ln_supported(C.byref(_desc(**kw))) == 1
    kw["reserved"][2] = L.DTYPE_F16
    assert lib.glf_fusion_ln_supported(C.byref(_desc(**kw))) == 1
    assert _sizes(**kw)[0] == 0
    kw["reserved"][2] = L.DTYPE_F32
    assert lib.glf_fusion_ln_supported(C.byref(_desc(**kw))) == 0
    rc, _ = _sizes(**kw)
    assert rc < 0 and "reserved[2]" in lib.glf_last_error().decode()
    # the blocks' own x stays bf16 token-major for the fused pass: fp16 x_g / x_l are not its input
    kw["reserved"][2] = L.DTYPE_F16
    assert lib.glf_fusion_ln_supported(C.byref(_desc(io_dtype=L.DTYPE_F16, **kw))) == 0
