"""glf_desc.reserved[3] (GLF_PARAMS_*) at the C ABI, host-only: the parameter dtype sizes an fp32 parameter copy into
`saved` and an fp32 gradient staging area into ws_bwd, is validated, and is refused by the fp32-exact arm.  No compute
calls here."""
import ctypes as C

import pytest

import glfusion_b200
from glfusion_b200 import _lib as L

C_, CI = 256, 128
PARAM_FLOATS = 4 * C_ * CI + 3 * CI + 5 * C_       # the twelve tensors of glf_grads


def _sizes(**kw):
    d = L.GlfDesc()
    d.B, d.T, d.H, d.W, d.C, d.Ci = 2, 4, 28, 28, C_, CI
    d.mode, d.io_dtype, d.x_layout, d.dz_layout = L.MODE_DOT, L.DTYPE_BF16, L.LAYOUT_TOKEN, L.LAYOUT_TOKEN
    d.training, d.bn_layer = 1, 1
    d.eps_bn = d.eps_ln = 1e-5
    d.momentum = 0.1
    for k, v in kw.pop("reserved", {}).items():
        d.reserved[k] = v
    for k, v in kw.items():
        setattr(d, k, v)
    s = L.GlfSizes()
    rc = glfusion_b200.load_library().glf_tpavi_sizes(C.byref(d), C.byref(s))
    return rc, s


def test_param_dtype_codes():
    assert (L.PARAMS_F32, L.PARAMS_BF16, L.PARAMS_F16) == (0, 1, 2)


@pytest.mark.parametrize("algo", [1, 2])
@pytest.mark.parametrize("code", [L.PARAMS_BF16, L.PARAMS_F16])
def test_half_params_grow_saved_and_ws_bwd(algo, code):
    rc_f, sf = _sizes(reserved={1: algo})
    rc_h, sh = _sizes(reserved={1: algo, 3: code})
    assert rc_f == rc_h == 0
    assert sh.saved_bytes >= sf.saved_bytes + 4 * PARAM_FLOATS          # fp32 copy of the parameters, kept for backward
    assert sh.ws_fwd_bytes >= sf.ws_fwd_bytes + 4 * PARAM_FLOATS        # ... and in the no-`saved` fallback
    assert sh.ws_bwd_bytes >= sf.ws_bwd_bytes + 4 * PARAM_FLOATS        # fp32 gradients before rounding
    assert sh.saved_bytes < sf.saved_bytes + 4 * PARAM_FLOATS + 12 * 256


@pytest.mark.parametrize("code", [3, -1, 7])
def test_unknown_param_dtype_fails(code):
    rc, _ = _sizes(reserved={3: code})
    assert rc < 0
    assert "reserved[3]" in glfusion_b200.load_library().glf_last_error().decode()


def test_f32x3_with_half_params_is_refused():
    rc, _ = _sizes(io_dtype=L.DTYPE_F32, precision=L.PRECISION_F32X3, reserved={3: L.PARAMS_BF16})
    assert rc < 0
    assert "fp32 parameters" in glfusion_b200.load_library().glf_last_error().decode()
    assert _sizes(io_dtype=L.DTYPE_F32, precision=L.PRECISION_F32X3)[0] == 0
