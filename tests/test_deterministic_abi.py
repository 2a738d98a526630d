"""GLF_DETERMINISTIC (glf_desc.reserved[1] | 0x100) on the host side: which descriptors accept it, which bits are
refused, and the workspace it adds.  The slab space is the witness that a shape really takes a split path: it appears
exactly where a product sums partials of several K slices or batch entries, and nowhere else."""
import ctypes as C

import pytest

import glfusion_b200
from glfusion_b200 import _lib as L

DET = L.DETERMINISTIC


def _desc(**kw):
    d = L.GlfDesc()
    d.B, d.T, d.H, d.W, d.C, d.Ci = 2, 4, 28, 28, 256, 128
    d.mode, d.io_dtype, d.x_layout, d.dz_layout = L.MODE_DOT, L.DTYPE_BF16, L.LAYOUT_TOKEN, L.LAYOUT_TOKEN
    d.training, d.bn_layer = 1, 1
    d.eps_bn = d.eps_ln = 1e-5
    d.momentum = 0.1
    d.reserved[1] = kw.pop("algo", 0) | (DET if kw.pop("det", False) else 0)
    d.reserved[0] = kw.pop("defer_ln", 0)
    d.reserved[3] = kw.pop("params", L.PARAMS_F32)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _sizes(**kw):
    s = L.GlfSizes()
    rc = glfusion_b200.load_library().glf_tpavi_sizes(C.byref(_desc(**kw)), C.byref(s))
    assert rc == 0, glfusion_b200.load_library().glf_last_error().decode()
    return s.saved_bytes, s.ws_fwd_bytes, s.ws_bwd_bytes


# the shapes tests/test_gpu_deterministic.py runs: each takes a split path, so the flag adds slab space to ws_bwd
SPLIT_SHAPES = {
    "dot_token_c256_b16": dict(B=16, algo=1),
    "dot_gram_b4": dict(B=4, algo=2),
    "dot_gram_b2_t16": dict(B=2, T=16, algo=2),
    "embedded_c256": dict(mode=L.MODE_EMBEDDED),
    "embedded_c192": dict(mode=L.MODE_EMBEDDED, C=192, Ci=96, T=2, H=14, W=14),
    "gaussian_c128": dict(mode=L.MODE_GAUSSIAN, C=128, Ci=64, T=2, H=14, W=14),
    "gaussian_c256": dict(mode=L.MODE_GAUSSIAN, T=2, H=14, W=14),
    "width2048": dict(C=2048, Ci=1024, T=3, H=28, W=28),
    "f32x3": dict(C=128, Ci=64, T=2, H=14, W=14, algo=1, precision=L.PRECISION_F32X3, io_dtype=L.DTYPE_F32),
    "half_params": dict(B=16, algo=1, params=L.PARAMS_F16),
    "fusion_pair": dict(B=2, T=4, H=14, W=14, defer_ln=1, algo=1),
}


@pytest.mark.parametrize("name", sorted(SPLIT_SHAPES))
def test_flag_is_accepted_and_adds_slabs_only_to_workspace(name):
    kw = SPLIT_SHAPES[name]
    off, on = _sizes(**kw), _sizes(det=True, **kw)
    assert on[0] == off[0], "the saved blob does not depend on the flag"
    assert on[1] >= off[1]
    assert on[2] > off[2], "a split path of the backward must get slab space"
    assert on[2] % 256 == 0 and on[1] % 256 == 0


@pytest.mark.parametrize("algo", [0, 1, 2])
def test_flag_is_accepted_with_every_dot_algorithm(algo):
    off, on = _sizes(algo=algo), _sizes(algo=algo, det=True)
    assert on[0] == off[0]


def test_no_split_no_slab():
    """The Gram form at 128 sequences (the benchmark's configuration) writes every output once: no slab, same sizes."""
    kw = dict(B=128, algo=2)
    assert _sizes(det=True, **kw) == _sizes(**kw)


def test_flag_off_sizes_do_not_depend_on_the_flag_bit_position():
    for kw in SPLIT_SHAPES.values():
        d = _desc(**dict(kw))
        s1, s2 = L.GlfSizes(), L.GlfSizes()
        lib = glfusion_b200.load_library()
        assert lib.glf_tpavi_sizes(C.byref(d), C.byref(s1)) == 0
        d.reserved[1] = d.reserved[1] & 0xFF
        assert lib.glf_tpavi_sizes(C.byref(d), C.byref(s2)) == 0
        assert (s1.saved_bytes, s1.ws_fwd_bytes, s1.ws_bwd_bytes) == (s2.saved_bytes, s2.ws_fwd_bytes, s2.ws_bwd_bytes)


def test_wide_split_slabs_are_sized_for_every_k_slice():
    """dWcat at C = 2048 is 3 * 1024 x 2048 fp32 (25 MB) per K slice; the 3-view shape picks three slices."""
    off, on = _sizes(**SPLIT_SHAPES["width2048"]), _sizes(det=True, **SPLIT_SHAPES["width2048"])
    assert on[2] - off[2] >= 3 * 3 * 1024 * 2048 * 4


@pytest.mark.parametrize("value", [DET | 3, 0x200, 0x200 | 1, DET | 0x200, 0x10000 | 2, -1, 3])
def test_stray_bits_are_refused_with_a_message(value):
    lib = glfusion_b200.load_library()
    d = _desc()
    d.reserved[1] = value
    s = L.GlfSizes()
    rc = lib.glf_tpavi_sizes(C.byref(d), C.byref(s))
    assert rc < 0
    msg = lib.glf_last_error().decode()
    assert "reserved[1]" in msg and "GLF_DETERMINISTIC" in msg


def test_fused_layernorm_pair_accepts_and_ignores_the_flag():
    lib = glfusion_b200.load_library()
    kw = dict(defer_ln=1, algo=1)
    assert lib.glf_fusion_ln_supported(C.byref(_desc(**kw))) == 1
    assert lib.glf_fusion_ln_supported(C.byref(_desc(det=True, **kw))) == 1
    assert lib.glf_fusion_ln_bwd_views_supported(C.byref(_desc(det=True, **kw))) == \
        lib.glf_fusion_ln_bwd_views_supported(C.byref(_desc(**kw)))


def test_state_reads_the_torch_switch():
    """TPAVIState sets the bit from torch.are_deterministic_algorithms_enabled(), and backward re-reads it."""
    import torch
    from glfusion_b200.tpavi import TPAVIState
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        args = (16, 256, 4, 28, 28, 128, L.MODE_DOT, L.DTYPE_BF16, L.LAYOUT_TOKEN, True, True)
        torch.use_deterministic_algorithms(False)
        st_off = TPAVIState(*args)
        assert st_off.desc.reserved[1] & DET == 0
        torch.use_deterministic_algorithms(True, warn_only=True)
        st_on = TPAVIState(*args)
        assert st_on.desc.reserved[1] & DET == DET
        assert st_on.sizes.ws_bwd_bytes >= st_off.sizes.ws_bwd_bytes
        torch.use_deterministic_algorithms(False)
        st_on.refresh_deterministic()
        assert st_on.desc.reserved[1] & DET == 0
        assert st_on.sizes.ws_bwd_bytes == st_off.sizes.ws_bwd_bytes
        assert st_on.desc.reserved[1] & 0xFF == st_off.desc.reserved[1] & 0xFF
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)
