"""Host-side behaviour of mode='gaussian' (f = x x^T on the block input itself, ours.py:869-873): the descriptor is
accepted with the bf16 arm and refused with the fp32-exact arm and the Gram form, the blob sizes reflect that only the
g projection is kept, the standalone attention entry points size their scratch and refuse bad arguments, and
TPAVIModule(mode='gaussian') is the reference's parameter container.  No compute calls here."""
import ctypes as C

import pytest
import torch

import glfusion_b200
from glfusion_b200 import _lib as L
from glfusion_b200 import TPAVIModule
from glfusion_b200.tpavi import TPAVIState

FAKE = C.c_void_p(1 << 20)       # a 256-byte aligned non-NULL address; never dereferenced (refused before any launch)


def _desc(**kw):
    d = L.GlfDesc()
    d.B, d.T, d.H, d.W, d.C, d.Ci = 2, 4, 28, 28, 256, 128
    d.mode, d.io_dtype, d.x_layout, d.dz_layout = L.MODE_GAUSSIAN, L.DTYPE_BF16, L.LAYOUT_TOKEN, L.LAYOUT_TOKEN
    d.training, d.bn_layer = 1, 1
    d.eps_bn = d.eps_ln = 1e-5
    d.momentum = 0.1
    d.reserved[1] = kw.pop("algo", 0)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _sizes(**kw):
    lib = glfusion_b200.load_library()
    s = L.GlfSizes()
    rc = lib.glf_tpavi_sizes(C.byref(_desc(**kw)), C.byref(s))
    return rc, s


@pytest.mark.parametrize("kw", [dict(), dict(io_dtype=L.DTYPE_F32), dict(io_dtype=L.DTYPE_F16),
                                dict(x_layout=L.LAYOUT_NCTHW), dict(C=2048, Ci=1024), dict(C=128, Ci=64),
                                dict(bn_layer=0), dict(training=0)])
def test_sizes_succeed(kw):
    rc, s = _sizes(**kw)
    assert rc == 0, glfusion_b200.load_library().glf_last_error()
    assert s.saved_bytes > 0 and s.saved_bytes % 256 == 0 and s.ws_fwd_bytes % 256 == 0 and s.ws_bwd_bytes % 256 == 0


def test_half_parameters_and_deferred_layernorm_are_accepted():
    lib = glfusion_b200.load_library()
    for pdt in (L.PARAMS_BF16, L.PARAMS_F16):
        d = _desc()
        d.reserved[3] = pdt
        assert lib.glf_tpavi_sizes(C.byref(d), C.byref(L.GlfSizes())) == 0
    d = _desc()
    d.reserved[0] = 1
    assert lib.glf_fusion_ln_supported(C.byref(d)) == 1


def test_saved_blob_keeps_g_alone():
    """gaussian keeps G [rows, C'] where embedded keeps [Theta | Phi | G] [rows, 3C']; its backward scratch holds
    [dS X | dS^T X | dG] [rows, 2C + C'] instead of [rows, 3C']."""
    rows, C_, Ci = 2 * 4 * 28 * 28, 256, 128
    rc, sg = _sizes()
    assert rc == 0
    rc, se = _sizes(mode=L.MODE_EMBEDDED)
    assert rc == 0
    # P: 2 C' fewer bf16 columns per token; the weight copy [C, 2C + C'] is C (2C - 2C') larger than [C, 3C']
    assert se.saved_bytes - sg.saved_bytes >= rows * 2 * Ci * 2 - C_ * (2 * C_ - 2 * Ci) * 2 - 4096
    assert sg.ws_bwd_bytes - se.ws_bwd_bytes >= rows * (2 * C_ + Ci - 3 * Ci) * 2 - 4096


@pytest.mark.parametrize("kw,frag", [
    (dict(precision=L.PRECISION_F32X3, io_dtype=L.DTYPE_F32), "F32X3"),
    (dict(algo=2), "Gram form"),
    (dict(mode=3), "mode"),
])
def test_unsupported_combinations_are_errors_with_messages(kw, frag):
    lib = glfusion_b200.load_library()
    rc, _ = _sizes(**kw)
    assert rc < 0
    assert frag.lower() in lib.glf_last_error().decode().lower()
    with pytest.raises(L.GlfError):
        L.check(rc)


def test_fp32_precision_is_refused_before_any_launch():
    with pytest.raises(L.GlfError, match="F32X3"):
        TPAVIState(2, 128, 2, 4, 4, 64, L.MODE_GAUSSIAN, L.DTYPE_F32, L.LAYOUT_TOKEN, True, True,
                   precision=L.PRECISION_F32X3)


def test_state_dict_matches_the_reference_container():
    C_ = 256
    g = TPAVIModule(in_channels=C_, mode='gaussian')
    d = TPAVIModule(in_channels=C_, mode='dot')
    assert g.inter_channels == C_ // 2
    assert {k: tuple(v.shape) for k, v in g.state_dict().items()} == {k: tuple(v.shape) for k, v in d.state_dict().items()}
    assert list(g.state_dict().keys()) == list(d.state_dict().keys())
    assert "theta.weight" in g.state_dict() and "phi.bias" in g.state_dict()


@pytest.mark.parametrize("C_,bn", [(128, True), (96, False)])
def test_same_seed_draws_the_same_weights_as_dot(C_, bn):
    """Same holders created in the same order: the constructor consumes the RNG stream exactly as mode='dot' does."""
    torch.manual_seed(11)
    g = TPAVIModule(C_, mode='gaussian', bn_layer=bn)
    after_g = torch.rand(4)
    torch.manual_seed(11)
    d = TPAVIModule(C_, mode='dot', bn_layer=bn)
    after_d = torch.rand(4)
    sg, sd = g.state_dict(), d.state_dict()
    for k in sd:
        assert torch.equal(sg[k], sd[k]), k
    assert torch.equal(after_g, after_d)


def test_other_modes_unchanged():
    with pytest.raises(NotImplementedError):
        TPAVIModule(64, mode='concatenate')
    with pytest.raises(NotImplementedError):
        TPAVIModule(64, mode='gaussian', dimension=2)
    assert TPAVIModule(64, mode='gaussian')._mode_id == L.MODE_GAUSSIAN
    assert TPAVIModule(64, mode='embedded')._mode_id == L.MODE_EMBEDDED
    assert TPAVIModule(64)._mode_id == L.MODE_DOT


def test_gaussian_fusion_module_builds():
    f = glfusion_b200.GlobalLocalFusion(128, mode='gaussian')
    assert f.global_attn._mode_id == f.local_attn._mode_id == L.MODE_GAUSSIAN


# ---- standalone entry points (glf_attention_gaussian_*) -----------------------------------------------------------

def _ld(N):
    return (N + 7) & ~7


@pytest.mark.parametrize("N,C_,Ci", [(3136, 256, 128), (1000, 96, 48), (64, 128, 64)])
def test_scratch_bytes(N, C_, Ci):
    lib = glfusion_b200.load_library()
    for B in (1, 2, 5):
        f = lib.glf_attention_gaussian_scratch_bytes(B, N, C_, Ci, 0)
        b = lib.glf_attention_gaussian_scratch_bytes(B, N, C_, Ci, 1)
        assert f > 0 and f % 256 == 0 and b % 256 == 0
        # the backward also holds the [B N, 2C] pair dS X | dS^T X and the score scratch of the chunked path
        assert b >= f + B * N * 2 * C_ * 2
        assert b >= lib.glf_attention_scratch_bytes(B, N, Ci, 1) + B * N * 2 * C_ * 2


def _refusal(fn, *args):
    lib = glfusion_b200.load_library()
    rc = getattr(lib, fn)(*args)
    assert rc < 0
    with pytest.raises(L.GlfError):
        L.check(rc)
    return lib.glf_last_error().decode()


@pytest.mark.parametrize("B,N,C_,Ci,frag", [
    (2, 64, 128, 36, "positive multiple of 8, at most 2048 (got 36)"),
    (2, 64, 100, 64, "positive multiple of 8, at most 2048 (got 100)"),
    (2, 64, 4096, 64, "positive multiple of 8, at most 2048 (got 4096)"),
    (2, 0, 128, 64, "empty input"),
    (0, 64, 128, 64, "empty input"),
])
def test_bad_shapes_are_refused(B, N, C_, Ci, frag):
    lib = glfusion_b200.load_library()
    assert lib.glf_attention_gaussian_scratch_bytes(B, N, C_, Ci, 1) == 0
    assert frag in _refusal("glf_attention_gaussian_fwd", FAKE, FAKE, FAKE, FAKE, B, N, C_, Ci, FAKE, None)
    assert frag in _refusal("glf_attention_gaussian_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, B, N, C_, Ci,
                            FAKE, None)


def test_null_and_misaligned_pointers_are_refused():
    assert "X is NULL" in _refusal("glf_attention_gaussian_fwd", None, FAKE, FAKE, FAKE, 2, 64, 128, 64, FAKE, None)
    assert "G is NULL" in _refusal("glf_attention_gaussian_bwd", FAKE, None, FAKE, FAKE, FAKE, FAKE, FAKE, None, 2, 64,
                                   128, 64, FAKE, None)
    assert "dX is NULL" in _refusal("glf_attention_gaussian_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, None, FAKE, None, 2, 64,
                                    128, 64, FAKE, None)
    assert "scratch is NULL" in _refusal("glf_attention_gaussian_fwd", FAKE, FAKE, FAKE, FAKE, 2, 64, 128, 64, None,
                                         None)
    assert "256-byte aligned" in _refusal("glf_attention_gaussian_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, 2,
                                          64, 128, 64, C.c_void_p((1 << 20) + 16), None)
    assert "16-byte aligned" in _refusal("glf_attention_gaussian_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, FAKE,
                                         C.c_void_p((1 << 20) + 4), None, 2, 64, 128, 64, FAKE, None)
