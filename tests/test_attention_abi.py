"""Host-side behaviour of the standalone softmax-attention entry points (glf_attention_*): scratch sizing follows the
chunk rule of the materialised path, and bad arguments are refused, with a message naming the fault, before any device
work.  No compute calls here."""
import ctypes as C

import pytest

import glfusion_b200
from glfusion_b200 import _lib as L

FAKE = C.c_void_p(1 << 20)       # a 256-byte aligned non-NULL address; never dereferenced (refused before any launch)


def _ld(N):
    return (N + 7) & ~7


def _chunk(N):
    """Sequences per chunk of the materialised path: the backward's 12 bytes per score stay under 2 GiB."""
    return max(1, (2 << 30) // (12 * _ld(N) * N))


@pytest.mark.parametrize("N,Ci", [(3136, 96), (1000, 48), (3136, 128), (72, 32)])
def test_scratch_follows_the_chunk_rule(N, Ci):
    lib = glfusion_b200.load_library()
    chunk = _chunk(N)
    per_seq_bwd = 12 * _ld(N) * N
    Bs = sorted(set(range(1, min(chunk, 40) + 1)) | {chunk, chunk + 1, chunk + 2, 2 * chunk + 3})
    fwd = [lib.glf_attention_scratch_bytes(B, N, Ci, 0) for B in Bs]
    bwd = [lib.glf_attention_scratch_bytes(B, N, Ci, 1) for B in Bs]
    for f, b in zip(fwd, bwd):
        assert f > 0 and f % 256 == 0 and b % 256 == 0 and b > f
    for i in range(1, len(Bs)):
        assert fwd[i] >= fwd[i - 1] and bwd[i] >= bwd[i - 1]          # monotone in B
        if Bs[i] <= chunk:                                            # every sequence of a chunk has its score tile
            assert fwd[i] - fwd[i - 1] >= 6 * _ld(N) * N * (Bs[i] - Bs[i - 1]) - 256
            assert bwd[i] - bwd[i - 1] >= per_seq_bwd * (Bs[i] - Bs[i - 1]) - 256
        elif Bs[i - 1] >= chunk:                                      # saturated: only per-token bookkeeping grows
            assert fwd[i] == fwd[i - 1]
            assert bwd[i] - bwd[i - 1] < per_seq_bwd // 4 * (Bs[i] - Bs[i - 1])
    if (N, Ci) == (3136, 96):
        assert chunk == 18                                            # B = 20 runs as chunks of 18 + 2 sequences
        b20 = lib.glf_attention_scratch_bytes(20, N, Ci, 1)
        assert 18 * per_seq_bwd <= b20 < 2.2e9


def _refusal(fn, *args):
    lib = glfusion_b200.load_library()
    rc = getattr(lib, fn)(*args)
    assert rc < 0
    with pytest.raises(L.GlfError):
        L.check(rc)
    return lib.glf_last_error().decode()


@pytest.mark.parametrize("B,N,Ci,frag", [
    (2, 64, 36, "Ci must be a positive multiple of 8, at most 2048 (got 36)"),
    (2, 64, 0, "Ci must be a positive multiple of 8, at most 2048 (got 0)"),
    (2, 64, 2056, "Ci must be a positive multiple of 8, at most 2048 (got 2056)"),
    (2, 0, 64, "empty input"),
    (0, 64, 64, "empty input"),
])
def test_bad_shapes_are_refused(B, N, Ci, frag):
    lib = glfusion_b200.load_library()
    assert lib.glf_attention_scratch_bytes(B, N, Ci, 1) == 0
    assert frag in lib.glf_last_error().decode()
    assert frag in _refusal("glf_attention_fwd", FAKE, FAKE, FAKE, B, N, Ci, FAKE, None)
    assert frag in _refusal("glf_attention_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, B, N, Ci, FAKE, None)


def test_null_and_misaligned_pointers_are_refused():
    assert "P3 is NULL" in _refusal("glf_attention_fwd", None, FAKE, FAKE, 2, 64, 64, FAKE, None)
    assert "P3 is NULL" in _refusal("glf_attention_bwd", None, FAKE, FAKE, FAKE, FAKE, FAKE, 2, 64, 64, FAKE, None)
    assert "lse is NULL" in _refusal("glf_attention_fwd", FAKE, FAKE, None, 2, 64, 64, FAKE, None)
    assert "dY is NULL" in _refusal("glf_attention_bwd", FAKE, FAKE, None, FAKE, FAKE, None, 2, 64, 64, FAKE, None)
    assert "scratch is NULL" in _refusal("glf_attention_fwd", FAKE, FAKE, FAKE, 2, 64, 64, None, None)
    assert "256-byte aligned" in _refusal("glf_attention_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, None, 2, 64, 64,
                                          C.c_void_p((1 << 20) + 16), None)
    assert "16-byte aligned" in _refusal("glf_attention_bwd", FAKE, FAKE, FAKE, FAKE, FAKE, C.c_void_p((1 << 20) + 4),
                                         2, 64, 64, FAKE, None)
