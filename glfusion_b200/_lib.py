"""ctypes binding of libglf_sm100a.so (include/glfusion.h).  There is no fallback: if the library is missing or a
call fails, the caller gets an exception."""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libglf_sm100a.so")

MODE_DOT, MODE_EMBEDDED, MODE_GAUSSIAN = 0, 1, 2
DTYPE_BF16, DTYPE_F32, DTYPE_F16 = 0, 1, 2
LAYOUT_NCTHW, LAYOUT_TOKEN = 0, 1
PRECISION_BF16, PRECISION_F32X3 = 0, 1
PRECISIONS = {"bf16": PRECISION_BF16, "fp32": PRECISION_F32X3}
PARAMS_F32, PARAMS_BF16, PARAMS_F16 = 0, 1, 2      # glf_desc.reserved[3]: dtype of the parameter tensors

EXPORTS = ("glf_version", "glf_last_error", "glf_tpavi_sizes", "glf_tpavi_fwd", "glf_tpavi_bwd",
           "glf_gate_concat_fwd", "glf_gate_concat_bwd", "glf_gate_concat_cl_fwd", "glf_gate_concat_cl_bwd",
           "glf_views_to_tokens", "glf_gemm_bf16", "glf_transpose", "glf_bn_res_ln_fwd",
           "glf_bn_res_ln_bwd", "glf_bn_res_ln_bwd_max_blocks", "glf_gate_concat_bwd_scratch_bytes",
           "glf_fusion_ln_supported", "glf_fusion_ln_fwd", "glf_fusion_ln_fwd_parts", "glf_fusion_ln_bwd", "glf_fusion_ln_bwd_views",
           "glf_fusion_ln_bwd_views_supported",
           "glf_bn_res_ln_pair_fwd",
           "glf_bn_res_ln_pair_bwd", "glf_gemm_bf16_ex", "glf_gram_contraction", "glf_p2p_signal_bytes", "glf_p2p_max_floats",
           "glf_p2p_export", "glf_p2p_open", "glf_p2p_close", "glf_p2p_allreduce", "glf_spatial_sums",
           "glf_cycle_loss_scratch_bytes", "glf_cycle_loss", "glf_attention_scratch_bytes", "glf_attention_fwd",
           "glf_attention_bwd", "glf_attention_gaussian_scratch_bytes", "glf_attention_gaussian_fwd",
           "glf_attention_gaussian_bwd")


class GlfDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "T", "H", "W", "C", "Ci", "mode", "io_dtype", "x_layout", "dz_layout",
                                         "precision", "training", "bn_layer", "accumulate")] + \
               [("eps_bn", C.c_float), ("eps_ln", C.c_float), ("momentum", C.c_float), ("reserved", C.c_int32 * 4)]


class GlfWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "wz_w", "wz_b",
                                          "bn_w", "bn_b", "bn_running_mean", "bn_running_var",
                                          "bn_num_batches_tracked", "ln_w", "ln_b")]


class GlfGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "wz_w", "wz_b",
                                          "bn_w", "bn_b", "ln_w", "ln_b")]


class GlfSizes(C.Structure):
    _fields_ = [("saved_bytes", C.c_size_t), ("ws_fwd_bytes", C.c_size_t), ("ws_bwd_bytes", C.c_size_t)]


class GlfError(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None


def load() -> C.CDLL:
    """Load the shared library (building it is `python -m glfusion_b200.build`); raises if it is absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise GlfError(f"{LIB_PATH} not found: build it with `python -m glfusion_b200.build` "
                           "(nvcc, sm_100a). glfusion_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.glf_version.restype = C.c_int
        lib.glf_last_error.restype = C.c_char_p
        vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
        lib.glf_tpavi_sizes.argtypes = [C.POINTER(GlfDesc), C.POINTER(GlfSizes)]
        lib.glf_tpavi_fwd.argtypes = [C.POINTER(GlfDesc), vp, C.POINTER(GlfWeights), vp, vp, vp, vp]
        lib.glf_tpavi_bwd.argtypes = [C.POINTER(GlfDesc), vp, vp, C.POINTER(GlfWeights), vp, vp, C.POINTER(GlfGrads),
                                      vp, vp]
        lib.glf_fusion_ln_supported.argtypes = [C.POINTER(GlfDesc)]
        lib.glf_fusion_ln_fwd.argtypes = [C.POINTER(GlfDesc), vp, vp, C.POINTER(GlfWeights), C.POINTER(GlfWeights), vp,
                                          vp, vp, vp]
        lib.glf_fusion_ln_fwd_parts.argtypes = [C.POINTER(GlfDesc), vp, vp, C.POINTER(GlfWeights), C.POINTER(GlfWeights),
                                                vp, vp, vp, vp, vp]
        lib.glf_fusion_ln_bwd.argtypes = [C.POINTER(GlfDesc), vp, vp, vp, C.POINTER(GlfWeights), C.POINTER(GlfWeights),
                                          vp, vp, vp, vp, vp]
        pp = C.POINTER(C.c_void_p)
        lib.glf_fusion_ln_bwd_views.argtypes = [C.POINTER(GlfDesc), vp, pp, vp, vp, vp, C.POINTER(GlfWeights),
                                                C.POINTER(GlfWeights), vp, vp, vp, vp, vp]
        lib.glf_fusion_ln_bwd_views_supported.argtypes = [C.POINTER(GlfDesc)]
        lib.glf_bn_res_ln_pair_fwd.argtypes = [i64, i32, pp, pp, pp, pp, pp, pp, vp, pp, pp, f32, i32, vp]
        lib.glf_bn_res_ln_pair_bwd.argtypes = [i64, i32, vp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp, pp,
                                               C.POINTER(C.c_int), vp]
        lib.glf_gate_concat_fwd.argtypes = [i32] * 6 + [f32, i32, i32, pp, pp, pp, vp, vp, vp, vp]
        lib.glf_gate_concat_bwd.argtypes = [i32] * 6 + [f32, i32, i32, pp, pp, pp, vp, vp, vp, pp, pp, pp, vp, vp]
        lib.glf_gate_concat_bwd_scratch_bytes.argtypes = [i32] * 5
        lib.glf_gate_concat_bwd_scratch_bytes.restype = C.c_size_t
        lib.glf_gemm_bf16.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, vp, f32,
                                      vp, i64, i64, i32, i32, vp, vp]
        lib.glf_gemm_bf16_ex.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, vp, i64,
                                         f32, i32, i32, vp, vp]
        lib.glf_gram_contraction.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
        lib.glf_p2p_signal_bytes.argtypes = [i32]
        lib.glf_p2p_signal_bytes.restype = C.c_size_t
        lib.glf_p2p_max_floats.argtypes = []
        lib.glf_p2p_max_floats.restype = C.c_int64
        lib.glf_p2p_export.argtypes = [vp, C.c_char_p, C.POINTER(C.c_uint64)]
        lib.glf_p2p_open.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p)]
        lib.glf_p2p_close.argtypes = [vp, C.c_uint64]
        lib.glf_p2p_allreduce.argtypes = [pp, pp, i32, i32, i64, f32, vp]
        lib.glf_transpose.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp]
        lib.glf_spatial_sums.argtypes = [vp, i32, i32, i32, i32, i64, i64, i64, vp, vp]
        lib.glf_cycle_loss_scratch_bytes.argtypes = [i32, i32, i32]
        lib.glf_cycle_loss_scratch_bytes.restype = C.c_size_t
        lib.glf_cycle_loss.argtypes = [vp, i32, i32, i32, i32, i32, f32, i32, i32, i32, i32, f32, vp, vp, vp, vp]
        lib.glf_gate_concat_cl_fwd.argtypes = [i32, i32, i32, i32, i32, i32, f32, i32, pp, vp, vp, pp, pp, vp, vp, vp, vp]
        lib.glf_gate_concat_cl_bwd.argtypes = [i32, i32, i32, i32, i32, i32, f32, i32, pp, vp, vp, pp, pp, vp, vp, vp, pp, vp,
                                               vp, pp, pp, vp, vp]
        lib.glf_views_to_tokens.argtypes = [i32, i32, i32, i32, i32, pp, vp, vp, vp, vp, vp]
        lib.glf_bn_res_ln_fwd.argtypes = [i64, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, f32, i32, vp]
        lib.glf_bn_res_ln_bwd.argtypes = [i64, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                          C.POINTER(C.c_int), vp]
        lib.glf_bn_res_ln_bwd_max_blocks.argtypes = []
        lib.glf_attention_scratch_bytes.argtypes = [i32, i32, i32, i32]
        lib.glf_attention_scratch_bytes.restype = C.c_size_t
        lib.glf_attention_fwd.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
        lib.glf_attention_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp]
        lib.glf_attention_gaussian_scratch_bytes.argtypes = [i32, i32, i32, i32, i32]
        lib.glf_attention_gaussian_scratch_bytes.restype = C.c_size_t
        lib.glf_attention_gaussian_fwd.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
        lib.glf_attention_gaussian_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
        for name in EXPORTS:
            fn = getattr(lib, name)
            if name not in ("glf_last_error", "glf_gate_concat_bwd_scratch_bytes", "glf_p2p_signal_bytes",
                            "glf_p2p_max_floats", "glf_attention_scratch_bytes",
                            "glf_attention_gaussian_scratch_bytes"):
                fn.restype = C.c_int
        _lib = lib
        return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().glf_last_error()
        raise GlfError(f"libglf_sm100a error {rc}: {msg.decode() if msg else '?'}")


def ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr() if t is not None else None)


def ptr_table(tensors):
    arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr
