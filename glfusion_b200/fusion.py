"""Fused global-local cross-view fusion: the hot-path section of ``Global_and_Local.forward``
(R/models/ours.py:1802-1837) as one autograd node.

    gate  a_v = sigmoid(w * max_c sigmoid(cls_v) * sigmoid(ctr_v))          ours.py:1802-1815
    X_g   = cat_v f4_v ,  X_l = cat_v f4_v * a_v                              ours.py:1816-1820, 1826-1827
    out_v = MGFM(X_g)[:, :, v] + MLFM(X_l)[:, :, v]                           ours.py:1821-1834

Inputs are what the reference has at that point: per-view backbone features ``f4[v]`` [B,C,h,w] (NCHW), the
classifier logits ``cls[v]`` [B,5,h,w] and the centerness logits ``ctr[v]`` [B,1,h,w] (both *before* the sigmoid).
One gate+concat kernel produces both token-major operands, the two TPAVI blocks run on them, and the second block's
LayerNorm epilogue accumulates into the first one's output (the `+` of ours.py:1834 costs no extra pass).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch
from torch import nn

from . import _lib as L
import threading

from .tpavi import (_IO_DTYPES, TPAVIModule, TPAVIState, _blob, _check_precision_dtype, _io_dtype, _stream_ptr,
                    _weights_struct, claim_grad_out, tpavi_backward_raw, tpavi_forward_raw)

_HALF = (torch.bfloat16, torch.float16)     # the 2-byte activation dtypes: 8 elements per 16 bytes


_SIDE_STREAMS = {}
_SIDE_LOCK = threading.Lock()      # nn.DataParallel drives one Python thread per GPU through this module


def _side_stream(device) -> "torch.cuda.Stream":
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    with _SIDE_LOCK:
        if key not in _SIDE_STREAMS:
            _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
        return _SIDE_STREAMS[key]


def _pair_ln_ok(mg, ml, shape, x, prec) -> bool:
    """True when the MGFM / MLFM LayerNorm stages can run as one fused pass (glf_fusion_ln_fwd / _bwd)."""
    if mg.inter_channels != ml.inter_channels or mg._mode_id != ml._mode_id or mg._bn_layer != ml._bn_layer:
        return False
    B, T, H, W, C_ = shape
    if mg._norm_config() != ml._norm_config():
        return False
    st = TPAVIState(B, C_, T, H, W, mg.inter_channels, mg._mode_id, _io_dtype(x), L.LAYOUT_TOKEN,
                    mg._norm_config()["training"], mg._bn_layer, precision=prec, defer_ln=True)
    return bool(L.load().glf_fusion_ln_supported(C.byref(st.desc)))


def _channels_last_rows(views: Sequence[torch.Tensor], x_dtype) -> Optional[tuple]:
    """(batch strides, token strides) when every [B,C,h,w] view is made of 16-byte aligned rows of C channels
    (channels_last tensors, or views of a token-major stack): the case the row kernels glf_gate_concat_cl_* take
    without any transposition (SURVEY.md section 8 f1).  None otherwise."""
    if x_dtype != torch.bfloat16 or len(views) > 8:
        return None
    dt = views[0].dtype
    if dt not in (torch.bfloat16, torch.float16, torch.float32):
        return None
    per16 = 8 if dt in _HALF else 4
    B, C_, h, w = views[0].shape
    if C_ % 8 or B * len(views) > 65535:
        return None
    sb, st = [], []
    for t in views:
        b_, c_, h_, w_ = t.stride()
        if (t.dtype != dt or tuple(t.shape) != (B, C_, h, w) or c_ != 1 or h_ != w * w_ or w_ < C_ or w_ % per16
                or b_ % per16 or t.data_ptr() % 16 or (B > 1 and b_ < 1)):
            return None
        sb.append(b_); st.append(w_)
    return sb, st


def _f32(t: torch.Tensor) -> torch.Tensor:
    """Contiguous fp32 logits, with no cast call when they already are (the fused node then makes no aten::to)."""
    return t if t.dtype == torch.float32 and t.is_contiguous() else t.float().contiguous()


def gate_concat_forward(f4: Sequence[torch.Tensor], cls: Sequence[torch.Tensor], ctr: Sequence[torch.Tensor],
                        weight: float, x_dtype=torch.bfloat16):
    lib = L.load()
    V = len(f4)
    B, C_, h, w = f4[0].shape
    dev = f4[0].device
    if not all(t.is_cuda for t in list(f4) + list(cls) + list(ctr)):
        raise L.GlfError("glfusion_b200 runs on CUDA (sm_100) tensors only; there is no CPU path")
    if any(t.dtype != f4[0].dtype for t in f4):
        # the kernels read every view with one element type: a mix would be misread, not converted
        raise TypeError(f"the f4 views must share one dtype, got {sorted({str(t.dtype) for t in f4})}")
    cls = [_f32(t) for t in cls]
    ctr = [_f32(t) for t in ctr]
    ncls = cls[0].shape[1]
    xg = torch.empty((B, V, h, w, C_), dtype=x_dtype, device=dev)
    xl = torch.empty_like(xg)
    gate = torch.empty((B, V, h, w), dtype=torch.float32, device=dev)
    rows = _channels_last_rows(f4, x_dtype)
    if rows is not None:
        # channels_last hand-off: the views are already rows of C channels, nothing is transposed
        f4 = list(f4)
        i64 = C.c_int64 * V
        with torch.cuda.device(dev):
            L.check(lib.glf_gate_concat_cl_fwd(B, C_, V, h, w, ncls, float(weight), _io_dtype(f4[0]), L.ptr_table(f4),
                                               i64(*rows[0]), i64(*rows[1]), L.ptr_table(cls), L.ptr_table(ctr),
                                               L.ptr(xg), L.ptr(xl), L.ptr(gate), _stream_ptr()))
        return xg, xl, gate, f4, cls, ctr
    f4 = [t.contiguous() for t in f4]
    with torch.cuda.device(dev):
        L.check(lib.glf_gate_concat_fwd(B, C_, V, h, w, ncls, float(weight), _io_dtype(f4[0]), _io_dtype(xg),
                                        L.ptr_table(f4),
                                        L.ptr_table(cls), L.ptr_table(ctr), L.ptr(xg), L.ptr(xl), L.ptr(gate),
                                        _stream_ptr()))
    return xg, xl, gate, f4, cls, ctr


_GATHER_DTYPES = (torch.bfloat16, torch.float32)


def views_to_tokens(views: Sequence[Optional[torch.Tensor]], out: torch.Tensor, dtypes=_GATHER_DTYPES) -> bool:
    """Gather per-view [B,C,h,w] tensors (NCHW or channels-last strides, of one of `dtypes`; None = zeros) into the
    token-major bf16 buffer `out` [B,V,h,w,C] with one kernel (glf_views_to_tokens) — the inverse of handing the
    dict-keyed caller one [B,C,h,w] view per key.  Returns False, having done nothing, when the kernel does not cover
    the case (other dtypes / strides); the caller then copies view by view.  The kernel also reads float16; the fused
    backward asks for it with dtypes=(torch.bfloat16, torch.float16, torch.float32)."""
    if out.dtype != torch.bfloat16 or not out.is_contiguous():
        return False
    B, V, h, w, Cn = out.shape
    live = [g for g in views if g is not None]
    if not live or Cn % 64 or V > 8 or B > 65535:
        return False
    dt = live[0].dtype
    if dt not in dtypes:
        return False
    sb, sc, st = [], [], []
    for g in views:
        if g is None:
            sb.append(0); sc.append(0); st.append(0)
            continue
        if g.dtype != dt or tuple(g.shape) != (B, Cn, h, w) or g.device != out.device:
            return False
        b_, c_, h_, w_ = g.stride()
        if h_ != w * w_ or (c_ != 1 and w_ != 1) or min(b_, c_) < 1 or w_ < 0:   # h*w must collapse; one unit stride
            return False                   # (w_ == 0: the broadcast gradient of a spatial sum, R/main.py:229)
        sb.append(b_); sc.append(c_); st.append(w_)
    ptrs = (C.c_void_p * V)(*[None if g is None else g.data_ptr() for g in views])
    i64 = C.c_int64 * V
    with torch.cuda.device(out.device):
        L.check(L.load().glf_views_to_tokens(B, Cn, V, h * w, _io_dtype(live[0]), ptrs, i64(*sb), i64(*sc), i64(*st), L.ptr(out),
                                             _stream_ptr()))
    return True


def _views_as_rows(grads, xg: torch.Tensor, st) -> Optional[tuple]:
    """The V per-view gradients as (tensors, batch strides) when the fused LayerNorm backward can read them in place
    (glf_fusion_ln_bwd_views): all present, one 2-byte dtype (bf16 or fp16), rows of C contiguous channels with
    contiguous tokens (channels_last or views of a token-major stack), 16-byte aligned, h*w a multiple of the pass's row
    tile.  None otherwise: the caller gathers them into one token-major buffer first."""
    B, V, h, w, Cn = xg.shape
    if any(g is None for g in grads) or xg.dtype != torch.bfloat16 or grads[0].dtype not in _HALF:
        return None
    if not L.load().glf_fusion_ln_bwd_views_supported(C.byref(st.desc)):
        return None
    sb = []
    for g in grads:
        if g.dtype != grads[0].dtype or tuple(g.shape) != (B, Cn, h, w) or g.device != xg.device:
            return None
        b_, c_, h_, w_ = g.stride()
        if c_ != 1 or w_ != Cn or h_ != w * Cn or b_ % 8 or g.data_ptr() % 16 or (B > 1 and b_ < h * w * Cn):
            return None
        sb.append(b_)
    return list(grads), sb


def gate_concat_backward(f4, cls, ctr, gate, dxg, dxl, weight: float):
    lib = L.load()
    V = len(f4)
    B, C_, h, w = f4[0].shape
    ncls = cls[0].shape[1]
    dcls = [torch.empty_like(t) for t in cls]
    dctr = [torch.empty_like(t) for t in ctr]
    scratch = torch.empty(max(int(lib.glf_gate_concat_bwd_scratch_bytes(B, C_, V, h, w)), 256), dtype=torch.uint8,
                          device=f4[0].device)
    rows = _channels_last_rows(f4, dxg.dtype)
    if rows is not None and dxg.is_contiguous() and dxl.is_contiguous():
        # gradients go back in the views' own memory format (channels_last), so the conv backward stays channels_last
        df4 = [torch.empty((B, h, w, C_), dtype=t.dtype, device=t.device).permute(0, 3, 1, 2) for t in f4]
        i64 = C.c_int64 * V
        dsb, dst = [h * w * C_] * V, [C_] * V
        with torch.cuda.device(f4[0].device):
            L.check(lib.glf_gate_concat_cl_bwd(B, C_, V, h, w, ncls, float(weight), _io_dtype(f4[0]), L.ptr_table(f4),
                                               i64(*rows[0]), i64(*rows[1]), L.ptr_table(cls), L.ptr_table(ctr),
                                               L.ptr(gate), L.ptr(dxg), L.ptr(dxl), L.ptr_table(df4), i64(*dsb),
                                               i64(*dst), L.ptr_table(dcls), L.ptr_table(dctr), L.ptr(scratch),
                                               _stream_ptr()))
        return df4, dcls, dctr
    f4 = [t.contiguous() for t in f4]
    df4 = [torch.empty_like(t) for t in f4]
    with torch.cuda.device(f4[0].device):
        L.check(lib.glf_gate_concat_bwd(B, C_, V, h, w, ncls, float(weight), _io_dtype(f4[0]), _io_dtype(dxg),
                                        L.ptr_table(f4),
                                        L.ptr_table(cls), L.ptr_table(ctr), L.ptr(gate), L.ptr(dxg), L.ptr(dxl),
                                        L.ptr_table(df4), L.ptr_table(dcls), L.ptr_table(dctr), L.ptr(scratch),
                                        _stream_ptr()))
    return df4, dcls, dctr


class _FusionFunction(torch.autograd.Function):
    """ONE autograd node for gate + concat + MGFM + MLFM + sum.  With ``parts`` it has a second output, the MGFM part
    on its own (f4_global_fusion, ours.py:1823), written by the same fused LayerNorm pass; gradients that arrive
    through that output (the cycle-consistency pass, R/main.py:211-235) take the per-block LayerNorm backward, and a
    backward that carries NO gradient for the fused sum skips the MLFM block altogether."""

    @staticmethod
    def forward(ctx, fusion, V, ng, parts, per_view, *tensors):
        ctx.set_materialize_grads(False)
        ctx.per_view = bool(per_view)
        f4, cls, ctr = tensors[:V], tensors[V:2 * V], tensors[2 * V:3 * V]
        pg, pl = tensors[3 * V:3 * V + ng], tensors[3 * V + ng:]
        mg, ml = fusion.global_attn, fusion.local_attn
        mg._grad_out_claimed = ml._grad_out_claimed = False      # a new autograd graph (tpavi.claim_grad_out)
        prec = mg._precision_id()
        if ml._precision_id() != prec:
            raise ValueError("global_attn and local_attn must use the same compute_precision")
        # one parameter dtype for both blocks (the fused LayerNorm pass reads both with one descriptor): 2-byte only when
        # both blocks hold it throughout, fp32 copies otherwise
        pdt = mg._storage_dtype(pg)
        if ml._storage_dtype(pl) != pdt:
            pdt = torch.float32
        _check_precision_dtype(prec, f4[0].dtype, pdt)
        tg, tl = mg._param_table(pg, pdt), ml._param_table(pl, pdt)
        bg, bl = mg._buffer_table(pdt), ml._buffer_table(pdt)
        xdt = torch.float32 if prec == L.PRECISION_F32X3 else torch.bfloat16
        xg, xl, gate, f4c, clsc, ctrc = gate_concat_forward(f4, cls, ctr, fusion.center_aware_weight, xdt)
        B, V_, h, w, C_ = xg.shape
        need = any(ctx.needs_input_grad)
        shape = (B, V_, h, w, C_)
        pair = _pair_ln_ok(mg, ml, shape, xg, prec)
        # fp16 f4: the fused LayerNorm pass writes the fp16 outputs itself (its z dtype, desc.reserved[2]); no cast pass
        zdt = torch.float16 if pair and f4[0].dtype == torch.float16 else xg.dtype
        zsum = torch.empty(shape, dtype=zdt, device=xg.device)
        parts = bool(parts) and pair
        zglob = torch.empty(shape, dtype=zdt, device=xg.device) if parts else None
        # MGFM and MLFM are independent up to the fused LayerNorm: the local block runs on a side stream (a parallel
        # branch when the step is captured in a CUDA graph), so one block's short latency-bound kernels (BN statistics,
        # the per-sequence W' products) overlap the other's streaming GEMMs
        side = _side_stream(xg.device) if pair and fusion.overlap_blocks else None
        if side is not None:
            cur = torch.cuda.current_stream(xg.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                _, stl, svl, _ = tpavi_forward_raw(xl, tl, bl, mode=ml._mode_id, **ml._norm_config(),
                                                   bn_layer=ml._bn_layer, Ci=ml.inter_channels,
                                                   keep_for_backward=True, z_out=zsum, accumulate=False,
                                                   token_shape=shape, precision=prec, defer_ln=True)
        _, stg, svg, _ = tpavi_forward_raw(xg, tg, bg, mode=mg._mode_id, **mg._norm_config(),
                                           bn_layer=mg._bn_layer, Ci=mg.inter_channels,
                                           keep_for_backward=need or pair, z_out=zsum, token_shape=shape,
                                           precision=prec, defer_ln=pair)
        if side is not None:
            cur.wait_stream(side)
        else:
            _, stl, svl, _ = tpavi_forward_raw(xl, tl, bl, mode=ml._mode_id, **ml._norm_config(),
                                               bn_layer=ml._bn_layer, Ci=ml.inter_channels,
                                               keep_for_backward=need or pair, z_out=zsum, accumulate=not pair,
                                               token_shape=shape, precision=prec, defer_ln=pair)
        if pair:
            # both blocks' BN + residual + LayerNorm and the `global + local` sum (ours.py:1834) in one HBM pass
            wg, wl = _weights_struct(tg, bg), _weights_struct(tl, bl)
            stg.desc.reserved[2] = _io_dtype(zsum)
            with torch.cuda.device(xg.device):
                L.check(L.load().glf_fusion_ln_fwd_parts(C.byref(stg.desc), L.ptr(xg), L.ptr(xl), C.byref(wg),
                                                         C.byref(wl), L.ptr(zsum), L.ptr(zglob), L.ptr(svg), L.ptr(svl),
                                                         _stream_ptr()))
            if not need:
                svg = svl = None
        ctx.pair = pair
        ctx.pdt = pdt
        ctx.fusion, ctx.V, ctx.ng = fusion, V, ng
        ctx.states = (stg, svg, stl, svl)
        ctx.io_dtype = f4[0].dtype
        ctx.save_for_backward(xg, xl, gate, *f4c, *clsc, *ctrc, *pg, *pl)
        out = zsum if zsum.dtype == f4[0].dtype else zsum.to(f4[0].dtype)
        ctx.parts = parts
        og = None
        if parts:
            og = zglob if zglob.dtype == f4[0].dtype else zglob.to(f4[0].dtype)
        if ctx.per_view:
            # one output per view ([B,C,h,w] views of the token-major buffers): the dict-keyed callers then get one
            # gradient per view in backward, instead of autograd materialising V full-size zero tensors for V slices
            res = [out[:, v].permute(0, 3, 1, 2) for v in range(V_)]
            if parts:
                res += [og[:, v].permute(0, 3, 1, 2) for v in range(V_)]
            return tuple(res)
        if parts:
            return out.permute(0, 4, 1, 2, 3), og.permute(0, 4, 1, 2, 3)
        return out.permute(0, 4, 1, 2, 3)          # [B, C, V, h, w] view of the token-major buffer

    @staticmethod
    def backward(ctx, *grads):
        V, ng = ctx.V, ctx.ng
        saved = ctx.saved_tensors
        xg, xl, gate = saved[:3]
        rest = saved[3:]
        f4, cls, ctr = rest[:V], rest[V:2 * V], rest[2 * V:3 * V]
        pg, pl = rest[3 * V:3 * V + ng], rest[3 * V + ng:]
        mg, ml = ctx.fusion.global_attn, ctx.fusion.local_attn
        stg, svg, stl, svl = ctx.states
        if svg is None:
            raise L.GlfError("backward called on a forward that ran without grad")
        def token(t, ln_pair=False):                # [B,C,V,h,w] gradient -> token-major [B,V,h,w,C] in the x dtype
            if ctx.per_view:
                return t                            # assembled token-major below
            t = t.permute(0, 2, 3, 4, 1)
            if t.dtype != xg.dtype and not (ln_pair and t.dtype == torch.float16):
                t = t.to(xg.dtype)                  # (the fused LayerNorm backward reads an fp16 dz itself)
            return t.contiguous()

        def assemble(gs):                           # per-view [B,C,h,w] gradients -> one token-major [B,V,h,w,C] buffer
            if all(g is None for g in gs):
                return None
            buf = torch.empty(xg.shape, dtype=xg.dtype, device=xg.device)
            if views_to_tokens(gs, buf, dtypes=tuple(_IO_DTYPES)):
                return buf
            for v, g in enumerate(gs):
                if g is None:
                    buf[:, v].zero_()
                else:
                    buf[:, v].copy_(g.permute(0, 2, 3, 1))
            return buf
        dz_rows = None          # per-view gradients that the fused LayerNorm backward can read where they lie
        if ctx.per_view:
            dglob = assemble(grads[V:2 * V]) if ctx.parts else None
            if dglob is None and ctx.pair:
                dz_rows = _views_as_rows(grads[:V], xg, stg)
            dout = grads[0] if dz_rows is not None else assemble(grads[:V])
        else:
            dout = grads[0]
            dglob = grads[1] if len(grads) > 1 else None
        n_in = 5 + 3 * V + 2 * ng
        if dout is None and dglob is None:
            return (None,) * n_in
        stg.refresh_deterministic()                 # (the ws blobs below are sized from the backward's flag)
        stl.refresh_deterministic()
        tg, tl = mg._param_table(pg, ctx.pdt), ml._param_table(pl, ctx.pdt)
        bg, bl = mg._buffer_table(ctx.pdt), ml._buffer_table(ctx.pdt)
        gl = None
        if dglob is None:
            # both blocks see the same dz (ours.py:1834); with dz_rows it stays where autograd delivered it, one tensor
            # per view, and `dz` is only a placeholder (the blocks' backward continues from dV, it never reads dz)
            dz = xg if dz_rows is not None else token(dout, ln_pair=ctx.pair)
            wsg = wsl = None
            if ctx.pair:
                # LayerNorm backward of both blocks in one pass (dz is read once); fills dV / partials inside each ws blob
                stg.desc.dz_layout = stl.desc.dz_layout = L.LAYOUT_TOKEN
                stg.desc.reserved[0] = stl.desc.reserved[0] = 1
                stg.desc.reserved[2] = _io_dtype(dz_rows[0][0] if dz_rows is not None else dz)
                wsg, wsl = _blob(stg.sizes.ws_bwd_bytes, xg.device), _blob(stl.sizes.ws_bwd_bytes, xg.device)
                wg, wl = _weights_struct(tg, bg), _weights_struct(tl, bl)
                with torch.cuda.device(xg.device):
                    if dz_rows is not None:
                        views, sb = dz_rows
                        L.check(L.load().glf_fusion_ln_bwd_views(C.byref(stg.desc), None, L.ptr_table(views),
                                                                 (C.c_int64 * V)(*sb), L.ptr(xg), L.ptr(xl), C.byref(wg),
                                                                 C.byref(wl), L.ptr(svg), L.ptr(svl), L.ptr(wsg),
                                                                 L.ptr(wsl), _stream_ptr()))
                    else:
                        L.check(L.load().glf_fusion_ln_bwd(C.byref(stg.desc), L.ptr(dz), L.ptr(xg), L.ptr(xl),
                                                           C.byref(wg), C.byref(wl), L.ptr(svg), L.ptr(svl), L.ptr(wsg),
                                                           L.ptr(wsl), _stream_ptr()))
            gout_g, gout_l = claim_grad_out(mg), claim_grad_out(ml)
            side = _side_stream(xg.device) if ctx.pair and ctx.fusion.overlap_blocks else None
            if side is not None:   # after the fused LayerNorm backward the two blocks' chains are independent again
                cur = torch.cuda.current_stream(xg.device)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    dxl, gl = tpavi_backward_raw(dz, L.LAYOUT_TOKEN, xl, stl, svl, tl, bl, ws=wsl,
                                                 grad_out=gout_l)
            dxg, gg = tpavi_backward_raw(dz, L.LAYOUT_TOKEN, xg, stg, svg, tg, bg, ws=wsg,
                                         grad_out=gout_g)
            if side is not None:
                cur.wait_stream(side)
            else:
                dxl, gl = tpavi_backward_raw(dz, L.LAYOUT_TOKEN, xl, stl, svl, tl, bl, ws=wsl,
                                             grad_out=gout_l)
            hook = ctx.fusion.on_weight_grads_ready
            if hook is not None and gout_g is not None and gout_l is not None:
                hook()  # the gradients sit in the bucket views: the all-reduce may start now, beside the gate backward
        else:
            # a gradient arrived through the MGFM part (cycle-consistency pass): the two blocks no longer share dz, so
            # each runs its own LayerNorm backward (reserved[0] = 0); without a gradient for the fused sum the MLFM
            # block is not on the path at all
            dzg = token(dglob) if dout is None else token(dout) + token(dglob)
            stg.desc.reserved[0] = 0
            dxg, gg = tpavi_backward_raw(dzg, L.LAYOUT_TOKEN, xg, stg, svg, tg, bg,
                                         grad_out=claim_grad_out(mg))
            if dout is not None:
                stl.desc.reserved[0] = 0
                dxl, gl = tpavi_backward_raw(token(dout), L.LAYOUT_TOKEN, xl, stl, svl, tl, bl,
                                             grad_out=claim_grad_out(ml))
            else:
                dxl = torch.zeros_like(dxg)
        df4, dcls, dctr = gate_concat_backward(f4, cls, ctr, gate, dxg, dxl, ctx.fusion.center_aware_weight)
        out = [None, None, None, None, None] + list(df4) + list(dcls) + list(dctr)
        for mod, plist, gr in ((mg, pg, gg), (ml, pl, gl)):
            for name, p in zip(mod._plist_names(), plist):
                if gr is None or mod._grad_key(name) not in gr:    # (gaussian: theta / phi receive no gradient)
                    out.append(None)
                    continue
                t = gr[mod._grad_key(name)].reshape(p.shape)
                out.append(t if t.dtype == p.dtype else t.to(p.dtype))
        return tuple(out)


class _GateConcatFunction(torch.autograd.Function):
    """gate + view concat alone (ours.py:1802-1820, 1826-1827): -> X_g, X_l as [B,C,V,h,w] views of token-major buffers."""

    @staticmethod
    def forward(ctx, weight, V, x_dtype, *tensors):
        f4, cls, ctr = tensors[:V], tensors[V:2 * V], tensors[2 * V:3 * V]
        xg, xl, gate, f4c, clsc, ctrc = gate_concat_forward(f4, cls, ctr, weight, x_dtype)
        ctx.weight, ctx.V = weight, V
        ctx.save_for_backward(gate, *f4c, *clsc, *ctrc)
        return xg.permute(0, 4, 1, 2, 3), xl.permute(0, 4, 1, 2, 3)

    @staticmethod
    def backward(ctx, dxg, dxl):
        V = ctx.V
        saved = ctx.saved_tensors
        gate, rest = saved[0], saved[1:]
        f4, cls, ctr = rest[:V], rest[V:2 * V], rest[2 * V:3 * V]

        def tok(t, like):
            t = torch.zeros_like(like) if t is None else t
            return t.permute(0, 2, 3, 4, 1).contiguous()
        like = torch.empty((f4[0].shape[0], f4[0].shape[1], V) + tuple(f4[0].shape[2:]), dtype=dxg.dtype if dxg is not None
                           else dxl.dtype, device=f4[0].device)
        df4, dcls, dctr = gate_concat_backward(f4, cls, ctr, gate, tok(dxg, like), tok(dxl, like), ctx.weight)
        return (None, None, None) + tuple(df4) + tuple(dcls) + tuple(dctr)


class GlobalLocalFusion(nn.Module):
    """MGFM + MLFM (attribute names follow ``Global_and_Local``: ``global_attn`` / ``local_attn``, ours.py:1746-1747,
    so the corresponding slice of a reference checkpoint loads unchanged)."""

    def __init__(self, in_channels: int = 2048, mode: str = 'dot', center_aware_weight: float = 20,
                 inter_channels=None):
        super().__init__()
        self.center_aware_weight = center_aware_weight
        self.overlap_blocks = True      # run MGFM / MLFM on two streams between the fused stages
        # data-parallel hook: called from the fused backward as soon as BOTH blocks' parameter gradients are final
        # (before the gate backward), so that a gradient all-reduce can run beside the rest of the backward pass
        # (dp.GradBucket.overlap_with).  None = no hook.
        self.on_weight_grads_ready = None
        self.global_attn = TPAVIModule(in_channels=in_channels, inter_channels=inter_channels, mode=mode)
        self.local_attn = TPAVIModule(in_channels=in_channels, inter_channels=inter_channels, mode=mode)

    def load_reference_checkpoint(self, ckpt, strict: bool = True):
        """Load the MGFM / MLFM slice of a reference checkpoint: ``torch.load('net_%05d.pth')`` as written by
        ``Trainer.save`` (R/main.py:857-872: ``{'network': model.module.state_dict()}``), the bare state dict, or one
        whose keys carry the ``module.`` prefix that ``Trainer.test`` adds (main.py:454-457).  Keys of the rest of the
        network (backbones, heads) are ignored; the fusion keys must match exactly when ``strict``."""
        sd = ckpt.get("network", ckpt) if isinstance(ckpt, dict) else ckpt
        picked = {}
        for k, v in sd.items():
            if k.startswith("module."):
                k = k[len("module."):]
            if k.startswith("global_attn.") or k.startswith("local_attn."):
                picked[k] = v
        return self.load_state_dict(picked, strict=strict)

    def forward_stacked(self, f4: Sequence[torch.Tensor], cls_logits: Sequence[torch.Tensor],
                        ctr_logits: Sequence[torch.Tensor]) -> torch.Tensor:
        """Returns f4_fusion stacked over views: [B, C, V, h, w] (memory is token-major [B,V,h,w,C])."""
        V = len(f4)
        if not (len(cls_logits) == V and len(ctr_logits) == V and V >= 1):
            raise ValueError("f4, cls_logits and ctr_logits need one entry per view")
        pg, pl = self.global_attn._plist(), self.local_attn._plist()
        return _FusionFunction.apply(self, V, len(pg), False, False, *f4, *cls_logits, *ctr_logits, *pg, *pl)

    def forward_parts(self, f4: Dict[str, torch.Tensor], mask_bb_logits: Dict[str, torch.Tensor],
                      ctr_logits: Dict[str, torch.Tensor], need_local: bool = True):
        """Like ``forward`` but also returns the two parts the reference network hands back to its trainer
        (ours.py:1843 ``return mask, mask_bb, f4_global_fusion, f4_local_fusion``; the cycle-consistency pass of
        R/main.py:211-235 uses ``f4_global_fusion`` alone): ``(f4_fusion, f4_global_fusion, f4_local_fusion)``, dicts
        view -> [B,C,h,w].  It is the same single fused autograd node as ``forward``: the fused LayerNorm pass stores the
        MGFM part beside the sum (glf_fusion_ln_fwd_parts), the MLFM part is their difference (``need_local=False``
        skips forming it: the trainer ignores it, main.py:220).  A backward that arrives only through
        ``f4_global_fusion`` (the cycle pass) never touches the MLFM block."""
        views: List[str] = list(f4.keys())
        V = len(views)
        xs = [f4[v] for v in views]
        pg, pl = self.global_attn._plist(), self.local_attn._plist()
        res = _FusionFunction.apply(self, V, len(pg), True, True, *xs, *[mask_bb_logits[v] for v in views],
                                    *[ctr_logits[v] for v in views], *pg, *pl)
        if len(res) == 2 * V:
            # the single fused node, with the MGFM parts as further outputs (one more store in the LayerNorm pass)
            fus = {v: res[i] for i, v in enumerate(views)}
            glob = {v: res[V + i] for i, v in enumerate(views)}
            loc = {v: fus[v] - glob[v] for v in views} if need_local else None
            return fus, glob, loc
        # shapes / precisions the fused LayerNorm pair does not cover: the two blocks as separate autograd nodes
        x_dtype = torch.float32 if self.global_attn._precision_id() == L.PRECISION_F32X3 else torch.bfloat16
        xg, xl = _GateConcatFunction.apply(self.center_aware_weight, V, x_dtype, *xs,
                                           *[mask_bb_logits[v] for v in views], *[ctr_logits[v] for v in views])
        zg, _ = self.global_attn(xg)
        zl, _ = self.local_attn(xl)
        if zg.dtype != xs[0].dtype:
            zg, zl = zg.to(xs[0].dtype), zl.to(xs[0].dtype)
        glob = {v: zg[:, :, i] for i, v in enumerate(views)}
        loc = {v: zl[:, :, i] for i, v in enumerate(views)}
        return {v: glob[v] + loc[v] for v in views}, glob, loc

    def forward(self, f4: Dict[str, torch.Tensor], mask_bb_logits: Dict[str, torch.Tensor],
                ctr_logits: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Dict-keyed like the reference (view id -> tensor): returns f4_fusion[view] = global + local."""
        views: List[str] = list(f4.keys())
        V = len(views)
        pg, pl = self.global_attn._plist(), self.local_attn._plist()
        res = _FusionFunction.apply(self, V, len(pg), False, True, *[f4[v] for v in views],
                                    *[mask_bb_logits[v] for v in views], *[ctr_logits[v] for v in views], *pg, *pl)
        return {v: res[i] for i, v in enumerate(views)}
