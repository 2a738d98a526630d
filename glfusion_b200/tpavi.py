"""Drop-in ``TPAVIModule`` (the reference's MGFM / MLFM block) backed by libglf_sm100a.so.

Mirrors ``R/models/ours.py:770-917`` (duplicate: ``R/models/TPAVI.py:6-155``):

* same constructor ``TPAVIModule(in_channels, inter_channels=None, mode='dot', dimension=3, bn_layer=True)``;
* same ``state_dict`` keys / shapes / init (the parameter containers are the same ``nn`` layers created in the same
  order, so a reference checkpoint loads with ``strict=True`` and the RNG stream at construction is identical);
* same ``forward(x, audio=None) -> (z, audio_temp)`` with ``z.shape == x.shape`` and ``z`` a permuted view of a
  ``[B,T,H,W,C]`` buffer, exactly the strides the reference's LayerNorm output has (ours.py:913-915).

The ``nn`` layers are parameter holders only: forward/backward are the CUDA kernels behind the C ABI
(``include/glfusion.h``).  There is no PyTorch / CPU fallback — on a machine without the library or without an
sm_100 GPU every call raises.
"""
from __future__ import annotations

import os

import ctypes as C
from typing import Optional, Tuple

import torch
from torch import nn

from . import _lib as L

DEFAULT_PRECISION = "bf16"


def set_default_precision(name: str) -> None:
    """Default `compute_precision` of modules constructed afterwards ('bf16' or 'fp32')."""
    global DEFAULT_PRECISION
    if name not in L.PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(L.PRECISIONS)}")
    DEFAULT_PRECISION = name


_PARAM_ORDER = ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "wz_w", "wz_b", "bn_w", "bn_b", "ln_w", "ln_b")
# mode='gaussian' scores the block input against itself (f = x x^T, ours.py:869-873): theta / phi are state_dict entries
# that take no part, so the kernels neither read them nor write a gradient for them (their .grad stays None)
_UNUSED_BY_MODE = {L.MODE_GAUSSIAN: frozenset(("theta_w", "theta_b", "phi_w", "phi_b"))}
_MODE_IDS = {"dot": L.MODE_DOT, "embedded": L.MODE_EMBEDDED, "gaussian": L.MODE_GAUSSIAN}


_IO_DTYPES = {torch.bfloat16: L.DTYPE_BF16, torch.float32: L.DTYPE_F32, torch.float16: L.DTYPE_F16}


def _io_dtype(t: torch.Tensor) -> int:
    """GLF_DTYPE_* of an activation.  float16 (torch.autocast's default) is an I/O dtype only: the kernels convert it to
    bf16 where they read it and round to fp16 where they write; the products and statistics in between are unchanged."""
    try:
        return _IO_DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"glfusion_b200 supports float32, bfloat16 and float16 activations, got {t.dtype}") from None


# Parameter dtypes the kernels read and write as they are (glf_desc.reserved[3]); anything else runs on fp32 copies.
_PARAM_DTYPES = {torch.float32: L.PARAMS_F32, torch.bfloat16: L.PARAMS_BF16, torch.float16: L.PARAMS_F16}


def _check_precision_dtype(precision: int, dtype: torch.dtype, param_dtype: torch.dtype = torch.float32) -> None:
    """The fp32-exact arm is an fp32 contract: float16 inputs or 2-byte parameters would defeat it (the library rejects
    both too)."""
    if precision == L.PRECISION_F32X3 and dtype == torch.float16:
        raise TypeError("compute_precision='fp32' takes float32 or bfloat16 activations, not float16; keep the default "
                        "compute_precision='bf16' for float16 (autocast) inputs")
    if precision == L.PRECISION_F32X3 and param_dtype != torch.float32:
        raise TypeError(f"compute_precision='fp32' takes float32 parameters, not {param_dtype}; keep the default "
                        "compute_precision='bf16' for a .half() / .bfloat16() module")


def _is_token_major(t: torch.Tensor) -> bool:
    """[B,C,T,H,W] tensor whose memory is a dense [B,T,H,W,C] array."""
    return t.permute(0, 2, 3, 4, 1).is_contiguous()


def _stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _blob(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


# Algorithm for mode='dot' (glf_desc.reserved[1]): 0 = the library chooses (Gram form when N >= 3 C at C = 256, 5 C below, 8 C above), 1 = token-space
# form (theta/phi/g per token), 2 = Gram form (channel-space products only).  Tests pin it; users leave it alone.
DOT_ALGO = int(os.environ.get("GLF_DOT_ALGO", "0"))


def _deterministic_bit() -> int:
    # torch.use_deterministic_algorithms(True) is the switch: the blocks then sum split products in a fixed order
    # (GLF_DETERMINISTIC) and give bitwise identical results from run to run.  warn_only changes nothing: the
    # deterministic implementation always exists.
    return L.DETERMINISTIC if torch.are_deterministic_algorithms_enabled() else 0


class TPAVIState:
    """Everything one forward/backward pair shares: descriptor, weights table, saved blob."""

    def __init__(self, B, C_, T, H, W, Ci, mode, io_dtype, x_layout, training, bn_layer, accumulate=False,
                 eps_bn=1e-5, eps_ln=1e-5, momentum=0.1, precision=L.PRECISION_BF16, defer_ln=False,
                 param_dtype=L.PARAMS_F32):
        d = L.GlfDesc()
        d.B, d.T, d.H, d.W, d.C, d.Ci = B, T, H, W, C_, Ci
        d.mode = mode
        d.io_dtype = io_dtype
        d.x_layout = x_layout
        d.dz_layout = L.LAYOUT_TOKEN
        d.precision = precision
        d.training = int(training)
        d.bn_layer = int(bn_layer)
        d.accumulate = int(accumulate)
        d.eps_bn, d.eps_ln, d.momentum = eps_bn, eps_ln, momentum
        d.reserved[0] = 1 if defer_ln else 0     # LayerNorm stage run for MGFM + MLFM together (glf_fusion_ln_*)
        d.reserved[1] = DOT_ALGO | _deterministic_bit()   # dot algorithm (0 / 1 / 2) | GLF_DETERMINISTIC
        d.reserved[3] = param_dtype              # dtype of the parameter tensors, gradients and running statistics
        self.desc = d
        self._resize()

    def _resize(self):
        sz = L.GlfSizes()
        L.check(L.load().glf_tpavi_sizes(C.byref(self.desc), C.byref(sz)))
        self.sizes = sz

    def refresh_deterministic(self):
        """Backward reads torch.are_deterministic_algorithms_enabled() again, as forward did: the flag only changes
        workspace sizes and reduction order, never the saved blob, so it may differ between the two."""
        bit = _deterministic_bit()
        if (self.desc.reserved[1] & L.DETERMINISTIC) != bit:
            self.desc.reserved[1] = (self.desc.reserved[1] & 0xFF) | bit
            self._resize()


def _weights_struct(p, buffers) -> L.GlfWeights:
    w = L.GlfWeights()
    for name in _PARAM_ORDER:
        setattr(w, name, p[name].data_ptr() if p.get(name) is not None else None)
    rm, rv, nbt = buffers
    w.bn_running_mean = rm.data_ptr() if rm is not None else None
    w.bn_running_var = rv.data_ptr() if rv is not None else None
    w.bn_num_batches_tracked = nbt.data_ptr() if nbt is not None else None
    return w


def tpavi_forward_raw(x: torch.Tensor, params: dict, buffers, *, mode: int, training: bool, bn_layer: bool,
                      Ci: int, keep_for_backward: bool, z_out: Optional[torch.Tensor] = None,
                      accumulate: bool = False, token_shape=None, precision: int = L.PRECISION_BF16,
                      defer_ln: bool = False, eps_bn: float = 1e-5, eps_ln: float = 1e-5, momentum: float = 0.1):
    """Run glf_tpavi_fwd.  ``x`` is either NCTHW-contiguous or token-major (see ``_is_token_major``), or, when
    ``token_shape=(B,T,H,W,C)`` is given, a dense token-major buffer of that shape.
    Returns (z_buffer [B,T,H,W,C], state, saved_blob)."""
    lib = L.load()
    if not x.is_cuda:
        raise L.GlfError("glfusion_b200 runs on CUDA (sm_100) tensors only; there is no CPU path")
    pdt = params["ln_w"].dtype      # _param_table: one dtype for every tensor of the table
    _check_precision_dtype(precision, x.dtype, pdt)
    if token_shape is not None:
        B, T, H, W, C_ = token_shape
        layout = L.LAYOUT_TOKEN
    else:
        B, C_, T, H, W = x.shape
        if _is_token_major(x):
            layout = L.LAYOUT_TOKEN
        else:
            x = x.contiguous()
            layout = L.LAYOUT_NCTHW
    st = TPAVIState(B, C_, T, H, W, Ci, mode, _io_dtype(x), layout, training, bn_layer, accumulate,
                    eps_bn=eps_bn, eps_ln=eps_ln, momentum=momentum, precision=precision, defer_ln=defer_ln,
                    param_dtype=_PARAM_DTYPES[pdt])
    dev = x.device
    if z_out is None:
        z_out = torch.empty((B, T, H, W, C_), dtype=x.dtype, device=dev)
    saved = _blob(st.sizes.saved_bytes, dev) if keep_for_backward else None
    ws = _blob(st.sizes.ws_fwd_bytes, dev)
    w = _weights_struct(params, buffers)
    with torch.cuda.device(dev):
        L.check(lib.glf_tpavi_fwd(C.byref(st.desc), L.ptr(x), C.byref(w), L.ptr(z_out), L.ptr(saved), L.ptr(ws),
                                  _stream_ptr()))
    return z_out, st, saved, x


def tpavi_backward_raw(dz: torch.Tensor, dz_layout: int, x: torch.Tensor, st: TPAVIState, saved: torch.Tensor,
                       params: dict, buffers, dx_out: Optional[torch.Tensor] = None,
                       ws: Optional[torch.Tensor] = None, grad_out: Optional[dict] = None):
    """Run glf_tpavi_bwd.  Returns (dx buffer in the layout of x, dict of parameter gradients in the dtype of `params`).
    `grad_out` (optional): name -> preallocated tensor of that dtype the kernels write that gradient into (e.g. views of
    a data-parallel all-reduce bucket, dp.GradBucket.bind): the returned gradient then aliases it."""
    lib = L.load()
    dev = x.device
    st.refresh_deterministic()
    d = st.desc
    d.dz_layout = dz_layout
    grads = {}
    gdt = params["ln_w"].dtype
    g = L.GlfGrads()
    unused = _UNUSED_BY_MODE.get(d.mode, ())
    for name in _PARAM_ORDER:
        if name in unused:
            setattr(g, name, None)
            continue
        ref = params.get(name)
        if ref is None:
            # bn_layer=False: no BN affine; the kernels still want a scratch target
            ref = params["ln_w"]
        dst = grad_out.get(name) if grad_out is not None and params.get(name) is not None else None
        if dst is not None and dst.dtype == gdt and dst.shape == ref.shape and dst.is_contiguous():
            t = dst.detach()        # fresh alias: autograd may adopt it as .grad without a copy
        else:
            t = torch.empty(ref.shape, dtype=gdt, device=dev)
        grads[name] = t
        setattr(g, name, t.data_ptr())
    if dx_out is None:
        if d.x_layout == L.LAYOUT_TOKEN:
            dx_out = torch.empty((d.B, d.T, d.H, d.W, d.C), dtype=x.dtype, device=dev)
        else:
            dx_out = torch.empty((d.B, d.C, d.T, d.H, d.W), dtype=x.dtype, device=dev)
    sz = L.GlfSizes()
    L.check(lib.glf_tpavi_sizes(C.byref(d), C.byref(sz)))
    if ws is None:
        ws = _blob(sz.ws_bwd_bytes, dev)
    w = _weights_struct(params, buffers)
    with torch.cuda.device(dev):
        L.check(lib.glf_tpavi_bwd(C.byref(d), L.ptr(dz), L.ptr(x), C.byref(w), L.ptr(saved), L.ptr(dx_out),
                                  C.byref(g), L.ptr(ws), _stream_ptr()))
    return dx_out, grads


def claim_grad_out(module):
    """dp.GradBucket.bind() lets a block's backward write its parameter gradients straight into the all-reduce bucket.
    The kernels ASSIGN (they never accumulate), so the bucket views may be handed out only to the FIRST backward node of
    a step that touches the module, and only while no gradient has been accumulated yet:

      * a module used twice before one backward (the reference's cycle pass, R/main.py:209 and :221): the second node
        gets fresh tensors and autograd adds the two contributions;
      * gradient accumulation / zero_grad(set_to_none=False): p.grad already exists (it may even alias the bucket), so
        the node writes to fresh tensors and autograd accumulates into p.grad.

    The claim is released by the next forward of the module (a new autograd graph)."""
    table = getattr(module, "_grad_out", None)
    if not table or getattr(module, "_grad_out_claimed", False):
        return None
    if any(p.grad is not None for p in module._plist()):
        return None
    module._grad_out_claimed = True
    return table


class _TPAVIFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, module, *plist):
        module._grad_out_claimed = False
        pdt = module._storage_dtype(plist)
        params = module._param_table(plist, pdt)
        buffers = module._buffer_table(pdt)
        need_grad = any(ctx.needs_input_grad)      # grad mode is off inside Function.forward
        z, st, saved, x_used = tpavi_forward_raw(x, params, buffers, mode=module._mode_id,
                                                 bn_layer=module._bn_layer,
                                                 Ci=module.inter_channels, keep_for_backward=need_grad,
                                                 precision=module._precision_id(), **module._norm_config())
        ctx.module = module
        ctx.pdt = pdt
        ctx.st = st
        ctx.saved_blob = saved
        ctx.x_dtype = x.dtype
        ctx.save_for_backward(x_used, *plist)
        out = z.permute(0, 4, 1, 2, 3)      # [B,C,T,H,W] view, strides identical to the reference's output
        return out

    @staticmethod
    def backward(ctx, dz):
        x_used, *plist = ctx.saved_tensors
        module = ctx.module
        params = module._param_table(plist, ctx.pdt)
        if ctx.saved_blob is None:
            raise L.GlfError("backward called on a forward that ran without grad")
        if dz.dtype != x_used.dtype:
            dz = dz.to(x_used.dtype)
        if _is_token_major(dz):
            layout = L.LAYOUT_TOKEN
        else:
            dz = dz.contiguous()
            layout = L.LAYOUT_NCTHW
        dx, grads = tpavi_backward_raw(dz, layout, x_used, ctx.st, ctx.saved_blob, params, module._buffer_table(ctx.pdt),
                                       grad_out=claim_grad_out(module))
        if ctx.st.desc.x_layout == L.LAYOUT_TOKEN:
            dx = dx.permute(0, 4, 1, 2, 3)
        out = [dx, None]
        for name, p in zip(module._plist_names(), plist):
            gname = module._grad_key(name)
            if gname not in grads:          # a parameter the mode does not use (gaussian: theta / phi)
                out.append(None)
                continue
            gr = grads[gname].reshape(p.shape)
            out.append(gr if gr.dtype == p.dtype else gr.to(p.dtype))
        return tuple(out)


class TPAVIModule(nn.Module):
    """B200-native drop-in for the reference's non-local fusion block (MGFM and MLFM are two instances of it)."""

    def __init__(self, in_channels, inter_channels=None, mode='dot', dimension=3, bn_layer=True):
        super(TPAVIModule, self).__init__()
        assert dimension in [1, 2, 3]
        if mode not in ['gaussian', 'embedded', 'dot', 'concatenate']:
            raise ValueError('`mode` must be one of `gaussian`, `embedded`, `dot` or `concatenate`')
        if dimension != 3:
            # ours.py:845-917 only works for dimension=3 (the LayerNorm permute is 5-D); 1/2 crash in the reference
            raise NotImplementedError("glfusion_b200.TPAVIModule supports dimension=3 (as the reference effectively does)")
        if mode == 'concatenate':
            raise NotImplementedError("mode='concatenate' is not built by any constructor site of the reference network; "
                                      "supported: 'dot' (MGFM/MLFM), 'embedded' and 'gaussian' (softmax)")
        self.mode = mode
        self.dimension = dimension
        self.in_channels = in_channels
        self.inter_channels = inter_channels
        if self.inter_channels is None:
            self.inter_channels = in_channels // 2
            if self.inter_channels == 0:
                self.inter_channels = 1
        # parameter holders, created in the reference's order (ours.py:800-843) so that init RNG use and
        # state_dict ordering are identical
        self.align_channel = nn.Linear(128, in_channels)
        self.norm_layer = nn.LayerNorm(in_channels)
        self.g = nn.Conv3d(in_channels=self.in_channels, out_channels=self.inter_channels, kernel_size=1)
        if bn_layer:
            self.W_z = nn.Sequential(
                nn.Conv3d(in_channels=self.inter_channels, out_channels=self.in_channels, kernel_size=1),
                nn.BatchNorm3d(self.in_channels))
            nn.init.constant_(self.W_z[1].weight, 0)
            nn.init.constant_(self.W_z[1].bias, 0)
        else:
            self.W_z = nn.Conv3d(in_channels=self.inter_channels, out_channels=self.in_channels, kernel_size=1)
            nn.init.constant_(self.W_z.weight, 0)
            nn.init.constant_(self.W_z.bias, 0)
        self.theta = nn.Conv3d(in_channels=self.in_channels, out_channels=self.inter_channels, kernel_size=1)
        self.phi = nn.Conv3d(in_channels=self.in_channels, out_channels=self.inter_channels, kernel_size=1)
        self._bn_layer = bool(bn_layer)
        self._mode_id = _MODE_IDS[mode]
        # tensor-core operand precision (not a reference ctor argument; set the attribute after construction):
        #   'bf16' — bf16 operands, fp32 accumulate (throughput arm, 2e-2 tolerance)
        #   'fp32' — fp32-exact products via 3-limb bf16 split on the same tcgen05 kernel (1e-4 tolerance, mode='dot')
        self.compute_precision = DEFAULT_PRECISION

    def _precision_id(self) -> int:
        try:
            return L.PRECISIONS[self.compute_precision]
        except KeyError:
            raise ValueError(f"compute_precision must be one of {sorted(L.PRECISIONS)}, got {self.compute_precision!r}")

    def _norm_config(self) -> dict:
        """eps / momentum / train-or-eval of the normalisation layers, read from the nn holders (not assumed): a loaded
        non-default configuration, or the usual 'freeze BatchNorm only' pattern (model.train(); bn.eval()), must act on
        the kernels exactly as it would on the reference's layers.  Configurations the kernels do not implement raise."""
        cfg = {"eps_bn": 1e-5, "eps_ln": float(self.norm_layer.eps), "momentum": 0.1, "training": bool(self.training)}
        if not self.norm_layer.elementwise_affine:
            raise NotImplementedError("LayerNorm without affine parameters is not supported")
        if self._bn_layer:
            bn = self.W_z[1]
            if bn.momentum is None or not bn.track_running_stats or not bn.affine:
                raise NotImplementedError("BatchNorm3d with momentum=None (cumulative average), track_running_stats=False "
                                          "or affine=False is not supported by the sm_100a kernels")
            cfg.update(eps_bn=float(bn.eps), momentum=float(bn.momentum), training=bool(bn.training))
        return cfg

    # ---- parameter plumbing -------------------------------------------------------------------------------------
    def _plist_names(self):
        names = ["theta.weight", "theta.bias", "phi.weight", "phi.bias", "g.weight", "g.bias"]
        if self._bn_layer:
            names += ["W_z.0.weight", "W_z.0.bias", "W_z.1.weight", "W_z.1.bias"]
        else:
            names += ["W_z.weight", "W_z.bias"]
        names += ["norm_layer.weight", "norm_layer.bias"]
        return names

    _KEYMAP = {"theta.weight": "theta_w", "theta.bias": "theta_b", "phi.weight": "phi_w", "phi.bias": "phi_b",
               "g.weight": "g_w", "g.bias": "g_b", "W_z.0.weight": "wz_w", "W_z.0.bias": "wz_b",
               "W_z.weight": "wz_w", "W_z.bias": "wz_b", "W_z.1.weight": "bn_w", "W_z.1.bias": "bn_b",
               "norm_layer.weight": "ln_w", "norm_layer.bias": "ln_b"}

    def _grad_key(self, name):
        return self._KEYMAP[name]

    def _plist(self):
        table = dict(self.named_parameters())
        return [table[n] for n in self._plist_names()]

    def _storage_dtype(self, plist) -> torch.dtype:
        """bfloat16 / float16 when every parameter of the block and both BatchNorm running statistics share that dtype
        (``.half()``, ``.bfloat16()``): the kernels read them, and write gradients and running statistics, in it.
        float32 otherwise, a mix such as bf16 convs beside fp32 norm layers included: that block runs on fp32 copies."""
        ts = list(plist)
        if self._bn_layer:
            ts += [self.W_z[1].running_mean, self.W_z[1].running_var]
        dts = {t.dtype for t in ts}
        dt = dts.pop() if len(dts) == 1 else torch.float32
        return dt if dt in (torch.bfloat16, torch.float16) else torch.float32

    def _param_table(self, plist, dtype=None):
        """Kernel-side name -> parameter tensor, all of `dtype` (default: _storage_dtype): fp32 copies where needed."""
        if dtype is None:
            dtype = self._storage_dtype(plist)
        out = {}
        for name, p in zip(self._plist_names(), plist):
            t = p.detach()
            if t.dtype != dtype:
                t = t.float()
            out[self._KEYMAP[name]] = t.contiguous()
        if not self._bn_layer:
            out["bn_w"] = None
            out["bn_b"] = None
        return out

    def _buffer_table(self, dtype=torch.float32):
        if not self._bn_layer:
            return (None, None, None)
        bn = self.W_z[1]
        if bn.running_mean.dtype != dtype or bn.running_var.dtype != dtype:
            raise L.GlfError("BatchNorm running statistics must stay float32 unless every parameter of the block "
                             "shares their bfloat16 / float16 dtype")
        return (bn.running_mean, bn.running_var, bn.num_batches_tracked)

    # ---- forward ------------------------------------------------------------------------------------------------
    def forward(self, x, audio=None) -> Tuple[torch.Tensor, int]:
        """
        args:
            x: (N, C, T, H, W)
            audio: must be None (the fusion network never passes it; ours.py:1821,1828)
        returns (z, audio_temp) with audio_temp == 0, as the reference does for audio=None (ours.py:851,917)
        """
        if audio is not None:
            raise NotImplementedError("the audio branch (align_channel) is not part of the GL-Fusion network path")
        if x.dim() != 5 or x.size(1) != self.in_channels:
            raise ValueError(f"expected x of shape [B,{self.in_channels},T,H,W], got {tuple(x.shape)}")
        z = _TPAVIFunction.apply(x, self, *self._plist())
        return z, 0
