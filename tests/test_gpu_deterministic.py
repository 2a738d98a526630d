"""torch.use_deterministic_algorithms(True): the blocks sum every split product in a fixed order (GLF_DETERMINISTIC), so
three runs on fresh copies of the inputs and fresh blobs give bitwise identical outputs, input gradients, parameter
gradients and running statistics.  Each case is one that takes a split path (tests/test_deterministic_abi.py checks
that the flag adds slab space for exactly these shapes), and the flag-on result is also held to the oracle (float64,
computed with the flag off: cuBLAS refuses to run under it without CUBLAS_WORKSPACE_CONFIG) within the suite's bounds.

The flag is process-global: every test takes it through the `deterministic` fixture, which restores both the flag and
its warn_only setting.  PyTorch's fill_uninitialized_memory stays on: every blob starts as NaN, so a kernel that read
scratch it did not write would show."""
import contextlib

import pytest
import torch

from glfusion_b200 import GlobalLocalFusion, TPAVIModule
from gpu_util import BF16_TOL, DEV, assert_close, dot_algo, grad_scale, grad_tol
from oracle import tpavi_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture
def deterministic():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


@contextlib.contextmanager
def _flag_off():
    """The oracle's float64 reference runs on the GPU with the flag off (cuBLAS)."""
    torch.use_deterministic_algorithms(False)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(True)


def _dev64(p):
    return {k: (v.to(DEV, torch.float64) if v.is_floating_point() else v.to(DEV)) for k, v in p.items()}


def _inputs(B, C_, T, H, W, seed, mode):
    gen = torch.Generator().manual_seed(seed)
    if mode == "gaussian":      # clustered tokens: a softmax over X X^T that is not one-hot
        from test_gpu_gaussian_attention import clustered_tokens
        x = clustered_tokens(B, T * H * W, C_, gen).reshape(B, T, H, W, C_).permute(0, 4, 1, 2, 3).contiguous()
    else:
        x = torch.randn(B, C_, T, H, W, generator=gen, dtype=torch.float64)
    dz = torch.randn(B, C_, T, H, W, generator=gen, dtype=torch.float64)
    return x, dz


def _block_run(p, mode, x, dz, algo, dtype, precision, pdtype):
    m = TPAVIModule(in_channels=x.shape[1], mode=mode, bn_layer=True)
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m = m.to(DEV).train()
    m.compute_precision = precision
    if pdtype is not None:
        m = m.to(pdtype)
    xi = x.to(DEV, dtype).requires_grad_(True)
    with dot_algo(algo):
        z, _ = m(xi)
    z.backward(dz.to(DEV, dtype))
    torch.cuda.synchronize()
    out = {"z": z.detach().clone(), "dx": xi.grad.detach().clone(),
           "running_mean": m.W_z[1].running_mean.clone(), "running_var": m.W_z[1].running_var.clone()}
    for name, t in m.named_parameters():
        if t.grad is not None:
            out["grad:" + name] = t.grad.detach().clone()
    return out


def _bits(t):
    t = t.contiguous().reshape(-1)
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def _assert_bitwise(runs):
    for i, r in enumerate(runs[1:], 1):
        assert set(r) == set(runs[0])
        for k in sorted(r):
            a, b = runs[0][k], r[k]
            assert a.dtype == b.dtype and a.shape == b.shape, k
            assert torch.equal(_bits(a), _bits(b)), f"{k}: run {i} differs from run 0"


BLOCK_CASES = [
    # id, mode, C, (T, H, W), B, dot algorithm, io dtype, compute_precision, parameter dtype
    ("dot-token-c256", "dot", 256, (4, 28, 28), 16, "token", torch.bfloat16, "bf16", None),
    ("dot-gram-b4", "dot", 256, (4, 28, 28), 4, "gram", torch.bfloat16, "bf16", None),
    ("dot-gram-b2-t16", "dot", 256, (16, 28, 28), 2, "gram", torch.bfloat16, "bf16", None),
    ("embedded-c256-flash", "embedded", 256, (4, 28, 28), 2, "auto", torch.bfloat16, "bf16", None),
    ("embedded-c192-chunked", "embedded", 192, (2, 14, 14), 2, "auto", torch.bfloat16, "bf16", None),
    ("gaussian-c128-flash", "gaussian", 128, (2, 14, 14), 2, "auto", torch.bfloat16, "bf16", None),
    ("gaussian-c256-chunked", "gaussian", 256, (2, 14, 14), 2, "auto", torch.bfloat16, "bf16", None),
    ("width2048-3views", "dot", 2048, (3, 28, 28), 2, "auto", torch.bfloat16, "bf16", None),
    ("fp32-exact", "dot", 128, (2, 14, 14), 2, "token", torch.float32, "fp32", None),
    ("half-module", "dot", 256, (4, 28, 28), 16, "token", torch.float16, "bf16", torch.float16),
]


@pytest.mark.parametrize("case", BLOCK_CASES, ids=[c[0] for c in BLOCK_CASES])
def test_block_is_bitwise_reproducible_and_matches_the_oracle(deterministic, case):
    _, mode, C_, (T, H, W), B, algo, dtype, precision, pdtype = case
    p = O.init_params(C_, seed=11)
    if pdtype is not None:      # the oracle sees the values the 2-byte parameters hold
        p = {k: (v.to(pdtype).float() if v.is_floating_point() else v) for k, v in p.items()}
    x, dz = _inputs(B, C_, T, H, W, seed=12, mode=mode)
    runs = [_block_run(p, mode, x, dz, algo, dtype, precision, pdtype) for _ in range(3)]
    _assert_bitwise(runs)

    q = _dev64(p)
    with _flag_off():
        z, dx, g = O.tpavi_fwd_bwd(x.to(dtype).to(DEV, torch.float64), dz.to(dtype).to(DEV, torch.float64), q,
                                   mode=mode, training=True, bn_layer=True)
    r = runs[0]
    tol = 1e-4 if precision == "fp32" else BF16_TOL
    omode = "embedded" if mode == "embedded" else "dot"
    if mode == "gaussian":      # the bounds of test_gpu_gaussian_module: the oracle's own bf16 floor, capped at 4e-2
        from test_gpu_gaussian_module import _floors, _tol
        with _flag_off():
            floors = _floors(x, dz, p, True, True, (z, dx, g))
        bound = lambda name: _tol(name, floors)
    else:
        bound = lambda name: tol if precision == "fp32" or name in ("z", "dx") else grad_tol(name, omode)
    assert_close("z", r["z"], z, bound("z"))
    assert_close("dx", r["dx"], dx, bound("dx"))
    scale = grad_scale(g.values())
    for name, ref in g.items():
        assert_close("grad:" + name, r["grad:" + name].reshape(ref.shape), ref, bound(name), zero_scale=scale)
    assert_close("running_mean", r["running_mean"], q["W_z.1.running_mean"], tol, abs_floor=1e-3)
    assert_close("running_var", r["running_var"], q["W_z.1.running_var"], tol)


def _fusion_inputs(C_, V, B, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    f4 = [torch.randn(B, C_, h, w, generator=gen) for _ in range(V)]
    cl = [torch.randn(B, 5, h, w, generator=gen) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, generator=gen) for _ in range(V)]
    do = [torch.randn(B, C_, h, w, generator=gen) for _ in range(V)]
    return f4, cl, ct, do


def _fusion(C_, pg, pl):
    f = GlobalLocalFusion(in_channels=C_)
    f.global_attn.load_state_dict({k: v.clone() for k, v in pg.items()}, strict=True)
    f.local_attn.load_state_dict({k: v.clone() for k, v in pl.items()}, strict=True)
    return f.to(DEV).train()


def _fusion_run(kind, C_, pg, pl, f4, cl, ct, do):
    f = _fusion(C_, pg, pl)
    V = len(f4)
    f4d = [t.to(DEV, torch.bfloat16).requires_grad_(True) for t in f4]
    cld = [t.to(DEV).requires_grad_(True) for t in cl]
    ctd = [t.to(DEV).requires_grad_(True) for t in ct]
    views = [f"v{i}" for i in range(V)]
    if kind == "stacked":
        out = f.forward_stacked(f4d, cld, ctd)
        out.backward(torch.stack(do, dim=2).to(DEV, torch.bfloat16))
        outs = [out[:, :, v] for v in range(V)]
    elif kind == "dict":
        res = f(dict(zip(views, f4d)), dict(zip(views, cld)), dict(zip(views, ctd)))
        outs = [res[v] for v in views]
        torch.autograd.backward(outs, [t.to(DEV, torch.bfloat16) for t in do])
    else:   # forward_parts, backward through the global part only (the cycle-consistency pass)
        _, glob, _ = f.forward_parts(dict(zip(views, f4d)), dict(zip(views, cld)), dict(zip(views, ctd)),
                                     need_local=False)
        outs = [glob[v] for v in views]
        torch.autograd.backward(outs, [t.to(DEV, torch.bfloat16) for t in do])
    torch.cuda.synchronize()
    r = {f"out{v}": o.detach().clone() for v, o in enumerate(outs)}
    for v in range(V):
        for tag, t in (("df4", f4d[v]), ("dcls", cld[v]), ("dctr", ctd[v])):
            if t.grad is not None:
                r[f"{tag}_{v}"] = t.grad.detach().clone()
    for tag, mod in (("g", f.global_attn), ("l", f.local_attn)):
        r[f"{tag}:running_mean"] = mod.W_z[1].running_mean.clone()
        r[f"{tag}:running_var"] = mod.W_z[1].running_var.clone()
        for name, t in mod.named_parameters():
            if t.grad is not None:
                r[f"{tag}:grad:{name}"] = t.grad.detach().clone()
    return r


@pytest.mark.parametrize("kind", ["stacked", "dict", "parts"])
def test_fusion_is_bitwise_reproducible(deterministic, kind):
    C_, V, B, h, w = 256, 4, 2, 14, 14
    pg, pl = O.init_params(C_, seed=21), O.init_params(C_, seed=22)
    f4, cl, ct, do = _fusion_inputs(C_, V, B, h, w, seed=23)
    with dot_algo("token"):     # N = 784 per sequence: a split token contraction and a batch-reduced dWz per block
        runs = [_fusion_run(kind, C_, pg, pl, f4, cl, ct, do) for _ in range(3)]
    _assert_bitwise(runs)
    r = runs[0]
    d64 = lambda ts, cast=False: [(t.to(torch.bfloat16) if cast else t).to(DEV, torch.float64) for t in ts]
    if kind == "parts":
        with _flag_off():
            with torch.no_grad():
                xg, _ = O.gate_concat(d64(f4, True), d64(cl), d64(ct))
            z, _, _ = O.tpavi_fwd_bwd(xg, torch.stack(d64(do, True), dim=2), _dev64(pg))
        for v in range(V):
            assert_close(f"glob{v}", r[f"out{v}"], z[:, :, v], BF16_TOL)
        return
    with _flag_off():
        outs, df4, dcls, dctr, gg, gl = O.fusion_fwd_bwd(d64(f4, True), d64(cl), d64(ct), d64(do, True), _dev64(pg),
                                                        _dev64(pl))
    for v in range(V):
        assert_close(f"out{v}", r[f"out{v}"], outs[v], BF16_TOL)
        assert_close(f"df4_{v}", r[f"df4_{v}"], df4[v], BF16_TOL)
    for tag, ref in (("g", gg), ("l", gl)):
        scale = grad_scale(ref.values())
        for name, t in ref.items():
            assert_close(f"{tag}:{name}", r[f"{tag}:grad:{name}"].reshape(t.shape), t, grad_tol(name), zero_scale=scale)


def test_cuda_graph_replays_the_deterministic_path(deterministic):
    C_, V, B, h, w = 256, 4, 2, 14, 14
    pg, pl = O.init_params(C_, seed=31), O.init_params(C_, seed=32)
    f4, cl, ct, do = _fusion_inputs(C_, V, B, h, w, seed=33)
    with dot_algo("token"):
        eager = _fusion_run("stacked", C_, pg, pl, f4, cl, ct, do)
        f = _fusion(C_, pg, pl)
        f4d = [t.to(DEV, torch.bfloat16).requires_grad_(True) for t in f4]
        cld, ctd = [t.to(DEV) for t in cl], [t.to(DEV) for t in ct]
        dzd = torch.stack(do, dim=2).to(DEV, torch.bfloat16)
        params = [p for p in f.parameters() if p.requires_grad]
        holder = {}

        def compute():
            for t in f4d:
                t.grad = None
            for p in params:
                p.grad = None
            holder["out"] = f.forward_stacked(f4d, cld, ctd)
            holder["out"].backward(dzd)

        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                compute()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            compute()
        graph.replay()
        torch.cuda.synchronize()
    out = holder["out"].detach()
    for v in range(V):
        assert torch.equal(out[:, :, v], eager[f"out{v}"]), f"out{v}"
        assert torch.equal(f4d[v].grad, eager[f"df4_{v}"]), f"df4_{v}"
    for tag, mod in (("g", f.global_attn), ("l", f.local_attn)):
        for name, t in mod.named_parameters():
            if t.grad is not None:
                assert torch.equal(t.grad, eager[f"{tag}:grad:{name}"]), f"{tag}:{name}"


def test_default_path_returns_after_the_flag_is_restored():
    """The same module under the flag, then with it restored (off): the default path's sizes and results again."""
    C_, T, H, W, B = 256, 4, 28, 28, 16
    p = O.init_params(C_, seed=41)
    x, dz = _inputs(B, C_, T, H, W, seed=42, mode="dot")
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        on = _block_run(p, "dot", x, dz, "token", torch.bfloat16, "bf16", None)
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)
    from glfusion_b200 import _lib as L
    from glfusion_b200.tpavi import TPAVIState
    st = TPAVIState(B, C_, T, H, W, C_ // 2, L.MODE_DOT, L.DTYPE_BF16, L.LAYOUT_NCTHW, True, True)
    assert st.desc.reserved[1] & L.DETERMINISTIC == 0
    off = _block_run(p, "dot", x, dz, "token", torch.bfloat16, "bf16", None)
    for k in on:
        assert_close(k, off[k], on[k], BF16_TOL, abs_floor=1e-3)
