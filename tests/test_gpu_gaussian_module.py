"""TPAVIModule(mode='gaussian') and GlobalLocalFusion(mode='gaussian') against the oracle's literal restatement of the
reference (oracle/tpavi_oracle.py: tpavi_fwd_bwd / fusion_fwd_bwd with mode='gaussian', f = x x^T on the block input
itself) in float64, on clustered tokens whose softmax is non-trivial (test_gpu_gaussian_attention.clustered_tokens).

Tolerance: 2e-2 relative L2, as for the other modes.  Where a tensor is ill-conditioned in bf16 for any implementation,
the bound is the oracle's own error under torch.autocast(bfloat16) against its float64 run on the same inputs, measured
here, capped at 4e-2.  theta / phi take no part in mode='gaussian': their .grad must stay None."""
import copy
import json

import pytest
import torch

from glfusion_b200 import GlobalLocalFusion, TPAVIModule
from glfusion_b200.dp import GradBucket
from gpu_util import BF16_TOL, DEV, assert_close, grad_scale
from oracle import tpavi_oracle as O
from test_gpu_gaussian_attention import clustered_tokens, witness

pytestmark = pytest.mark.gpu

UNUSED = ("theta.weight", "theta.bias", "phi.weight", "phi.bias")


def _tol(name, floors):
    f = floors.get(name, 0.0)
    return BF16_TOL if f <= BF16_TOL else min(f, 4e-2)


def _oracle(x, dz, p, training, bn_layer, dtype, autocast=False):
    """z, dx, grads and the updated parameter dict of the oracle on DEV in `dtype` (optionally under bf16 autocast)."""
    q = {k: (v.to(DEV, dtype) if v.is_floating_point() else v.to(DEV)) for k, v in p.items()}
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        z, dx, g = O.tpavi_fwd_bwd(x.to(DEV, dtype), dz.to(DEV, dtype), q, mode="gaussian", training=training,
                                   bn_layer=bn_layer)
    return z, dx, g, q


def _floors(x, dz, p, training, bn_layer, ref):
    z32, dx32, g32, _ = _oracle(x, dz, p, training, bn_layer, torch.float32, autocast=True)
    z, dx, g = ref
    out = {"z": O.rel_err(z32, z), "dx": O.rel_err(dx32, dx)}
    out.update({k: O.rel_err(g32[k], g[k]) for k in g})
    return out


def _inputs(B, C_, T, H, W, seed):
    gen = torch.Generator().manual_seed(seed)
    N = T * H * W
    x = clustered_tokens(B, N, C_, gen).reshape(B, T, H, W, C_).permute(0, 4, 1, 2, 3)
    dz = torch.randn(B, C_, T, H, W, generator=gen, dtype=torch.float64)
    return x, dz


CASES = [
    # C, (T, H, W), B, training, bn_layer, io dtype, token-major input
    (128, (2, 8, 16), 2, True, True, torch.bfloat16, False),      # flash (128, 64)
    (128, (2, 8, 16), 2, False, True, torch.float32, True),       # eval: running statistics
    (128, (3, 5, 7), 2, True, False, torch.float16, False),       # bn_layer=False, N = 105 (masked tail)
    (64, (2, 8, 8), 3, True, True, torch.float32, True),          # chunked (64, 32)
    (256, (4, 28, 28), 2, True, True, torch.bfloat16, True),      # chunked (256, 128): cfg2's N = 3136
    (192, (2, 10, 10), 2, False, False, torch.bfloat16, False),   # chunked (192, 96), eval without BatchNorm
]


def _id(c):
    return f"C{c[0]}-N{c[1][0] * c[1][1] * c[1][2]}-{'train' if c[3] else 'eval'}-{'bn' if c[4] else 'nobn'}-" \
           f"{str(c[5]).split('.')[-1]}-{'token' if c[6] else 'ncthw'}"


def _run_module(m, x, dz, dtype, token_major):
    xi = x.to(DEV, dtype)
    if token_major:
        xi = xi.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
    xi = xi.detach().requires_grad_(True)
    z, _ = m(xi)
    z.backward(dz.to(DEV, dtype))
    torch.cuda.synchronize()
    return z.detach(), xi.grad.detach()


def _check_module(tag, m, x, dz, p, training, bn_layer, dtype, token_major):
    z, dx = _run_module(m, x, dz, dtype, token_major)
    # the oracle reads the values the module read
    xr = x.to(dtype).double()
    dzr = dz.to(dtype).double()
    pr = {k: (v.to(m.g.weight.dtype).double() if v.is_floating_point() else v) for k, v in p.items()}
    zr, dxr, gr, q = _oracle(xr, dzr, pr, training, bn_layer, torch.float64)
    wit = witness(((xr[0].reshape(xr.shape[1], -1).T) @ xr[0].reshape(xr.shape[1], -1)).to(DEV))
    floors = _floors(xr, dzr, pr, training, bn_layer, (zr, dxr, gr))
    report = {"case": tag, "pmax": round(wit[0], 3), "not_self": round(wit[1], 3),
              "z": O.rel_err(z, zr), "dx": O.rel_err(dx, dxr)}
    assert_close("z", z, zr, _tol("z", floors))
    assert_close("dx", dx, dxr, _tol("dx", floors))
    grads = {k: p_.grad for k, p_ in m.named_parameters() if not k.startswith("align_channel")}
    for k in UNUSED:
        assert grads[k] is None, f"{k}.grad must stay None in mode='gaussian'"
    scale = grad_scale(gr.values())
    used = [k for k in grads if k not in UNUSED]
    assert sorted(used) == sorted(gr), (used, list(gr))
    assert len(used) == (8 if bn_layer else 6)
    for k in used:
        report[k] = O.rel_err(grads[k], gr[k])
        assert_close("grad:" + k, grads[k], gr[k], _tol(k, floors), zero_scale=scale)
    if bn_layer:
        bn = m.W_z[1]
        assert_close("running_mean", bn.running_mean, q["W_z.1.running_mean"], BF16_TOL, abs_floor=1e-3)
        assert_close("running_var", bn.running_var, q["W_z.1.running_var"], BF16_TOL)
        assert int(bn.num_batches_tracked) == int(q["W_z.1.num_batches_tracked"])
    print("GAUSS-MODULE " + json.dumps({k: (float(f"{v:.3e}") if isinstance(v, float) else v)
                                         for k, v in report.items()}))


@pytest.mark.parametrize("case", CASES, ids=_id)
def test_module_against_oracle(case):
    C_, (T, H, W), B, training, bn_layer, dtype, token_major = case
    p = O.init_params(C_, seed=41 + C_, randomize_affine=True, bn_layer=bn_layer)
    x, dz = _inputs(B, C_, T, H, W, seed=42 + C_)
    m = TPAVIModule(C_, mode="gaussian", bn_layer=bn_layer)
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m = m.to(DEV).train(training)
    _check_module(_id(case), m, x, dz, p, training, bn_layer, dtype, token_major)


def test_half_module_against_oracle():
    """A .half() module: fp16 parameters, BatchNorm buffers and gradients, fp16 activations."""
    C_, T, H, W, B = 128, 2, 8, 16, 2
    p = O.init_params(C_, seed=51, randomize_affine=True)
    x, dz = _inputs(B, C_, T, H, W, seed=52)
    m = TPAVIModule(C_, mode="gaussian")
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m = m.to(DEV).half().train()
    _check_module("half-C128", m, x, dz, p, True, True, torch.float16, False)
    assert m.g.weight.grad.dtype == torch.float16 and m.W_z[1].running_mean.dtype == torch.float16


def test_grad_bucket_leaves_theta_phi_none():
    """dp.GradBucket over gaussian blocks: after allreduce_mean() the unused parameters' .grad is still None and the
    used ones carry their gradients (single process: the mean over one rank is the gradient itself)."""
    C_ = 128
    p = O.init_params(C_, seed=61, randomize_affine=True)
    m = TPAVIModule(C_, mode="gaussian")
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m = m.to(DEV).train()
    bucket = GradBucket(m._plist())
    bucket.bind([m])
    x, dz = _inputs(2, C_, 2, 8, 8, seed=62)
    _run_module(m, x, dz, torch.bfloat16, False)
    want = {k: p_.grad.clone() for k, p_ in m.named_parameters() if p_.grad is not None}
    bucket.allreduce_mean()
    torch.cuda.synchronize()
    for k, p_ in m.named_parameters():
        if k in UNUSED:
            assert p_.grad is None, k
    for k, g in want.items():
        assert torch.equal(dict(m.named_parameters())[k].grad, g), k


def test_cuda_graph_replay_equals_eager():
    """z, dx and the BatchNorm buffers bitwise; the weight gradients are token contractions that the GEMM reduces over
    K slices with fp32 atomics (as in every mode), so they agree to fp32 summation order."""
    C_, T, H, W, B = 128, 2, 8, 16, 2
    p = O.init_params(C_, seed=71, randomize_affine=True)
    m = TPAVIModule(C_, mode="gaussian")
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m = m.to(DEV).train()
    x, dz = _inputs(B, C_, T, H, W, seed=72)
    xd = x.to(DEV, torch.bfloat16).detach().requires_grad_(True)
    dzd = dz.to(DEV, torch.bfloat16)
    params = [q for k, q in m.named_parameters() if k.split(".")[0] not in ("align_channel", "theta", "phi")]
    state0 = copy.deepcopy(m.state_dict())
    holder = {}

    def step():
        xd.grad = None
        for q in m.parameters():
            q.grad = None
        holder["z"], _ = m(xd)
        holder["z"].backward(dzd)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    m.load_state_dict(state0)       # the warm-up steps moved the running statistics
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    m.load_state_dict(state0)
    holder["z"].detach().zero_()
    xd.grad.detach().zero_()
    graph.replay()
    torch.cuda.synchronize()
    got = (holder["z"].detach().clone(), xd.grad.clone(), [q.grad.clone() for q in params],
           m.W_z[1].running_mean.clone(), m.W_z[1].running_var.clone())
    m.load_state_dict(state0)
    step()
    torch.cuda.synchronize()
    ref = (holder["z"].detach(), xd.grad, [q.grad for q in params], m.W_z[1].running_mean, m.W_z[1].running_var)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for a, b in zip(got[2], ref[2]):
        assert O.rel_err(a, b) < 1e-5
    assert torch.equal(got[3], ref[3]) and torch.equal(got[4], ref[4])
    assert m.theta.weight.grad is None and m.phi.bias.grad is None


def _fusion_inputs(B, C_, V, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    x = clustered_tokens(B, V * h * w, C_, gen).reshape(B, V, h, w, C_)
    f4 = [x[:, v].permute(0, 3, 1, 2).contiguous() for v in range(V)]
    cl = [torch.randn(B, 5, h, w, generator=gen, dtype=torch.float64) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, generator=gen, dtype=torch.float64) for _ in range(V)]
    do = [torch.randn(B, C_, h, w, generator=gen, dtype=torch.float64) for _ in range(V)]
    return f4, cl, ct, do


@pytest.mark.parametrize("api", ["stacked", "dict", "parts"])
@pytest.mark.parametrize("C_", [128, 256])
def test_fusion_against_oracle(api, C_):
    B, V, h, w = 2, 4, 8, 8
    pg = O.init_params(C_, seed=81, randomize_affine=True)
    pl = O.init_params(C_, seed=82, randomize_affine=True)
    f4, cl, ct, do = _fusion_inputs(B, C_, V, h, w, seed=83)
    f4b = [t.to(torch.bfloat16) for t in f4]
    dob = [t.to(torch.bfloat16) for t in do]
    def oracle(dt, autocast):
        q = lambda p: {k: (v.to(DEV, dt) if v.is_floating_point() else v.to(DEV)) for k, v in p.items()}
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            return O.fusion_fwd_bwd([t.to(DEV, dt) for t in f4b], [t.to(DEV, dt) for t in cl],
                                    [t.to(DEV, dt) for t in ct], [t.to(DEV, dt) for t in dob], q(pg), q(pl),
                                    mode="gaussian")
    outs, df4, _, _, gg, gl = oracle(torch.float64, False)
    # the oracle's own bf16 error on these inputs: the bound of the tensors that are ill-conditioned in bf16
    o32, d32, _, _, g32, l32 = oracle(torch.float32, True)
    floors = {"out": max(O.rel_err(a, b) for a, b in zip(o32, outs)), "df4": max(O.rel_err(a, b) for a, b in zip(d32, df4))}
    gfloor = [{k: O.rel_err(a[k], b[k]) for k in b} for a, b in ((g32, gg), (l32, gl))]
    f = GlobalLocalFusion(in_channels=C_, mode="gaussian")
    f.global_attn.load_state_dict(pg, strict=True)
    f.local_attn.load_state_dict(pl, strict=True)
    f = f.to(DEV).train()
    f4d = [t.to(DEV).requires_grad_(True) for t in f4b]
    cld, ctd = [t.to(DEV, torch.float32) for t in cl], [t.to(DEV, torch.float32) for t in ct]
    if api == "stacked":
        out = f.forward_stacked(f4d, cld, ctd)
        out.backward(torch.stack(dob, dim=2).to(DEV))
        got = [out[:, :, v] for v in range(V)]
    else:
        views = [f"v{i}" for i in range(V)]
        args = ({k: t for k, t in zip(views, f4d)}, {k: t for k, t in zip(views, cld)},
                {k: t for k, t in zip(views, ctd)})
        res = f(*args) if api == "dict" else f.forward_parts(*args)[0]
        got = [res[k] for k in views]
        torch.autograd.backward(got, [t.to(DEV) for t in dob])
    torch.cuda.synchronize()
    print("GAUSS-FUSION " + json.dumps(dict(api=api, C=C_, floor_out=float(f"{floors['out']:.3e}"),
                                            floor_df4=float(f"{floors['df4']:.3e}"),
                                            df4=float(f"{max(O.rel_err(f4d[v].grad, df4[v]) for v in range(V)):.3e}"))))
    for v in range(V):
        assert_close(f"out:{v}", got[v], outs[v], _tol("out", floors))
        assert_close(f"df4:{v}", f4d[v].grad, df4[v], _tol("df4", floors))
    for mod, ref, fl in ((f.global_attn, gg, gfloor[0]), (f.local_attn, gl, gfloor[1])):
        scale = grad_scale(ref.values())
        for k, p_ in mod.named_parameters():
            if k.startswith("align_channel"):
                continue
            if k in UNUSED:
                assert p_.grad is None, k
                continue
            assert_close("grad:" + k, p_.grad, ref[k], _tol(k, fl), zero_scale=scale)
