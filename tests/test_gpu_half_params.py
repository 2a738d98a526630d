"""TPAVIModule and GlobalLocalFusion cast as a whole (``.half()``, ``.bfloat16()``): 2-byte parameters, BatchNorm running
statistics and gradients.  Such a block computes what an fp32-parameter block holding the same values computes; the
only new roundings are the stores of the gradients and of the updated running statistics."""
import copy

import pytest
import torch

from gpu_util import BF16_TOL, DEV, assert_close, dot_algo, grad_scale, grad_tol, load_module_from_params
from glfusion_b200 import GlobalLocalFusion, TPAVIModule
from oracle import tpavi_oracle as O

pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
IDS = ["bf16", "fp16"]


def _round(p, dt):
    """The parameters / buffers rounded to `dt`, kept in fp32 (the oracle's and the fp32 module's values)."""
    return {k: (v.to(dt).float() if v.is_floating_point() else v.clone()) for k, v in p.items()}


def _assert_dtypes(mod, dt):
    for k, p in mod.named_parameters():
        assert p.dtype == dt, k
        if p.grad is not None:
            assert p.grad.dtype == dt, k
    for k, b in mod.named_buffers():
        assert b.dtype == (torch.int64 if k.endswith("num_batches_tracked") else dt), k


def _within_ulp(got, ref, dt):
    """|got - ref| <= 1 ulp of dt at ref (both already representable in dt)."""
    got, ref = got.float(), ref.to(dt).float()
    ulp = torch.finfo(dt).eps * ref.abs() + torch.finfo(dt).tiny
    assert ((got - ref).abs() <= ulp).all(), float((got - ref).abs().max())


# ------------------------------------------------------------------------------------------------ bitwise equivalence
@pytest.mark.parametrize("dt", HALF, ids=IDS)
def test_half_block_equals_fp32_block_on_the_same_values(dt):
    """Dot mode, Gram form, 96 sequences (every reduction fixed-order, DESIGN.md §4): z and dx bitwise equal, each
    gradient is the fp32 block's gradient rounded to dt, the running statistics agree within 1 ulp."""
    B, C, T, H, W = 96, 256, 1, 8, 8
    p = _round(O.init_params(C, seed=201, randomize_affine=True), dt)
    p["W_z.1.running_mean"] = (torch.randn(C, generator=torch.Generator().manual_seed(202)) * 0.1).to(dt).float()
    mf = load_module_from_params(TPAVIModule, p, C, "dot", True).train()
    mh = copy.deepcopy(mf).to(dt)
    gen = torch.Generator().manual_seed(203)
    x = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    dz = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    res = {}
    for tag, m in (("f32", mf), ("half", mh)):
        xd = x.clone().requires_grad_(True)
        with dot_algo("gram"):
            z, _ = m(xd)
            z.backward(dz)
        torch.cuda.synchronize()
        res[tag] = (z.detach(), xd.grad)
    assert torch.equal(res["f32"][0], res["half"][0])
    assert torch.equal(res["f32"][1], res["half"][1])
    _assert_dtypes(mh, dt)
    pf, ph = dict(mf.named_parameters()), dict(mh.named_parameters())
    for k in ph:
        if k.startswith("align_channel"):
            continue
        assert torch.equal(ph[k].grad, pf[k].grad.to(dt)), k
    bf, bh = mf.W_z[1], mh.W_z[1]
    _within_ulp(bh.running_mean, bf.running_mean, dt)
    _within_ulp(bh.running_var, bf.running_var, dt)
    assert int(bh.num_batches_tracked) == int(bf.num_batches_tracked) == 1


# ------------------------------------------------------------------------------------------------ oracle parity
@pytest.mark.parametrize("dt", HALF, ids=IDS)
@pytest.mark.parametrize("cfg", ["dot-token", "dot-gram", "embedded"])
@pytest.mark.parametrize("layout", ["ncthw", "token"])
@pytest.mark.parametrize("state", ["train", "eval", "frozen_bn", "nobn"])
def test_tpavi_half_module_vs_oracle(dt, cfg, layout, state):
    mode, algo = (cfg.split("-") + ["auto"])[:2]
    B, C, T, H, W = 2, 128, 2, 8, 8
    bn = state != "nobn"
    p = O.init_params(C, seed=211, randomize_affine=True, bn_layer=bn)
    if bn:
        p["W_z.1.running_mean"] = torch.randn(C, generator=torch.Generator().manual_seed(212)) * 0.1
    p = _round(p, dt)
    gen = torch.Generator().manual_seed(213)
    x = torch.randn(B, C, T, H, W, generator=gen).to(dt).float()
    dz = torch.randn(B, C, T, H, W, generator=gen).to(dt).float()
    bn_training = state in ("train", "nobn")
    pref = {k: v.clone() for k, v in p.items()}
    zo, dxo, go = O.tpavi_fwd_bwd(x, dz, pref, mode=mode, training=bn_training, bn_layer=bn)
    kw = dict(zero_scale=grad_scale(go.values())) if mode == "embedded" else dict(abs_floor=1e-3)
    m = load_module_from_params(TPAVIModule, p, C, mode, bn).to(dt).train(state != "eval")
    if state == "frozen_bn":
        m.W_z[1].eval()                     # model.train(); bn.eval(): BatchNorm on its running statistics
    xd, dzd = x.to(DEV, dt), dz.to(DEV, dt)
    if layout == "token":
        xd = xd.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
        dzd = dzd.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
    xd.requires_grad_(True)
    with dot_algo(algo):
        z, _ = m(xd)
        z.backward(dzd)
    torch.cuda.synchronize()
    assert z.dtype == dt and xd.grad.dtype == dt
    assert_close("z", z, zo, BF16_TOL)
    assert_close("dx", xd.grad, dxo, BF16_TOL)
    for k, q in m.named_parameters():
        if not k.startswith("align_channel"):
            assert_close("grad:" + k, q.grad, go[k], grad_tol(k, mode), **kw)
    _assert_dtypes(m, dt)
    if bn:
        sd = m.state_dict()
        for k in ("W_z.1.running_mean", "W_z.1.running_var"):
            assert_close(k, sd[k], pref[k], 1e-2)
        assert int(sd["W_z.1.num_batches_tracked"]) == int(pref["W_z.1.num_batches_tracked"])


def _fusion(C, pg, pl, dt):
    f = GlobalLocalFusion(in_channels=C)
    f.global_attn.load_state_dict({k: v.clone() for k, v in pg.items()}, strict=True)
    f.local_attn.load_state_dict({k: v.clone() for k, v in pl.items()}, strict=True)
    return f.to(DEV).to(dt).train()


def _fusion_inputs(B, C, V, h, w, seed, dt):
    gen = torch.Generator().manual_seed(seed)
    f4 = [torch.randn(B, C, h, w, generator=gen).to(dt).float() for _ in range(V)]
    cl = [torch.randn(B, 5, h, w, generator=gen) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, generator=gen) for _ in range(V)]
    do = [torch.randn(B, C, h, w, generator=gen).to(dt).float() for _ in range(V)]
    return f4, cl, ct, do


# C = 256: the bulk-copy LayerNorm pair and the Gram form;  C = 2048: the wide-row ring LayerNorm and the token-space form
@pytest.mark.parametrize("dt", HALF, ids=IDS)
@pytest.mark.parametrize("shape", [(2, 256, 4, 28, 28), (2, 2048, 2, 4, 4)], ids=["C256", "C2048"])
@pytest.mark.parametrize("entry", ["stacked", "dict", "parts"])
def test_fusion_half_module_vs_oracle(dt, shape, entry):
    B, C, V, h, w = shape
    pg = _round(O.init_params(C, seed=221, randomize_affine=True), dt)
    pl = _round(O.init_params(C, seed=222, randomize_affine=True), dt)
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 223, dt)
    gref, lref = {k: v.clone() for k, v in pg.items()}, {k: v.clone() for k, v in pl.items()}
    outs, df4, _, _, gg, gl = O.fusion_fwd_bwd(f4, cl, ct, do, gref, lref)
    f = _fusion(C, pg, pl, dt)
    f4d = [t.to(DEV, dt).requires_grad_(True) for t in f4]
    cld, ctd = [t.to(DEV) for t in cl], [t.to(DEV) for t in ct]
    keys = [str(v) for v in range(V)]
    if entry == "stacked":
        out = f.forward_stacked(f4d, cld, ctd)
        out.backward(torch.stack(do, dim=2).to(DEV, dt))
        res = [out[:, :, v] for v in range(V)]
    else:
        fwd = f if entry == "dict" else f.forward_parts
        o = fwd(dict(zip(keys, f4d)), dict(zip(keys, cld)), dict(zip(keys, ctd)))
        if entry == "parts":
            o, glob, loc = o
            with torch.no_grad():
                zg = O.tpavi_forward(O.gate_concat(f4, cl, ct)[0], {k: v.clone() for k, v in pg.items()})
            for i, k in enumerate(keys):
                assert glob[k].dtype == dt and loc[k].dtype == dt
                assert_close(f"global:{k}", glob[k], zg[:, :, i], BF16_TOL)
        res = [o[k] for k in keys]
        torch.autograd.backward(res, [t.to(DEV, dt) for t in do])
    torch.cuda.synchronize()
    for v in range(V):
        assert res[v].dtype == dt and f4d[v].grad.dtype == dt
        assert_close(f"out:{v}", res[v], outs[v], BF16_TOL)
        assert_close(f"df4:{v}", f4d[v].grad, df4[v], BF16_TOL)
    for mod, ref, rp in ((f.global_attn, gg, gref), (f.local_attn, gl, lref)):
        _assert_dtypes(mod, dt)
        for k, q in mod.named_parameters():
            if not k.startswith("align_channel"):
                assert_close("grad:" + k, q.grad, ref[k], grad_tol(k), abs_floor=1e-3)
        sd = mod.state_dict()
        for k in ("W_z.1.running_mean", "W_z.1.running_var"):
            assert_close(k, sd[k], rp[k], 1e-2)


# ------------------------------------------------------------------------------------------------ no casts, launches
def _profile(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    events = list(prof.events())
    ops = [e.name for e in events if e.device_type == torch.autograd.DeviceType.CPU]
    kernels = sum(1 for e in events if e.device_type == torch.autograd.DeviceType.CUDA)
    return ops, kernels


def test_fused_step_makes_no_casts_and_two_launches_per_block():
    B, C, V, h, w = 2, 256, 4, 28, 28
    pg = _round(O.init_params(C, seed=231, randomize_affine=True), torch.bfloat16)
    pl = _round(O.init_params(C, seed=232, randomize_affine=True), torch.bfloat16)
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 233, torch.bfloat16)
    cld, ctd = [t.to(DEV) for t in cl], [t.to(DEV) for t in ct]
    xs = [t.to(DEV, torch.bfloat16).requires_grad_(True) for t in f4]
    # dz token-major, as the node's own output is: the backward then copies no activation either
    dz = torch.stack(do, dim=2).to(DEV, torch.bfloat16).permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
    res = {}
    for pdt in (torch.float32, torch.bfloat16):
        f = _fusion(C, pg, pl, pdt)

        def step():
            f.forward_stacked(xs, cld, ctd).backward(dz)
        step()                                   # warm-up (module loads, attribute set-up)
        f.zero_grad(set_to_none=True)
        for t in xs:
            t.grad = None
        res[pdt] = _profile(step)
        _assert_dtypes(f.global_attn, pdt)
        _assert_dtypes(f.local_attn, pdt)
    ops, kernels = res[torch.bfloat16]
    casts = [o for o in ops if o in ("aten::to", "aten::_to_copy", "aten::copy_")]
    assert not casts, casts
    assert kernels <= res[torch.float32][1] + 2 * 2, (kernels, res[torch.float32][1])


# ------------------------------------------------------------------------------------------------ CUDA graphs
def test_bf16_training_step_replays_from_a_cuda_graph():
    """Forward, backward and AdamW.step of a bf16 block captured once and replayed: the same parameters as the same
    steps run eagerly (96 sequences, Gram form: every reduction is fixed-order)."""
    B, C, T, H, W = 96, 256, 1, 8, 8
    p = O.init_params(C, seed=241, randomize_affine=True)
    base = load_module_from_params(TPAVIModule, p, C, "dot", True).to(torch.bfloat16).train()
    gen = torch.Generator().manual_seed(242)
    x = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    dz = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    models = {k: copy.deepcopy(base) for k in ("eager", "graph")}
    opts = {k: torch.optim.AdamW(m.parameters(), lr=1e-2, capturable=True) for k, m in models.items()}

    def step(k):
        opts[k].zero_grad(set_to_none=True)
        z, _ = models[k](x)
        z.backward(dz)
        opts[k].step()
    with dot_algo("gram"):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):                  # warm-up: optimizer state, module loads
                step("graph")
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        opts["graph"].zero_grad(set_to_none=True)
        with torch.cuda.graph(g):
            step("graph")
        for _ in range(3):
            g.replay()
        for _ in range(5):
            step("eager")
    torch.cuda.synchronize()
    me, mg = dict(models["eager"].named_parameters()), dict(models["graph"].named_parameters())
    for k in me:
        assert me[k].dtype == torch.bfloat16
        assert torch.equal(me[k], mg[k]), k
    be, bg = models["eager"].W_z[1], models["graph"].W_z[1]
    assert torch.equal(be.running_mean, bg.running_mean) and torch.equal(be.running_var, bg.running_var)
    assert int(be.num_batches_tracked) == int(bg.num_batches_tracked) == 5


# ------------------------------------------------------------------------------------------------ mixed dtypes, fp32 arm
def test_mixed_parameter_dtypes_keep_the_fp32_path():
    """bf16 convs beside fp32 norm layers (the usual 'keep normalisation in fp32' recipe): fp32 copies as before, so the
    block computes exactly what the fp32 block on the same values computes, and each gradient comes back in its
    parameter's dtype."""
    B, C, T, H, W = 96, 256, 1, 8, 8
    p = O.init_params(C, seed=251, randomize_affine=True)
    mf = load_module_from_params(TPAVIModule, p, C, "dot", True).train()
    mm = copy.deepcopy(mf).to(torch.bfloat16)
    mm.norm_layer.float()
    mm.W_z[1].float()
    with torch.no_grad():
        for k, q in mf.named_parameters():
            q.copy_(dict(mm.named_parameters())[k].float())
    gen = torch.Generator().manual_seed(252)
    x = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    dz = torch.randn(B, C, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    res = {}
    for tag, m in (("f32", mf), ("mixed", mm)):
        xd = x.clone().requires_grad_(True)
        with dot_algo("gram"):
            z, _ = m(xd)
            z.backward(dz)
        torch.cuda.synchronize()
        res[tag] = (z.detach(), xd.grad)
    assert torch.equal(res["f32"][0], res["mixed"][0]) and torch.equal(res["f32"][1], res["mixed"][1])
    pf = dict(mf.named_parameters())
    for k, q in mm.named_parameters():
        if k.startswith("align_channel"):
            continue
        assert q.grad.dtype == q.dtype, k
        assert torch.equal(q.grad, pf[k].grad.to(q.dtype)), k
    assert torch.equal(mm.W_z[1].running_mean, mf.W_z[1].running_mean)
    assert torch.equal(mm.W_z[1].running_var, mf.W_z[1].running_var)


@pytest.mark.parametrize("dt", HALF, ids=IDS)
def test_fp32_precision_refuses_half_parameters_before_any_launch(dt):
    B, C, V, h, w = 2, 128, 2, 8, 8
    m = TPAVIModule(C).to(DEV).to(dt)
    m.compute_precision = "fp32"
    with pytest.raises(TypeError, match="float32 parameters"):
        m(torch.randn(B, C, 2, h, w, device=DEV))
    f = GlobalLocalFusion(in_channels=C).to(DEV).to(dt)
    f.global_attn.compute_precision = f.local_attn.compute_precision = "fp32"
    f4 = [torch.randn(B, C, h, w, device=DEV) for _ in range(V)]
    cl = [torch.randn(B, 5, h, w, device=DEV) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, device=DEV) for _ in range(V)]
    with pytest.raises(TypeError, match="float32 parameters"):
        f.forward_stacked(f4, cl, ct)
