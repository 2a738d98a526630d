"""float16 activations (torch.autocast's default dtype, paired with torch.amp.GradScaler) through TPAVIModule and
GlobalLocalFusion.  fp16 is an I/O dtype only: the inputs are rounded to fp16 here, the CPU oracle runs on those same
values, and the bounds are the bf16 arm's (the products in between are bf16 in both)."""
import pytest
import torch

from gpu_util import BF16_TOL, DEV, assert_close, dot_algo, grad_scale, grad_tol, load_module_from_params
from glfusion_b200 import GlobalLocalFusion, TPAVIModule, cycle
from oracle import cycle_oracle as CO
from oracle import tpavi_oracle as O

pytestmark = pytest.mark.gpu

H16 = torch.float16
FP16_MAX = 65504.0


def _h(t):
    """fp16-rounded values, kept in fp32 for the oracle."""
    return t.to(H16).float()


def _fusion(C, pg, pl):
    f = GlobalLocalFusion(in_channels=C)
    f.global_attn.load_state_dict({k: v.clone() for k, v in pg.items()}, strict=True)
    f.local_attn.load_state_dict({k: v.clone() for k, v in pl.items()}, strict=True)
    return f.to(DEV).train()


def _fusion_inputs(B, C, V, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    f4 = [_h(torch.randn(B, C, h, w, generator=gen)) for _ in range(V)]
    cl = [torch.randn(B, 5, h, w, generator=gen) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, generator=gen) for _ in range(V)]
    do = [_h(torch.randn(B, C, h, w, generator=gen)) for _ in range(V)]
    return f4, cl, ct, do


def _to_dev(t, fmt):
    t = t.to(DEV, H16)
    return t.contiguous(memory_format=torch.channels_last) if fmt == "cl" else t


def _check_params(f, gg, gl):
    for mod, ref in ((f.global_attn, gg), (f.local_attn, gl)):
        for k, p in mod.named_parameters():
            if not k.startswith("align_channel"):
                assert_close("grad:" + k, p.grad, ref[k], grad_tol(k), abs_floor=1e-3)


# ------------------------------------------------------------------------------------------------ TPAVIModule
@pytest.mark.parametrize("cfg", ["dot-token", "dot-gram", "embedded"])
@pytest.mark.parametrize("layout", ["ncthw", "token"])
@pytest.mark.parametrize("state", ["train", "eval", "nobn"])
def test_tpavi_module_fp16_in_and_out(cfg, layout, state):
    mode, algo = (cfg.split("-") + ["auto"])[:2]
    B, C, T, H, W = 2, 128, 2, 8, 8
    bn = state != "nobn"
    p = O.init_params(C, seed=101, randomize_affine=True, bn_layer=bn)
    if bn:
        p["W_z.1.running_mean"] = torch.randn(C, generator=torch.Generator().manual_seed(5)) * 0.1
    gen = torch.Generator().manual_seed(102)
    x = _h(torch.randn(B, C, T, H, W, generator=gen))
    dz = _h(torch.randn(B, C, T, H, W, generator=gen))
    training = state != "eval"
    pref = {k: v.clone() for k, v in p.items()}
    zo, dxo, go = O.tpavi_fwd_bwd(x, dz, pref, mode=mode, training=training, bn_layer=bn)
    # softmax mode: the biases whose shift the softmax / BatchNorm cancels are ~0, bounded against the real gradients
    kw = dict(zero_scale=grad_scale(go.values())) if mode == "embedded" else dict(abs_floor=1e-3)
    m = load_module_from_params(TPAVIModule, p, C, mode, bn).train(training)

    def run(dt):
        xd, dzd = x.to(DEV, dt), dz.to(DEV, dt)
        if layout == "token":
            xd = xd.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
            dzd = dzd.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
        xd.requires_grad_(True)
        with dot_algo(algo):
            z, _ = m(xd)
            z.backward(dzd)
        torch.cuda.synchronize()
        return z.detach(), xd.grad
    z, dx = run(H16)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    grads = {k: q.grad.clone() for k, q in m.named_parameters() if q.grad is not None}
    assert z.dtype == H16 and dx.dtype == H16
    assert_close("z", z, zo, BF16_TOL)
    assert_close("dx", dx, dxo, BF16_TOL)
    for k, g in grads.items():
        assert_close("grad:" + k, g, go[k], grad_tol(k, mode), **kw)
    if bn:
        for k in ("W_z.1.running_mean", "W_z.1.running_var"):
            assert_close(k, sd[k], pref[k], 1e-2)
    m.zero_grad(set_to_none=True)
    zb, dxb = run(torch.bfloat16)                       # the strides the bf16 path returns
    assert z.stride() == zb.stride() and dx.stride() == dxb.stride()


# ------------------------------------------------------------------------------------------------ GlobalLocalFusion
SHAPES = [(2, 256, 4, 28, 28), (3, 128, 3, 5, 7), (2, 512, 2, 4, 4), (2, 2048, 2, 4, 4)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"C{s[1]}_{s[3]}x{s[4]}")
@pytest.mark.parametrize("fmt", ["nchw", "cl"])
@pytest.mark.parametrize("entry", ["stacked", "dict"])
def test_fusion_fp16_f4(shape, fmt, entry):
    B, C, V, h, w = shape
    pg = O.init_params(C, seed=111, randomize_affine=True)
    pl = O.init_params(C, seed=112, randomize_affine=True)
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 113)
    outs, df4, dcls, dctr, gg, gl = O.fusion_fwd_bwd(f4, cl, ct, do, {k: v.clone() for k, v in pg.items()},
                                                     {k: v.clone() for k, v in pl.items()})
    f = _fusion(C, pg, pl)
    f4d = [_to_dev(t, fmt).requires_grad_(True) for t in f4]
    cld = [t.to(DEV).requires_grad_(True) for t in cl]
    ctd = [t.to(DEV).requires_grad_(True) for t in ct]
    if entry == "stacked":
        out = f.forward_stacked(f4d, cld, ctd)
        out.backward(torch.stack(do, dim=2).to(DEV, H16))
        res = [out[:, :, v] for v in range(V)]
    else:
        keys = [str(v) for v in range(V)]
        o = f(dict(zip(keys, f4d)), dict(zip(keys, cld)), dict(zip(keys, ctd)))
        res = [o[k] for k in keys]
        torch.autograd.backward(res, [_to_dev(t, fmt) for t in do])
    torch.cuda.synchronize()
    for v in range(V):
        assert res[v].dtype == H16 and f4d[v].grad.dtype == H16
        # df4 comes back in f4's own memory format
        assert f4d[v].grad.is_contiguous(memory_format=torch.channels_last if fmt == "cl" else torch.contiguous_format)
        assert_close(f"out:{v}", res[v], outs[v], BF16_TOL)
        assert_close(f"df4:{v}", f4d[v].grad, df4[v], BF16_TOL)
        assert_close(f"dcls:{v}", cld[v].grad, dcls[v], 4e-2)
        assert_close(f"dctr:{v}", ctd[v].grad, dctr[v], 4e-2)
    _check_params(f, gg, gl)


@pytest.mark.parametrize("fmt", ["nchw", "cl"])
def test_fusion_fp16_parts_and_cycle_pass(fmt):
    """forward_parts -> cycle.spatial_sum -> dense_seg_cycle -> backward with fp16 f4 (the cycle pass reads the fp16
    MGFM part, and its broadcast gradient is gathered by views_to_tokens at token stride 0).  The oracle chain is driven
    by the loss gradient of the features the GPU path computed (the cycle loss is sharp: a gradient taken at slightly
    different features would measure the loss, not the fusion node)."""
    B, C, V, h, w = 20, 256, 2, 4, 4
    R, off, ch, temp = 12, 2, 3, 10.0
    pg = O.init_params(C, seed=121, randomize_affine=True)
    pl = O.init_params(C, seed=122, randomize_affine=True)
    f4, cl, ct, _ = _fusion_inputs(B, C, V, h, w, 123)
    f = _fusion(C, pg, pl)
    keys = [str(i) for i in range(V)]
    f4d = [_to_dev(t, fmt).requires_grad_(True) for t in f4]
    fus, glob, loc = f.forward_parts(dict(zip(keys, f4d)), dict(zip(keys, [t.to(DEV) for t in cl])),
                                     dict(zip(keys, [t.to(DEV) for t in ct])))
    feats = [cycle.spatial_sum(glob[k]) for k in keys]
    loss = sum(cycle.dense_seg_cycle(ft, R, off, ch, temp) for ft in feats)
    loss.backward()
    torch.cuda.synchronize()
    # oracle: the reference's lines on CPU
    f4o = [t.clone().requires_grad_(True) for t in f4]
    qg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and k not in O.BUFFER_KEYS else v.clone())
          for k, v in pg.items()}
    xg, xl = O.gate_concat(f4o, cl, ct)
    zg = O.tpavi_forward(xg, qg)
    lo, tot = 0.0, 0
    for i, ft in enumerate(feats):
        l_i, g_i = CO.dense_seg_cycle(ft.detach().cpu().numpy(), R, off, ch, temp)
        lo += float(l_i)
        tot = tot + (zg[:, :, i].sum(dim=(2, 3)) * torch.from_numpy(g_i).float()).sum()
    tot.backward()
    assert abs(float(loss.detach()) - lo) <= 1e-3 * abs(lo) + 1e-5
    for i, k in enumerate(keys):
        assert glob[k].dtype == H16 and fus[k].dtype == H16
        assert_close(f"global:{k}", glob[k], zg[:, :, i], BF16_TOL)
    for i in range(V):
        assert f4d[i].grad.dtype == H16
        assert_close(f"df4:{i}", f4d[i].grad, f4o[i].grad, 3e-2)
    assert f.local_attn.theta.weight.grad is None
    assert_close("grad_g:theta.weight", f.global_attn.theta.weight.grad, qg["theta.weight"].grad, 3e-2)


def test_fp16_and_bf16_forward_agree():
    """The same (fp16-representable) inputs as fp16 and as bf16: only the output rounding separates the two, so a
    wrong-dtype read anywhere would miss by orders of magnitude."""
    B, C, V, h, w = 2, 256, 4, 28, 28
    pg = O.init_params(C, seed=131, randomize_affine=True)
    pl = O.init_params(C, seed=132, randomize_affine=True)
    f4, cl, ct, _ = _fusion_inputs(B, C, V, h, w, 133)
    f = _fusion(C, pg, pl)
    cld, ctd = [t.to(DEV) for t in cl], [t.to(DEV) for t in ct]
    with torch.no_grad():
        for fmt in ("nchw", "cl"):
            a = f.forward_stacked([_to_dev(t, fmt) for t in f4], cld, ctd).float()
            b = f.forward_stacked([_to_dev(t, fmt).to(torch.bfloat16) for t in f4], cld, ctd).float()
            assert O.rel_err(a, b) < 1e-2


def _kernel_count(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


@pytest.mark.parametrize("fmt", ["nchw", "cl"])
def test_fp16_adds_no_conversion_pass(fmt):
    """One fused forward + backward launches as many kernels with fp16 f4 as with bf16 f4 (same fp32 logits)."""
    B, C, V, h, w = 2, 256, 4, 28, 28
    pg = O.init_params(C, seed=141, randomize_affine=True)
    pl = O.init_params(C, seed=142, randomize_affine=True)
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 143)
    f = _fusion(C, pg, pl)
    cld, ctd = [t.to(DEV) for t in cl], [t.to(DEV) for t in ct]
    counts = {}
    for dt in (H16, torch.bfloat16):
        xs = [_to_dev(t, fmt).to(dt).requires_grad_(True) for t in f4]
        dz = torch.stack(do, dim=2).to(DEV, dt)

        def step():
            out = f.forward_stacked(xs, cld, ctd)
            out.backward(dz)
        step()                                   # warm-up (module loads, attribute set-up)
        f.zero_grad(set_to_none=True)
        for t in xs:
            t.grad = None
        counts[dt] = _kernel_count(step)
        f.zero_grad(set_to_none=True)
    assert counts[H16] == counts[torch.bfloat16], counts


@pytest.mark.parametrize("fmt", ["nchw", "cl"])
def test_gradscaler_overflow_becomes_signed_inf(fmt):
    """A scaled dz that pushes parts of df4 beyond the fp16 range: those are +-inf with the reference's sign (not
    clamped to 65504, not NaN), the rest stays finite."""
    B, C, V, h, w = 2, 256, 4, 28, 28
    pg = O.init_params(C, seed=151, randomize_affine=True)
    pl = O.init_params(C, seed=152, randomize_affine=True)
    for p in (pg, pl):
        p["norm_layer.weight"] = p["norm_layer.weight"] * 8.0     # LayerNorm gain: df4 well above dz
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 153)
    s = 0.9 * FP16_MAX / max(float(t.abs().max()) for t in do)
    dzs = [_h(t * s) for t in do]
    assert all(torch.isfinite(t.to(H16)).all() for t in dzs)
    _, df4, _, _, _, _ = O.fusion_fwd_bwd(f4, cl, ct, dzs, {k: v.clone() for k, v in pg.items()},
                                          {k: v.clone() for k, v in pl.items()})
    f = _fusion(C, pg, pl)
    f4d = [_to_dev(t, fmt).requires_grad_(True) for t in f4]
    out = f.forward_stacked(f4d, [t.to(DEV) for t in cl], [t.to(DEV) for t in ct])
    out.backward(torch.stack(dzs, dim=2).to(DEV, H16))
    torch.cuda.synchronize()
    n_big = n_small = 0
    for v in range(V):
        got = f4d[v].grad.float().cpu()
        ref = df4[v]
        big = ref.abs() > 1.05 * 65520.0
        small = ref.abs() < 0.95 * FP16_MAX
        n_big += int(big.sum())
        n_small += int(small.sum())
        assert torch.isinf(got[big]).all()
        assert torch.equal(torch.sign(got[big]), torch.sign(ref[big]))
        assert torch.isfinite(got[small]).all()
    assert n_big > 0 and n_small > 0


def test_gradscaler_skips_a_step_with_an_inf_gradient():
    B, C, V, h, w = 2, 256, 4, 28, 28
    pg = O.init_params(C, seed=161, randomize_affine=True)
    pl = O.init_params(C, seed=162, randomize_affine=True)
    f4, cl, ct, do = _fusion_inputs(B, C, V, h, w, 163)
    f = _fusion(C, pg, pl)
    opt = torch.optim.Adam(f.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=1.0)
    before = {k: v.detach().clone() for k, v in f.named_parameters()}
    g = torch.stack(do, dim=2).to(DEV, H16)
    g[0, 3, 1, 5, 7] = float("inf")
    out = f.forward_stacked([t.to(DEV, H16).requires_grad_(True) for t in f4], [t.to(DEV) for t in cl],
                            [t.to(DEV) for t in ct])
    scaler.scale((out.float() * g.float()).sum()).backward()
    torch.cuda.synchronize()
    for name, p in f.named_parameters():
        if name.endswith("align_channel.weight") or name.endswith("align_channel.bias"):
            continue
        if name.endswith("W_z.0.bias"):
            assert torch.equal(p.grad, torch.zeros_like(p.grad))     # exactly 0 by construction in training mode
        else:
            assert not torch.isfinite(p.grad).all(), name
    scaler.unscale_(opt)
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() < 1.0
    for k, v in f.named_parameters():
        assert torch.equal(v.detach(), before[k]), k


def test_amp_recipe_end_to_end():
    """torch.autocast("cuda") (fp16) + GradScaler + Adam around a tiny stand-in network: per-view conv backbones,
    classifier / centerness heads, GlobalLocalFusion and a 1x1 head.  The fusion node sees fp16 f4 and logits and an
    fp16 output gradient; its unscaled parameter gradients match the oracle run on the captured tensors."""
    torch.manual_seed(0)
    B, C, V, h, w = 2, 128, 2, 8, 8
    keys = ["a", "b"]
    nn = torch.nn
    backbone = nn.ModuleDict({k: nn.Conv2d(3, C, 3, padding=1) for k in keys})
    classifier = nn.ModuleDict({k: nn.Conv2d(C, 5, 1) for k in keys})
    centerness = nn.ModuleDict({k: nn.Conv2d(C, 1, 1) for k in keys})
    head = nn.Conv2d(C, 2, 1)
    fusion = GlobalLocalFusion(in_channels=C)
    net = nn.ModuleList([backbone, classifier, centerness, head, fusion]).to(DEV).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda")
    gen = torch.Generator().manual_seed(7)
    img = {k: torch.randn(B, 3, h, w, generator=gen).to(DEV) for k in keys}
    for _ in range(2):
        opt.zero_grad(set_to_none=True)
        params = {m: {k: v.detach().float().cpu().clone() for k, v in getattr(fusion, m).state_dict().items()}
                  for m in ("global_attn", "local_attn")}
        cap = {}
        with torch.autocast("cuda"):
            f4 = {k: backbone[k](img[k]) for k in keys}
            cls = {k: classifier[k](f4[k]) for k in keys}
            ctr = {k: centerness[k](f4[k]) for k in keys}
            out = fusion(f4, cls, ctr)
            for k in keys:
                out[k].register_hook(lambda g, k=k: cap.__setitem__(k, g.detach().clone()))
            loss = sum(head(out[k]).float().pow(2).mean() for k in keys)
        assert all(f4[k].dtype == H16 and out[k].dtype == H16 for k in keys)
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        scale = scaler.get_scale()
        assert all(cap[k].dtype == H16 and torch.isfinite(cap[k]).all() for k in keys)
        _, _, _, _, gg, gl = O.fusion_fwd_bwd([f4[k].detach().float().cpu() for k in keys],
                                              [cls[k].detach().float().cpu() for k in keys],
                                              [ctr[k].detach().float().cpu() for k in keys],
                                              [cap[k].float().cpu() / scale for k in keys],
                                              params["global_attn"], params["local_attn"])
        _check_params(fusion, gg, gl)
        scaler.step(opt)
        scaler.update()


def test_mixed_view_dtypes_are_refused():
    B, C, V, h, w = 2, 128, 2, 8, 8
    f = GlobalLocalFusion(in_channels=C).to(DEV)
    gen = torch.Generator().manual_seed(171)
    f4 = [torch.randn(B, C, h, w, generator=gen).to(DEV, dt) for dt in (torch.bfloat16, H16)]
    cl = [torch.randn(B, 5, h, w, generator=gen).to(DEV) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, generator=gen).to(DEV) for _ in range(V)]
    with pytest.raises(TypeError, match="dtype"):
        f.forward_stacked(f4, cl, ct)


def test_fp32_precision_refuses_fp16_before_any_launch():
    B, C, V, h, w = 2, 128, 2, 8, 8
    f = GlobalLocalFusion(in_channels=C).to(DEV)
    f.global_attn.compute_precision = f.local_attn.compute_precision = "fp32"
    f4 = [torch.randn(B, C, h, w, device=DEV, dtype=H16) for _ in range(V)]
    cl = [torch.randn(B, 5, h, w, device=DEV) for _ in range(V)]
    ct = [torch.randn(B, 1, h, w, device=DEV) for _ in range(V)]
    with pytest.raises(TypeError, match="float16"):
        f.forward_stacked(f4, cl, ct)
    m = TPAVIModule(C).to(DEV)
    m.compute_precision = "fp32"
    with pytest.raises(TypeError, match="float16"):
        m(torch.randn(B, C, 2, h, w, device=DEV, dtype=H16))
