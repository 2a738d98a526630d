"""SURVEY 8(f)2 / BASELINE configs[0]: the reference's full network ``Global_and_Local`` (R/models/ours.py:1708-1843),
built UNMODIFIED from the staged reference sources (oracle/_ref, git-ignored, staged by build()) through the harness
shim of SURVEY 8(c), with the fusion blocks swapped for the B200 path by ``glfusion_b200.install(models.ours)``:

* the patched network takes the unpatched network's ``state_dict`` with ``strict=True`` (the wire format of R/main.py:857-872);
* one training step of the plumbing configuration (2 views x 8 frames x 112 x 112, BCE-with-logits sum loss as in
  R/main.py:87,209-211) gives the same masks, fused features, loss and gradients as the unpatched fp32 network on the
  same weights, within the bf16 bound of the fusion path."""
import pytest
import torch

import glfusion_b200
from gpu_util import BF16_TOL, DEV, assert_close, grad_tol
from oracle import build_ref
from oracle import tpavi_oracle as O

pytestmark = pytest.mark.gpu

VIEWS = ["1", "3"]


def _build(ours, patched: bool, seed: int = 0):
    orig = ours.TPAVIModule
    try:
        if patched:
            glfusion_b200.install(ours)          # ours.py:1746-1747 resolve the class name at construction time
        torch.manual_seed(seed)
        net = ours.Global_and_Local(VIEWS)
    finally:
        ours.TPAVIModule = orig
    return net


def _step(net, imgs, target, seed):
    net.zero_grad(set_to_none=True)
    torch.manual_seed(seed)                      # DeepLabHead has a Dropout(0.5) (R/models/deeplabv3.py:159)
    mask, mask_bb, fg, fl = net(imgs)
    loss = sum(torch.nn.functional.binary_cross_entropy_with_logits(mask[v], target[v], reduction="sum") for v in VIEWS)
    loss.backward()
    torch.cuda.synchronize()
    return mask, fg, fl, loss.detach()


class _Bf16Block(torch.nn.Module):
    """A reference fusion block run under torch.autocast(bfloat16): the reference's OWN bf16 sensitivity of every
    network output / gradient (the yardstick of this end-to-end comparison, as tests/golden/bf16_floor.json is for the
    bare module)."""

    def __init__(self, block):
        super().__init__()
        self.block = block

    def forward(self, x, audio=None):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            z, a = self.block(x)
        return z.float(), a


def _rel(a, b):
    a, b = a.detach().float(), b.detach().float()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def test_install_full_network_cfg1_step():
    ours = build_ref.import_reference_network()
    if ours is None:
        pytest.skip("oracle/_ref was not staged (build() found no upstream GL-Fusion sources)")
    ref = _build(ours, patched=False)
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():                        # SURVEY F3: BN gamma / beta of the fusion blocks are 0 at init
        for blk in (ref.global_attn, ref.local_attn):
            for p, mean in ((blk.W_z[1].weight, 1.0), (blk.W_z[1].bias, 0.0), (blk.norm_layer.weight, 1.0),
                            (blk.norm_layer.bias, 0.0)):
                p.copy_(mean + 0.2 * torch.randn(p.shape, generator=gen))
    ours_net = _build(ours, patched=True)
    assert isinstance(ours_net.global_attn, glfusion_b200.TPAVIModule)
    assert isinstance(ours_net.local_attn, glfusion_b200.TPAVIModule)
    missing = ours_net.load_state_dict(ref.state_dict(), strict=True)      # identical keys and shapes, whole network
    assert not missing.missing_keys and not missing.unexpected_keys
    ref, ours_net = ref.to(DEV).train(), ours_net.to(DEV).train()

    F_, H = 8, 112
    imgs = {v: torch.rand(F_, 1, H, H, generator=gen).to(DEV) for v in VIEWS}            # loader: pixels / 255
    target = {v: (torch.rand(F_, 5, H, H, generator=gen) > 0.7).float().to(DEV) for v in VIEWS}
    m0, fg0, fl0, loss0 = _step(ref, imgs, target, seed=11)
    g0 = {k: (p.grad.detach().clone() if p.grad is not None else None) for k, p in ref.named_parameters()}
    m1, fg1, fl1, loss1 = _step(ours_net, imgs, target, seed=11)
    g1 = {k: p.grad for k, p in ours_net.named_parameters()}
    # the reference's own bf16 sensitivity: the same network with ONLY its two fusion blocks under bf16 autocast
    ref.global_attn, ref.local_attn = _Bf16Block(ref.global_attn), _Bf16Block(ref.local_attn)
    m2, fg2, fl2, loss2 = _step(ref, imgs, target, seed=11)
    g2 = {k.replace("_attn.block.", "_attn."): p.grad for k, p in ref.named_parameters()}

    def check(name, ours_t, ref_t, floor_t, tol):
        floor = _rel(floor_t, ref_t)
        err = _rel(ours_t, ref_t)
        # within north_star's bf16 bound, or within 2.5x the reference's own bf16 error on this tensor: gradients that
        # travel back through 50 backbone layers, train-mode BatchNorm over 8 frames and Dropout are chaotic in any
        # reduced precision (the reference's own first-conv gradient moves by 15 % under autocast of the two fusion
        # blocks alone), and the bf16 arm additionally stores x / z / dz in bf16, which autocast keeps in fp32
        assert err < max(tol, 2.5 * floor), f"{name}: rel err {err:.3e} (reference's own bf16 error {floor:.3e})"
        return err, floor

    assert abs(float(loss1) - float(loss0)) / abs(float(loss0)) < 5e-3
    worst = {}
    dice_rows = []
    for v in VIEWS:
        check(f"f4_global_fusion:{v}", fg1[v], fg0[v], fg2[v], BF16_TOL)
        check(f"f4_local_fusion:{v}", fl1[v], fl0[v], fl2[v], BF16_TOL)
        # the masks sit behind the DeepLab head (ASPP + Dropout + 1x1, R/models/deeplabv3.py:102-166): at random init its
        # logits are small differences of large activations, which amplifies the error of the fused features
        # (measured: 2.4e-2 for a 4e-3 error of the fused features; the bf16 arm also rounds the residual input x, which
        # autocast keeps in fp32, so the reference's own figure, 7.5e-3, is not reachable here)
        worst[f"mask:{v}"] = check(f"mask:{v}", m1[v], m0[v], m2[v], 5e-2)
        # segmentation agreement through the reference's OWN classifier heads, with its Dice definition (R/main.py:800-815)
        # and the unpatched fp32 network's prediction as the target: at least what the reference's own bf16 run reaches
        # (minus half a point), and never less than 98 % at random init, where the logits hover around zero
        seg0 = (m0[v] > 0).float()
        d_ours, d_floor = O.dice(m1[v], seg0), O.dice(m2[v], seg0)
        dice_rows.append((v, round(100 * d_ours, 2), round(100 * d_floor, 2)))
        assert d_ours >= min(0.98, d_floor - 0.005), f"Dice vs the fp32 network's masks: ours {d_ours:.4f}, reference bf16 {d_floor:.4f}"
    unused = 0
    rest0, rest1, rest2 = [], [], []
    for k, a in g0.items():
        if a is None:                            # the template network / align_channel never receive a gradient
            assert g1[k] is None, k
            unused += 1
            continue
        if k.startswith("global_attn.") or k.startswith("local_attn."):
            if k.endswith("W_z.0.bias"):
                continue                         # analytically zero (BatchNorm cancels it): noise on both sides
            worst[k] = check("grad:" + k, g1[k], a, g2[k], BF16_TOL)
        else:
            rest0.append(a.flatten()); rest1.append(g1[k].flatten()); rest2.append(g2[k].flatten())
    # everything the backbones and heads receive through the fusion blocks, as ONE vector (single small tensors, e.g. a
    # BatchNorm bias inside the ASPP pooling branch, are sums of cancelling terms and move by 10 - 25 % under any bf16
    # rounding, the reference's own included)
    worst["grad:backbones+heads"] = check("grad:backbones+heads", torch.cat(rest1), torch.cat(rest0), torch.cat(rest2), 5e-2)
    assert unused > 0
    top = sorted(worst.items(), key=lambda kv: -kv[1][0])[:5]
    print("Dice (%) against the fp32 network's masks (view, ours, reference's own bf16):", dice_rows)
    print("largest errors (ours, reference's own bf16):", [(k, round(e, 4), round(f, 4)) for k, (e, f) in top])
