"""Generate golden input/output vectors from the UNMODIFIED reference module.

Run in the build container only (needs /root/reference):

    python oracle/gen_golden.py

It imports ``/root/reference/GLfusion/models/TPAVI.py`` (torch-only; semantically identical to the copy at
R/models/ours.py:770-917), loads seeded weights into it through ``load_state_dict(strict=True)``, re-randomises
the zero-initialised BatchNorm gamma/beta and the LayerNorm affine (SURVEY.md F3), runs forward + autograd
backward on CPU in fp32 and writes ``tests/golden/<case>.npz`` with every input, output, gradient and BN buffer
(the OUTPUTS_ONLY cases without their seeded inputs and weights, which ``seeded_inputs`` rebuilds).  ``init_dot_c96``
holds the constructor's own state dict under a fixed seed.

The glue case additionally restates, literally, lines 1802-1834 of R/models/ours.py around two reference
modules (the enclosing class cannot be constructed offline: it downloads ImageNet weights and imports monai).
TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = "/root/reference/GLfusion"

from oracle import tpavi_oracle as O  # noqa: E402

CASES = {
    # name: (B, C, T, H, W, mode, training, bn_layer)
    "dot_train_c128": (2, 128, 2, 8, 8, "dot", True, True),
    "dot_train_c256": (2, 256, 3, 4, 8, "dot", True, True),
    "dot_eval_c128": (2, 128, 2, 8, 8, "dot", False, True),
    "dot_nobn_c128": (2, 128, 2, 8, 8, "dot", True, False),
    "embedded_train_c128": (2, 128, 2, 8, 8, "embedded", True, True),
    "embedded_eval_c128": (1, 128, 3, 8, 8, "embedded", False, True),
    "dot_ragged_c128": (3, 128, 3, 5, 7, "dot", True, True),     # N = 105: not a multiple of any tile
}


def load_reference_module():
    sys.path.insert(0, REF)
    from models.TPAVI import TPAVIModule  # type: ignore
    return TPAVIModule


def make_module(TPAVIModule, C, mode, bn_layer, params):
    m = TPAVIModule(in_channels=C, mode=mode, bn_layer=bn_layer)
    sd = {k: v.clone() for k, v in params.items()}
    m.load_state_dict(sd, strict=True)
    return m


GLUE_SEED = 7
# cases whose .npz holds only what the reference computed: their seeded inputs and weights are rebuilt by
# seeded_inputs() (keeps every golden file under 1 MB)
OUTPUTS_ONLY = ("dot_train_c256", "glue_dot_c128")


def seeded_inputs(name: str) -> dict:
    """The seeded inputs and weights of golden case `name`, keyed as in its .npz, as torch tensors."""
    out = {}
    if name == "glue_dot_c128":
        B, C, V, h, w = 2, 128, 3, 6, 6
        for tag, s in (("g", GLUE_SEED), ("l", GLUE_SEED + 100)):
            out.update({f"param_{tag}:{k}": v for k, v in O.init_params(C, seed=s, randomize_affine=True).items()})
        gen = torch.Generator().manual_seed(GLUE_SEED + 2)
        for key, c in (("f4", C), ("cls", 5), ("ctr", 1), ("d_out", C)):
            out.update({f"{key}:{v}": torch.randn(B, c, h, w, generator=gen) for v in range(V)})
        return out
    B, C, T, H, W, mode, training, bn_layer = CASES[name]
    seed = 100 + list(CASES).index(name)
    params = O.init_params(C, seed=seed, randomize_affine=True, bn_layer=bn_layer)
    if bn_layer and not training:
        # eval mode reads running stats: make them non-trivial
        g = torch.Generator().manual_seed(seed + 1)
        params["W_z.1.running_mean"] = torch.randn(C, generator=g) * 0.1
        params["W_z.1.running_var"] = torch.rand(C, generator=g) * 0.5 + 0.5
    out.update({"param:" + k: v for k, v in params.items()})
    g = torch.Generator().manual_seed(seed + 2)
    out["x"] = torch.randn(B, C, T, H, W, generator=g)
    out["dz"] = torch.randn(B, C, T, H, W, generator=g)
    return out


def run_case(TPAVIModule, name, B, C, T, H, W, mode, training, bn_layer, seed):
    torch.manual_seed(seed)
    inp = seeded_inputs(name)
    params = {k[len("param:"):]: v for k, v in inp.items() if k.startswith("param:")}
    m = make_module(TPAVIModule, C, mode, bn_layer, params)
    m.train(training)
    x, dz = inp["x"], inp["dz"]
    x.requires_grad_(True)
    z, audio_temp = m(x)
    assert audio_temp == 0
    z.backward(dz)
    out = {"x": x.detach().numpy(), "dz": dz.numpy(), "z": z.detach().numpy(), "dx": x.grad.numpy()}
    for k, v in params.items():
        out["param:" + k] = v.numpy()
    for k, v in m.named_parameters():
        if k.startswith("align_channel"):
            continue
        out["grad:" + k] = (v.grad if v.grad is not None else torch.zeros_like(v)).numpy()
    for k, v in m.named_buffers():
        out["buf_after:" + k] = v.numpy()
    out["meta"] = np.array([B, C, T, H, W, int(training), int(bn_layer)], dtype=np.int64)
    out["mode"] = np.array(mode)
    z_strides = np.array(z.stride(), dtype=np.int64)
    out["z_strides"] = z_strides
    return out


def run_glue_case(TPAVIModule):
    """ours.py:1802-1834 restated literally around two reference TPAVIModule instances."""
    from torch import nn
    B, C, V, h, w = 2, 128, 3, 6, 6
    inp = seeded_inputs("glue_dot_c128")
    pg = {k[len("param_g:"):]: v for k, v in inp.items() if k.startswith("param_g:")}
    pl = {k[len("param_l:"):]: v for k, v in inp.items() if k.startswith("param_l:")}
    global_attn = make_module(TPAVIModule, C, "dot", True, pg)
    local_attn = make_module(TPAVIModule, C, "dot", True, pl)
    f4, cls_l, ctr_l, d_out = ([inp[f"{key}:{v}"] for v in range(V)] for key in ("f4", "cls", "ctr", "d_out"))
    for t in f4 + cls_l + ctr_l:
        t.requires_grad_(True)
    center_aware_weight = 20
    mask_bb, ctr, f4_local = [], [], []
    for v in range(V):
        mb = nn.Sigmoid()(cls_l[v])                                    # :1803
        n, c, hh, ww = mb.shape
        mb = nn.AdaptiveMaxPool3d((1, hh, ww))(mb)                     # :1805-1806
        mask_bb.append(mb)
        ctr.append(nn.Sigmoid()(ctr_l[v]))                             # :1810
    for v in range(V):
        atten = (center_aware_weight * mask_bb[v] * ctr[v]).sigmoid()  # :1815
        f4_local.append(f4[v].clone() * atten)                         # :1816
    gcat = torch.cat([f.unsqueeze(2) for f in f4], dim=2)              # :1819-1820
    gfeat, _ = global_attn(gcat)                                       # :1821
    lcat = torch.cat([f.unsqueeze(2) for f in f4_local], dim=2)        # :1826-1827
    lfeat, _ = local_attn(lcat)                                        # :1828
    outs = [gfeat[:, :, i] + lfeat[:, :, i] for i in range(V)]         # :1823,1830,1834
    torch.autograd.backward(outs, d_out)
    out = {"meta": np.array([B, C, V, h, w], dtype=np.int64)}
    for v in range(V):
        out[f"f4:{v}"] = f4[v].detach().numpy()
        out[f"cls:{v}"] = cls_l[v].detach().numpy()
        out[f"ctr:{v}"] = ctr_l[v].detach().numpy()
        out[f"d_out:{v}"] = d_out[v].numpy()
        out[f"out:{v}"] = outs[v].detach().numpy()
        out[f"df4:{v}"] = f4[v].grad.numpy()
        out[f"dcls:{v}"] = cls_l[v].grad.numpy()
        out[f"dctr:{v}"] = ctr_l[v].grad.numpy()
    for tag, p, m in (("g", pg, global_attn), ("l", pl, local_attn)):
        for k, t in p.items():
            out[f"param_{tag}:{k}"] = t.numpy()
        for k, t in m.named_parameters():
            if not k.startswith("align_channel"):
                out[f"grad_{tag}:{k}"] = t.grad.numpy()
        for k, t in m.named_buffers():
            out[f"buf_after_{tag}:{k}"] = t.numpy()
    return out


def run_init_case(TPAVIModule, C=96, seed=1234):
    """The constructor's state dict under torch.manual_seed(seed): the weights its initialisers draw from the global RNG."""
    torch.manual_seed(seed)
    return {k: v.numpy() for k, v in TPAVIModule(in_channels=C, mode="dot").state_dict().items()}


def save(outdir, name, out):
    if name in OUTPUTS_ONLY:
        out = {k: v for k, v in out.items() if k not in seeded_inputs(name)}
    np.savez_compressed(os.path.join(outdir, name + ".npz"), **out)


def main():
    TPAVIModule = load_reference_module()
    outdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    for i, (name, cfg) in enumerate(CASES.items()):
        out = run_case(TPAVIModule, name, *cfg, seed=100 + i)
        save(outdir, name, out)
        print(name, "z", out["z"].shape, "strides", out["z_strides"])
    save(outdir, "glue_dot_c128", run_glue_case(TPAVIModule))
    save(outdir, "init_dot_c96", run_init_case(TPAVIModule))
    print("glue_dot_c128, init_dot_c96 done")


if __name__ == "__main__":
    main()
