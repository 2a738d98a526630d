"""Recipe for ``oracle/_ref/``: the UNMODIFIED reference module of the hot path, staged for the GPU box.

TEST INFRASTRUCTURE ONLY (see oracle/tpavi_oracle.py).  The reference is pure Python: its fusion block
``R/models/TPAVI.py`` (identical to ``R/models/ours.py:770-917``, SURVEY.md F5) imports only torch.  There is nothing to
compile; "building" the reference arm means staging that one file where it lies under ``/root/reference`` into the
git-ignored (NOT gpurun-ignored) ``oracle/_ref/`` so that it travels to the GPU box with the snapshot.  No reference
source is ever committed: ``oracle/_ref/`` is in ``.gitignore`` and this script is the only writer.

    python oracle/build_ref.py         # no-op (returns False) when /root/reference is absent, e.g. on the GPU box
"""
from __future__ import annotations

import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = "/root/reference/GLfusion/models/TPAVI.py"
REF_DIR = os.path.join(HERE, "_ref")
REF_DST = os.path.join(REF_DIR, "models", "TPAVI.py")
REF_MAIN = os.path.join(REF_DIR, "main.py")          # the trainer, for its cycle-consistency methods


def build_ref() -> bool:
    """Stage the reference's ``models/`` package (the fusion block and, for the full-network harness of
    tests/test_gpu_network.py, the network that calls it) and its ``main.py`` (the trainer's cycle-consistency methods,
    for tests/test_oracle_cycle.py); True when oracle/_ref holds the fusion block afterwards."""
    src_dir = os.path.dirname(REF_SRC)
    if os.path.exists(REF_SRC):
        os.makedirs(os.path.dirname(REF_DST), exist_ok=True)
        for name in sorted(os.listdir(src_dir)):
            if name.endswith(".py"):
                shutil.copyfile(os.path.join(src_dir, name), os.path.join(os.path.dirname(REF_DST), name))
        main = os.path.join(os.path.dirname(src_dir), "main.py")
        if os.path.exists(main):
            shutil.copyfile(main, REF_MAIN)
    return os.path.exists(REF_DST)


def import_reference_network():
    """``models.ours`` of the staged reference, importable in this image: the harness-side shim of SURVEY.md 8(c) —
    stub modules for the packages the file imports but the fusion network never uses (monai, matplotlib, tensorboardX)
    and ``resnet50(weights=None)`` instead of the ImageNet download (no network here).  Nothing of the reference is
    edited.  Returns the module, or None when oracle/_ref was never staged."""
    import importlib
    import sys
    import types
    if not os.path.exists(os.path.join(REF_DIR, "models", "ours.py")):
        return None
    for name in ("monai", "monai.data", "matplotlib", "matplotlib.pyplot", "tensorboardX"):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    sys.modules["monai.data"].DataLoader = getattr(sys.modules["monai.data"], "DataLoader", object)
    sys.modules["monai"].data = sys.modules["monai.data"]
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["tensorboardX"].SummaryWriter = getattr(sys.modules["tensorboardX"], "SummaryWriter", object)
    import torchvision.models.resnet as tvr
    if not getattr(tvr, "_glf_no_download", False):
        orig = tvr.resnet50

        def resnet50_no_download(*args, **kwargs):
            kwargs.pop("pretrained", None)
            kwargs["weights"] = None
            return orig(*args, **kwargs)
        tvr.resnet50 = resnet50_no_download
        tvr.__dict__["resnet50"] = resnet50_no_download
        tvr._glf_no_download = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
        if not getattr(sys.modules[k], "__file__", "").startswith(REF_DIR):
            del sys.modules[k]
    return importlib.import_module("models.ours")


def load_reference_tpavi():
    """The reference's own ``TPAVIModule`` class from oracle/_ref (None when it was never staged)."""
    if not os.path.exists(REF_DST):
        return None
    import importlib.util
    spec = importlib.util.spec_from_file_location("glf_reference_tpavi", REF_DST)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.TPAVIModule


def reference_fusion_fwd_bwd(TPAVI, f4, cls_logits, ctr_logits, d_out, p_global, p_local, weight=20.0):
    """One fwd+bwd of the fusion call site around two UNMODIFIED reference modules: the literal glue lines
    R/models/ours.py:1802-1834 (sigmoid / max over the class channels / sigmoid, gate, per-view concat, MGFM and MLFM,
    split, sum) on whatever device the inputs live on.  Returns (per-view outputs, per-view input gradients)."""
    import torch
    C = f4[0].shape[1]
    dev = f4[0].device
    mg = TPAVI(in_channels=C, mode="dot").to(dev)
    ml = TPAVI(in_channels=C, mode="dot").to(dev)
    mg.load_state_dict(p_global, strict=True)
    ml.load_state_dict(p_local, strict=True)
    mg.train()
    ml.train()
    xs = [t.detach().clone().requires_grad_(True) for t in f4]
    cls_logits = [t.detach().clone().requires_grad_(True) for t in cls_logits]   # the gate back-propagates to both heads
    ctr_logits = [t.detach().clone().requires_grad_(True) for t in ctr_logits]
    loc = []
    for v, x in enumerate(xs):
        m = torch.sigmoid(cls_logits[v]).amax(dim=1, keepdim=True)          # ours.py:1802-1806 (AdaptiveMaxPool3d over classes)
        c = torch.sigmoid(ctr_logits[v])                                     # ours.py:1808-1811
        a = (weight * m * c).sigmoid()                                       # ours.py:1814-1815
        loc.append(x.clone() * a)                                            # ours.py:1816
    xg = torch.cat([x.unsqueeze(2) for x in xs], dim=2)                      # ours.py:1819-1820
    xl = torch.cat([x.unsqueeze(2) for x in loc], dim=2)                     # ours.py:1826-1827
    zg, _ = mg(xg)                                                           # ours.py:1821
    zl, _ = ml(xl)                                                           # ours.py:1828
    outs = [zg[:, :, v] + zl[:, :, v] for v in range(len(xs))]               # ours.py:1822-1834
    torch.autograd.backward(outs, list(d_out))
    return outs, [x.grad for x in xs]


if __name__ == "__main__":
    print("oracle/_ref staged" if build_ref() else "reference not available; oracle/_ref not staged")
