"""The oracle (oracle/tpavi_oracle.py) against the golden vectors produced by the real reference module
(oracle/gen_golden.py), and against the live reference module when it is staged in oracle/_ref."""
import pytest
import torch

from conftest import load_golden
from oracle import tpavi_oracle as O

CASES = ["dot_train_c128", "dot_train_c256", "dot_eval_c128", "dot_nobn_c128", "embedded_train_c128",
         "embedded_eval_c128", "dot_ragged_c128"]
TOL = 2e-5   # fp32 vs fp32, different op order only


def _params(g, prefix="param:"):
    p = {}
    for k, v in g.items():
        if k.startswith(prefix):
            p[k[len(prefix):]] = v.clone() if isinstance(v, torch.Tensor) else torch.tensor(v.item())
    return p


def _meta(g):
    B, C, T, H, W, training, bn = [int(v) for v in g["meta"]]
    return B, C, T, H, W, bool(training), bool(bn), str(g["mode"])


def _check_oracle(g, mode, training, bn):
    """The oracle against one run of the reference module: z, dx, every parameter gradient and the BN buffers after."""
    p = _params(g)
    z, dx, grads = O.tpavi_fwd_bwd(g["x"], g["dz"], p, mode=mode, training=training, bn_layer=bn)
    assert O.rel_err(z, g["z"]) < TOL
    assert O.rel_err(dx, g["dx"]) < TOL
    for k, v in grads.items():
        ref = g["grad:" + k]
        if ref.abs().max() < 1e-3:
            # analytically zero (train-mode BN cancels any per-channel shift of U: W_z.0.bias always, and g.bias
            # and phi.bias under softmax: rows sum to 1, row-constant logit shifts cancel); reference value = rounding noise
            assert k in ("W_z.0.bias", "g.bias", "phi.bias") and v.abs().max() < 1e-3
            continue
        assert O.rel_err(v, ref) < 5e-5, k
    if bn:
        assert O.rel_err(p["W_z.1.running_mean"], g["buf_after:W_z.1.running_mean"]) < TOL
        assert O.rel_err(p["W_z.1.running_var"], g["buf_after:W_z.1.running_var"]) < TOL
        assert int(p["W_z.1.num_batches_tracked"]) == int(g["buf_after:W_z.1.num_batches_tracked"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    g = load_golden(name)
    B, C, T, H, W, training, bn, mode = _meta(g)
    _check_oracle(g, mode, training, bn)


@pytest.mark.parametrize("name", ["dot_train_c128", "dot_train_c256", "dot_eval_c128", "dot_ragged_c128"])
def test_closed_form_dot_matches_golden(name):
    """The reassociated O(N) algorithm + hand-derived backward == the reference (fp64 closed form vs fp32 ref)."""
    g = load_golden(name)
    B, C, T, H, W, training, bn, mode = _meta(g)
    p = {k: (v.double() if v.is_floating_point() else v) for k, v in _params(g).items()}
    z, dx, grads, _ = O.tpavi_dot_closed_form(g["x"].double(), g["dz"].double(), p, training=training)
    assert O.rel_err(z, g["z"]) < TOL
    assert O.rel_err(dx, g["dx"]) < TOL
    for k, v in grads.items():
        ref = g["grad:" + k]
        if k == "W_z.0.bias" and training:
            assert v.abs().max() < 1e-9
            continue
        assert O.rel_err(v, ref) < 5e-5, k


@pytest.mark.parametrize("name", ["dot_train_c128", "dot_train_c256", "dot_eval_c128", "dot_ragged_c128",
                                  "dot_nobn_c128"])
def test_gram_form_dot_matches_golden(name):
    """The Gram-matrix reassociation (channel-space products only; what the CUDA path runs when N >> C) + its
    hand-derived backward == the reference module's outputs and all 13 gradients (fp64 restatement vs fp32 golden)."""
    g = load_golden(name)
    B, C, T, H, W, training, bn, mode = _meta(g)
    p = {k: (v.double() if v.is_floating_point() else v) for k, v in _params(g).items()}
    z, dx, grads, aux = O.tpavi_dot_gram_form(g["x"].double(), g["dz"].double(), p, training=training, bn_layer=bn)
    assert O.rel_err(z, g["z"]) < TOL
    assert O.rel_err(dx, g["dx"]) < TOL
    for k, v in grads.items():
        ref = g["grad:" + k]
        if k == "W_z.0.bias" and training:
            assert v.abs().max() < 1e-9 * max(1.0, float(g["grad:W_z.0.weight"].abs().max()))
            continue
        assert O.rel_err(v, ref) < 5e-5, k
    if bn and training:
        n = B * T * H * W
        rm = 0.9 * g["param:W_z.1.running_mean"].double() + 0.1 * aux["mean"]
        rv = 0.9 * g["param:W_z.1.running_var"].double() + 0.1 * aux["var"] * n / (n - 1)
        assert O.rel_err(rm, g["buf_after:W_z.1.running_mean"]) < TOL
        assert O.rel_err(rv, g["buf_after:W_z.1.running_var"]) < TOL


def test_glue_matches_golden():
    g = load_golden("glue_dot_c128")
    B, C, V, h, w = [int(v) for v in g["meta"]]
    pg, pl = _params(g, "param_g:"), _params(g, "param_l:")
    f4 = [g[f"f4:{v}"] for v in range(V)]
    cl = [g[f"cls:{v}"] for v in range(V)]
    ct = [g[f"ctr:{v}"] for v in range(V)]
    do = [g[f"d_out:{v}"] for v in range(V)]
    outs, df4, dcls, dctr, gg, gl = O.fusion_fwd_bwd(f4, cl, ct, do, pg, pl)
    for v in range(V):
        assert O.rel_err(outs[v], g[f"out:{v}"]) < TOL
        assert O.rel_err(df4[v], g[f"df4:{v}"]) < TOL
        assert O.rel_err(dcls[v], g[f"dcls:{v}"]) < 1e-4
        assert O.rel_err(dctr[v], g[f"dctr:{v}"]) < 1e-4
    for tag, gr in (("g", gg), ("l", gl)):
        for k, val in gr.items():
            if k == "W_z.0.bias":
                continue
            assert O.rel_err(val, g[f"grad_{tag}:{k}"]) < 5e-5, (tag, k)


def test_zero_init_trap():
    """SURVEY F3: with the reference's default init (BN gamma=beta=0) the block is exactly LayerNorm(x)."""
    p = O.init_params(64, seed=3, randomize_affine=False)
    x = torch.randn(2, 64, 2, 4, 4)
    z = O.tpavi_forward(x, p)
    ln = torch.nn.functional.layer_norm(x.permute(0, 2, 3, 4, 1), (64,)).permute(0, 4, 1, 2, 3)
    assert (z - ln).abs().max() < 1e-6


def test_dice_definition():
    pred = torch.tensor([3.0, -2.0, 1.0, -1.0])
    tgt = torch.tensor([1.0, 0.0, 0.0, 1.0])
    assert abs(O.dice(pred, tgt) - 2 * 1 / (2 * 1 + 1 + 1 + 1e-5)) < 1e-9


@pytest.mark.parametrize("mode", ["dot", "embedded"])
def test_oracle_matches_live_reference(mode):
    """The oracle against the reference module in train mode: on the run the reference recorded
    (tests/golden/<mode>_train_c128.npz) and, when the reference module is staged in oracle/_ref, on a live run of it
    with fresh random inputs."""
    _check_oracle(load_golden(f"{mode}_train_c128"), mode, True, True)
    from oracle import build_ref
    TPAVI = build_ref.load_reference_tpavi()
    if TPAVI is None:
        return
    C = 64
    p = O.init_params(C, seed=11, randomize_affine=True)
    m = TPAVI(in_channels=C, mode=mode)
    m.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    m.train()
    x = torch.randn(3, C, 2, 5, 6)
    dz = torch.randn_like(x)
    xr = x.clone().requires_grad_(True)
    z, _ = m(xr)
    z.backward(dz)
    live = {"x": x, "dz": dz, "z": z.detach(), "dx": xr.grad}
    live.update({"param:" + k: v for k, v in p.items()})
    live.update({"grad:" + k: v.grad for k, v in m.named_parameters() if not k.startswith("align_channel")})
    live.update({"buf_after:" + k: v for k, v in m.named_buffers()})
    _check_oracle(live, mode, True, True)


class _OracleTPAVI(torch.nn.Module):
    """The oracle's restatement of TPAVIModule behind the reference module's interface (constructor, strict state-dict
    load, ``(z, audio) = m(x)``), for driving the call-site wrapper when the reference module is not staged."""

    def __init__(self, in_channels, mode="dot"):
        super().__init__()
        self.mode, self.p = mode, None

    def load_state_dict(self, state_dict, strict=True):
        self.p = {k: v.clone().requires_grad_(k not in O.BUFFER_KEYS) for k, v in state_dict.items()}

    def forward(self, x):
        return O.tpavi_forward(x, self.p, mode=self.mode, training=self.training), 0


def test_reference_arm_wrapper_matches_oracle():
    """bench.py's reference arm / cpu_baseline / gpu_reference leg run a module pair inside the literal call-site lines
    ours.py:1802-1834 (oracle/build_ref.py::reference_fusion_fwd_bwd): driven by the UNMODIFIED reference module (the
    staged oracle/_ref copy) or, without it, by the oracle's restatement, it must reproduce the outputs and input
    gradients the reference recorded for the same call site (tests/golden/glue_dot_c128.npz)."""
    from oracle import build_ref
    TPAVI = build_ref.load_reference_tpavi() or _OracleTPAVI
    g = load_golden("glue_dot_c128")
    V = int(g["meta"][2])
    f4, cl, ct, do = ([g[f"{key}:{v}"] for v in range(V)] for key in ("f4", "cls", "ctr", "d_out"))
    r_out, r_df4 = build_ref.reference_fusion_fwd_bwd(TPAVI, f4, cl, ct, do, _params(g, "param_g:"), _params(g, "param_l:"))
    for v in range(V):
        assert O.rel_err(r_out[v].detach(), g[f"out:{v}"]) < TOL
        assert O.rel_err(r_df4[v], g[f"df4:{v}"]) < TOL
