"""Host-side mirror of the reference interface: constructor, state_dict, init, error behaviour (no GPU needed)."""
import os

import pytest
import torch

from conftest import GOLDEN, load_golden

import glfusion_b200
from glfusion_b200 import GlfError, GlobalLocalFusion, TPAVIModule


def test_state_dict_keys_shapes_match_reference_contract():
    C = 256
    m = TPAVIModule(in_channels=C, mode='dot')
    sd = m.state_dict()
    expect = {
        "align_channel.weight": (C, 128), "align_channel.bias": (C,),
        "norm_layer.weight": (C,), "norm_layer.bias": (C,),
        "g.weight": (C // 2, C, 1, 1, 1), "g.bias": (C // 2,),
        "theta.weight": (C // 2, C, 1, 1, 1), "theta.bias": (C // 2,),
        "phi.weight": (C // 2, C, 1, 1, 1), "phi.bias": (C // 2,),
        "W_z.0.weight": (C, C // 2, 1, 1, 1), "W_z.0.bias": (C,),
        "W_z.1.weight": (C,), "W_z.1.bias": (C,), "W_z.1.running_mean": (C,), "W_z.1.running_var": (C,),
        "W_z.1.num_batches_tracked": (),
    }
    assert {k: tuple(v.shape) for k, v in sd.items()} == expect
    assert sd["W_z.1.num_batches_tracked"].dtype == torch.int64
    # reference init: BN gamma = beta = 0 (ours.py:826-827)
    assert sd["W_z.1.weight"].abs().max() == 0 and sd["W_z.1.bias"].abs().max() == 0


@pytest.mark.parametrize("name", ["dot_train_c128", "dot_nobn_c128", "embedded_train_c128"])
def test_reference_checkpoint_loads_strict(name):
    g = load_golden(name)
    B, C, T, H, W, training, bn = [int(v) for v in g["meta"]]
    m = TPAVIModule(in_channels=C, mode=str(g["mode"]), bn_layer=bool(bn))
    sd = {k[len("param:"):]: (v if isinstance(v, torch.Tensor) else torch.tensor(v.item())) for k, v in g.items()
          if k.startswith("param:")}
    m.load_state_dict(sd, strict=True)


def test_constructor_argument_errors_match_reference():
    with pytest.raises(ValueError):
        TPAVIModule(64, mode='softmax')
    with pytest.raises(AssertionError):
        TPAVIModule(64, dimension=4)
    with pytest.raises(NotImplementedError):
        TPAVIModule(64, mode='concatenate')
    m = TPAVIModule(3)
    assert m.inter_channels == 1          # ours.py:789-791
    assert TPAVIModule(64, inter_channels=16).inter_channels == 16


def test_cpu_tensors_fail_loudly_no_fallback():
    m = TPAVIModule(64)
    with pytest.raises(GlfError):
        m(torch.randn(1, 64, 2, 4, 4))
    f = GlobalLocalFusion(64)
    with pytest.raises(GlfError):
        f.forward_stacked([torch.randn(1, 64, 4, 4)], [torch.randn(1, 5, 4, 4)], [torch.randn(1, 1, 4, 4)])
    with pytest.raises(NotImplementedError):
        m(torch.randn(1, 64, 2, 4, 4), audio=torch.randn(1, 2, 128))


def test_fusion_module_uses_reference_attribute_names():
    f = GlobalLocalFusion(128)
    keys = set(f.state_dict().keys())
    assert "global_attn.theta.weight" in keys and "local_attn.W_z.1.running_var" in keys   # ours.py:1746-1747


def test_reference_network_checkpoint_slice_loads():
    """A checkpoint in the reference's wire format (main.py:857-872, optionally with the 'module.' prefix of
    main.py:454-457) holds the whole network; the fusion blocks take their slice with strict=True."""
    torch.manual_seed(7)
    src = GlobalLocalFusion(64)
    for p in src.parameters():
        torch.nn.init.normal_(p, std=0.1)
    net = {"module." + k: v.clone() for k, v in src.state_dict().items()}
    net["module.backbone.conv1.weight"] = torch.zeros(8, 1, 7, 7)          # other parts of Global_and_Local
    net["module.classifier.1.4.weight"] = torch.zeros(5, 256, 1, 1)
    dst = GlobalLocalFusion(64)
    res = dst.load_reference_checkpoint({"network": net})
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in src.state_dict().items():
        assert torch.equal(dst.state_dict()[k], v), k
    broken = {k: v for k, v in net.items() if not k.endswith("local_attn.theta.bias")}
    with pytest.raises(RuntimeError):
        GlobalLocalFusion(64).load_reference_checkpoint({"network": broken})


def test_init_rng_stream_identical_to_reference():
    """Under torch.manual_seed the constructor draws the same weights as the reference's (the same nn holders created
    in the same order): the state dict must equal tests/golden/init_dot_c96.npz (oracle/gen_golden.py::run_init_case)
    bit for bit, and, when the reference module is staged in oracle/_ref, the reference's own state dict."""
    import numpy as np
    from oracle import build_ref
    from oracle import gen_golden as G
    golden = np.load(os.path.join(GOLDEN, "init_dot_c96.npz"))
    so = G.run_init_case(TPAVIModule)
    assert list(so) == golden.files
    for k in so:
        assert so[k].dtype == golden[k].dtype and np.array_equal(so[k], golden[k]), k
    Ref = build_ref.load_reference_tpavi()
    if Ref is not None:
        sr = G.run_init_case(Ref)
        assert list(sr) == list(so)
        for k in sr:
            assert np.array_equal(sr[k], so[k]), k


def test_install_patches_reference_namespace():
    import types
    fake = types.SimpleNamespace(TPAVIModule=None)
    glfusion_b200.install(fake)
    assert fake.TPAVIModule is TPAVIModule
