"""The cycle-consistency oracle (oracle/cycle_oracle.py) against golden vectors produced by the reference's own
Trainer.seg_cycle / Trainer.dense_seg_cycle (R/main.py:650-798, oracle/gen_golden_cycle.py), and against the live
reference methods when they are staged in oracle/_ref.  CPU only."""
import glob
import os

import numpy as np
import pytest

from oracle import cycle_oracle as CO

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cycle_*.npz")))


def run_oracle(d, feat=None):
    feat = d["feat"] if feat is None else feat
    R, off, ch, temp = int(d["target_region"]), int(d["cyc_off"]), int(d["chunk_size"]), float(d["temperature"])
    if int(d["dense"]):
        return CO.dense_seg_cycle(feat, R, off, ch, temp, bool(d["soft_label"]), bool(d["is_overlap"]))
    return CO.seg_cycle(feat, R, off, ch, temp, int(d["target_strtpt"]))


def test_golden_fixtures_exist():
    assert len(GOLDEN) == 5


def check_oracle(d):
    loss, g = run_oracle(d)
    assert abs(loss - float(d["loss"])) <= 2e-6 * abs(float(d["loss"]))           # the reference ran in fp32
    assert np.abs(g - d["dfeat"]).max() <= 5e-5 * np.abs(d["dfeat"]).max()


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_matches_reference_golden(path):
    check_oracle(np.load(path))


@pytest.mark.parametrize("path", GOLDEN[:2] + GOLDEN[-1:], ids=lambda p: os.path.basename(p)[:-4])
def test_oracle_gradient_is_the_derivative_of_its_loss(path):
    """Central differences in fp64 along random directions: the hand-derived backward is the gradient of the loss."""
    d = np.load(path)
    feat = d["feat"].astype(np.float64)
    _, g = run_oracle(d, feat)
    rng = np.random.default_rng(0)
    for _ in range(3):
        v = rng.standard_normal(feat.shape)
        eps = 1e-5
        lp, _ = run_oracle(d, feat + eps * v)
        lm, _ = run_oracle(d, feat - eps * v)
        num = (lp - lm) / (2 * eps)
        assert abs(num - (g * v).sum()) <= 1e-6 * max(1.0, abs(num))


def test_spatial_sum_restatement():
    x = np.arange(2 * 3 * 4 * 5, dtype=np.float32).reshape(2, 3, 4, 5)
    assert np.array_equal(CO.spatial_sum(x), x.astype(np.float64).reshape(2, 3, -1).sum(-1))


def test_rejects_too_few_frames():
    with pytest.raises(ValueError):
        CO.seg_cycle(np.zeros((18, 8)), 16, 2, 3, 10.0, 0)          # key region shorter than chunk + offset


def test_oracle_matches_live_reference_methods():
    """The oracle against the reference's Trainer.seg_cycle / dense_seg_cycle: on the runs they recorded
    (tests/golden/cycle_*.npz) and, when the reference's main.py is staged in oracle/_ref, on live runs of them."""
    import types

    import torch
    from oracle import build_ref
    from oracle import gen_golden_cycle as G
    for path in GOLDEN:
        check_oracle(np.load(path))
    if not os.path.exists(build_ref.REF_MAIN):
        return
    seg_cycle, dense_seg_cycle = G.load_reference_methods(build_ref.REF_MAIN)
    me = types.SimpleNamespace(device=torch.device("cpu"))
    feat = G.features(34, 48, seed=21)
    for kw in ({"soft_label": False, "is_overlap": True}, {"soft_label": True, "is_overlap": False}):
        f = feat.clone().requires_grad_(True)
        loss = dense_seg_cycle(me, f, target_region=14, cyc_off=1, chunk_size=2, temperature=7.0, **kw)
        loss.backward()
        lo, go = CO.dense_seg_cycle(feat.numpy(), 14, 1, 2, 7.0, **kw)
        assert abs(lo - loss.item()) <= 2e-6 * abs(lo)
        assert np.abs(go - f.grad.numpy()).max() <= 5e-5 * np.abs(go).max()
    np.random.seed(5)
    start = int(np.random.choice(CO.positions(14, 1, 2)))
    np.random.seed(5)
    f = feat.clone().requires_grad_(True)
    loss = seg_cycle(me, f, target_region=14, cyc_off=1, chunk_size=2, temperature=7.0)
    loss.backward()
    lo, go = CO.seg_cycle(feat.numpy(), 14, 1, 2, 7.0, start)
    assert abs(lo - loss.item()) <= 2e-6 * abs(lo)
    assert np.abs(go - f.grad.numpy()).max() <= 5e-5 * np.abs(go).max()
