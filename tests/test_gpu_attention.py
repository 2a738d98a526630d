"""The softmax attention of mode='embedded' (csrc/glf_flash.cu) through glf_attention_fwd / glf_attention_bwd, against a
float64 reference evaluated on exactly the bf16 bytes the kernels read (P3 = [Theta | Phi | G], dY, and the Y the
backward reads):  S = Theta Phi^T (no 1/sqrt(d)), P = softmax(S), Y = P G, lse = logsumexp(S);  delta = rowsum(dY o Y),
dS = P o (dY G^T - delta), dTheta = dS Phi, dPhi = dS^T Theta, dG = P^T dY.

Errors are per row (Y and dTheta per query, dPhi and dG per key), each relative to max(|ref row|, 1e-2 * median row
norm); lse is compared as an absolute error.  The bounds follow from the kernels' roundings (P and dS rounded to bf16,
fp32 accumulation, bf16 stores, ex2.approx): 1e-2 for Y, 2e-3 for lse, 2e-2 for the gradients.

The inputs are built so that S has a known structure, and each regime asserts a witness on its reference that the
inputs reach what the regime is named for:
  random      |S| up to about 20 nats;
  shift       every score moved by a constant ab (Theta[:, 0] = a, Phi[:, 0] = b, exact in bf16).  At ab = -60 every
              real score is below -40, so a key past N that escaped the mask (score 0, value 0) would take nearly all
              of the softmax weight.  Y must not move and lse must move by exactly ab;
  late maxima a ramp over the last key tiles (Theta[:, 0] * Phi[:, 0]): the running maximum rises by more than 8 in
              log2 units from tile to tile, the largest score lies in the last, possibly partial, key tile;
  near one-hot  each query's winning key leads by at least 6 nats (and by not much more in the closest row, so the
              losing keys keep weights that dTheta and dPhi resolve above fp32 noise).
Every output buffer has 256 guard rows filled with a NaN bit pattern that must survive, and every call runs twice:
both paths write without atomics (the flash kernels and the chunked path's GEMMs store their tiles, split_k = 1; the
column statistics are per-CTA partials reduced in a fixed order), so the two results must be bitwise equal."""
import ctypes as C
import json
import math

import pytest
import torch

from glfusion_b200 import TPAVIModule
from glfusion_b200 import _lib as L
from gpu_util import BF16_TOL, DEV, assert_close, grad_scale, grad_tol, load_module_from_params, stream
from oracle import tpavi_oracle as O

pytestmark = pytest.mark.gpu

Y_TOL, LSE_TOL, GRAD_TOL = 1e-2, 2e-3, 2e-2
BIAS_TOL = 1e-4          # bias_grad against the fp64 column sums of the dP3 it was reduced from (fp32 partial sums)
GUARD = 256
LN2 = math.log(2.0)
SHIFTS = {0: (0.0, 0.0), -60: (6.0, -10.0), -20: (4.0, -5.0), 20: (4.0, 5.0), 60: (6.0, 10.0)}
RAMP_STEP = 10.0         # nats per key tile: 14.4 in log2 units, above the kernel's lazy-rescale threshold of 8
# The ramp is split as Theta[:, 0] = 8 times Phi[:, 0] = 1.25 per tile (both exact in bf16).  dTheta = dS Phi sums
# bf16-rounded dS against Phi's common column, dPhi = dS^T Theta against Theta's: a rounding error of about 2^-9 per dS
# entry times that column's size, against rows as long as the rest of Phi / Theta.  All of the 40-nat ramp on Phi
# (Theta[:, 0] = 1) would make that 40 x 2^-9 / |Phi row|, several 1e-2.  So the ramp is split, and Theta and Phi carry
# RAMP_FREE-long components on disjoint columns, which lengthen the rows and leave the scores unchanged.
RAMP_THETA = 8.0
RAMP_FREE = 8.0
ONE_HOT_LEAD = 6.5       # the closest row's lead; bf16 rounding of the unit vectors moves a score by ~0.05

FLASH_N = (64, 127, 128, 129, 255, 256, 257, 385, 1000, 3136)
FLASH = [(D, N, 1 if N in (127, 1000) else 3, None) for D in (64, 128) for N in FLASH_N]
# chunked exact path (head widths other than 64 / 128); B = 20 at N = 3136 runs as chunks of 18 + 2 sequences, and
# B = 70 at N = 1000 is 70 000 score rows in one chunk, more than one launch of softmax_bwd_kernel may cover (65 535)
CHUNKED = [(Ci, N, 2, None) for Ci in (32, 48, 96, 192) for N in (72, 129, 1000)] + \
          [(96, 3136, 20, (0, 17, 18, 19)), (48, 1000, 70, (0, 34, 65, 69))]
EXTRA_SHIFTS = {(64, 257), (128, 3136), (48, 129), (192, 1000)}


def _id(case):
    return f"D{case[0]}-N{case[1]}-B{case[2]}"


def _nan_rows(rows, cols, dtype):
    t = torch.empty(rows + GUARD, cols, dtype=dtype, device=DEV)
    t.view(torch.int16 if dtype == torch.bfloat16 else torch.int32).fill_(-1)    # all-ones: a NaN in bf16 and fp32
    return t


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


class Result:
    pass


def _attention(P3, dY, B, N, D):
    """Forward twice, backward twice (on the first forward's Y / lse); guard rows, finiteness and bitwise equality."""
    lib = L.load()
    rows = B * N
    nbytes = max(lib.glf_attention_scratch_bytes(B, N, D, 0), lib.glf_attention_scratch_bytes(B, N, D, 1))
    assert nbytes > 0
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    fw, bw = [], []
    for _ in range(2):
        Y, lse = _nan_rows(rows, D, torch.bfloat16), _nan_rows(rows, 1, torch.float32)
        L.check(lib.glf_attention_fwd(L.ptr(P3), L.ptr(Y), L.ptr(lse), B, N, D, L.ptr(scratch), stream()))
        fw.append((Y, lse))
    Y, lse = fw[0]
    for _ in range(2):
        dP3, bias = _nan_rows(rows, 3 * D, torch.bfloat16), _nan_rows(1, 3 * D, torch.float32)
        L.check(lib.glf_attention_bwd(L.ptr(P3), L.ptr(Y), L.ptr(dY), L.ptr(lse), L.ptr(dP3), L.ptr(bias), B, N, D,
                                      L.ptr(scratch), stream()))
        bw.append((dP3, bias))
    torch.cuda.synchronize()
    for name, (a, b), n in (("Y", (fw[0][0], fw[1][0]), rows), ("lse", (fw[0][1], fw[1][1]), rows),
                            ("dP3", (bw[0][0], bw[1][0]), rows), ("bias_grad", (bw[0][1], bw[1][1]), 1)):
        for t in (a, b):
            assert bool((_bits(t[n:]) == -1).all()), f"{name}: a guard row past the output was written"
        assert bool(torch.isfinite(a[:n]).all()), f"{name}: non-finite or unwritten entries"
        assert torch.equal(_bits(a[:n]), _bits(b[:n])), f"{name}: two calls on the same inputs differ"
    r = Result()
    r.Y = Y[:rows].view(B, N, D)
    r.lse = lse[:rows].view(B, N)
    r.dP3 = bw[0][0][:rows].view(B, N, 3 * D)
    r.bias = bw[0][1][0]
    return r


def _reference(p3, y, dy, D):
    """float64 attention of one sequence; delta from the bf16 Y the backward reads."""
    p = p3.double()
    th, ph, g = p[:, :D], p[:, D:2 * D], p[:, 2 * D:]
    S = th @ ph.T
    lse = torch.logsumexp(S, 1)
    P = torch.exp(S - lse[:, None])
    dy = dy.double()
    delta = (dy * y.double()).sum(1)
    dS = P * (dy @ g.T - delta[:, None])
    return dict(S=S, lse=lse, Y=P @ g, dTheta=dS @ ph, dPhi=dS.T @ th, dG=P.T @ dy)


def _row_err(got, ref):
    rn = ref.norm(dim=1)
    floor = max(1e-2 * float(rn.median()), 1e-30)
    return float(((got.double() - ref).norm(dim=1) / rn.clamp(min=floor)).max())


def _ramp(N):
    """Scores added by the ramp: flat, then RAMP_STEP more per key tile over the last (up to four) 128-key tiles."""
    T = (N + 127) // 128
    t = torch.arange(N, device=DEV) // 128
    return RAMP_STEP * (t - (T - 1 - min(T - 1, 4))).clamp(min=0).double()


def _inputs(regime, B, N, D, seed, ab=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    th, ph, gv, dy = (torch.randn(B, N, D, device=DEV, generator=g, dtype=torch.float64) for _ in range(4))
    if regime == "one_hot":   # key perm[i] = c * unit(Theta_i): S_i,perm[i] = c, every other score c * cos(angle)
        th = th / th.norm(dim=-1, keepdim=True)
        cos = th @ th.transpose(1, 2) - 3.0 * torch.eye(N, device=DEV, dtype=th.dtype)
        c = ONE_HOT_LEAD / float((1.0 - cos.max(-1).values).min())
        perm = torch.stack([torch.randperm(N, device=DEV, generator=g) for _ in range(B)])
        ph = torch.empty_like(th).scatter_(1, perm[..., None].expand(B, N, D), c * th)
    else:
        sigma = {"random": 4.0, "shift": 3.0, "ramp": 1.0}[regime]    # standard deviation of the random scores
        s = math.sqrt(sigma / math.sqrt(D))
        th, ph = th * s, ph * s
        if regime == "shift":
            th[..., 0], ph[..., 0] = SHIFTS[ab]
        elif regime == "ramp":   # columns 1 :: 3 carry the random scores, 2 :: 3 only Theta, 3 :: 3 only Phi
            th[..., 0] = RAMP_THETA
            ph[..., 0] = _ramp(N) / RAMP_THETA
            for t, own, other in ((th, 2, 3), (ph, 3, 2)):
                free = t[..., own::3]
                t[..., own::3] = free * (RAMP_FREE / free.norm(dim=-1, keepdim=True))
                t[..., other::3] = 0.0
    P3 = torch.cat([th, ph, gv], -1).to(torch.bfloat16).contiguous()
    return P3, dy.to(torch.bfloat16).contiguous()


def _witness(regime, ab=0):
    def check(S, N):
        if regime == "random":
            assert 8.0 < float(S.abs().max()) < 30.0
        elif regime == "shift" and ab == -60:
            assert float(S.max()) < -40.0                     # every real score; a padding key would score 0
        elif regime == "ramp":
            T = (N + 127) // 128
            if T == 1:
                return
            tmax = torch.stack([S[:, t * 128:(t + 1) * 128].max(1).values for t in range(T)], 1)
            events = torch.zeros(N, dtype=torch.int64, device=S.device)
            for t in range(1, T):
                events += (tmax[:, t] > tmax[:, :t].max(1).values + 8.0 * LN2).long()
            assert float((events >= min(2, T - 1)).double().mean()) >= 0.8, "the running maximum rarely rises by 8 (log2)"
            assert int(S.argmax(1).min()) >= (T - 1) * 128, "a row's largest score is not in the last key tile"
        elif regime == "one_hot":
            top = torch.topk(S, 2, dim=1).values
            assert float((top[:, 0] - top[:, 1]).min()) >= 6.0
    return check


def _check(tag, regime, case, ab=0, seed=1):
    D, N, B, seqs = case
    P3, dY = _inputs(regime, B, N, D, seed, ab)
    k = _attention(P3, dY, B, N, D)
    wit = _witness(regime, ab)
    err = dict(Y=0.0, lse=0.0, dTheta=0.0, dPhi=0.0, dG=0.0)
    for b in (range(B) if seqs is None else seqs):
        ref = _reference(P3[b], k.Y[b], dY[b], D)
        wit(ref["S"], N)
        err["Y"] = max(err["Y"], _row_err(k.Y[b], ref["Y"]))
        err["lse"] = max(err["lse"], float((k.lse[b].double() - ref["lse"]).abs().max()))
        for i, name in enumerate(("dTheta", "dPhi", "dG")):
            err[name] = max(err[name], _row_err(k.dP3[b, :, i * D:(i + 1) * D], ref[name]))
        del ref
    dp = k.dP3.reshape(B * N, 3 * D).double()
    err["bias"] = float(((k.bias.double() - dp.sum(0)).abs() / (dp.abs().sum(0) + 1e-30)).max())
    print("ATTN " + json.dumps(dict(case=tag, regime=regime, ab=ab, D=D, N=N, B=B,
                                    **{n: float(f"{v:.3e}") for n, v in err.items()})))
    assert err["Y"] < Y_TOL, f"{tag}: Y per-row error {err['Y']:.3e}"
    assert err["lse"] < LSE_TOL, f"{tag}: lse error {err['lse']:.3e}"
    for name in ("dTheta", "dPhi", "dG"):
        assert err[name] < GRAD_TOL, f"{tag}: {name} per-row error {err[name]:.3e}"
    assert err["bias"] < BIAS_TOL, f"{tag}: bias_grad vs the column sums of dP3: {err['bias']:.3e}"
    return k


@pytest.mark.parametrize("case", FLASH + CHUNKED, ids=_id)
def test_shifted_scores(case):
    """Softmax is invariant to a per-row shift: Y must not move, lse must move by ab.  At ab = -60 the key mask of
    every path decides the result."""
    D, N = case[0], case[1]
    base = _check(_id(case), "shift", case, ab=0)
    for ab in ((-60, -20, 20, 60) if (D, N) in EXTRA_SHIFTS else (-60,)):
        k = _check(_id(case), "shift", case, ab=ab)
        dy = max(_row_err(k.Y[b], base.Y[b].double()) for b in range(case[2]))
        dl = float((k.lse.double() - base.lse.double() - ab).abs().max())
        print("ATTN " + json.dumps(dict(case=_id(case), regime="shift-metamorphic", ab=ab, Y=float(f"{dy:.3e}"),
                                        lse=float(f"{dl:.3e}"))))
        assert dy < Y_TOL, f"ab = {ab}: Y moved by {dy:.3e} per row"
        assert dl < LSE_TOL, f"ab = {ab}: lse(shifted) - lse - ab = {dl:.3e}"


@pytest.mark.parametrize("case", FLASH + CHUNKED, ids=_id)
def test_late_maxima(case):
    """The running maximum rises several times per row and peaks in the last key tile: the forward's lazy rescale of
    O, and the last tile's mask where N % 128 != 0."""
    _check(_id(case), "ramp", case, seed=2)


@pytest.mark.parametrize("case", [(64, 1000, 1, None), (128, 257, 3, None), (128, 3136, 3, None), (32, 129, 2, None),
                                  (192, 1000, 2, None)], ids=_id)
def test_random_scores(case):
    _check(_id(case), "random", case, seed=3)


@pytest.mark.parametrize("case", [(64, 3136, 3, None), (128, 385, 3, None), (64, 129, 3, None), (48, 1000, 2, None),
                                  (96, 72, 2, None)], ids=_id)
def test_near_one_hot(case):
    _check(_id(case), "one_hot", case, seed=4)


@pytest.mark.parametrize("D", [64, 128, 32])
def test_single_token(D):
    """N = 1: the only key takes all the weight, so Y = G exactly, lse = S, dTheta = dPhi = 0 and dG = dY."""
    P3, dY = _inputs("random", 3, 1, D, seed=5)
    k = _attention(P3, dY, 3, 1, D)
    th, ph, g = P3[..., :D].double(), P3[..., D:2 * D].double(), P3[..., 2 * D:]
    assert torch.equal(k.Y, g)
    assert float((k.lse.double() - (th * ph).sum(-1)).abs().max()) < LSE_TOL
    assert float(k.dP3[..., :2 * D].double().abs().max()) < 1e-3 * float(dY.double().abs().max())
    assert _row_err(k.dP3[..., 2 * D:].reshape(3, D), dY.reshape(3, D).double()) < GRAD_TOL


def _per_token(got, ref):
    """[B, C, T, H, W] -> worst per-token relative error (rows of C channels)."""
    C_ = got.shape[1]
    return _row_err(got.permute(0, 2, 3, 4, 1).reshape(-1, C_), ref.permute(0, 2, 3, 4, 1).reshape(-1, C_).double())


@pytest.mark.parametrize("C_", [128, 256, 192])
@pytest.mark.parametrize("T,H,W", [(3, 5, 7), (4, 28, 28)], ids=["N105", "N3136"])
def test_module_shifted_scores(C_, T, H, W):
    """TPAVIModule(mode='embedded') with every score moved by -36 (theta.bias[0] = 6, phi.bias[0] = -6, row 0 of both
    weights zero) against the same module without the shift: the saved lse, delta from the stored Y and the bias sums
    in the regime where the key mask decides the result.  phi.weight's row 0 is the one gradient the shift changes
    (6 times the column sums of dS against x), so it is left out; every other entry must agree.  phi.bias is
    analytically zero with or without the shift (every row of dS sums to zero), so both must be rounding noise.
    C = 192 (head width 96) takes the chunked path; at N = 3136 its dTheta GEMM runs 256-row super-tiles and leaves a
    different number of column-statistic rows than the dPhi / dG GEMMs."""
    B = 2
    p = O.init_params(C_, seed=31, randomize_affine=True, bn_layer=False)
    p["theta.weight"][0] = 0.0
    p["phi.weight"][0] = 0.0
    gen = torch.Generator().manual_seed(32)
    x = torch.randn(B, C_, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    dz = torch.randn(B, C_, T, H, W, generator=gen).to(DEV, torch.bfloat16)
    out = []
    for a, b in ((0.0, 0.0), (6.0, -6.0)):
        q = {k: v.clone() for k, v in p.items()}
        q["theta.bias"][0], q["phi.bias"][0] = a, b
        m = load_module_from_params(TPAVIModule, q, C_, "embedded", False).eval()
        xi = x.clone().requires_grad_(True)
        z, _ = m(xi)
        z.backward(dz)
        torch.cuda.synchronize()
        out.append((z.detach(), xi.grad.detach(), {k: v.grad.detach() for k, v in m.named_parameters()
                                                   if not k.startswith("align_channel")}))
    (z0, dx0, g0), (z1, dx1, g1) = out
    ez, edx = _per_token(z1, z0), _per_token(dx1, dx0)
    print("ATTN " + json.dumps(dict(case=f"module-C{C_}-N{T * H * W}", regime="shift-36", z=float(f"{ez:.3e}"),
                                    dx=float(f"{edx:.3e}"))))
    assert ez < BF16_TOL and edx < BF16_TOL
    g0["phi.weight"], g1["phi.weight"] = g0["phi.weight"][1:], g1["phi.weight"][1:]
    scale = grad_scale(g0.values())
    zb = [float(g["phi.bias"].abs().max()) / scale for g in (g0, g1)]
    print("ATTN " + json.dumps(dict(case=f"module-C{C_}-N{T * H * W}", regime="phi.bias/scale", base=float(f"{zb[0]:.3e}"),
                                    shifted=float(f"{zb[1]:.3e}"))))
    assert max(zb) < grad_tol("phi.bias", "embedded"), f"phi.bias is not rounding noise: {zb}"
    del g0["phi.bias"], g1["phi.bias"]
    for k in g0:
        assert_close("grad:" + k, g1[k], g0[k], grad_tol(k, "embedded"), zero_scale=scale)
