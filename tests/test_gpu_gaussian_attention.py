"""The softmax attention of mode='gaussian' (csrc/glf_flash.cu) through glf_attention_gaussian_fwd / _bwd, against a
float64 reference evaluated on exactly the bf16 bytes the kernels read (X, G, dY, and the Y the backward reads):
S = X X^T (no projection, no 1/sqrt(C)), P = softmax(S), Y = P G, lse = logsumexp(S);  delta = rowsum(dY o Y),
dS = P o (dY G^T - delta), dX = dS X + dS^T X, dG = P^T dY.

With N(0, 1) tokens the self score |x|^2 ~ C dominates every row, P is the identity and no gradient flows through the
softmax.  So the tokens are clustered: x = centre of its cluster (8 tokens each, entries of variance 1/2) + noise, the
centres far apart (other clusters' scores lie C/2 nats, less a few standard deviations of C^(1/2)/2, below), the noise
scaled so that a token's self score leads its cluster's other keys by about one nat, against a spread of about one nat
that the noise puts on those keys.  Each case asserts that witness on its reference: the mean largest probability per query lies in
(0.1, 0.9), and for at least a tenth of the queries the largest score is not the self key.

Errors are per row, relative to max(|ref row|, 1e-2 * median row norm); lse as an absolute error.  Bounds as for
mode='embedded' (tests/test_gpu_attention.py): 1e-2 for Y, 2e-3 for lse, 2e-2 for the gradients, except where dX is
ill-conditioned: a row of dS sums to zero, so dS X is a small difference of the keys' shared cluster centre, and the
bf16 rounding of dS (every bf16 implementation rounds it) does not cancel there.  That rounding's own effect is
measured per case on the fp64 reference (dS rounded to bf16, then the products in fp64: 2e-2 to 8e-2 on these inputs,
growing with C); the dX bound is that floor times 1.1 plus 5e-3, at least 2e-2.  So the kernels may add little beyond
the rounding of dS itself (measured on B200: at most 1e-3 beyond it).  Every output buffer
has 256 NaN guard rows that must survive, and every call runs twice: no path uses atomics, so the two results must be
bitwise equal."""
import json
import math

import pytest
import torch

from glfusion_b200 import _lib as L
from gpu_util import DEV, stream

pytestmark = pytest.mark.gpu

Y_TOL, LSE_TOL, GRAD_TOL = 1e-2, 2e-3, 2e-2
BIAS_TOL = 1e-4
GUARD = 256
CLUSTER = 8              # tokens per cluster
CENTRE_VAR = 0.5         # per-entry variance of a centre: |centre|^2 = C / 2
SELF_LEAD = 1.0          # |noise|^2: the self score's expected lead over the rest of its cluster

FLASH_N = (64, 127, 129, 257, 1000, 3136)
FLASH = [(C_, Ci, N, 1 if N in (127, 1000) else 3, None) for C_, Ci in ((64, 64), (128, 64), (128, 128))
         for N in FLASH_N]
# chunked exact path (every other width pair); B = 20 at N = 3136 runs as chunks of 18 + 2 sequences, and B = 70 at
# N = 1000 is 70 000 score rows in one chunk, more than one launch of softmax_bwd_kernel covers (65 535)
CHUNKED = [(C_, Ci, N, 2, None) for C_, Ci in ((64, 32), (96, 48), (192, 96), (256, 128)) for N in (64, 129, 1000)] + \
          [(256, 128, 3136, 20, (0, 17, 18, 19)), (96, 48, 1000, 70, (0, 34, 65, 69)), (256, 32, 257, 2, None)]


def _id(case):
    return f"C{case[0]}-Ci{case[1]}-N{case[2]}-B{case[3]}"


def _nan_rows(rows, cols, dtype):
    t = torch.empty(rows + GUARD, cols, dtype=dtype, device=DEV)
    t.view(torch.int16 if dtype == torch.bfloat16 else torch.int32).fill_(-1)    # all-ones: a NaN in bf16 and fp32
    return t


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def clustered_tokens(B, N, C_, gen, dtype=torch.float64):
    """[B, N, C] tokens x = centre + noise (CLUSTER tokens per centre, randomly placed): a non-trivial softmax of x x^T."""
    nc = max(1, N // CLUSTER)
    centres = torch.randn(B, nc, C_, generator=gen, dtype=torch.float64) * math.sqrt(CENTRE_VAR)
    assign = torch.stack([torch.randperm(N, generator=gen) % nc for _ in range(B)])
    x = torch.gather(centres, 1, assign[..., None].expand(B, N, C_))
    x = x + torch.randn(B, N, C_, generator=gen, dtype=torch.float64) * math.sqrt(SELF_LEAD / C_)
    return x.to(dtype)


def witness(S):
    """S [N, N] float64 scores of one sequence: the softmax is neither uniform nor the identity."""
    P = torch.softmax(S, 1)
    pmax = float(P.max(1).values.mean())
    not_self = float((S.argmax(1) != torch.arange(S.shape[0], device=S.device)).double().mean())
    assert 0.1 < pmax < 0.9, f"mean largest probability {pmax:.3f}"
    assert not_self >= 0.1, f"the self key is the largest score for {1 - not_self:.1%} of the queries"
    return pmax, not_self


class Result:
    pass


def _attention(X, G, dY, B, N, C_, Ci):
    lib = L.load()
    rows = B * N
    nbytes = max(lib.glf_attention_gaussian_scratch_bytes(B, N, C_, Ci, 0),
                 lib.glf_attention_gaussian_scratch_bytes(B, N, C_, Ci, 1))
    assert nbytes > 0
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    fw, bw = [], []
    for _ in range(2):
        Y, lse = _nan_rows(rows, Ci, torch.bfloat16), _nan_rows(rows, 1, torch.float32)
        L.check(lib.glf_attention_gaussian_fwd(L.ptr(X), L.ptr(G), L.ptr(Y), L.ptr(lse), B, N, C_, Ci, L.ptr(scratch),
                                               stream()))
        fw.append((Y, lse))
    Y, lse = fw[0]
    for _ in range(2):
        dX, dG, bias = (_nan_rows(rows, C_, torch.bfloat16), _nan_rows(rows, Ci, torch.bfloat16),
                        _nan_rows(1, Ci, torch.float32))
        L.check(lib.glf_attention_gaussian_bwd(L.ptr(X), L.ptr(G), L.ptr(Y), L.ptr(dY), L.ptr(lse), L.ptr(dX), L.ptr(dG),
                                               L.ptr(bias), B, N, C_, Ci, L.ptr(scratch), stream()))
        bw.append((dX, dG, bias))
    torch.cuda.synchronize()
    for name, (a, b), n in (("Y", (fw[0][0], fw[1][0]), rows), ("lse", (fw[0][1], fw[1][1]), rows),
                            ("dX", (bw[0][0], bw[1][0]), rows), ("dG", (bw[0][1], bw[1][1]), rows),
                            ("bias_grad", (bw[0][2], bw[1][2]), 1)):
        for t in (a, b):
            assert bool((_bits(t[n:]) == -1).all()), f"{name}: a guard row past the output was written"
        assert bool(torch.isfinite(a[:n]).all()), f"{name}: non-finite or unwritten entries"
        assert torch.equal(_bits(a[:n]), _bits(b[:n])), f"{name}: two calls on the same inputs differ"
    r = Result()
    r.Y = Y[:rows].view(B, N, Ci)
    r.lse = lse[:rows].view(B, N)
    r.dX = bw[0][0][:rows].view(B, N, C_)
    r.dG = bw[0][1][:rows].view(B, N, Ci)
    r.bias = bw[0][2][0]
    return r


def _reference(x, g, y, dy):
    x, g, dy = x.double(), g.double(), dy.double()
    S = x @ x.T
    lse = torch.logsumexp(S, 1)
    P = torch.exp(S - lse[:, None])
    delta = (dy * y.double()).sum(1)
    dS = P * (dy @ g.T - delta[:, None])
    dSb = dS.to(torch.bfloat16).double()
    dX = dS @ x + dS.T @ x
    return dict(S=S, lse=lse, Y=P @ g, dX=dX, dG=P.T @ dy, dX_floor=_row_err(dSb @ x + dSb.T @ x, dX))


def _row_err(got, ref):
    rn = ref.norm(dim=1)
    floor = max(1e-2 * float(rn.median()), 1e-30)
    return float(((got.double() - ref).norm(dim=1) / rn.clamp(min=floor)).max())


def _inputs(B, N, C_, Ci, seed):
    gen = torch.Generator().manual_seed(seed)
    X = clustered_tokens(B, N, C_, gen)
    G = torch.randn(B, N, Ci, generator=gen, dtype=torch.float64)
    dY = torch.randn(B, N, Ci, generator=gen, dtype=torch.float64)
    return tuple(t.to(DEV, torch.bfloat16).contiguous() for t in (X, G, dY))


@pytest.mark.parametrize("case", FLASH + CHUNKED, ids=_id)
def test_clustered_tokens(case):
    C_, Ci, N, B, seqs = case
    X, G, dY = _inputs(B, N, C_, Ci, seed=7 + N)
    k = _attention(X, G, dY, B, N, C_, Ci)
    err = dict(Y=0.0, lse=0.0, dX=0.0, dG=0.0)
    wit = []
    floor = 0.0
    for b in (range(B) if seqs is None else seqs):
        ref = _reference(X[b], G[b], k.Y[b], dY[b])
        wit.append(witness(ref["S"]))
        err["Y"] = max(err["Y"], _row_err(k.Y[b], ref["Y"]))
        err["lse"] = max(err["lse"], float((k.lse[b].double() - ref["lse"]).abs().max()))
        err["dX"] = max(err["dX"], _row_err(k.dX[b], ref["dX"]))
        floor = max(floor, ref["dX_floor"])
        err["dG"] = max(err["dG"], _row_err(k.dG[b], ref["dG"]))
        del ref
    dg = k.dG.reshape(B * N, Ci).double()
    err["bias"] = float(((k.bias.double() - dg.sum(0)).abs() / (dg.abs().sum(0) + 1e-30)).max())
    print("GAUSS " + json.dumps(dict(case=_id(case), pmax=round(min(w[0] for w in wit), 3),
                                     not_self=round(min(w[1] for w in wit), 3), dX_floor=float(f"{floor:.3e}"),
                                     **{n: float(f"{v:.3e}") for n, v in err.items()})))
    assert err["Y"] < Y_TOL, f"Y per-row error {err['Y']:.3e}"
    assert err["lse"] < LSE_TOL, f"lse error {err['lse']:.3e}"
    dx_tol = max(GRAD_TOL, 1.1 * floor + 5e-3)
    assert err["dX"] < dx_tol, f"dX per-row error {err['dX']:.3e} (dS rounding alone: {floor:.3e})"
    assert err["dG"] < GRAD_TOL, f"dG per-row error {err['dG']:.3e}"
    assert err["bias"] < BIAS_TOL, f"bias_grad vs the column sums of dG: {err['bias']:.3e}"


@pytest.mark.parametrize("C_,Ci", [(128, 64), (96, 48)])
def test_single_token(C_, Ci):
    """N = 1: the only key takes all the weight, so Y = G exactly, lse = |x|^2, dX = 0 and dG = dY."""
    X, G, dY = _inputs(3, 1, C_, Ci, seed=5)
    k = _attention(X, G, dY, 3, 1, C_, Ci)
    assert torch.equal(k.Y, G)
    assert float((k.lse.double() - (X.double() ** 2).sum(-1)).abs().max()) < LSE_TOL * max(1.0, float(k.lse.abs().max()))
    assert float(k.dX.double().abs().max()) < 1e-3 * float(dY.double().abs().max()) * float(X.double().abs().max())
    assert _row_err(k.dG.reshape(3, Ci), dY.reshape(3, Ci).double()) < GRAD_TOL
