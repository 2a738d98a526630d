"""S = X^T X (one input) and R = dV^T X (two inputs) of gram_kernel at the bench shape, timed alone."""
import sys, os, ctypes as C, torch
sys.path.insert(0, os.getcwd())
from glfusion_b200 import _lib as L
lib = L.load()
dev = "cuda:0"
B, N, Cc = 128, 3136, 256
X = torch.randn(B, N, Cc, device=dev).to(torch.bfloat16)
dV = torch.randn(B, N, Cc, device=dev).to(torch.bfloat16)
D = torch.empty(B, Cc, Cc, device=dev, dtype=torch.bfloat16)
rs = torch.empty(B, Cc, device=dev)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
def t(a):
    for _ in range(3):
        L.check(lib.glf_gram_contraction(L.ptr(a), L.ptr(X), L.ptr(D), L.ptr(rs), B, N, Cc, Cc, st))
    ts = []
    for _ in range(10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); L.check(lib.glf_gram_contraction(L.ptr(a), L.ptr(X), L.ptr(D), L.ptr(rs), B, N, Cc, Cc, st)); e1.record()
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort(); return ts[len(ts) // 2]
print("S %.1f us  R %.1f us" % (t(X), t(dV)))
