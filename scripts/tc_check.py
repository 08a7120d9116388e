"""Standalone check of the tcgen05 GEMMs against fp64 (run under `timeout`; a deadlock must not hang the box)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from spgnn_b200 import ops
from spgnn_b200._lib import lib, ptr, stream

def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())

def check(M, K1, K2, N, seed=0):
    g = torch.Generator().manual_seed(seed)
    x1 = torch.randn(M, K1, generator=g); x2 = torch.randn(M, K2, generator=g) if K2 else None
    W = torch.randn(N, K1 + K2, generator=g) / (K1 + K2) ** 0.5
    go = torch.randn(M, N, generator=g)
    xs = [t.cuda().requires_grad_() for t in ([x1, x2] if K2 else [x1])]
    Wc = W.cuda().requires_grad_()
    ops.GEMM_MODE = 1
    y = ops.linear(xs[0], Wc, None, None, x2=xs[1] if K2 else None)
    torch.cuda.synchronize()
    xd = torch.cat([x1, x2], 1).double() if K2 else x1.double()
    yd = xd @ W.double().t()
    e_f = rel(y.detach().cpu(), yd)
    y.backward(go.cuda()); torch.cuda.synchronize()
    dxd = go.double() @ W.double()
    dWd = go.double().t() @ xd
    e_x = rel(torch.cat([t.grad for t in xs], 1).cpu(), dxd)
    e_w = rel(Wc.grad.cpu(), dWd)
    print(f"M={M} K={K1}+{K2} N={N}: fwd {e_f:.2e}  dX {e_x:.2e}  dW {e_w:.2e}", flush=True)
    return max(e_f, e_x, e_w)

if __name__ == "__main__":
    print(torch.cuda.get_device_name(0))
    worst = 0
    for shp in [(128, 64, 0, 16), (300, 64, 0, 48), (1000, 1024, 39, 130), (257, 39, 0, 258), (513, 100, 8, 22),
                (5000, 1024, 40, 1028), (4096, 192, 0, 4100), (3001, 768, 0, 516)]:
        worst = max(worst, check(*shp))
    print("worst", worst)
