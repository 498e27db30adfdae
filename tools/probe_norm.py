"""Bring-up probe: LayerNorm fwd/bwd (+quant), colsum, patchify vs torch/oracle."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200")); sys.path.insert(0, ROOT)
import numpy as np, torch
import torch.nn.functional as F
import mv_native as mv
from oracle import quant_oracle as qo
dev = "cuda"
torch.manual_seed(0)
def q(t, e=5, m=10):
    return mv.float_quantize(t, e, m)
for D in (192, 384, 768, 128):
    rows = 1000
    x = torch.randn(rows, D, device=dev) * 3; g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    y, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    xq = q(x)
    ref = F.layer_norm(xq.double(), (D,), g.double(), b.double(), 1e-5).float()
    refq = q(ref)
    d = (y.float() - refq).abs()
    print("ln fwd D%d: max diff %.3e  frac mismatch %.2e (fp16 ulp flips expected at ~1e-3)" % (D, d.max().item(), (d > 0).float().mean().item()))
    y32, _, _ = mv.layernorm_q_fwd(x, g, b, q_in=None, q_post=None, out_dtype=torch.float32)
    print("   fp32 no-quant max err %.3e" % (y32 - F.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-5).float()).abs().max().item())
    # backward
    dy = torch.randn(rows, D, device=dev); dres = torch.randn(rows, D, device=dev)
    xr = xq.double().requires_grad_(True); gr = g.double().requires_grad_(True); br = b.double().requires_grad_(True)
    out = F.layer_norm(xr, (D,), gr, br, 1e-5); out.backward(dy.double())
    dg = torch.zeros(D, device=dev); db = torch.zeros(D, device=dev); dp = torch.zeros(D, device=dev)
    dx, dx16 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dgamma=dg, dbeta=db, dbias_prev=dp)
    want = (xr.grad + dres.double())
    print("ln bwd D%d: dx err %.3e (max %.2f) f16copy err %.3e dgamma err %.3e dbeta err %.3e dbias_prev err %.3e" % (
        D, (dx.double() - want).abs().max().item(), want.abs().max().item(), (dx16.double() - want).abs().max().item(),
        (dg.double() - gr.grad).abs().max().item(), (db.double() - br.grad).abs().max().item(), (dp.double() - want.sum(0)).abs().max().item()))
# colsum
for dt in (torch.float16, torch.float32):
    a = torch.randn(65792 // 8, 1152, device=dev).to(dt); o = torch.zeros(1152, device=dev)
    mv.colsum(a, o)
    print("colsum", dt, "err %.3e" % (o.double() - a.double().sum(0)).abs().max().item())
# patchify
img = torch.randn(4, 3, 64, 96, device=dev)
pt = mv.patchify_q(img, 16, q_in=(5, 10))
ref = img.reshape(4, 3, 4, 16, 6, 16).permute(0, 2, 4, 3, 5, 1).reshape(4 * 24, 768)
print("patchify mismatches", int((pt.float() != q(ref.contiguous())).sum()))
# timing LN fwd/bwd at flagship size
rows, D = 65792, 384
x = torch.randn(rows, D, device=dev); g = torch.ones(D, device=dev); b = torch.zeros(D, device=dev)
dy = torch.randn(rows, D, device=dev)
y, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
dg = torch.zeros(D, device=dev); db = torch.zeros(D, device=dev); dp = torch.zeros(D, device=dev)
dx = torch.empty(rows, D, device=dev); dx16 = torch.empty(rows, D, device=dev, dtype=torch.float16)
def timeit(fn, n=20):
    for _ in range(3): fn()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
ms = timeit(lambda: mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10)))
print("ln fwd 65792x384: %.3f ms, %.0f GB/s (6 B/elem)" % (ms, rows * D * 6 / ms / 1e6))
ms = timeit(lambda: mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dy, q_in=(5, 10), dgamma=dg, dbeta=db, dbias_prev=dp, dx=dx, dx_f16=dx16))
print("ln bwd 65792x384: %.3f ms, %.0f GB/s (18 B/elem)" % (ms, rows * D * 18 / ms / 1e6))
