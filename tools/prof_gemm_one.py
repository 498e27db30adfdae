"""Profiling driver: a few launches of one GEMM shape.  usage: prof_gemm_one.py N K mode
mode: plain | res | gelu | dgelu | wgrad"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200")); sys.path.insert(0, ROOT)
import torch
import mv_native as mv
N, K, mode = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
M = 65792
dev, h = "cuda", torch.float16
torch.manual_seed(0)
nbuf = 3
if mode == "wgrad":
    dY = [torch.randn(M, N, device=dev).to(h) for _ in range(nbuf)]
    X = [torch.randn(M, K, device=dev).to(h) for _ in range(nbuf)]
    out = torch.zeros(N, K, device=dev)
    for i in range(2 * nbuf):
        mv.gemm(dY[i % nbuf], X[i % nbuf], out, a_major=1, b_major=1, accumulate=True)
else:
    A = [torch.randn(M, K, device=dev).to(h) for _ in range(nbuf)]
    # fc1 + GELU: u = fc1's output with the spread of the benchmark's random init (std 0.4); randn weights would put half of
    # the GELU outputs below fp16's normal range (the quantiser's rare branch on every group)
    B = (torch.randn(N, K, device=dev) * (0.4 / K ** 0.5 if mode == "gelu" else 1.0)).to(h)
    odt = torch.float32 if mode == "res" else h
    out = [torch.empty(M, N, device=dev, dtype=odt) for _ in range(nbuf)]
    aux = [torch.randn(M, N, device=dev).to(h) for _ in range(nbuf)]
    res = [torch.randn(M, N, device=dev) for _ in range(nbuf)] if mode == "res" else None
    bias = torch.randn(N, device=dev) * (0.02 if mode == "gelu" else 1.0)
    for i in range(2 * nbuf):
        j = i % nbuf
        if mode == "gelu": mv.gemm(A[j], B, out[j], bias=bias, aux=aux[j], epilogue=mv.EPI_GELU, q_res=(5, 10))
        elif mode == "dgelu": mv.gemm(A[j], B, out[j], aux=aux[j], epilogue=mv.EPI_DGELU)
        elif mode == "res": mv.gemm(A[j], B, out[j], bias=bias, residual=res[j])
        else: mv.gemm(A[j], B, out[j], bias=bias)
torch.cuda.synchronize()
print("ok")
