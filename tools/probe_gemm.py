"""Bring-up probe (not a test): runs the tcgen05 GEMM over many layouts/shapes on the GPU and
prints error statistics instead of asserting, so one gpurun call tells us as much as possible."""
import os, sys, time, traceback
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200")); sys.path.insert(0, ROOT)
import torch
import mv_native as mv

torch.manual_seed(0)
dev = "cuda"

def ref_mm(A, B, a_major, b_major):
    Af = A.double(); Bf = B.double()
    if a_major: Af = Af.t()
    if b_major: Bf = Bf.t()
    return Af @ Bf.t()

def report(name, got, want):
    got = got.double(); err = (got - want).abs()
    denom = want.abs().max().item() + 1e-30
    bad = (err > 1e-2 * denom)
    print("%-58s max_abs_err %.3e  (ref max %.3e)  rel %.3e  bad %d/%d" % (name, err.max().item(), denom, err.max().item()/denom, int(bad.sum()), bad.numel()), flush=True)
    if bad.any():
        idx = bad.nonzero()[:6].tolist()
        print("    first bad idx:", idx, "rows bad:", int(bad.any(1).sum()), "cols bad:", int(bad.any(0).sum()))
        rows = bad.any(1).nonzero().flatten()[:20].tolist(); cols = bad.any(0).nonzero().flatten()[:20].tolist()
        print("    bad rows", rows, "bad cols", cols)

def run(name, fn):
    try:
        fn(); torch.cuda.synchronize()
    except Exception as e:
        print(name, "EXC", repr(e)); traceback.print_exc()

def case(M, N, K, adt, bdt, a_major, b_major, **kw):
    def f():
        A = (torch.randn((K, M) if a_major else (M, K), device=dev)).to(adt)
        B = (torch.randn((K, N) if b_major else (N, K), device=dev)).to(bdt)
        out = torch.full((M, N), float("nan"), device=dev)
        mv.gemm(A, B, out, a_major=a_major, b_major=b_major, **kw)
        torch.cuda.synchronize()
        report("M%d N%d K%d %s x %s amaj%d bmaj%d" % (M, N, K, str(adt)[6:], str(bdt)[6:], a_major, b_major), out, ref_mm(A, B, a_major, b_major))
    run("case", f)

h, f32 = torch.float16, torch.float32
case(128, 128, 64, h, h, 0, 0)
case(128, 128, 128, h, h, 0, 0)
case(256, 256, 384, h, h, 0, 0)
case(128, 128, 64, h, h, 1, 0)
case(128, 128, 64, h, h, 0, 1)
case(128, 128, 64, h, h, 1, 1)
case(256, 384, 512, h, h, 1, 1)
case(128, 128, 32, f32, f32, 0, 0)
case(256, 128, 256, f32, f32, 0, 0)
case(128, 128, 32, f32, f32, 1, 1)
case(256, 256, 128, f32, f32, 1, 1)
case(200, 45, 384, h, h, 0, 0)
case(1000, 384, 1536, h, h, 0, 0)
case(65792, 1152, 384, h, h, 0, 0)
case(1000, 1536, 384, h, h, 0, 0)
case(1000, 256, 384, h, h, 0, 0)
case(512, 512, 4096, h, h, 1, 1)

# split-K accumulate (wgrad shape): dW[N_out, K_in] = dY^T X
def wgrad():
    T, No, Ki = 8192, 384, 1536
    dY = torch.randn(T, No, device=dev).to(h); X = torch.randn(T, Ki, device=dev).to(h)
    out = torch.zeros(No, Ki, device=dev)
    mv.gemm(dY, X, out, a_major=1, b_major=1, accumulate=True)
    torch.cuda.synchronize()
    report("wgrad splitK T8192 384x1536", out, dY.double().t() @ X.double())
run("wgrad", wgrad)

# epilogue: bias + residual + quant
def epi():
    M, N, K = 512, 384, 384
    A = torch.randn(M, K, device=dev).to(h); B = (torch.randn(N, K, device=dev) * 0.05).to(h)
    bias = torch.randn(N, device=dev); res = torch.randn(M, N, device=dev)
    out = torch.empty(M, N, device=dev)
    mv.gemm(A, B, out, bias=bias, residual=res)
    report("epi bias+res", out, A.double() @ B.double().t() + bias.double() + res.double())
    outh = torch.empty(M, N, device=dev, dtype=h)
    mv.gemm(A, B, outh, bias=bias, q_out=(5, 10))
    want = mv.float_quantize((A.float() @ B.float().t() + bias), 5, 10)
    report("epi bias+q_out->f16", outh, want.double())
    u = torch.empty(M, N, device=dev, dtype=h); hh = torch.empty(M, N, device=dev, dtype=h)
    mv.gemm(A, B, hh, bias=bias, aux=u, epilogue=mv.EPI_GELU, q_res=(5, 10))
    uu = (A.double() @ B.double().t() + bias.double()).requires_grad_(True)
    torch.nn.functional.gelu(uu).sum().backward()
    report("epi gelu' (aux)", u, uu.grad)
    report("epi gelu h", hh, torch.nn.functional.gelu(uu).detach())
run("epi", epi)

# timing of the flagship shapes
def bench(M, N, K, iters=20):
    A = torch.randn(M, K, device=dev).to(h); B = torch.randn(N, K, device=dev).to(h)
    out = torch.empty(M, N, device=dev, dtype=h)
    for _ in range(3): mv.gemm(A, B, out)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): mv.gemm(A, B, out)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    print("bench M%d N%d K%d f16 out: %.3f ms  %.1f TFLOP/s  %.1f GB/s" % (M, N, K, ms, 2.0*M*N*K/ms/1e9, (M*K*2+N*K*2+M*N*2)/ms/1e6), flush=True)
    Af, Bf = A.float(), B.float()
    torch.backends.cuda.matmul.allow_tf32 = True
    for _ in range(3): Ah = A @ B.t()
    e0.record()
    for _ in range(iters): Ah = A @ B.t()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    print("   cuBLAS f16: %.3f ms  %.1f TFLOP/s" % (ms, 2.0*M*N*K/ms/1e9), flush=True)
for shp in [(65792, 1152, 384), (65792, 384, 384), (65792, 1536, 384), (65792, 384, 1536), (8192, 8192, 8192)]:
    run("bench", lambda: bench(*shp))

def bench_cold(name, M, N, K, nbuf=6, **kw):
    """rotate over nbuf operand/output sets so every launch reads from HBM (as inside the step)"""
    As = [torch.randn(M, K, device=dev).to(h) for _ in range(nbuf)]
    Bm = torch.randn(N, K, device=dev).to(h)
    odt = kw.pop("odt", h)
    outs = [torch.empty(M, N, device=dev, dtype=odt) for _ in range(nbuf)]
    extra = {}
    if kw.get("gelu"):
        auxs = [torch.empty(M, N, device=dev, dtype=h) for _ in range(nbuf)]
    if kw.get("res"):
        ress = [torch.randn(M, N, device=dev) for _ in range(nbuf)]
    bias = torch.randn(N, device=dev)
    def call(i):
        j = i % nbuf
        if kw.get("gelu"):
            mv.gemm(As[j], Bm, outs[j], bias=bias, aux=auxs[j], epilogue=mv.EPI_GELU, q_res=(5, 10))
        elif kw.get("res"):
            mv.gemm(As[j], Bm, outs[j], bias=bias, residual=ress[j])
        else:
            mv.gemm(As[j], Bm, outs[j], bias=bias)
    for i in range(nbuf): call(i)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(3 * nbuf): call(i)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (3 * nbuf)
    print("cold %-28s M%d N%d K%d: %.3f ms  %.1f TFLOP/s" % (name, M, N, K, ms, 2.0*M*N*K/ms/1e9), flush=True)
run("c", lambda: bench_cold("qkv fwd (f16 out)", 65792, 1152, 384))
run("c", lambda: bench_cold("proj fwd (+res, f32 out)", 65792, 384, 384, res=True, odt=f32))
run("c", lambda: bench_cold("fc1 fwd (gelu)", 65792, 1536, 384, gelu=True))
run("c", lambda: bench_cold("fc2 fwd (+res, f32 out)", 65792, 384, 1536, res=True, odt=f32))
def wgrad_cold(T, No, Ki, nbuf=4):
    dYs = [torch.randn(T, No, device=dev).to(h) for _ in range(nbuf)]; Xs = [torch.randn(T, Ki, device=dev).to(h) for _ in range(nbuf)]
    out = torch.zeros(No, Ki, device=dev)
    for i in range(nbuf): mv.gemm(dYs[i], Xs[i], out, a_major=1, b_major=1, accumulate=True)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(3 * nbuf): mv.gemm(dYs[i % nbuf], Xs[i % nbuf], out, a_major=1, b_major=1, accumulate=True)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (3 * nbuf)
    print("cold wgrad T%d %dx%d: %.3f ms %.1f TFLOP/s" % (T, No, Ki, ms, 2.0*T*No*Ki/ms/1e9), flush=True)
run("w", lambda: wgrad_cold(65792, 1536, 384))
run("w", lambda: wgrad_cold(65792, 384, 1536))
run("w", lambda: wgrad_cold(65792, 1152, 384))
run("w", lambda: wgrad_cold(65792, 384, 384))
