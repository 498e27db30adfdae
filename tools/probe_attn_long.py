"""Long-sequence attention timing (detection config: B=8, H=6, N=2501): forward, backward with fused dQ
red.add."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200")); sys.path.insert(0, ROOT)
import torch
import mv_native as mv
B, H, N = (int(a) for a in sys.argv[1:4]) if len(sys.argv) > 3 else (8, 6, 2501)
D = H * 64
torch.manual_seed(0)
qkv = torch.randn(B * N, 3 * D, device="cuda").half()
do = torch.randn(B * N, D, device="cuda").half()
out, lse = mv.attention_fwd(qkv, B, H, N, q_out=(5, 10))
def timeit(fn, n=10):
    for _ in range(3): fn()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
fl = 4.0 * B * H * N * N * 64
ms = timeit(lambda: mv.attention_fwd(qkv, B, H, N, q_out=(5, 10)))
print("fwd %.3f ms  %.0f TFLOP/s" % (ms, fl / ms / 1e9))
ms = timeit(lambda: mv.attention_bwd(qkv, out, do, lse, B, H, N))
print("bwd %.3f ms  %.0f TFLOP/s (2.5x fwd flops)" % (ms, 2.5 * fl / ms / 1e9))
