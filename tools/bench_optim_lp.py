"""Cost of the low-precision optimizer step (qtorch.optim.OptimLP's fused path, mv_adamw_lp_step) against plain
FusedAdamW (mv_adamw_step) on ViT-Small's parameters (256 x 256, FP16_32: 21.76 M, the Linear weights updated by
32x32 tiles that also emit the next step's fp16 q(W) / q(W)^T).  Variants, alternating launch by launch in one
process so that all see the same clocks and neighbours:
  plain          FusedAdamW alone
  lp_stochastic  all five sites (grad, exp_avg, exp_avg_sq, acc, weight) at FloatingPoint(8, 7), stochastic
  lp_nearest     the same sites with nearest rounding: the same bytes without Philox
  lp_identity    OptimLP's kernel with no quantiser (28 B/param, as plain): the cost of its structure alone
Each launch is timed with CUDA events around the kernel alone (tables built once, launches back to back).  The working
set (~0.9 GB) is far above the 126 MB L2.  Byte floors: 28 B/param plain, 40 B/param with the accumulator read and
written and the gradient written back, plus 4 B per Linear-weight element for the two fp16 operands.  Prints one JSON
line; the card name and power limit are part of it.

    python tools/bench_optim_lp.py [--launches 300] [--out results/bench_optim_lp.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "myrtle-vision_b200")]

import torch                                   # noqa: E402

COPY_BW = 6.54e12                              # B/s, the copy bandwidth DESIGN.md section 5 measured on a B200


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optim_lp.py measures the B200 optimizer step: no CUDA device")
    import mv_native as mv
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from myrtle_vision.utils.optim import add_weight_decay
    from qtorch import FloatingPoint
    from qtorch.optim import OptimLP
    from qtorch.quant import quantizer
    dev = "cuda"
    launches = {}
    n_params = n_linear = 0
    for name in ("plain", "lp_stochastic", "lp_nearest", "lp_identity"):
        torch.manual_seed(0)
        m = ViT(decoder="classification", image_size=256, patch_size=16, num_classes=45, dim=384, depth=12, heads=6,
                mlp_dim=1536, q_format="FP16_32").to(dev).train()
        for p in m.parameters():
            p.grad = torch.randn_like(p) * 1e-3
        inner = FusedAdamW(add_weight_decay(m, 0.05), lr=1e-3, model=m)
        opt = inner
        if name == "lp_identity":
            opt = OptimLP(inner, seed=1)
        elif name != "plain":
            q = quantizer(FloatingPoint(8, 7), forward_rounding=name[3:])
            opt = OptimLP(inner, weight_quant=q, grad_quant=q, momentum_quant=q, acc_quant=q, seed=1)
            assert opt.fused
        opt.step()                                     # builds the tables and the device hyper-parameters
        rows = len(inner._updated)
        chunks = sum(((t.rows + 31) // 32) * ((t.cols + 31) // 32) if t.wq else (t.n + 1023) // 1024
                     for t, _ in inner._updated)
        base, hy = inner._table[1].data_ptr(), mv._ptr(inner._hyper)
        if name == "plain":
            n_params = sum(t.n for t, _ in inner._updated)
            n_linear = sum(t.n for t, _ in inner._updated if t.wq)
            launches[name] = (lambda b=base, r=rows, c=chunks, h=hy: mv.lib().mv_adamw_step(
                ctypes.c_void_p(b), r, c, h, mv._stream()), (m, opt))
        else:
            lp_base = base + inner._table[3]
            launches[name] = (lambda b=base, lb=lp_base, r=rows, c=chunks, h=hy, o=opt: mv.lib().mv_adamw_lp_step(
                ctypes.c_void_p(b), ctypes.c_void_p(lb), r, c, h, ctypes.byref(o.spec), mv._stream()), (m, opt))
    times = {k: [] for k in launches}
    for _ in range(10):                                # warm-up
        for fn, _ in launches.values():
            assert fn() == 0
    torch.cuda.synchronize()
    for _ in range(args.launches):
        for k, (fn, _) in launches.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            assert fn() == 0
            e1.record()
            times[k].append((e0, e1))
    torch.cuda.synchronize()
    ms = {k: statistics.median(a.elapsed_time(b) for a, b in v) for k, v in times.items()}
    floors = {"plain": (28 * n_params + 4 * n_linear) / COPY_BW * 1e3,
              "lp": (40 * n_params + 4 * n_linear) / COPY_BW * 1e3}
    res = {"bench": "optim_lp", "card": card(), "params": n_params, "linear_weight_elems": n_linear,
           "launches": args.launches, "median_ms": {k: round(v, 4) for k, v in ms.items()},
           "floor_ms_at_6.54TBps": {k: round(v, 4) for k, v in floors.items()},
           "lp_stochastic_over_floor": round(ms["lp_stochastic"] / floors["lp"], 3),
           "plain_over_floor": round(ms["plain"] / floors["plain"], 3)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
