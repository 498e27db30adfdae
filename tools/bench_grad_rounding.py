"""Cost of stochastic gradient rounding on the fused training step: ViT-Small, 256 x 256, FP16_32, batch 256, gradient
format E5M2, the step captured as a CUDA graph (GraphedTrainStep: zero_grad -> forward -> loss x 65536 -> backward), with
backward_rounding "nearest" and "stochastic" on the same weights, alternating in one process so both see the same clocks
and neighbours.  Also the per-launch times of an eager step (mv_native.enable_timing) for the kernels the rounding
changes: the four dgrad GEMMs (fc2 input with gelu', fc1 input, to_out input, to_qkv input) and the LayerNorm backward.
Prints one JSON line; the card name and power limit are part of it.

    python tools/bench_grad_rounding.py [--batch 256] [--rounds 5] [--steps 20] [--out results/bench_grad_rounding.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "myrtle-vision_b200")]

import torch                                   # noqa: E402
import torch.nn.functional as F                # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--format", default="5,2", help="gradient format exp,man")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_grad_rounding.py measures the B200 step: no CUDA device")
    import mv_native
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.graph import GraphedTrainStep
    dev = "cuda"
    torch.manual_seed(0)
    img = torch.randn(args.batch, 3, 256, 256, device=dev).clamp(-1, 1)
    tgt = torch.randint(0, 45, (args.batch,), device=dev)
    gfmt = tuple(int(v) for v in args.format.split(","))
    loss_fn = lambda out, t: F.cross_entropy(out, t) * 65536.0     # the reference's GradScaler(65536); noqa: E731
    models, steps = {}, {}
    state = None
    for p in ("nearest", "stochastic"):
        m = ViT(decoder="classification", image_size=256, patch_size=16, num_classes=45, dim=384, depth=12, heads=6,
                mlp_dim=1536, q_format="FP16_32", backward_format=gfmt, backward_rounding=p)
        if state is None:
            state = m.state_dict()
        m.load_state_dict(state)
        models[p] = m.to(dev).train()
    # per-kernel times of an eager step (timing events around every library call; separate from the graphed timing)
    kernels = {}
    for p, m in models.items():
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            loss_fn(m(img), tgt).backward()
        torch.cuda.synchronize()
        mv_native.enable_timing(True)
        for _ in range(3):
            m.zero_grad(set_to_none=True)
            loss_fn(m(img), tgt).backward()
        torch.cuda.synchronize()
        summ = mv_native.timing_summary()
        mv_native.enable_timing(False)
        M = args.batch * 257
        names = {"dgrad_fc2_in_gelu": "gemm_dgrad_%dx1536x384" % M, "dgrad_fc1_in": "gemm_dgrad_%dx384x1536" % M,
                 "dgrad_out_in": "gemm_dgrad_%dx384x384" % M, "dgrad_qkv_in": "gemm_dgrad_%dx384x1152" % M,
                 "ln_bwd": "ln_bwd"}
        kernels[str(p)] = {k: (round(summ[v][1] / summ[v][0] * 1e3, 2) if v in summ else None)
                           for k, v in names.items()}          # us per launch
        kernels[str(p)]["launches_per_step"] = {k: summ[v][0] // 3 for k, v in names.items() if v in summ}
    for p, m in models.items():
        steps[p] = GraphedTrainStep(m, loss_fn, img, tgt)
        for _ in range(10):
            steps[p](img, tgt)
    times = {p: [] for p in models}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for p in models:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                steps[p](img, tgt)
            e1.record()
            torch.cuda.synchronize()
            times[p].append(e0.elapsed_time(e1) / args.steps)
    res = {"workload": "ViT-Small 256x256 FP16_32 batch %d, gradient format %r, graphed fwd+loss+bwd" % (args.batch, gfmt),
           "card": card()}
    for p in models:
        ms = statistics.median(times[p])
        res[p] = {"ms_per_step": round(ms, 3), "img_per_s": round(args.batch / ms * 1e3, 1),
                           "ms_rounds": [round(t, 3) for t in times[p]], "kernel_us": kernels[str(p)]}
    res["stochastic_overhead_pct"] = round(
        100.0 * (statistics.median(times["stochastic"]) / statistics.median(times["nearest"]) - 1), 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
