"""Cost of Mixup / CutMix / label smoothing (utils/mixup.py) on the graphed training step, and of its two kernels.

ViT-Small 256 x 256, FP16_32, batch 256, one captured step (forward, loss, backward) per variant, the variants
alternating round by round in one process:
  plain     - F.cross_entropy, no mixing
  smoothing - label smoothing 0.1 alone (mv_mix_ce_loss without records)
  deit      - DeiT's defaults: mixup 0.8, cutmix 1.0, switch 0.5, smoothing 0.1 (draw, mixing gather, soft-target loss)
and per launch (CUDA events over 200 launches, median of 5):
  the plain patch gather (mv_patchify_q) against the mixing one (mv_patchify_mix_q) with every image Mixup-mixed, and
  with every image CutMix-mixed (records fixed: lam = 0.6 / a centred box of lam = 0.6);
  the loss kernel (forward and backward in one pass) against the ATen composite (-t * log_softmax(x)).sum(-1).mean()
  with its backward.
Prints one JSON line, with the card name and its power limit read in the same run.
Usage: python tools/bench_mixup.py [--batch 256] [--steps 20] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "myrtle-vision_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np                              # noqa: E402
import torch                                    # noqa: E402
import torch.nn.functional as F                 # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def fixed_recs(B, H, W, cutmix, dev):
    rec = np.zeros((B, 8), dtype=np.int32)
    f = rec[:, :3].view(np.float32)
    if cutmix:
        h, w = int(H * 0.4 ** 0.5), int(W * 0.4 ** 0.5)
        y0, x0 = (H - h) // 2, (W - w) // 2
        rec[:, 3:] = (1, y0, y0 + h, x0, x0 + w)
        f[:, 0], f[:, 1] = 1.0 - h * w / (H * W), 1.0
    else:
        f[:] = (0.6, 0.6, np.float32(1.0 - 0.6))
    return torch.from_numpy(rec).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.graph import GraphedTrainStep
    from myrtle_vision.utils.mixup import Mixup, MixupLoss, MixupWrapper
    import mv_native as mv

    dev, B, C = torch.device("cuda"), args.batch, 45
    torch.manual_seed(0)

    def vit():
        return ViT(decoder="classification", image_size=256, patch_size=16, num_classes=C, dim=384, depth=12, heads=6,
                   mlp_dim=1536, q_format="FP16_32").to(dev).train()
    img = torch.randn(B, 3, 256, 256, device=dev).clamp(-1, 1)
    tgt = torch.randint(0, C, (B,), device=dev)
    steps = {
        "plain": GraphedTrainStep(vit(), F.cross_entropy, img, tgt),
        "smoothing": GraphedTrainStep(vit(), MixupLoss(0.1), img, tgt),
        "deit": GraphedTrainStep(MixupWrapper(vit(), Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, switch_prob=0.5,
                                                           label_smoothing=0.1)), MixupLoss(0.1), img, tgt),
    }
    times = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, step in steps.items():
            step()
            times[k].append(timed(step, args.steps))
    ms = {k: statistics.median(v) for k, v in times.items()}

    # per launch: the patch gathers (fp16 container, the FP16_32 step's) ...
    fmt = (5, 10)
    recs = {"mixup": fixed_recs(B, 256, 256, False, dev), "cutmix": fixed_recs(B, 256, 256, True, dev)}
    calls = {"patchify": lambda: mv.patchify_q(img, 16, q_in=fmt, cls_slot=1),
             "patchify_mix_mixup": lambda: mv.patchify_mix_q(img, recs["mixup"], 16, q_in=fmt, cls_slot=1),
             "patchify_mix_cutmix": lambda: mv.patchify_mix_q(img, recs["cutmix"], 16, q_in=fmt, cls_slot=1)}
    # ... and the loss: the fused kernel against the ATen composite with its backward
    x = torch.randn(B, C, device=dev)
    xr = x.clone().requires_grad_()
    draw = Mixup(mixup_alpha=0.8, cutmix_alpha=1.0).draw(B, 256, 256, seed=1)
    lam = mv.mix_records(draw)["lam"]

    def aten():
        s = torch.full((B, C), 0.1 / C, device=dev).scatter_(1, tgt[:, None], 1.0 - 0.1 + 0.1 / C)
        t = lam[:, None] * s + (1.0 - lam[:, None]) * s.flip(0)
        xr.grad = None
        (-t * F.log_softmax(xr, dim=-1)).sum(-1).mean().backward()
    calls["loss_fused"] = lambda: mv.mix_ce_loss(x, tgt, draw, 0.1)
    calls["loss_aten"] = aten
    for f in calls.values():
        timed(f, 20)
    launch_ms = {k: statistics.median(timed(f, 200) for _ in range(5)) for k, f in calls.items()}
    base = ms["plain"]
    print(json.dumps({"card": card(), "batch": B, "step_ms": {k: round(v, 3) for k, v in ms.items()},
                      "over_plain": {k: round(v / base - 1.0, 4) for k, v in ms.items()},
                      "launch_ms": {k: round(v, 4) for k, v in launch_ms.items()}}))


if __name__ == "__main__":
    main()
