"""Cost of knowledge distillation (models/distill.py) on the graphed training step, and of its fused loss kernel.

ViT-Small 256 x 256, FP16_32, batch 256, one captured step (teacher forward, student forward, loss, backward) per
variant, the variants alternating round by round in one process:
  none     - no distillation: the student and F.cross_entropy
  student  - distillation token and head, the teacher replaced by constant logits: the student-side cost alone
  vit      - a ViT-Small FP16_32 teacher
  resnet50 - a torchvision resnet50 teacher
and the loss kernel (mv_distill_loss, forward and backward in one pass) against the ATen composite it replaces
(cross_entropy + log_softmax / softmax / kl_div, forward and backward).  Prints one JSON line, with the card name and
its power limit read in the same run.  Usage: python tools/bench_distill.py [--batch 256] [--steps 20] [--rounds 5]
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

import torch                                    # noqa: E402
import torch.nn.functional as F                 # noqa: E402
from torch import nn                            # noqa: E402


class ConstTeacher(nn.Module):
    def __init__(self, logits):
        super().__init__()
        self.register_buffer("logits", logits)

    def forward(self, img):
        return self.logits


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torchvision
    from myrtle_vision.models.distill import DistillLoss, DistillWrapper
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.graph import GraphedTrainStep
    import mv_native as mv

    dev, B, C = torch.device("cuda"), args.batch, 45
    torch.manual_seed(0)

    def vit():
        return ViT(decoder="classification", image_size=256, patch_size=16, num_classes=C, dim=384, depth=12, heads=6,
                   mlp_dim=1536, q_format="FP16_32")
    img = torch.randn(B, 3, 256, 256, device=dev).clamp(-1, 1)
    tgt = torch.randint(0, C, (B,), device=dev)
    crit = DistillLoss(temperature=3.0, alpha=0.5)
    teachers = {"student": ConstTeacher(torch.randn(B, C)), "vit": vit(),
                "resnet50": torchvision.models.resnet50(weights=None, num_classes=C)}
    steps = {}
    m = vit().to(dev).train()
    steps["none"] = GraphedTrainStep(m, F.cross_entropy, img, tgt)
    for name, t in teachers.items():
        w = DistillWrapper(student=vit(), teacher=t).to(dev).train()
        steps[name] = GraphedTrainStep(w, crit, img, tgt)
    times = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, step in steps.items():
            step()
            times[k].append(timed(step, args.steps))
    ms = {k: statistics.median(v) for k, v in times.items()}

    # the loss alone: the fused kernel (one pass writes the loss and both gradients) against the ATen composite
    s, d, t = (torch.randn(B, C, device=dev) for _ in range(3))
    sr, dr = s.clone().requires_grad_(), d.clone().requires_grad_()

    def fused():
        mv.distill_loss(s, d, t, tgt, 3.0, 0.5, False)

    def aten():
        loss = 0.5 * F.cross_entropy(sr, tgt) + 0.5 * 9.0 * F.kl_div(
            F.log_softmax(dr / 3.0, dim=-1), F.softmax(t / 3.0, dim=-1), reduction="batchmean")
        sr.grad = dr.grad = None
        loss.backward()
    for f in (fused, aten):
        timed(f, 20)
    loss_ms = {"fused": statistics.median(timed(fused, 200) for _ in range(5)),
               "aten": statistics.median(timed(aten, 200) for _ in range(5))}
    base = ms["none"]
    print(json.dumps({"card": card(), "batch": B, "step_ms": {k: round(v, 3) for k, v in ms.items()},
                      "over_none": {k: round(v / base - 1.0, 4) for k, v in ms.items()},
                      "loss_ms": {k: round(v, 4) for k, v in loss_ms.items()}}))


if __name__ == "__main__":
    main()
