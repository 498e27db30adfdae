"""Mixup, CutMix and label smoothing (DeiT's regularisers; timm 0.5.4's `Mixup`, `mixup_target` and
`SoftTargetCrossEntropy`), with the batch mixed inside the patch gather and the soft targets in one loss kernel.

`Mixup(mixup_alpha, cutmix_alpha, prob, switch_prob, mode, label_smoothing, num_classes)` takes timm's arguments.
`Mixup.draw(B, H, W)` draws the per-image records on the device (mv_mix_draw): each says how image b is mixed with
image B - 1 - b and the weight lam of its own label.  `ViT.forward(img, mix=recs)` runs the encoder on the mixed batch
without materialising it (mv_patchify_mix_q), and `mix_cross_entropy(logits, labels, recs, smoothing)` is the
soft-target loss

    t_b = lam_b s(y_b) + (1 - lam_b) s(y_{B-1-b}),   s(y) = smoothing / C + (1 - smoothing) e_y,
    loss = mean_b sum_c -t_bc log_softmax(x_b)_c

in one kernel (mv_mix_ce_loss; recs=None: F.cross_entropy(x, y, label_smoothing=smoothing)).  `MixupWrapper(vit,
mixup)` draws the records per training forward and returns `(logits, recs)` for `MixupLoss`.  The randomness is the
"mix stream" of include/mv_b200.h, keyed by a seed drawn on the device from torch's CUDA generator: a replayed CUDA graph
mixes differently every step and torch.manual_seed repeats a run.  DESIGN.md section 7 lists where this differs from
timm.
"""
import numbers

import torch
from torch import nn

import mv_native as mv

MODES = tuple(mv.MIX_MODES)


def _real(v):
    return isinstance(v, numbers.Real) and not isinstance(v, bool)


def check_mix_args(mixup_alpha, cutmix_alpha, prob, switch_prob, mode, label_smoothing):
    """ValueError unless the arguments describe a valid Mixup (at least one alpha > 0)."""
    for name, v in (("mixup_alpha", mixup_alpha), ("cutmix_alpha", cutmix_alpha)):
        if not _real(v) or not v >= 0:
            raise ValueError("%s must be a number >= 0, got %r" % (name, v))
    if not (mixup_alpha > 0 or cutmix_alpha > 0):
        raise ValueError("Mixup needs mixup_alpha > 0 or cutmix_alpha > 0")
    for name, v in (("prob", prob), ("switch_prob", switch_prob), ("label_smoothing", label_smoothing)):
        if not _real(v) or not 0.0 <= v <= 1.0:
            raise ValueError("%s must be a number in [0, 1], got %r" % (name, v))
    if mode not in mv.MIX_MODES:
        raise ValueError("mode must be one of %s, got %r" % (", ".join(MODES), mode))


class Mixup:
    def __init__(self, mixup_alpha=1.0, cutmix_alpha=0.0, prob=1.0, switch_prob=0.5, mode="batch",
                 label_smoothing=0.1, num_classes=1000):
        check_mix_args(mixup_alpha, cutmix_alpha, prob, switch_prob, mode, label_smoothing)
        self.mixup_alpha, self.cutmix_alpha = float(mixup_alpha), float(cutmix_alpha)
        self.mix_prob, self.switch_prob, self.mode = float(prob), float(switch_prob), mode
        self.label_smoothing, self.num_classes = float(label_smoothing), num_classes
        self.spec = mv.MixSpec(self.mixup_alpha, self.cutmix_alpha, self.mix_prob, self.switch_prob,
                               mv.MIX_MODES[mode])

    def draw(self, B, H, W, seed=None, rank=0, device=None):
        """The records of one batch of B images of H x W (int32 [B, 8] on the device; mv_native.mix_records reads
        them).  seed: None draws a 64-bit seed on the device from torch's CUDA generator; an int or a 1-element int64
        CUDA tensor fixes it.  rank: the data-parallel rank (ranks sharing a seed mix independently)."""
        if B % 2:
            raise ValueError("Mixup needs an even batch (image b is mixed with image B - 1 - b), got %d" % B)
        device = torch.device("cuda") if device is None else torch.device(device)
        if seed is None:
            seed = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=device)
        elif not isinstance(seed, torch.Tensor):
            seed = torch.tensor([int(seed)], dtype=torch.int64, device=device)
        return mv.mix_draw(seed, B, H, W, self.spec, rank=rank)


class _MixCrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, recs, smoothing):
        loss, dx = mv.mix_ce_loss(logits, labels, recs, smoothing)
        ctx.save_for_backward(dx)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad):
        (dx,) = ctx.saved_tensors
        return dx * grad, None, None, None


def mix_cross_entropy(logits, labels, recs=None, smoothing=0.0):
    """The soft-target cross-entropy of a mixed batch (mv_mix_ce_loss); recs=None: label smoothing alone."""
    if not _real(smoothing) or not 0.0 <= smoothing <= 1.0:
        raise ValueError("smoothing must be a number in [0, 1], got %r" % (smoothing,))
    return _MixCrossEntropy.apply(logits, labels, recs, float(smoothing))


class MixupLoss:
    """criterion(outputs, labels): outputs = (logits, recs) from MixupWrapper, or bare logits (unmixed)."""

    def __init__(self, smoothing=0.0):
        if not _real(smoothing) or not 0.0 <= smoothing <= 1.0:
            raise ValueError("smoothing must be a number in [0, 1], got %r" % (smoothing,))
        self.smoothing = float(smoothing)

    def __call__(self, outputs, labels):
        logits, recs = outputs if isinstance(outputs, tuple) else (outputs, None)
        return mix_cross_entropy(logits, labels, recs, self.smoothing)


class MixupWrapper(nn.Module):
    """Training: draws a seed and the records on the device, runs `vit(img, mix=recs)`, keeps the records in
    `last_mix` and returns `(logits, recs)`.  Eval: `(vit(img), None)`, drawing nothing.  No parameters of its own."""

    def __init__(self, vit, mixup):
        super().__init__()
        if getattr(vit, "task", None) != "classification":
            raise ValueError("Mixup / CutMix needs a classification ViT")
        self.vit, self.mixup = vit, mixup
        self.last_mix = None

    # the ViT's fused engine stands for the wrapper (utils.graph.GraphedTrainStep, utils.parallel.DataParallel)
    def engine(self):
        return self.vit.engine()

    @property
    def _engine(self):
        return self.vit._engine

    def forward(self, img):
        if not self.training:
            return self.vit(img), None
        b, _, h, w = img.shape
        recs = self.mixup.draw(b, h, w, rank=self.engine().rank, device=img.device)
        self.last_mix = recs
        return self.vit(img, mix=recs), recs


# ------------------------------------------------------------------------------------------- config
MIX_KEYS = {"mixup": 0.0, "cutmix": 0.0, "cutmix_minmax": None, "mixup_prob": 1.0, "mixup_switch_prob": 0.5,
            "mixup_mode": "batch", "smoothing": 0.0}


def parse_mix_config(train_config, decoder, local_batch_size, distiller=False):
    """DeiT's argument names in train_config -> {key: value} with MIX_KEYS' defaults.  Mixing is on when mixup > 0 or
    cutmix > 0.  ValueError for values out of range, an unknown mode, an odd local batch with mixing, a non-
    classification decoder with mixing or smoothing, or mixing with distillation; NotImplementedError for
    cutmix_minmax."""
    cfg = {k: train_config.get(k, d) for k, d in MIX_KEYS.items()}
    if cfg["cutmix_minmax"] is not None:
        raise NotImplementedError("cutmix_minmax is not supported (only the Beta-distributed CutMix box)")
    for k in ("mixup", "cutmix"):
        if not _real(cfg[k]) or not cfg[k] >= 0:
            raise ValueError("train_config.%s must be a number >= 0, got %r" % (k, cfg[k]))
    for k in ("mixup_prob", "mixup_switch_prob", "smoothing"):
        if not _real(cfg[k]) or not 0.0 <= cfg[k] <= 1.0:
            raise ValueError("train_config.%s must be a number in [0, 1], got %r" % (k, cfg[k]))
    if cfg["mixup_mode"] not in mv.MIX_MODES:
        raise ValueError("train_config.mixup_mode must be one of %s, got %r" % (", ".join(MODES), cfg["mixup_mode"]))
    mixing = cfg["mixup"] > 0 or cfg["cutmix"] > 0
    if (mixing or cfg["smoothing"] > 0) and decoder != "classification":
        raise ValueError("Mixup, CutMix and label smoothing are classification methods, the decoder is %r" % (decoder,))
    if mixing and distiller:
        raise ValueError("Mixup / CutMix together with distiller_config is not supported")
    if mixing and local_batch_size % 2:
        raise ValueError("Mixup / CutMix needs an even local batch (image b is mixed with image B - 1 - b), got %d"
                         % local_batch_size)
    cfg["active"] = mixing
    return cfg


def build_mixup(cfg, num_classes):
    """The Mixup of a parse_mix_config result with mixing active."""
    return Mixup(mixup_alpha=cfg["mixup"], cutmix_alpha=cfg["cutmix"], prob=cfg["mixup_prob"],
                 switch_prob=cfg["mixup_switch_prob"], mode=cfg["mixup_mode"], label_smoothing=cfg["smoothing"],
                 num_classes=num_classes)
