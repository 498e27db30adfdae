"""Knowledge distillation with a distillation token (DeiT; the reference's models/distill.py, a restatement of
lucidrains' vit-pytorch `DistillWrapper`, whose forward is broken upstream: SURVEY.md section 2 row 11).

`DistillWrapper(student=vit, teacher=t, temperature=T, alpha=a, hard=False)` owns a `distillation_token` [1, 1, dim]
and a `distill_mlp = Sequential(LayerNorm(dim), Linear(dim, num_classes))`.  Its forward runs the frozen teacher under
no_grad, the student with the token appended as the last row of its sequence (`ViT.forward(img, distill_token=...)`),
and the head on that row's encoder output; it returns `(student_logits, distill_logits, teacher_logits)`, which
`DistillLoss` turns into

    (1 - a) CE(student_logits, labels) + a D,   D = T^2 KL(log_softmax(distill / T) || softmax(teacher / T)) (batchmean)
                                                  or, hard, CE(distill_logits, argmax(teacher_logits))

in one kernel (mv_distill_loss).  Evaluation and inference use the student alone (`vit(img)`), as upstream.  The
teacher is kept out of the module tree: it is not in `parameters()` (so no optimizer sees it) nor in `state_dict()`,
but `.to()` / `.cuda()` move it and `.train()` leaves it in eval mode.  DESIGN.md section 7 has the details.
"""
import numbers

import torch
from torch import nn

import mv_native as mv
from myrtle_vision.models.vit import ViT
from myrtle_vision.utils.quantize import QFormat, QuantStubSlot

# gradient-quantiser sites of the head continue the decoder's (ViT._gfmt): 10 depth + 1 + j
DISTILL_NORM_SITE, DISTILL_LINEAR_SITE = 3, 4        # LayerNorm input; Linear input (its weight: 5)


def _check_hyper(temperature, alpha, hard):
    if not isinstance(temperature, numbers.Real) or isinstance(temperature, bool) or not temperature > 0:
        raise ValueError("distillation temperature must be a number > 0, got %r" % (temperature,))
    if not isinstance(alpha, numbers.Real) or isinstance(alpha, bool) or not 0.0 <= alpha <= 1.0:
        raise ValueError("distillation alpha must be a number in [0, 1], got %r" % (alpha,))
    if not isinstance(hard, bool):
        raise ValueError("distillation hard must be true or false, got %r" % (hard,))


class _DistillLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, student, distill, teacher, labels, temperature, alpha, hard):
        loss, ds, dd = mv.distill_loss(student, distill, teacher, labels, temperature, alpha, hard)
        ctx.save_for_backward(ds, dd)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad):
        ds, dd = ctx.saved_tensors
        return ds * grad, dd * grad, None, None, None, None, None


def distill_loss(student_logits, distill_logits, teacher_logits, labels, temperature=1.0, alpha=0.5, hard=False):
    """The fused distillation loss (mv_distill_loss); gradients flow to the student and distillation logits."""
    _check_hyper(temperature, alpha, hard)
    return _DistillLoss.apply(student_logits, distill_logits, teacher_logits.detach(), labels, float(temperature),
                              float(alpha), hard)


class DistillLoss:
    """criterion(outputs, labels) for the outputs of DistillWrapper.forward (utils.graph.GraphedTrainStep's loss_fn)."""

    def __init__(self, temperature=1.0, alpha=0.5, hard=False):
        _check_hyper(temperature, alpha, hard)
        self.temperature, self.alpha, self.hard = float(temperature), float(alpha), hard

    def __call__(self, outputs, labels):
        student, distill, teacher = outputs
        return distill_loss(student, distill, teacher, labels, self.temperature, self.alpha, self.hard)


class DistillWrapper(nn.Module):
    def __init__(self, *, student, teacher, temperature=1.0, alpha=0.5, hard=False):
        super().__init__()
        _check_hyper(temperature, alpha, hard)
        if not isinstance(student, ViT) or student.task != "classification":
            raise ValueError("distillation needs a classification ViT student")
        self.student = student
        self.__dict__["teacher"] = teacher.eval().requires_grad_(False)      # not a submodule: see the module doc
        self.temperature, self.alpha, self.hard = float(temperature), float(alpha), hard
        dim = student.dim
        num_classes = _unwrap_linear(student.decoder.linear).out_features
        self.distillation_token = nn.Parameter(torch.randn(1, 1, dim))
        self.distill_mlp = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, num_classes))
        if student.quantizer.q_format != QFormat.FP32:
            # the student's quantised layout: Sequential(QuantStubSlot, module), keys distill_mlp.<i>.1.<param>
            fmt = student.quantizer.plan.inp
            for i in range(2):
                self.distill_mlp[i] = nn.Sequential(QuantStubSlot(fmt), self.distill_mlp[i])

    # the student's fused engine stands for the wrapper (utils.graph.GraphedTrainStep, utils.parallel.DataParallel,
    # utils.fused_adamw.FusedAdamW)
    def engine(self):
        return self.student.engine()

    @property
    def _engine(self):
        return self.student._engine

    def _apply(self, fn, *args, **kwargs):
        self.teacher._apply(fn, *args, **kwargs)
        return super()._apply(fn, *args, **kwargs)

    def train(self, mode=True):
        super().train(mode)
        self.teacher.eval()
        return self

    def teacher_logits(self, img):
        with torch.no_grad():
            if isinstance(self.teacher, ViT):
                self.teacher.engine().frozen_weights = True
            return self.teacher(img).float()

    def forward(self, img):
        teacher = self.teacher_logits(img)
        s = self.student
        student, dist_row = s(img, distill_token=self.distillation_token)
        distill = s._linear(self.distill_mlp[1], s._norm(self.distill_mlp[0], dist_row, DISTILL_NORM_SITE),
                            DISTILL_LINEAR_SITE)
        return student, distill, teacher

    def distiller_state_dict(self):
        """The wrapper's own parameters (distillation_token, distill_mlp.*): the checkpoint's "distiller" entry."""
        return {k: v for k, v in self.state_dict().items() if not k.startswith("student.")}

    def load_distiller_state_dict(self, state):
        missing, unexpected = self.load_state_dict(state, strict=False)
        missing = [k for k in missing if not k.startswith("student.")]
        if missing or unexpected:
            raise RuntimeError("distiller state: missing %s, unexpected %s" % (missing, unexpected))


def _unwrap_linear(m):
    return m[1] if isinstance(m, nn.Sequential) else m


# ------------------------------------------------------------------------------------------- config
DISTILLER_KEYS = ("teacher", "temperature", "alpha", "hard")
TEACHER_KEYS = {"vit": ("kind", "vit_config", "checkpoint"), "torchvision": ("kind", "arch", "checkpoint")}
TEACHER_VIT_KEYS = ("image_size", "patch_size", "embed_dim", "depth", "heads", "mlp_dim", "dropout", "emb_dropout",
                    "q_format", "decoder")


def parse_distiller_config(cfg, student_decoder):
    """Validate config["distiller_config"] (unknown keys are errors) ->
    {"teacher": {...}, "temperature": T, "alpha": a, "hard": bool}:

        {"teacher": {"kind": "vit", "vit_config": {...}, "checkpoint": path}
                  | {"kind": "torchvision", "arch": "resnet50", "checkpoint": path},
         "temperature": 1.0, "alpha": 0.5, "hard": false}

    temperature, alpha and hard default to 1.0, 0.5 and false.  Teacher weights come only from `checkpoint`."""
    if student_decoder != "classification":
        raise ValueError("distiller_config: distillation is a classification method, the decoder is %r"
                         % (student_decoder,))
    if not isinstance(cfg, dict):
        raise ValueError("distiller_config: expected an object, got %r" % (cfg,))
    unknown = set(cfg) - set(DISTILLER_KEYS)
    if unknown:
        raise ValueError("distiller_config: unknown keys %s (known: %s)" % (sorted(unknown), ", ".join(DISTILLER_KEYS)))
    out = {"temperature": cfg.get("temperature", 1.0), "alpha": cfg.get("alpha", 0.5), "hard": cfg.get("hard", False)}
    _check_hyper(out["temperature"], out["alpha"], out["hard"])
    t = cfg.get("teacher")
    if not isinstance(t, dict) or t.get("kind") not in TEACHER_KEYS:
        raise ValueError("distiller_config.teacher: expected an object with \"kind\": \"vit\" or \"torchvision\", got %r"
                         % (t,))
    keys = TEACHER_KEYS[t["kind"]]
    unknown, missing = set(t) - set(keys), set(keys) - set(t)
    if unknown or missing:
        raise ValueError("distiller_config.teacher (%s): unknown keys %s, missing keys %s"
                         % (t["kind"], sorted(unknown), sorted(missing)))
    if not isinstance(t["checkpoint"], str) or not t["checkpoint"]:
        raise ValueError("distiller_config.teacher.checkpoint: expected a file path, got %r" % (t["checkpoint"],))
    if t["kind"] == "vit":
        vc = t["vit_config"]
        if not isinstance(vc, dict):
            raise ValueError("distiller_config.teacher.vit_config: expected an object, got %r" % (vc,))
        unknown = set(vc) - set(TEACHER_VIT_KEYS)
        missing = {"image_size", "patch_size", "embed_dim", "depth", "heads", "mlp_dim", "q_format"} - set(vc)
        if unknown or missing:
            raise ValueError("distiller_config.teacher.vit_config: unknown keys %s, missing keys %s"
                             % (sorted(unknown), sorted(missing)))
        if vc.get("decoder", "classification") != "classification":
            raise ValueError("distiller_config.teacher.vit_config: the teacher must be a classification ViT")
        if vc["q_format"] not in QFormat.__members__:
            raise ValueError("distiller_config.teacher.vit_config.q_format: unknown format %r" % (vc["q_format"],))
    elif not isinstance(t["arch"], str):
        raise ValueError("distiller_config.teacher.arch: expected a torchvision model name, got %r" % (t["arch"],))
    out["teacher"] = dict(t)
    return out


def _load_state(path):
    state = torch.load(path, map_location="cpu", weights_only=True)
    if isinstance(state, dict):
        for key in ("model", "state_dict"):
            if key in state and isinstance(state[key], dict):
                return state[key]
    return state


def build_teacher(spec, num_classes):
    """The teacher of a parsed distiller_config["teacher"], its weights loaded from spec["checkpoint"] (a state dict,
    or a checkpoint holding one under "model" or "state_dict"; this project's checkpoints qualify)."""
    if spec["kind"] == "vit":
        vc = spec["vit_config"]
        teacher = ViT(decoder="classification", image_size=vc["image_size"], patch_size=vc["patch_size"],
                      num_classes=num_classes, dim=vc["embed_dim"], depth=vc["depth"], heads=vc["heads"],
                      mlp_dim=vc["mlp_dim"], dropout=vc.get("dropout", 0.0), emb_dropout=vc.get("emb_dropout", 0.0),
                      q_format=QFormat[vc["q_format"]])
    else:
        import torchvision
        ctor = getattr(torchvision.models, spec["arch"], None)
        if ctor is None or not callable(ctor):
            raise ValueError("distiller_config.teacher.arch: torchvision has no model %r" % (spec["arch"],))
        teacher = ctor(weights=None, num_classes=num_classes)
    teacher.load_state_dict(_load_state(spec["checkpoint"]))
    return teacher
