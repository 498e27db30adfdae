"""Knowledge distillation without a GPU: the distiller_config schema, the wrapper's parameters and state_dict keys,
get_models, the optimizer's parameter groups and the C ABI of the two new entry points."""
import argparse
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCH = dict(image_size=80, patch_size=16, embed_dim=128, depth=2, heads=2, mlp_dim=256, dropout=0.0, emb_dropout=0.0,
            decoder="classification")


def _vit(q_format="FP32", **kw):
    from myrtle_vision.models.vit import ViT
    return ViT(decoder=kw.get("decoder", "classification"), image_size=80, patch_size=16, num_classes=5, dim=128,
               depth=2, heads=2, mlp_dim=256, q_format=q_format)


def _teacher_ckpt(tmp_path, q_format="FP32"):
    path = str(tmp_path / "teacher.pt")
    torch.save({"model": _vit(q_format).state_dict()}, path)
    return path


def _cfg(tmp_path, **over):
    cfg = {"teacher": {"kind": "vit", "vit_config": dict(ARCH, q_format="FP32"), "checkpoint": _teacher_ckpt(tmp_path)},
           "temperature": 3.0, "alpha": 0.5, "hard": False}
    cfg.update(over)
    return cfg


# ------------------------------------------------------------------------------------------------ config
@pytest.mark.parametrize("over,match", [
    ({"alpha": 1.5}, "alpha"),
    ({"alpha": -0.1}, "alpha"),
    ({"alpha": "0.5"}, "alpha"),
    ({"temperature": 0.0}, "temperature"),
    ({"temperature": -1}, "temperature"),
    ({"temperature": True}, "temperature"),
    ({"hard": 1}, "hard"),
    ({"bogus": 1}, "unknown keys"),
    ({"teacher": {"kind": "timm", "checkpoint": "x"}}, "kind"),
    ({"teacher": {"kind": "torchvision", "arch": "resnet50"}}, "missing keys"),
    ({"teacher": {"kind": "torchvision", "arch": "resnet50", "checkpoint": "x", "pretrained": True}}, "unknown keys"),
    ({"teacher": {"kind": "vit", "vit_config": dict(ARCH, q_format="FP32", extra=1), "checkpoint": "x"}},
     "unknown keys"),
    ({"teacher": {"kind": "vit", "vit_config": dict(ARCH, q_format="FP8"), "checkpoint": "x"}}, "q_format"),
    ({"teacher": {"kind": "vit", "vit_config": dict(ARCH, q_format="FP32", decoder="segmentation"),
                  "checkpoint": "x"}}, "classification"),
])
def test_config_validation(tmp_path, over, match):
    from myrtle_vision.models.distill import parse_distiller_config
    with pytest.raises(ValueError, match=match):
        parse_distiller_config(_cfg(tmp_path, **over), "classification")


@pytest.mark.parametrize("decoder", ["segmentation", "detection"])
def test_distillation_is_classification_only(tmp_path, decoder):
    from myrtle_vision.models.distill import DistillWrapper, parse_distiller_config
    with pytest.raises(ValueError, match="classification"):
        parse_distiller_config(_cfg(tmp_path), decoder)
    from myrtle_vision.models.vit import ViT
    student = ViT(decoder=decoder, image_size=176, patch_size=16, num_classes=3, dim=128, depth=1, heads=2,
                  mlp_dim=256)
    with pytest.raises(ValueError, match="classification"):
        DistillWrapper(student=student, teacher=_vit())


def test_config_defaults(tmp_path):
    from myrtle_vision.models.distill import parse_distiller_config
    cfg = _cfg(tmp_path)
    for k in ("temperature", "alpha", "hard"):
        del cfg[k]
    out = parse_distiller_config(cfg, "classification")
    assert (out["temperature"], out["alpha"], out["hard"]) == (1.0, 0.5, False)


# ------------------------------------------------------------------------------------------------ module
@pytest.mark.parametrize("fmt", ["FP32", "FP16_32", "TF32", "FP16_16"])
def test_wrapper_state_dict_keys(fmt):
    from myrtle_vision.models.distill import DistillWrapper
    student, teacher = _vit(fmt), _vit("FP32")
    w = DistillWrapper(student=student, teacher=teacher)
    mid = "" if fmt == "FP32" else ".1"
    assert list(w.distiller_state_dict()) == [
        "distillation_token"] + ["distill_mlp.%d%s.%s" % (i, mid, p) for i in (0, 1) for p in ("weight", "bias")]
    assert w.distillation_token.shape == (1, 1, 128)
    # the student's own keys are unchanged, the teacher is in neither state dict
    assert list(student.state_dict()) == list(_vit(fmt).state_dict())
    names = {n for n, _ in w.named_parameters()}
    assert not any(n.startswith("teacher") for n in w.state_dict())
    assert {id(p) for p in teacher.parameters()}.isdisjoint({id(p) for p in w.parameters()})
    assert {"student.cls_token", "distillation_token"} <= names


def test_train_mode_leaves_the_teacher_in_eval():
    from myrtle_vision.models.distill import DistillWrapper
    w = DistillWrapper(student=_vit(), teacher=_vit())
    w.train()
    assert w.student.training and not w.teacher.training
    assert not any(p.requires_grad for p in w.teacher.parameters())


def test_resume_state_round_trip():
    from myrtle_vision.models.distill import DistillWrapper
    a = DistillWrapper(student=_vit("FP16_32"), teacher=_vit())
    b = DistillWrapper(student=_vit("FP16_32"), teacher=_vit())
    b.load_distiller_state_dict(a.distiller_state_dict())
    assert torch.equal(a.distillation_token, b.distillation_token)
    with pytest.raises(RuntimeError, match="missing"):
        b.load_distiller_state_dict({"distillation_token": a.distillation_token})


def test_get_models_returns_the_wrapper(tmp_path):
    from myrtle_vision.models.distill import DistillWrapper
    from myrtle_vision.utils.models import get_models
    cfg = {"vit_config": dict(ARCH, q_format="FP16_32"), "data_config": {"number_of_classes": 5},
           "distiller_config": _cfg(tmp_path, hard=True)}
    vit, w = get_models(cfg)
    assert isinstance(w, DistillWrapper) and w.student is vit and w.hard and w.temperature == 3.0
    sd = torch.load(cfg["distiller_config"]["teacher"]["checkpoint"])["model"]
    assert all(torch.equal(v, sd[k]) for k, v in w.teacher.state_dict().items())


def test_get_models_builds_a_torchvision_teacher_from_its_checkpoint(tmp_path):
    import torchvision
    from myrtle_vision.utils.models import get_models
    path = str(tmp_path / "resnet.pt")
    ref = torchvision.models.resnet18(weights=None, num_classes=5)
    torch.save(ref.state_dict(), path)
    cfg = {"vit_config": dict(ARCH, q_format="FP32"), "data_config": {"number_of_classes": 5},
           "distiller_config": {"teacher": {"kind": "torchvision", "arch": "resnet18", "checkpoint": path}}}
    _, w = get_models(cfg)
    assert torch.equal(w.teacher.fc.weight, ref.fc.weight)
    cfg["distiller_config"]["teacher"]["arch"] = "no_such_net"
    with pytest.raises(ValueError, match="no model"):
        get_models(cfg)


def test_the_teacher_is_absent_from_the_optimizer(tmp_path):
    from myrtle_vision.models.distill import DistillWrapper
    from myrtle_vision.utils.optim import create_optimizer
    w = DistillWrapper(student=_vit("FP16_32"), teacher=_vit())
    args = argparse.Namespace(opt="adamw", weight_decay=0.05, lr=1e-3, opt_eps=1e-8, opt_betas=None, momentum=0.9)
    opt = create_optimizer(args, w, fused=False)
    seen = {id(p) for g in opt.param_groups for p in g["params"]}
    assert seen == {id(p) for p in w.parameters()}
    assert seen.isdisjoint({id(p) for p in w.teacher.parameters()})
    decay = {id(p) for g in opt.param_groups if g["weight_decay"] > 0 for p in g["params"]}
    # the distillation token follows cls_token's weight-decay rule
    assert (id(w.distillation_token) in decay) == (id(w.student.cls_token) in decay)


# ------------------------------------------------------------------------------------------------ C ABI
_CTYPE = {"int": ctypes.c_int, "float": ctypes.c_float}


def _prototype(name):
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    args = re.search(r"int %s\(([^)]*)\);" % name, text).group(1)
    out = []
    for a in (x.strip() for x in args.split(",")):
        out.append(ctypes.c_void_p if "*" in a else _CTYPE[a.rsplit(" ", 1)[0]])
    return out


@pytest.mark.parametrize("name", ["mv_token_row", "mv_distill_loss"])
def test_ctypes_signatures_mirror_the_header(name):
    import mv_native
    assert mv_native.SIGNATURES[name] == _prototype(name)


def test_library_exports_and_checks_the_new_entry_points():
    import __graft_entry__
    __graft_entry__.build()
    import mv_native
    lib = mv_native.lib()
    assert lib.mv_token_row.argtypes == mv_native.SIGNATURES["mv_token_row"]
    assert lib.mv_token_row(None, None, 1, 2, 4, 0, 0, 0, None) != 0
    assert b"mv_token_row" in lib.mv_last_error()
    p = ctypes.c_void_p(16)
    assert lib.mv_distill_loss(p, p, p, p, 4, 1, 1.0, 0.5, 0, p, p, p, p, None) != 0
    assert b"C >= 2" in lib.mv_last_error()
    assert lib.mv_distill_loss(p, p, p, p, 4, 3, 0.0, 0.5, 0, p, p, p, p, None) != 0
    assert b"T > 0" in lib.mv_last_error()
    assert lib.mv_patchify_q(None, None, 1, 1, 3, 32, 32, 16, 0, 0, 3, None) != 0
    assert b"cls_slot" in lib.mv_last_error()
