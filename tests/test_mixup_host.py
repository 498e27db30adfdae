"""Mixup / CutMix / label smoothing without a GPU: the ctypes mirrors of the new structs and entry points against the
header, the entry points' argument checks, the Mixup arguments and the train_config keys."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    return re.sub(r"/\*.*?\*/", "", text, flags=re.S)


def declared_fields(struct):
    body = re.search(r"typedef struct \{([^}]*)\} %s;" % struct, _header()).group(1)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        first, *rest = decl.split(",")
        names += [re.findall(r"\w+", first)[-1]] + [r.strip() for r in rest]
    return names


def _prototype(name):
    import mv_native
    ctype = {"int": ctypes.c_int, "float": ctypes.c_float, "mv_mix_spec": mv_native.MixSpec}
    args = re.search(r"int %s\(([^)]*)\);" % name, _header()).group(1)
    return [ctypes.c_void_p if "*" in a else ctype[a.rsplit(" ", 1)[0]] for a in (x.strip() for x in args.split(","))]


# ------------------------------------------------------------------------------------------------ C ABI
@pytest.mark.parametrize("struct,cls", [("mv_mix_spec", "MixSpec"), ("mv_mix_rec", "MixRec")])
def test_ctypes_structs_mirror_the_header(struct, cls):
    import mv_native
    assert [f[0] for f in getattr(mv_native, cls)._fields_] == declared_fields(struct)


def test_record_layout_is_eight_words():
    import mv_native
    assert ctypes.sizeof(mv_native.MixRec) == 32 and ctypes.sizeof(mv_native.MixSpec) == 20
    assert [t for _, t in mv_native.MixRec._fields_[:3]] == [ctypes.c_float] * 3


@pytest.mark.parametrize("name", ["mv_mix_draw", "mv_patchify_mix_q", "mv_mix_ce_loss"])
def test_ctypes_signatures_mirror_the_header(name):
    import mv_native
    assert mv_native.SIGNATURES[name] == _prototype(name)


def test_modes_mirror_the_header():
    import mv_native
    defs = dict(re.findall(r"#define MV_MIX_(BATCH|PAIR|ELEM) (\d+)", _header()))
    assert {k.lower(): int(v) for k, v in defs.items()} == mv_native.MIX_MODES


def test_version_is_unchanged():
    api = open(os.path.join(ROOT, "myrtle-vision_b200", "csrc", "api.cu")).read()
    assert "return 105;" in api


def test_entry_points_reject_bad_arguments_without_a_device():
    import __graft_entry__
    __graft_entry__.build()
    import mv_native
    lib = mv_native.lib()
    assert lib.mv_version() == 105
    p = ctypes.c_void_p(16)
    good = mv_native.MixSpec(0.8, 1.0, 1.0, 0.5, 0)

    def err(rc, text):
        assert rc != 0
        assert text in lib.mv_last_error(), lib.mv_last_error()

    err(lib.mv_mix_draw(None, 0, 8, 32, 32, good, p, None), b"null pointer")
    err(lib.mv_mix_draw(p, 0, 7, 32, 32, good, p, None), b"even")
    err(lib.mv_mix_draw(p, 0, 8, 32, 32, mv_native.MixSpec(0.8, 1.0, 1.0, 0.5, 3), p, None), b"mode")
    err(lib.mv_mix_draw(p, 0, 8, 32, 32, mv_native.MixSpec(0.0, 0.0, 1.0, 0.5, 0), p, None), b"alphas")
    err(lib.mv_mix_draw(p, 0, 8, 32, 32, mv_native.MixSpec(-1.0, 1.0, 1.0, 0.5, 0), p, None), b"alphas")
    err(lib.mv_mix_draw(p, 0, 8, 32, 32, mv_native.MixSpec(0.8, 1.0, 1.5, 0.5, 0), p, None), b"prob")
    err(lib.mv_mix_draw(p, -1, 8, 32, 32, good, p, None), b"rank")
    err(lib.mv_patchify_mix_q(p, None, p, 1, 8, 3, 32, 32, 16, 0, 0, 1, None), b"null records")
    err(lib.mv_patchify_mix_q(p, p, p, 1, 7, 3, 32, 32, 16, 0, 0, 1, None), b"even")
    err(lib.mv_patchify_mix_q(p, p, p, 1, 8, 3, 32, 32, 16, 0, 0, 3, None), b"cls_slot")
    err(lib.mv_patchify_mix_q(p, p, p, 1, 8, 3, 30, 32, 16, 0, 0, 1, None), b"divisible")
    err(lib.mv_mix_ce_loss(p, p, None, 4, 1, 0.1, p, p, p, None), b"C >= 2")
    err(lib.mv_mix_ce_loss(p, p, p, 5, 3, 0.1, p, p, p, None), b"even")
    err(lib.mv_mix_ce_loss(p, p, None, 4, 3, 1.5, p, p, p, None), b"smoothing")
    err(lib.mv_mix_ce_loss(None, p, None, 4, 3, 0.1, p, p, p, None), b"null pointer")


# ------------------------------------------------------------------------------------------------ Mixup
@pytest.mark.parametrize("kw,match", [
    ({"mixup_alpha": 0.0, "cutmix_alpha": 0.0}, "mixup_alpha > 0 or cutmix_alpha > 0"),
    ({"mixup_alpha": -1.0}, "mixup_alpha"),
    ({"cutmix_alpha": "1"}, "cutmix_alpha"),
    ({"prob": 1.5}, "prob"),
    ({"switch_prob": -0.1}, "switch_prob"),
    ({"label_smoothing": 2.0}, "label_smoothing"),
    ({"mode": "row"}, "mode"),
    ({"prob": True}, "prob"),
])
def test_mixup_arguments(kw, match):
    from myrtle_vision.utils.mixup import Mixup
    with pytest.raises(ValueError, match=match):
        Mixup(**kw)


def test_mixup_defaults_are_timms():
    import inspect

    from myrtle_vision.utils.mixup import Mixup
    sig = inspect.signature(Mixup)
    assert {k: v.default for k, v in sig.parameters.items()} == {
        "mixup_alpha": 1.0, "cutmix_alpha": 0.0, "prob": 1.0, "switch_prob": 0.5, "mode": "batch",
        "label_smoothing": 0.1, "num_classes": 1000}
    m = Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, mode="pair")
    assert (m.spec.mixup_alpha, m.spec.cutmix_alpha, m.spec.prob, m.spec.switch_prob, m.spec.mode) == (
        pytest.approx(0.8), 1.0, 1.0, 0.5, 1)


def test_odd_batch_is_rejected_before_any_launch():
    from myrtle_vision.utils.mixup import Mixup
    with pytest.raises(ValueError, match="even"):
        Mixup().draw(7, 32, 32, seed=1)


def test_smoothing_is_checked():
    from myrtle_vision.utils.mixup import MixupLoss
    with pytest.raises(ValueError, match="smoothing"):
        MixupLoss(1.5)


def test_wrapper_is_classification_only_and_has_no_parameters():
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.mixup import Mixup, MixupWrapper
    seg = ViT(decoder="segmentation", image_size=176, patch_size=16, num_classes=3, dim=128, depth=1, heads=2,
              mlp_dim=256)
    with pytest.raises(ValueError, match="classification"):
        MixupWrapper(seg, Mixup())
    vit = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=1, heads=2,
              mlp_dim=256)
    w = MixupWrapper(vit, Mixup())
    assert {id(p) for p in w.parameters()} == {id(p) for p in vit.parameters()}
    assert list(vit.state_dict()) == [k[len("vit."):] for k in w.state_dict()]


# ------------------------------------------------------------------------------------------------ train_config
def test_config_defaults_leave_mixing_off():
    from myrtle_vision.utils.mixup import parse_mix_config
    cfg = parse_mix_config({}, "classification", 7)
    assert not cfg["active"] and cfg["smoothing"] == 0.0
    assert (cfg["mixup"], cfg["cutmix"], cfg["cutmix_minmax"], cfg["mixup_prob"], cfg["mixup_switch_prob"],
            cfg["mixup_mode"]) == (0.0, 0.0, None, 1.0, 0.5, "batch")
    # segmentation and detection parse without the keys, as before
    for decoder in ("segmentation", "detection"):
        assert not parse_mix_config({}, decoder, 3)["active"]


def test_config_deit_settings():
    from myrtle_vision.utils.mixup import build_mixup, parse_mix_config
    cfg = parse_mix_config({"mixup": 0.8, "cutmix": 1.0, "smoothing": 0.1, "mixup_mode": "elem"}, "classification", 256)
    assert cfg["active"]
    m = build_mixup(cfg, 45)
    assert (m.mixup_alpha, m.cutmix_alpha, m.mode, m.label_smoothing, m.num_classes) == (0.8, 1.0, "elem", 0.1, 45)
    assert parse_mix_config({"smoothing": 0.1}, "classification", 7)["active"] is False


@pytest.mark.parametrize("over,decoder,batch,distiller,exc,match", [
    ({"mixup": -0.1}, "classification", 8, False, ValueError, "mixup"),
    ({"cutmix": "1"}, "classification", 8, False, ValueError, "cutmix"),
    ({"mixup": 0.8, "mixup_prob": 1.2}, "classification", 8, False, ValueError, "mixup_prob"),
    ({"mixup": 0.8, "mixup_switch_prob": -1}, "classification", 8, False, ValueError, "mixup_switch_prob"),
    ({"smoothing": 1.1}, "classification", 8, False, ValueError, "smoothing"),
    ({"mixup": 0.8, "mixup_mode": "rows"}, "classification", 8, False, ValueError, "mixup_mode"),
    ({"mixup": 0.8}, "classification", 7, False, ValueError, "even local batch"),
    ({"cutmix": 1.0}, "segmentation", 8, False, ValueError, "classification"),
    ({"smoothing": 0.1}, "detection", 8, False, ValueError, "classification"),
    ({"mixup": 0.8}, "classification", 8, True, ValueError, "distiller_config"),
    ({"mixup": 0.8, "cutmix_minmax": [0.2, 0.8]}, "classification", 8, False, NotImplementedError, "cutmix_minmax"),
])
def test_config_rejections(over, decoder, batch, distiller, exc, match):
    from myrtle_vision.utils.mixup import parse_mix_config
    with pytest.raises(exc, match=match):
        parse_mix_config(over, decoder, batch, distiller)


def test_trainer_rejects_bad_keys_before_building_anything(tmp_path):
    from myrtle_vision.utils.trainer import train_deit
    vit = {"patch_size": 16, "embed_dim": 128, "depth": 1, "heads": 2, "mlp_dim": 256, "dropout": 0.0,
           "emb_dropout": 0.0, "decoder": "classification", "image_size": 80, "q_format": "FP32"}
    train = {"output_directory": str(tmp_path), "checkpoint_path": "", "epochs": 1, "local_batch_size": 3,
             "global_batch_size": 3, "seed": 1, "drop_last_batch": True, "mixup": 0.8}
    cfg = {"train_config": train, "dist_config": {}, "vit_config": vit,
           "data_config": {"number_of_classes": 5, "synthetic": {"train_length": 4, "val_length": 0}}}
    with pytest.raises(ValueError, match="even local batch"):
        train_deit(0, 1, cfg)
