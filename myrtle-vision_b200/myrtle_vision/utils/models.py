"""Model factory and checkpoint helpers (reference: src/myrtle_vision/utils/models.py:25-141).

`get_models(config)` keeps the JSON schema (`vit_config`, `data_config_path`) and returns
`(vit, None)`, or `(vit, DistillWrapper)` when the config has a `distiller_config` (models/distill.py; the
reference's wrapper is broken upstream, SURVEY.md §2 row 11, and is restated there)."""
import torch

from myrtle_vision.models.vit import ViT
from myrtle_vision.utils.quantize import QFormat
from myrtle_vision.utils.utils import parse_config


def get_models(config, profile=False):
    vit_config = config["vit_config"]
    data_config = config.get("data_config")
    if data_config is None:
        data_config = parse_config(config["data_config_path"])
    distiller = None
    if "distiller_config" in config:
        from myrtle_vision.models.distill import parse_distiller_config
        distiller = parse_distiller_config(config["distiller_config"], vit_config["decoder"])
    vit = ViT(
        decoder=vit_config["decoder"],
        image_size=vit_config["image_size"],
        patch_size=vit_config["patch_size"],
        num_classes=data_config["number_of_classes"],
        dim=vit_config["embed_dim"],
        depth=vit_config["depth"],
        heads=vit_config["heads"],
        mlp_dim=vit_config["mlp_dim"],
        dropout=vit_config["dropout"],
        emb_dropout=vit_config["emb_dropout"],
        profile=profile,
        q_format=QFormat[vit_config["q_format"]],
    )
    if distiller is None:
        return vit, None
    from myrtle_vision.models.distill import DistillWrapper, build_teacher
    teacher = build_teacher(distiller["teacher"], data_config["number_of_classes"])
    return vit, DistillWrapper(student=vit, teacher=teacher, temperature=distiller["temperature"],
                               alpha=distiller["alpha"], hard=distiller["hard"])


def save_checkpoint(model, optimizer, lr_scheduler, iteration, filepath, distiller=None):
    """distiller (a DistillWrapper): its own parameters go under "distiller"; "model" stays the student's."""
    state = {
        "model": model.state_dict(),
        "optimizer": optimizer.state_dict(),
        "lr_scheduler": lr_scheduler.state_dict() if lr_scheduler is not None else None,
        "iteration": iteration,
    }
    if distiller is not None:
        state["distiller"] = distiller.distiller_state_dict()
    torch.save(state, filepath)


def load_checkpoint(model, optimizer, lr_scheduler, filepath, distiller=None):
    checkpoint = torch.load(filepath, map_location="cpu")
    model.load_state_dict(checkpoint["model"])
    if distiller is not None:
        if "distiller" not in checkpoint:
            raise KeyError("%s has no \"distiller\" entry to resume the distillation head from" % filepath)
        distiller.load_distiller_state_dict(checkpoint["distiller"])
    if optimizer is not None:
        optimizer.load_state_dict(checkpoint["optimizer"])
    if lr_scheduler is not None and checkpoint.get("lr_scheduler") is not None:
        lr_scheduler.load_state_dict(checkpoint["lr_scheduler"])
    return checkpoint["iteration"]


def prepare_model_and_load_ckpt(train_config, model, optimizer=None, lr_scheduler=None, distiller=None):
    if train_config["checkpoint_path"] != "":
        return load_checkpoint(model=model, optimizer=optimizer, lr_scheduler=lr_scheduler,
                               filepath=train_config["checkpoint_path"], distiller=distiller)
    return 0


def get_optimizer_args(train_config):
    """train_config -> the Namespace the optimizer / scheduler factories read (reference :84-110)."""
    import argparse
    cfg = train_config
    return argparse.Namespace(
        opt=cfg["optimizer"], opt_eps=cfg["opt_eps"], opt_betas=cfg["opt_betas"], clip_grad=cfg["clip_grad"],
        momentum=cfg["momentum"], weight_decay=cfg["weight_decay"], sched=cfg["scheduler"], lr=cfg["lr"],
        lr_noise=cfg.get("lr_noise"), lr_noise_pct=cfg.get("lr_noise_pct"), lr_noise_std=cfg.get("lr_noise_std"),
        warmup_lr=cfg["warmup_lr"], min_lr=cfg["min_lr"], epochs=cfg["epochs"], decay_epochs=cfg["decay_epochs"],
        warmup_epochs=cfg["warmup_epochs"], cooldown_epochs=cfg["cooldown_epochs"],
        patience_epochs=cfg["patience_epochs"], decay_rate=cfg["decay_rate"])


# ---- pretrained-backbone key mapping (reference utils/models.py:144-223)
_TIMM_RULES = [
    (r"pos_embed", r"pos_embedding"),
    (r"patch_embed\.proj\.(weight|bias)", r"patch_to_embedding.\1"),
    (r"blocks\.([0-9]+)\.norm1\.(weight|bias)", r"transformer.layers.\1.0.fn.norm.\2"),
    (r"blocks\.([0-9]+)\.attn\.qkv\.(weight|bias)", r"transformer.layers.\1.0.fn.fn.to_qkv.\2"),
    (r"blocks\.([0-9]+)\.attn\.proj\.(weight|bias)", r"transformer.layers.\1.0.fn.fn.to_out.0.\2"),
    (r"blocks\.([0-9]+)\.norm2\.(weight|bias)", r"transformer.layers.\1.1.fn.norm.\2"),
    (r"blocks\.([0-9]+)\.mlp\.fc1\.(weight|bias)", r"transformer.layers.\1.1.fn.fn.net.0.\2"),
    (r"blocks\.([0-9]+)\.mlp\.fc2\.(weight|bias)", r"transformer.layers.\1.1.fn.fn.net.3.\2"),
]
_TIMM_HEAD = (r"norm\.weight", r"norm\.bias", r"head\.weight", r"head\.bias")


def apply_rules(name, rules):
    """Apply the first matching rule (regex substitution) to name."""
    import re
    for pattern, replacement in rules:
        if re.match(pattern, name) is not None:
            return re.sub(pattern, replacement, name)
    return name


def rename_timm_state_dict(timm_model_name, vit_config, num_classes, q_format=None):
    """State dict of a pretrained timm ViT under this package's parameter names.

    `timm_model_name`: a timm model name (needs timm, as in the reference) or an already loaded
    timm-style state dict.  The classifier head (`norm.*`, `head.*`) is dropped; the Conv2d patch
    embedding `(O, I, H, W)` becomes the Linear weight `(O, (H, W, I))`.  `q_format` (default: the
    config's) selects the key layout: quantised models wrap every Linear / LayerNorm in
    `Sequential(stub, module)`, so their parameters live under `<name>.1.<param>` — the
    reference maps to the unwrapped names only, which silently loads nothing into a quantised
    model (SURVEY.md fact 8)."""
    import re
    if isinstance(timm_model_name, str):
        try:
            import timm
        except ImportError as e:
            raise ImportError("rename_timm_state_dict(<model name>) needs timm; pass a timm-style "
                              "state dict instead") from e
        source = timm.create_model(timm_model_name, pretrained=True, num_classes=num_classes).state_dict()
    else:
        source = timm_model_name
    fmt = q_format if q_format is not None else vit_config.get("q_format", "FP32")
    fmt = QFormat[fmt] if isinstance(fmt, str) else fmt
    wrapped = fmt != QFormat.FP32
    out = {}
    for key, value in source.items():
        if any(re.match(pat, key) for pat in _TIMM_HEAD):
            continue
        new_key = apply_rules(key, _TIMM_RULES)
        if new_key.startswith("patch_to_embedding.weight") and value.dim() == 4:
            value = value.permute(0, 2, 3, 1).reshape(vit_config["embed_dim"],
                                                      vit_config["patch_size"] ** 2 * value.shape[1])
        if wrapped and new_key != key and not new_key.startswith("pos_embedding"):
            stem, param = new_key.rsplit(".", 1)
            new_key = f"{stem}.1.{param}"
        out[new_key] = value
    return out
