"""The training loop behind the three train.py entry points (reference classification/train.py:55-318,
segmentation/train.py, detection/train.py — one `train_deit(rank, num_gpus, config)` each, identical
in shape).  Same config schema, batch-size solving, seeding, checkpoint cadence and printed lines;
what differs is underneath:

* the model is the fused sm_100a ViT, wrapped in `utils.parallel.DataParallel` (NCCL bucket
  all-reduce overlapped with backward) instead of DistributedDataParallel;
* forward + loss + backward run as ONE captured CUDA graph when shapes are static
  (`train_config["cuda_graph"]`, default on for classification / segmentation);
* the optimizer is `FusedAdamW` (one launch, emits next step's quantised weight operands);
* the loss scale is applied inside the encoder backward (power-of-two, chosen on the device), so no
  GradScaler and no per-iteration host sync: losses are printed every `log_every` iterations;
* data: `data_config["synthetic"] = {"train_length": n, "val_length": m}` selects the synthetic datasets;
  a real dataset is plugged in with `data_config["dataset_factory"] = "module:function"` returning
  `(trainset, valset, collate_fn or None)`.
"""
import importlib
import os

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch.utils.data import DataLoader
from torch.utils.data.distributed import DistributedSampler

from qtorch.optim import OptimLP

from myrtle_vision.datasets.synthetic import SyntheticVision, detection_collate
from myrtle_vision.models.matcher import pad_targets
from myrtle_vision.utils.graph import GraphedTrainStep
from myrtle_vision.utils.mixup import MixupLoss, MixupWrapper, build_mixup, parse_mix_config
from myrtle_vision.utils.models import (get_models, get_optimizer_args, prepare_model_and_load_ckpt,
                                        save_checkpoint)
from myrtle_vision.utils.optim import create_optimizer, create_scheduler, wrap_optim_lp
from myrtle_vision.utils.parallel import DataParallel
from myrtle_vision.utils.utils import (cleanup_distributed, get_batch_sizes, init_distributed,
                                       parse_config, seed_everything)


def build_datasets(task, data_config, vit_config):
    if "dataset_factory" in data_config:
        mod, fn = data_config["dataset_factory"].split(":")
        return getattr(importlib.import_module(mod), fn)(data_config)
    syn = data_config.get("synthetic")
    if syn is None:
        raise NotImplementedError(
            "dataset loaders are outside the B200 hot path: set data_config['synthetic'] or "
            "data_config['dataset_factory'] = 'module:function'")
    size, classes = vit_config["image_size"], data_config["number_of_classes"]
    seed = syn.get("seed", 1234)
    train = SyntheticVision(task, syn["train_length"], size, classes, seed)
    val = SyntheticVision(task, syn.get("val_length", 0), size, classes, seed + 1)
    return train, val, detection_collate if task == "detection" else None


def build_criterion(task, train_config, num_classes, device):
    """-> loss(outputs, targets) returning a scalar."""
    if task == "segmentation" and train_config.get("fused_seg_loss", True):
        from myrtle_vision.models.losses import upsampled_cross_entropy

        def seg_loss(outputs, targets):
            # training: patch logits [B, gh*gw, C] (decoder.fused_loss); validation: the upsampled map
            return upsampled_cross_entropy(outputs, targets) if outputs.dim() == 3 else F.cross_entropy(outputs, targets)
        return seg_loss
    if task != "detection":
        return F.cross_entropy
    from myrtle_vision.models.detector import SetCriterion
    from myrtle_vision.models.matcher import HungarianMatcher
    weights = {k: train_config[k] for k in ("loss_ce", "class_error", "loss_bbox", "loss_giou",
                                            "cardinality_error") if k in train_config}
    # the reference matches with HungarianMatcher()'s default costs (1 / 1 / 1, detection/train.py:199) and applies
    # the weight_dict to the loss terms only; "matcher_costs": [class, bbox, giou] is an explicit opt-in
    mc = train_config.get("matcher_costs")
    matcher = HungarianMatcher(*mc) if mc else HungarianMatcher()
    crit = SetCriterion(num_classes, matcher, weights, train_config.get("eos_coef", 0.1),
                        ["labels", "boxes", "cardinality"]).to(device)

    def loss(outputs, targets):
        terms = crit(outputs, targets)
        return sum(terms[k] * weights[k] for k in terms if k in weights)
    return loss


def to_device(targets, device):
    if isinstance(targets, dict):
        return {k: v.to(device, non_blocking=True) for k, v in targets.items()}
    if isinstance(targets, list):
        return [{k: v.to(device, non_blocking=True) for k, v in t.items()} for t in targets]
    return targets.to(device, non_blocking=True)


@torch.no_grad()
def validation(task, loader, device, criterion, vit):
    """-> (mean loss, metric): accuracy (classification), mIoU (segmentation, reference
    segmentation/train.py:35-71), 0 for detection (COCO evaluation is outside the hot path)."""
    vit.eval()
    total, metric, n = 0.0, 0.0, max(1, len(loader))
    miou = None
    if task == "segmentation":
        from myrtle_vision.utils.miou import MIoU
        miou = MIoU(vit.decoder.linear[1].out_features if isinstance(vit.decoder.linear, torch.nn.Sequential)
                    else vit.decoder.linear.out_features, device)
    for imgs, targets in loader:
        imgs, targets = imgs.to(device), to_device(targets, device)
        out = vit(imgs)
        total += float(criterion(out, targets)) / n
        if task == "classification":
            metric += float((out.argmax(dim=1) == targets).float().mean()) / n
        elif miou is not None:
            miou.add_img(out.argmax(dim=1), targets)
    if miou is not None:
        metric = miou.get_miou()
    vit.train()
    return total, metric


def train_deit(rank, num_gpus, config, task=None, max_iterations=None):
    train_config, dist_config, vit_config = config["train_config"], config["dist_config"], config["vit_config"]
    task = task or vit_config["decoder"]
    data_config = config.get("data_config") or parse_config(config["data_config_path"])
    config["data_config"] = data_config
    seed_everything(train_config["seed"])
    batch_size, n_batch_accum = get_batch_sizes(train_config["local_batch_size"], num_gpus,
                                                train_config["global_batch_size"], verbose=(rank == 0))
    train_config["local_batch_size"] = batch_size
    train_config["global_batch_size"] = batch_size * n_batch_accum * max(1, num_gpus)
    train_config["n_batch_accum"] = n_batch_accum
    # Mixup / CutMix / label smoothing (DeiT's train_config keys, utils/mixup.py): validated before anything is built
    mix = parse_mix_config(train_config, task, batch_size, "distiller_config" in config)
    if num_gpus > 1:
        init_distributed(rank, num_gpus, **dist_config)
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    out_dir = train_config["output_directory"]
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        print("output directory:", out_dir)

    trainset, valset, collate = build_datasets(task, data_config, vit_config)
    sampler = DistributedSampler(trainset) if num_gpus > 1 else None
    train_loader = DataLoader(trainset, num_workers=train_config.get("num_workers", 1), shuffle=sampler is None,
                              sampler=sampler, batch_size=batch_size, pin_memory=True,
                              drop_last=train_config["drop_last_batch"], collate_fn=collate)
    val_loader = DataLoader(valset, num_workers=0, batch_size=batch_size, collate_fn=collate,
                            drop_last=train_config["drop_last_batch"]) if len(valset) else []

    vit, distiller = get_models(config)
    vit = vit.to(device)
    if task == "segmentation" and train_config.get("fused_seg_loss", True):
        vit.decoder.fused_loss = True        # training forward returns patch logits for the fused loss
    # distillation (config["distiller_config"], models/distill.py): the step trains the wrapper (student, token and
    # head; the frozen teacher runs inside it), evaluation and checkpoints' "model" stay the student's
    model = vit
    if distiller is not None:
        model = distiller.to(device)
    elif mix["active"]:
        # the step trains the wrapper, which mixes each training batch; it has no parameters of its own, so the
        # optimizer and checkpoints are the ViT's, and validation runs the bare ViT on unmixed images, as DeiT
        model = MixupWrapper(vit, build_mixup(mix, data_config["number_of_classes"]))
    net = DataParallel(model) if num_gpus > 1 else model
    optimizer_args = get_optimizer_args(train_config)
    optimizer = create_optimizer(optimizer_args, distiller if distiller is not None else vit)
    if train_config.get("optim_lp") is not None:
        # qtorch.optim.OptimLP: low-precision weights, gradients, moments and accumulator (DESIGN.md section 7)
        optimizer = wrap_optim_lp(optimizer, train_config["optim_lp"])
    lr_scheduler, _ = create_scheduler(optimizer_args, optimizer)
    criterion = build_criterion(task, train_config, data_config["number_of_classes"], device)
    train_criterion = criterion
    if distiller is not None:
        from myrtle_vision.models.distill import DistillLoss
        train_criterion = DistillLoss(distiller.temperature, distiller.alpha, distiller.hard)
    elif mix["active"] or mix["smoothing"] > 0:
        train_criterion = MixupLoss(mix["smoothing"])        # soft targets; smoothing alone: unmixed logits
    iteration = prepare_model_and_load_ckpt(train_config=train_config, model=vit, optimizer=optimizer,
                                            lr_scheduler=lr_scheduler, distiller=distiller)
    # detection: targets padded to a fixed [B, capacity] block and matched on the device (csrc/assign.cu),
    # so the criterion has no host synchronisation and the whole step is one CUDA graph like the other tasks;
    # "device_matching": false restores the host (SciPy) matcher between two captured graphs
    device_matching = task == "detection" and train_config.get("device_matching", True)
    det_capacity = 0
    # (the one-graph detection step is measured on one GPU; under data parallelism it is opt-in via "cuda_graph": true)
    use_graph = train_config.get("cuda_graph", task != "detection" or (device_matching and num_gpus <= 1)) \
        and n_batch_accum == 1 \
        and train_config["drop_last_batch"]
    split_graph = (task == "detection" and not device_matching and train_config.get("cuda_graph", True)
                   and n_batch_accum == 1 and train_config["drop_last_batch"] and num_gpus <= 1)
    iters_per_checkpoint = train_config.get("iters_per_checkpoint", 0)
    iters_per_val = train_config.get("iters_per_val", 0)
    log_every = train_config.get("log_every", 1)
    epoch_offset = max(0, int(batch_size * max(1, num_gpus) * iteration / max(1, len(trainset))))
    model.train()
    if num_gpus > 1:
        dist.barrier()
    graphed, n_accum, last_val, history = None, 0, (0.0, 0.0), []
    for epoch in range(epoch_offset, train_config["epochs"]):
        if sampler is not None:
            sampler.set_epoch(epoch)
        for imgs, targets in train_loader:
            if rank == 0 and n_accum == 0 and iters_per_checkpoint and iteration % iters_per_checkpoint == 0:
                save_checkpoint(model=vit, optimizer=optimizer, lr_scheduler=lr_scheduler,
                                iteration=iteration, filepath=f"{out_dir}/vit_{iteration:06}", distiller=distiller)
            if rank == 0 and n_accum == 0 and iters_per_val and iteration % iters_per_val == 0 and len(valset):
                last_val = validation(task, val_loader, device, criterion, vit)
            if device_matching:
                most = max([int(t["boxes"].shape[0]) for t in targets] + [1])
                if most > det_capacity:                     # grow the padded block: the graph is re-captured
                    det_capacity, graphed = -(-most // 16) * 16, None
                targets = pad_targets(targets, capacity=det_capacity)
            imgs, targets = imgs.to(device, non_blocking=True), to_device(targets, device)
            if use_graph:
                if graphed is None:
                    graphed = GraphedTrainStep(net, train_criterion, imgs, targets)
                loss = graphed(imgs, targets)
            elif split_graph:
                # detection: the matcher runs on the host between forward and backward, so the model's
                # forward and backward are two captured graphs around the eager criterion
                if graphed is None:
                    graphed = torch.cuda.make_graphed_callables(vit, (imgs,), allow_unused_input=True)
                vit.zero_grad(set_to_none=True)
                loss = criterion(graphed(imgs), targets)
                loss.backward()
            else:
                if n_accum == 0:
                    model.zero_grad(set_to_none=True)
                loss = train_criterion(net(imgs), targets)
                loss.backward()
            if optimizer_args.clip_grad is not None:
                torch.nn.utils.clip_grad_norm_(model.parameters(), optimizer_args.clip_grad)
            n_accum += 1
            if n_accum == n_batch_accum:
                n_accum = 0
                if hasattr(optimizer, "_operands") or isinstance(optimizer, OptimLP):
                    # FusedAdamW (or OptimLP): the backward's device-side overflow flag skips the update exactly like
                    # GradScaler.step() in the reference (classification/train.py:274-277), without a host sync
                    optimizer.step(found_inf=vit.engine().found_inf)
                    vit.engine().found_inf.zero_()
                else:
                    optimizer.step()
                iteration += 1
                if rank == 0 and iteration % log_every == 0:
                    history.append(float(loss.detach()))
                    print(f"Iteration {iteration}:\tloss={history[-1]:.4f}")
                if max_iterations is not None and iteration >= max_iterations:
                    break
        # after the epoch's batches, as the reference (classification/train.py:287): epoch e trains at lr(e - 1)
        lr_scheduler.step(epoch)
        if rank == 0:
            print(f"Epoch : {epoch + 1} - val_loss : {last_val[0]:.4f} - val_metric: {last_val[1]:.4f}\n")
        if max_iterations is not None and iteration >= max_iterations:
            break
    if num_gpus > 1:
        cleanup_distributed()
    return history
