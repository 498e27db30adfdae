"""Optimizer and learning-rate schedule of the train.py entry points.

The reference builds both with timm 0.5.4 (`timm.optim.create_optimizer`, `timm.scheduler.
create_scheduler`; classification/train.py:161-166) from the Namespace made by
`get_optimizer_args` (utils/models.py:84-110).  timm is not a dependency here; the two pieces the
shipped configs use are restated [recall of timm 0.5.4 — optim_factory.py / cosine_lr.py]:

* `adamw`: AdamW where parameters with ndim <= 1, names ending in ".bias" and names in
  `model.no_weight_decay()` get weight_decay 0, everything else `args.weight_decay`.
* `cosine`: per-epoch schedule, linear warm-up from `warmup_lr` over `warmup_epochs`, then
  `min_lr + 0.5 (lr - min_lr)(1 + cos(pi t / epochs))` (warm-up epochs are NOT a prefix), `min_lr`
  after `epochs`; training runs `epochs + cooldown_epochs` epochs.

`FusedAdamW` (utils/fused_adamw.py) is the B200-side optimizer the entry points use when the model
is on a CUDA device; the torch.optim path below is its parity reference.
"""
import math

import torch


def add_weight_decay(model, weight_decay=1e-5, skip_list=()):
    decay, no_decay = [], []
    for name, param in model.named_parameters():
        if not param.requires_grad:
            continue
        if param.ndim <= 1 or name.endswith(".bias") or name in skip_list:
            no_decay.append(param)
        else:
            decay.append(param)
    return [{"params": no_decay, "weight_decay": 0.0},
            {"params": decay, "weight_decay": weight_decay}]


def optimizer_kwargs(args):
    kw = dict(lr=args.lr, eps=args.opt_eps if args.opt_eps is not None else 1e-8)
    if getattr(args, "opt_betas", None) is not None:
        kw["betas"] = tuple(args.opt_betas)
    return kw


def create_optimizer(args, model, filter_bias_and_bn=True, fused=None):
    """args: the Namespace of get_optimizer_args.  fused=None picks FusedAdamW for CUDA models."""
    opt = args.opt.lower()
    weight_decay = args.weight_decay
    if weight_decay and filter_bias_and_bn:
        skip = model.no_weight_decay() if hasattr(model, "no_weight_decay") else ()
        params = add_weight_decay(model, weight_decay, skip)
        weight_decay = 0.0
    else:
        params = [{"params": [p for p in model.parameters() if p.requires_grad]}]
    if opt == "adamw":
        on_cuda = all(p.is_cuda for g in params for p in g["params"])
        if fused is None:
            fused = on_cuda
        if fused:
            from myrtle_vision.utils.fused_adamw import FusedAdamW
            return FusedAdamW(params, weight_decay=weight_decay, model=model, **optimizer_kwargs(args))
        return torch.optim.AdamW(params, weight_decay=weight_decay, **optimizer_kwargs(args))
    if opt in ("sgd", "nesterov", "momentum"):
        return torch.optim.SGD(params, lr=args.lr, momentum=args.momentum, weight_decay=weight_decay,
                               nesterov=opt != "momentum")
    raise NotImplementedError("optimizer %r (the shipped configs use adamw)" % args.opt)


_LP_KEYS = ("weight_quant", "grad_quant", "momentum_quant", "acc_quant", "grad_scaling", "seed")


def _lp_quantizer(site, spec):
    """train_config["optim_lp"][site] -> a qtorch.quant.quantizer (None for null)."""
    from qtorch import FixedPoint, FloatingPoint
    from qtorch.quant import quantizer
    if spec is None:
        return None
    if not isinstance(spec, dict):
        raise ValueError("optim_lp.%s: expected null or an object, got %r" % (site, spec))
    kinds = [k for k in ("float", "fixed") if k in spec]
    if len(kinds) != 1:
        raise ValueError("optim_lp.%s: give exactly one of \"float\": [exp, man] or \"fixed\": [wl, fl]" % site)
    allowed = {"float": {"float", "rounding"}, "fixed": {"fixed", "rounding", "clamp", "symmetric"}}[kinds[0]]
    unknown = set(spec) - allowed
    if unknown:
        raise ValueError("optim_lp.%s: unknown keys %s" % (site, sorted(unknown)))
    rounding = spec.get("rounding", "stochastic")
    if rounding not in ("stochastic", "nearest"):
        raise ValueError("optim_lp.%s: rounding must be \"stochastic\" or \"nearest\", got %r" % (site, rounding))
    bits = spec[kinds[0]]
    if not (isinstance(bits, (list, tuple)) and len(bits) == 2 and all(isinstance(b, int) for b in bits)):
        raise ValueError("optim_lp.%s: %s needs two integers, got %r" % (site, kinds[0], bits))
    if kinds[0] == "float":
        if not (1 <= bits[0] <= 8 and 1 <= bits[1] <= 22):
            raise ValueError("optim_lp.%s: float [exp, man] needs exp in 1..8 and man in 1..22, got %r" % (site, bits))
        number = FloatingPoint(exp=bits[0], man=bits[1])
    else:
        if not (1 <= bits[0] <= 32 and 1 <= bits[1] <= 100):
            raise ValueError("optim_lp.%s: fixed [wl, fl] needs wl in 1..32 and fl in 1..100, got %r" % (site, bits))
        number = FixedPoint(wl=bits[0], fl=bits[1], clamp=bool(spec.get("clamp", True)),
                            symmetric=bool(spec.get("symmetric", False)))
    return quantizer(forward_number=number, forward_rounding=rounding)


def wrap_optim_lp(optimizer, cfg):
    """train_config["optim_lp"] -> qtorch.optim.OptimLP around `optimizer` (DESIGN.md section 7):
    {"weight_quant": Q, "grad_quant": Q, "momentum_quant": Q, "acc_quant": Q, "grad_scaling": 1.0, "seed": null},
    Q = null | {"float": [exp, man], "rounding": ...} | {"fixed": [wl, fl], "clamp": true, "symmetric": false,
    "rounding": ...}, rounding "stochastic" (the default, as QPyTorch's) or "nearest".  Absent keys are null / 1.0."""
    from qtorch.optim import OptimLP
    if not isinstance(cfg, dict):
        raise ValueError("optim_lp: expected an object, got %r" % (cfg,))
    unknown = set(cfg) - set(_LP_KEYS)
    if unknown:
        raise ValueError("optim_lp: unknown keys %s (known: %s)" % (sorted(unknown), ", ".join(_LP_KEYS)))
    scaling = cfg.get("grad_scaling", 1.0)
    if not isinstance(scaling, (int, float)) or isinstance(scaling, bool) or not scaling > 0:
        raise ValueError("optim_lp.grad_scaling: expected a positive number, got %r" % (scaling,))
    seed = cfg.get("seed")
    if seed is not None and (not isinstance(seed, int) or isinstance(seed, bool) or not 0 <= seed < 2 ** 64):
        raise ValueError("optim_lp.seed: expected null or an integer in [0, 2^64), got %r" % (seed,))
    q = {k: _lp_quantizer(k, cfg.get(k)) for k in _LP_KEYS[:4]}
    return OptimLP(optimizer, weight_quant=q["weight_quant"], grad_scaling=float(scaling), grad_quant=q["grad_quant"],
                   momentum_quant=q["momentum_quant"], acc_quant=q["acc_quant"], seed=seed)


class CosineSchedule:
    """Epoch-indexed cosine decay with linear warm-up; `step(epoch)` sets the lr of every group."""

    def __init__(self, optimizer, t_initial, lr_min=0.0, warmup_t=0, warmup_lr_init=0.0):
        self.optimizer = optimizer
        self.t_initial, self.lr_min = t_initial, lr_min
        self.warmup_t, self.warmup_lr_init = warmup_t, warmup_lr_init
        for group in optimizer.param_groups:
            group.setdefault("initial_lr", group["lr"])
        self.base = [g["initial_lr"] for g in optimizer.param_groups]
        self.last_epoch = None
        if warmup_t > 0:
            self._apply([warmup_lr_init] * len(self.base))

    def values(self, t):
        if t < self.warmup_t:
            return [self.warmup_lr_init + t * (b - self.warmup_lr_init) / self.warmup_t for b in self.base]
        if t < self.t_initial:
            return [self.lr_min + 0.5 * (b - self.lr_min) * (1 + math.cos(math.pi * t / self.t_initial))
                    for b in self.base]
        return [self.lr_min] * len(self.base)

    def _apply(self, values):
        for group, lr in zip(self.optimizer.param_groups, values):
            group["lr"] = lr

    def step(self, epoch, metric=None):
        self.last_epoch = epoch
        self._apply(self.values(epoch))

    def get_cycle_length(self):
        return self.t_initial

    def state_dict(self):
        return {"last_epoch": self.last_epoch, "base": self.base}

    def load_state_dict(self, state):
        self.last_epoch, self.base = state["last_epoch"], state["base"]
        if self.last_epoch is not None:
            self._apply(self.values(self.last_epoch))


def create_scheduler(args, optimizer):
    """-> (scheduler, total epochs incl. cool-down), like timm.scheduler.create_scheduler."""
    if args.sched != "cosine":
        raise NotImplementedError("scheduler %r (the shipped configs use cosine)" % args.sched)
    sched = CosineSchedule(optimizer, t_initial=args.epochs, lr_min=args.min_lr,
                           warmup_t=args.warmup_epochs, warmup_lr_init=args.warmup_lr)
    return sched, sched.get_cycle_length() + args.cooldown_epochs
