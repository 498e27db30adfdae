"""qtorch.optim facade: `OptimLP` with QPyTorch 0.3.0's signature, keeping weights, the gradients the optimizer sees,
its moments and a weight accumulator in low precision (DESIGN.md section 7, "Low-precision optimizer").

For every parameter with a gradient, on each step that is not skipped, in this order:

1. grad: ``g = grad_quant(g * grad_scaling)`` after any un-scale (``inv_scale``); ``p.grad`` holds it afterwards.
   Without ``grad_quant`` the gradient is left alone and ``grad_scaling`` has no effect (as upstream).
2. update: on a full-precision accumulator (a copy of p made at construction) when ``acc_quant`` is set, else on p.
3. momentum: ``momentum_quant`` on ``exp_avg`` and ``exp_avg_sq`` (AdamW / Adam / FusedAdamW) or ``momentum_buffer``
   (SGD).  Upstream keys this on the class names "SGD" / "Adam" [recall]; AdamW gets Adam's treatment here.
4. accumulator: ``acc = acc_quant(acc)``.
5. weight: ``p = weight_quant(acc or p)``, written in place (the engine holds raw pointers to its parameters).

Stochastic rounding of a recognised quantiser (``qtorch.quant.quantizer`` / ``Quantizer`` with a FloatingPoint or
FixedPoint forward format) uses the optimizer rounding stream of include/mv_b200.h, not torch's RNG: site s (0 grad,
1 exp_avg, 2 exp_avg_sq, 3 acc, 4 weight) of parameter k (its position in the flattened ``param_groups``) rounds
with offset ``lp_offset(step, k, s)`` and the 64-bit ``seed`` (drawn once from torch's default generator when None,
and saved in ``state_dict``).  A run therefore repeats under ``torch.manual_seed``, data-parallel ranks holding the
same gradients keep bit-identical parameters, and a resumed run continues bit for bit.  Any other callable is called.

A step with a non-zero ``found_inf`` changes nothing and does not advance the step count.

Fused path (``fused=None`` with ``FusedAdamW`` and only recognised quantisers): one mv_adamw_lp_step launch does
steps 1-5 and emits the next forward's q(W) / q(W)^T of the final weights.  Composed path (everything else, or
``fused=False``): standalone quantiser calls around the inner ``step()``; it is the reference the fused path is held
to.  No CPU fallback: CPU parameters raise.
"""
import torch

import mv_native as _mv

from . import FixedPoint, FloatingPoint

__all__ = ["OptimLP", "lp_offset", "lp_format"]

SITES = ("grad", "exp_avg", "exp_avg_sq", "acc", "weight")


def lp_offset(step, k, site):
    """Offset of the optimizer rounding stream: (step << 32) | (k << 3) | site."""
    return (int(step) << 32) | (int(k) << 3) | int(site)


def lp_format(quant):
    """None for no quantiser; ("float", exp, man, rounding) / ("fixed", wl, fl, clamp, symmetric, rounding) for a
    quantiser made by qtorch.quant.quantizer / Quantizer with a FloatingPoint / FixedPoint forward format; "callable"
    for anything else (block floating point, lambdas)."""
    if quant is None:
        return None
    number = getattr(quant, "forward_number", None)
    rounding = getattr(quant, "forward_rounding", None)
    if rounding not in ("nearest", "stochastic"):
        return "callable"
    if isinstance(number, FloatingPoint):
        return ("float", number.exp, number.man, rounding)
    if isinstance(number, FixedPoint):
        return ("fixed", number.wl, number.fl, bool(number.clamp), bool(number.symmetric), rounding)
    return "callable"


def _is_adam(optim):
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    return isinstance(optim, (FusedAdamW, torch.optim.Adam, torch.optim.AdamW))


class OptimLP:
    def __init__(self, optim, weight_quant=None, grad_scaling=1.0, grad_quant=None, momentum_quant=None,
                 acc_quant=None, *, seed=None, fused=None):
        from myrtle_vision.utils.fused_adamw import FusedAdamW
        if grad_scaling <= 0:
            raise ValueError("need a positive grad_scaling, got {}".format(grad_scaling))
        if momentum_quant is not None and not (_is_adam(optim) or isinstance(optim, torch.optim.SGD)):
            raise NotImplementedError("momentum_quant for {} (supported: AdamW, Adam, SGD)".format(
                type(optim).__name__))
        for p in self._params_of(optim):
            if not p.is_cuda:
                raise _mv.MvError("OptimLP needs CUDA parameters (there is no CPU fallback)")
        self.optim = optim
        self.weight_quant, self.grad_quant = weight_quant, grad_quant
        self.momentum_quant, self.acc_quant = momentum_quant, acc_quant
        self.grad_scaling = float(grad_scaling)
        if seed is None:
            lo, hi = (int(v) for v in torch.randint(0, 2 ** 32, (2,), dtype=torch.int64))
            seed = (hi << 32) | lo
        self.seed = int(seed) & (2 ** 64 - 1)
        self._step = 0                 # steps taken (the composed path's count; the fused path's lives on the device)
        self._quants = (grad_quant, momentum_quant, momentum_quant, acc_quant, weight_quant)
        formats = [lp_format(q) for q in self._quants]
        recognised = all(f != "callable" for f in formats)
        if fused and not (isinstance(optim, FusedAdamW) and recognised):
            raise ValueError("fused=True needs FusedAdamW and FloatingPoint / FixedPoint quantisers")
        self.fused = isinstance(optim, FusedAdamW) and recognised if fused is None else bool(fused)
        self.acc = [p.detach().clone() if acc_quant is not None else None for p in self._params_of(optim)]
        if self.fused:
            from myrtle_vision.utils.fused_adamw import OptimLpSpec
            self.spec = OptimLpSpec()
            for name, f in zip(SITES, formats):
                self._fill(getattr(self.spec, name), f)
            self.spec.grad_scaling = self.grad_scaling if grad_quant is not None else 1.0
            self.spec.seed = self.seed

    @staticmethod
    def _params_of(optim):
        return [p for g in optim.param_groups for p in g["params"]]

    @staticmethod
    def _fill(q, f):
        if f is None:
            return
        if f[0] == "float":
            q.kind, q.exp_bits, q.man_bits = 1, f[1], f[2]
        else:
            q.kind, q.wl, q.fl, q.clamp, q.symmetric = 2, f[1], f[2], int(f[3]), int(f[4])
        q.rounding = _mv.ROUND_STOCHASTIC if f[-1] == "stochastic" else _mv.ROUND_NEAREST

    # ------------------------------------------------------------------ torch.optim.Optimizer surface
    @property
    def param_groups(self):
        return self.optim.param_groups

    @property
    def state(self):
        return self.optim.state

    def zero_grad(self, set_to_none=True):
        self.optim.zero_grad(set_to_none=set_to_none)

    # ------------------------------------------------------------------ fused path: side table of FusedAdamW
    def side(self, p, k, g):
        """(acc, grad_out) device pointers of parameter k for mv_adamw_lp_step."""
        acc = self.acc[k]
        return (acc.data_ptr() if acc is not None else None, g.data_ptr() if self.grad_quant is not None else None)

    # ------------------------------------------------------------------ composed path
    def _q(self, quant, x, step, k, site):
        f = lp_format(quant)
        if f == "callable":
            return quant(x)
        off = lp_offset(step, k, site)
        if f[0] == "float":
            return _mv.float_quantize(x, f[1], f[2], f[3], seed=self.seed, offset=off)
        return _mv.fixed_point_quantize(x, f[1], f[2], f[3], f[4], f[5], seed=self.seed, offset=off)

    def _composed(self, closure, inv_scale, found_inf):
        from myrtle_vision.utils.fused_adamw import FusedAdamW
        if found_inf is not None and float(found_inf.reshape(-1)[0]) != 0.0:
            return closure() if closure is not None else None
        step = self._step + 1
        live = [(k, p) for k, p in enumerate(self._params_of(self.optim)) if p.grad is not None]
        inner_scale = inv_scale
        fused_inner = isinstance(self.optim, FusedAdamW)
        if self.grad_quant is not None or (inv_scale is not None and not fused_inner):
            for k, p in live:
                g = p.grad if inv_scale is None else p.grad * inv_scale
                if self.grad_quant is not None:
                    if self.grad_scaling != 1.0:
                        g = g * self.grad_scaling
                    g = self._q(self.grad_quant, g, step, k, 0)
                p.grad.copy_(g)
            inner_scale = None
        for k, p in live:
            if self.acc[k] is not None:
                p.copy_(self.acc[k])
        loss = self.optim.step(closure, inv_scale=inner_scale) if fused_inner else self.optim.step(closure)
        for k, p in live:
            if self.momentum_quant is not None:
                st = self.optim.state[p]
                names = ("exp_avg", "exp_avg_sq") if _is_adam(self.optim) else ("momentum_buffer",)
                for site, name in enumerate(names, start=1):
                    if st.get(name) is not None:
                        st[name].copy_(self._q(self.momentum_quant, st[name], step, k, site))
            w = p
            if self.acc[k] is not None:
                self.acc[k].copy_(self._q(self.acc_quant, p, step, k, 3))
                w = self.acc[k]
            if self.weight_quant is not None:
                p.copy_(self._q(self.weight_quant, w, step, k, 4))
            elif w is not p:
                p.copy_(w)
        engine = getattr(self.optim, "_engine", None)
        if engine is not None:
            engine.invalidate_weights()            # p changed after the optimizer emitted its q(W) operands
        self._step = step
        return loss

    @torch.no_grad()
    def step(self, closure=None, inv_scale=None, found_inf=None):
        """inv_scale / found_inf: optional device scalars with GradScaler semantics (see FusedAdamW.step)."""
        if not self.fused:
            return self._composed(closure, inv_scale, found_inf)
        return self.optim._fused_step(closure, inv_scale, found_inf, lp=self)

    # ------------------------------------------------------------------ checkpoints
    def step_count(self):
        """Steps taken so far (skipped ones excluded): the `step` of the optimizer rounding stream's last step."""
        hy = getattr(self.optim, "_hyper", None)
        if self.fused and hy is not None:
            return int(hy[3].item())
        return self._step

    def state_dict(self):
        return {"optim": self.optim.state_dict(), "acc": [a.detach().clone() if a is not None else None
                                                            for a in self.acc],
                "seed": self.seed, "step": self.step_count()}

    def load_state_dict(self, state_dict):
        from myrtle_vision.utils.fused_adamw import FusedAdamW
        self.optim.load_state_dict(state_dict["optim"])
        if len(state_dict["acc"]) != len(self.acc):
            raise ValueError("OptimLP state has {} accumulators for {} parameters".format(
                len(state_dict["acc"]), len(self.acc)))
        for mine, saved in zip(self.acc, state_dict["acc"]):
            if (mine is None) != (saved is None):
                raise ValueError("OptimLP state and this optimizer disagree on acc_quant")
            if mine is not None:
                mine.copy_(saved)
        self.seed = int(state_dict["seed"])
        self._step = int(state_dict["step"])
        if self.fused:
            self.spec.seed = self.seed
        if isinstance(self.optim, FusedAdamW):
            self.optim._step0 = self._step         # the device step count FusedAdamW resumes from
