"""qtorch.quant facade: float_quantize / fixed_point_quantize / block_quantize / quantizer /
Quantizer with QPyTorch 0.3.0's signatures, executed by the sm_100a kernels of libmv_b200.so
(include/mv_b200.h: mv_float_quantize, mv_fixed_point_quantize, mv_block_quantize).

Stochastic rounding is reproducible: every call consumes one Philox stream
(seed, offset) from a module-level counter that `manual_seed` resets, where QPyTorch draws
an unseeded random tensor.
"""
import torch

import mv_native as _mv

from . import BlockFloatingPoint, FixedPoint, FloatingPoint

__all__ = ["float_quantize", "fixed_point_quantize", "block_quantize", "quantizer", "Quantizer",
           "manual_seed"]

_state = {"seed": 0, "offset": 0}


def manual_seed(seed, offset=0):
    _state["seed"], _state["offset"] = int(seed), int(offset)


def _stream():
    s = (_state["seed"], _state["offset"])
    _state["offset"] += 1
    return s


def _check_rounding(rounding):
    assert rounding in ("stochastic", "nearest"), "invalid rounding mode, {}".format(rounding)


def float_quantize(x, exp, man, rounding="stochastic"):
    _check_rounding(rounding)
    seed, off = _stream() if rounding == "stochastic" else (0, 0)
    return _mv.float_quantize(x, exp, man, rounding, seed=seed, offset=off).to(x.dtype)


def fixed_point_quantize(x, wl, fl, clamp=True, symmetric=False, rounding="stochastic"):
    _check_rounding(rounding)
    seed, off = _stream() if rounding == "stochastic" else (0, 0)
    return _mv.fixed_point_quantize(x, wl, fl, clamp, symmetric, rounding, seed=seed,
                                    offset=off).to(x.dtype)


def block_quantize(x, wl, dim=-1, rounding="stochastic"):
    _check_rounding(rounding)
    seed, off = _stream() if rounding == "stochastic" else (0, 0)
    return _mv.block_quantize(x, wl, dim, rounding, seed=seed, offset=off).to(x.dtype)


def _number_fn(number, rounding):
    if number is None:
        return None
    if isinstance(number, FloatingPoint):
        return lambda t: float_quantize(t, number.exp, number.man, rounding)
    if isinstance(number, FixedPoint):
        return lambda t: fixed_point_quantize(t, number.wl, number.fl, number.clamp,
                                              number.symmetric, rounding)
    if isinstance(number, BlockFloatingPoint):
        return lambda t: block_quantize(t, number.wl, number.dim, rounding)
    raise ValueError("unknown number format {}".format(number))


def quantizer(forward_number=None, backward_number=None, forward_rounding="stochastic",
              backward_rounding="stochastic", clamping_grad_zero=False, backward_hooks=[]):
    """Returns an autograd function: forward quantises with forward_number, backward quantises
    the incoming gradient with backward_number (identity when None)."""
    _check_rounding(forward_rounding)
    _check_rounding(backward_rounding)
    fwd = _number_fn(forward_number, forward_rounding)
    bwd = _number_fn(backward_number, backward_rounding)
    masked = clamping_grad_zero and isinstance(forward_number, FixedPoint)
    if clamping_grad_zero:
        assert isinstance(forward_number, FixedPoint), \
            "zeroing clamped gradients is only supported for fixed point"

    class _Rounding(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x):
            if fwd is None:
                return x
            if masked:
                rnd = forward_rounding
                seed, off = _stream() if rnd == "stochastic" else (0, 0)
                out, mask = _mv.fixed_point_quantize(x, forward_number.wl, forward_number.fl, True,
                                                     forward_number.symmetric, rnd, seed=seed,
                                                     offset=off, with_mask=True)
                ctx.mask = mask.bool()
                return out.to(x.dtype)
            return fwd(x.contiguous())

        @staticmethod
        def backward(ctx, grad):
            if not ctx.needs_input_grad[0]:
                return None
            if bwd is not None:
                grad = bwd(grad.contiguous())
            if masked:
                grad = grad.masked_fill(ctx.mask, 0)
            for hook in backward_hooks:
                grad = hook(grad)
            return grad

    def quantize(x):
        return _Rounding.apply(x)

    # what qtorch.optim.OptimLP reads to run a recognised format in its fused optimizer kernel
    quantize.forward_number, quantize.forward_rounding = forward_number, forward_rounding
    return quantize


class Quantizer(torch.nn.Module):
    def __init__(self, forward_number=None, backward_number=None, forward_rounding="stochastic",
                 backward_rounding="stochastic"):
        super().__init__()
        self.quantize = quantizer(forward_number, backward_number, forward_rounding,
                                  backward_rounding)
        self.forward_number, self.forward_rounding = forward_number, forward_rounding

    def forward(self, x):
        return self.quantize(x)
