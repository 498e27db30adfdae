"""Quantisation formats and the QAT preparation of the B200 ViT.

Drop-in for src/myrtle_vision/utils/quantize.py of the reference: same public names
(QFormat, NumberFormat, Quantizer, QuantizerFunction, ModelQuantizer with prepare_qat /
convert), same errors, same state_dict key layout per q_format (reference :215-228 wraps
every Linear/LayerNorm in Sequential(stub, module), which renames `x.weight` to
`x.1.weight`).  The difference is underneath: here the placement table (SURVEY.md
Appendix A) is recorded on the model as a `QuantPlan` that the fused sm_100a engine reads,
instead of a graph of observer hooks that launch one quant kernel each.
"""
import enum
from collections import namedtuple

import torch
from torch import nn

from qtorch import FixedPoint, FloatingPoint
from qtorch.quant import Quantizer as QTorchQuantizer


class QFormat(enum.IntEnum):
    """Quantization formats supported by ViT (reference utils/quantize.py:13-20)."""

    FP32 = 0
    PyTorchINT8 = 1
    FP16_16 = 2
    FP16_32 = 3
    TF32 = 4


class NumberFormat(enum.Enum):
    SymmetricInt8 = enum.auto()
    AsymmetricInt8 = enum.auto()
    HalfPrecisionFloat = enum.auto()
    SinglePrecisionFloat = enum.auto()
    TensorFloat32 = enum.auto()
    FixedPoint11Integral2 = enum.auto()
    FixedPoint11Integral3 = enum.auto()
    FixedPoint11Integral4 = enum.auto()

    @staticmethod
    def number(number_format):
        """The qtorch number a format simulates (None = fp32 identity); reference :46-72."""
        table = {
            NumberFormat.HalfPrecisionFloat: FloatingPoint(exp=5, man=10),
            NumberFormat.SinglePrecisionFloat: None,
            NumberFormat.TensorFloat32: FloatingPoint(exp=8, man=10),
            NumberFormat.FixedPoint11Integral2: FixedPoint(wl=11, fl=9),
            NumberFormat.FixedPoint11Integral3: FixedPoint(wl=11, fl=8),
            NumberFormat.FixedPoint11Integral4: FixedPoint(wl=11, fl=7),
        }
        if number_format not in table:
            raise NotImplementedError(number_format)
        return table[number_format]

    @staticmethod
    def quantizer(number_format):
        """A module that constrains an fp32 tensor to `number_format` (nearest rounding)."""
        number = NumberFormat.number(number_format)
        if number is None:
            return nn.Identity()
        return QTorchQuantizer(number, forward_rounding="nearest")


class QuantizerFunction(torch.autograd.Function):
    """Fake-quantise in forward, straight-through in backward (reference :77-89)."""

    @staticmethod
    def forward(ctx, X, quant):
        assert X.is_floating_point()
        return quant(X.data.float()).to(X.dtype)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None


class Quantizer(nn.Module):
    """Observer-shaped fake-quant module (standalone use; the fused engine does not call it)."""

    def __init__(self, number_format):
        super().__init__()
        self._number_format = number_format
        self._quant = NumberFormat.quantizer(number_format)

    def get_qparams(self):
        raise NotImplementedError()

    def forward(self, X):
        return QuantizerFunction.apply(X, self._quant)

    def forward_pre_hook(self, module, input):
        assert len(input) == 1, f"{self.__class__.__name__} only supports single tensor input"
        return self(input[0])

    def __repr__(self):
        return self.__class__.__name__ + f"({self._number_format})"


# (exp, man) of the float formats the engine understands; None = identity
_FLOAT_FMT = {
    NumberFormat.HalfPrecisionFloat: (5, 10),
    NumberFormat.TensorFloat32: (8, 10),
    NumberFormat.SinglePrecisionFloat: None,
}

# Where quantisers sit (SURVEY.md Appendix A):
#   inp : QuantStub in front of every Linear / LayerNorm, and every Linear weight
#   out : output observer of Linear / LayerNorm
#   ff  : FloatFunctional outputs (residual adds, cls/pos cat and add)
#   gelu: QuantStub in front of GELU
#   grad: gradient format of the `inp` quantisers (QPyTorch's backward_number; None = straight-through, the only
#         thing the reference configures, utils/quantize.py:47-72 — see ModelQuantizer.prepare_qat)
#   grad_rounding: QPyTorch's backward_rounding of those quantisers, "nearest" or "stochastic"
QuantPlan = namedtuple("QuantPlan", ["inp", "out", "ff", "gelu", "grad", "grad_rounding"], defaults=[None, "nearest"])
GRAD_ROUNDINGS = ("nearest", "stochastic")

_PLANS = {
    QFormat.FP32: QuantPlan(None, None, None, None),
    QFormat.FP16_32: QuantPlan((5, 10), None, None, None),
    QFormat.TF32: QuantPlan((8, 10), None, None, None),
    QFormat.FP16_16: QuantPlan((5, 10), (5, 10), (5, 10), (5, 10)),
}


class QuantStubSlot(nn.Module):
    """Parameter-free placeholder occupying index 0 of a wrapped Sequential, so that wrapped
    modules keep the reference's `<name>.1.<param>` state_dict keys."""

    def __init__(self, fmt):
        super().__init__()
        self.fmt = fmt

    def forward(self, x):
        if self.fmt is None:
            return x
        return Quantizer(NumberFormat.HalfPrecisionFloat if self.fmt == (5, 10)
                         else NumberFormat.TensorFloat32)(x)

    def extra_repr(self):
        return "fmt={}".format(self.fmt)


class QLinear(nn.Linear):
    """Linear holding a pre-quantised weight (result of ModelQuantizer.convert)."""

    def __init__(self, *args, activation_post_process=None, **kwargs):
        super().__init__(*args, **kwargs)
        self.activation_post_process = activation_post_process


class QLayerNorm(nn.LayerNorm):
    """LayerNorm holding a pre-quantised gamma (result of ModelQuantizer.convert)."""


class ModelQuantizer:
    def __init__(self, model):
        self.model = model

    def prepare_qat(self, q_format, backward_format=None, backward_rounding="nearest"):
        """Make the model simulate `q_format`.

        backward_format (extension; the reference builds every QPyTorch quantiser without a backward_number):
        (exp_bits, man_bits) of a float format that every input / weight quantiser of the plan also applies, with
        nearest rounding, to the gradient flowing back through it — qtorch.quant.Quantizer(forward_number,
        backward_number) at the QuantStubs in front of Linear / LayerNorm and at the weight fake-quant.  The
        quantiser sees the gradient as autograd presents it (loss scaling is the caller's, as with the reference's
        GradScaler): the engine's own power-of-two operand scale is switched off.  FP16_32 only.

        backward_rounding: QPyTorch's backward_rounding of those quantisers.  "stochastic" (QPyTorch's default) rounds
        every gradient-quantiser site with the Philox stream of include/mv_b200.h ("gradient rounding stream") under a
        seed drawn per training forward; "nearest" (the default here) rounds to nearest.  No effect without
        backward_format."""
        if backward_rounding not in GRAD_ROUNDINGS:
            raise ValueError("backward_rounding must be one of %s, got %r" % (GRAD_ROUNDINGS, backward_rounding))
        if hasattr(self, "q_format") and self.q_format != QFormat.FP32:
            raise ValueError("model already quantized")
        if isinstance(q_format, str):
            q_format = QFormat[q_format]
        if q_format == QFormat.PyTorchINT8:
            raise NotImplementedError(
                "PyTorchINT8 is torch's CPU-only int8 path, outside the B200 hot path")
        if q_format not in _PLANS:
            raise NotImplementedError(f"unknown q_format={q_format}")
        plan = _PLANS[q_format]
        if backward_format is not None:
            if q_format != QFormat.FP16_32:
                raise NotImplementedError("backward_format is implemented for q_format=FP16_32 (quantisers in front of "
                                          "Linear / LayerNorm and on the weights); got %s" % (q_format,))
            e, m = (int(v) for v in backward_format)
            if not (2 <= e <= 8 and 1 <= m <= 22):
                raise ValueError("backward_format must be (exp_bits in 2..8, man_bits in 1..22)")
            plan = plan._replace(grad=(e, m), grad_rounding=backward_rounding)
        if q_format != QFormat.FP32:
            self._wrap_modules(plan)
        self.plan = plan
        self.q_format = q_format
        self.converted = False
        if hasattr(self.model, "_invalidate_engine"):
            self.model._invalidate_engine()

    def _wrap_modules(self, plan):
        targets = []
        for name, module in self.model.named_modules():
            if isinstance(module, (nn.Linear, nn.LayerNorm)):
                targets.append((name, module, plan.inp))
            elif isinstance(module, nn.GELU) and plan.gelu is not None:
                targets.append((name, module, plan.gelu))
        for name, module, fmt in targets:
            parent = self.model
            parts = name.split(".")
            for part in parts[:-1]:
                parent = getattr(parent, part)
            setattr(parent, parts[-1], nn.Sequential(QuantStubSlot(fmt), module))

    def convert(self):
        """PTQ conversion for inference (reference :329-348, flow of classification/test_quantize.py:37-134).
        `torch.quantization.convert(mapping={qat.Linear: QLinear, LayerNorm: QLayerNorm})` does two things in the
        reference, both pinned by tests/golden/convert_*.npz (oracle/make_golden_convert.py runs it unmodified):
          * Linear weights and LayerNorm gammas are replaced by their fake-quantised values
            (QLinear.from_float / QLayerNorm.from_float, :134-166);
          * every hook-based quantiser disappears with its observer hook — the QuantStub in front of each
            Linear / LayerNorm / GELU and the Linear / LayerNorm output observers — while the FloatFunctional
            quantisers (FP16_16's residual adds and cat / pos adds), which are called inside FloatFunctional's
            own forward, stay.
        So the converted model computes in fp32 on quantised weights; the plan below says exactly that and the
        engine runs it on its fp32-grade (3xTF32) path."""
        if self.q_format == QFormat.FP32 or getattr(self, "converted", False):
            return
        fmt = self.plan.inp
        import mv_native
        with torch.no_grad():
            for module in self.model.modules():
                if isinstance(module, (nn.Linear, nn.LayerNorm)) and module.weight.is_cuda:
                    module.weight.copy_(mv_native.float_quantize(module.weight.data, fmt[0], fmt[1]))
                elif isinstance(module, (nn.Linear, nn.LayerNorm)):
                    raise RuntimeError("convert() needs the model on a CUDA device")
        self.plan = QuantPlan(None, None, self.plan.ff, None)
        self.converted = True
        if hasattr(self.model, "_invalidate_engine"):
            self.model._invalidate_engine()
