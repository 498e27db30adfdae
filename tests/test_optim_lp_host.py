"""qtorch.optim.OptimLP without a GPU: the C ABI mirrors, quantiser recognition, the rounding-stream offsets and the
trainer's optim_lp config."""
import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_fields(struct):
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\} %s;" % struct, text).group(1)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        first, *rest = decl.split(",")
        names += [re.findall(r"\w+", first)[-1]] + [r.strip() for r in rest]
    return names


@pytest.mark.parametrize("struct,cls", [("mv_adamw_lp_tensor", "AdamwLpTensor"), ("mv_lp_quant", "LpQuant"),
                                        ("mv_optim_lp", "OptimLpSpec")])
def test_ctypes_structs_mirror_the_header(struct, cls):
    from myrtle_vision.utils import fused_adamw
    assert [f[0] for f in getattr(fused_adamw, cls)._fields_] == declared_fields(struct)


def test_header_declares_the_entry_point_and_version():
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    assert re.search(r"int mv_adamw_lp_step\(const mv_adamw_tensor\* tensors_dev, const mv_adamw_lp_tensor\* lp_dev,",
                     text)
    api = open(os.path.join(ROOT, "myrtle-vision_b200", "csrc", "api.cu")).read()
    assert "return 105;" in api


def test_import_and_qtorch_signature():
    import qtorch.optim
    from qtorch.optim import OptimLP
    params = list(inspect.signature(OptimLP).parameters.values())
    assert [p.name for p in params[:6]] == ["optim", "weight_quant", "grad_scaling", "grad_quant", "momentum_quant",
                                            "acc_quant"]
    assert all(p.kind == p.POSITIONAL_OR_KEYWORD for p in params[:6])
    assert params[2].default == 1.0 and all(p.default is None for p in params[1:6] if p.name != "grad_scaling")
    assert {p.name for p in params[6:]} == {"seed", "fused"} and all(p.kind == p.KEYWORD_ONLY for p in params[6:])
    assert qtorch.optim.OptimLP is OptimLP


def test_quantiser_recognition():
    from qtorch import BlockFloatingPoint, FixedPoint, FloatingPoint
    from qtorch.optim import lp_format
    from qtorch.quant import Quantizer, quantizer
    assert lp_format(None) is None
    assert lp_format(quantizer(FloatingPoint(8, 7), forward_rounding="stochastic")) == ("float", 8, 7, "stochastic")
    assert lp_format(quantizer(FloatingPoint(5, 2), forward_rounding="nearest")) == ("float", 5, 2, "nearest")
    assert lp_format(quantizer(FixedPoint(11, 9))) == ("fixed", 11, 9, True, False, "stochastic")
    assert lp_format(Quantizer(FixedPoint(8, 4, clamp=False, symmetric=True), forward_rounding="nearest")) == \
        ("fixed", 8, 4, False, True, "nearest")
    assert lp_format(Quantizer(FloatingPoint(4, 3))) == ("float", 4, 3, "stochastic")
    assert lp_format(quantizer(BlockFloatingPoint(8))) == "callable"
    assert lp_format(quantizer(None)) == "callable"
    assert lp_format(lambda t: t) == "callable"
    q = quantizer(FloatingPoint(5, 10), forward_rounding="nearest")
    assert q.forward_number.exp == 5 and q.forward_rounding == "nearest"


def test_offsets():
    from qtorch.optim import lp_offset
    assert lp_offset(1, 0, 4) == (1 << 32) | 4
    assert lp_offset(3, 5, 2) == (3 << 32) | (5 << 3) | 2
    assert lp_offset(2 ** 24 - 1, 2 ** 29 - 1, 0) == ((2 ** 24 - 1) << 32) | ((2 ** 29 - 1) << 3)
    seen = {lp_offset(s, k, site) for s in range(1, 4) for k in range(40) for site in range(5)}
    assert len(seen) == 3 * 40 * 5


def test_cpu_parameters_raise():
    import mv_native
    from qtorch import FloatingPoint
    from qtorch.optim import OptimLP
    from qtorch.quant import quantizer
    p = torch.nn.Parameter(torch.zeros(4))
    with pytest.raises(mv_native.MvError, match="no CPU fallback"):
        OptimLP(torch.optim.SGD([p], lr=0.1), weight_quant=quantizer(FloatingPoint(8, 7)))
    with pytest.raises(mv_native.MvError, match="no CPU fallback"):
        OptimLP(torch.optim.AdamW([p], lr=0.1))


def test_momentum_quant_needs_a_known_optimizer():
    from qtorch import FloatingPoint
    from qtorch.optim import OptimLP
    from qtorch.quant import quantizer
    p = torch.nn.Parameter(torch.zeros(4))
    with pytest.raises(NotImplementedError, match="momentum_quant"):
        OptimLP(torch.optim.RMSprop([p], lr=0.1), momentum_quant=quantizer(FloatingPoint(8, 7)))


class _Opt:
    param_groups = [{"params": []}]


@pytest.mark.parametrize("cfg,match", [
    ({"weight_quant": None, "bogus": 1}, "unknown keys"),
    ({"weight_quant": {"float": [8, 7], "round": "nearest"}}, "unknown keys"),
    ({"weight_quant": {"float": [8, 7], "clamp": True}}, "unknown keys"),
    ({"grad_quant": {"float": [9, 7]}}, "exp in 1..8"),
    ({"grad_quant": {"float": [5, 23]}}, "man in 1..22"),
    ({"grad_quant": {"float": [5]}}, "two integers"),
    ({"acc_quant": {"fixed": [0, 4]}}, "wl in 1..32"),
    ({"acc_quant": {"fixed": [8, 0]}}, "fl in 1..100"),
    ({"acc_quant": {"float": [5, 2], "fixed": [8, 4]}}, "exactly one"),
    ({"acc_quant": {}}, "exactly one"),
    ({"momentum_quant": {"float": [5, 2], "rounding": "up"}}, "rounding"),
    ({"momentum_quant": [5, 2]}, "expected null or an object"),
    ({"grad_scaling": 0}, "grad_scaling"),
    ({"seed": -1}, "seed"),
    ([1, 2], "expected an object"),
])
def test_trainer_config_validation(cfg, match):
    from myrtle_vision.utils.optim import wrap_optim_lp
    with pytest.raises(ValueError, match=match):
        wrap_optim_lp(_Opt(), cfg)


def test_trainer_config_builds_recognised_quantisers(monkeypatch):
    import qtorch.optim
    from myrtle_vision.utils.optim import wrap_optim_lp
    seen = {}

    class Fake:
        def __init__(self, optim, **kw):
            seen.update(kw)

    monkeypatch.setattr(qtorch.optim, "OptimLP", Fake)
    wrap_optim_lp(_Opt(), {"weight_quant": {"float": [8, 7]}, "grad_quant": {"float": [5, 2], "rounding": "nearest"},
                           "acc_quant": {"fixed": [16, 12], "clamp": False, "symmetric": True}, "seed": 7,
                           "grad_scaling": 2})
    lp = qtorch.optim.lp_format
    assert lp(seen["weight_quant"]) == ("float", 8, 7, "stochastic")
    assert lp(seen["grad_quant"]) == ("float", 5, 2, "nearest")
    assert lp(seen["acc_quant"]) == ("fixed", 16, 12, False, True, "stochastic")
    assert seen["momentum_quant"] is None and seen["seed"] == 7 and seen["grad_scaling"] == 2.0
