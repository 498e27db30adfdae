"""Host side of stochastic gradient rounding (no GPU): argument validation, QuantPlan defaults, the decoder's site
table, the stream offsets with rank bits and the CPU reference (tests/grad_round_oracle.py)."""
import numpy as np
import pytest
import torch

import grad_round_oracle
from oracle import quant_oracle, vit_oracle
from oracle.golden_cases import ARCH, CASES, make_inputs


def _vit(decoder="classification", **kw):
    from myrtle_vision.models.vit import ViT
    return ViT(decoder=decoder, image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2, mlp_dim=256,
               num_det_tokens=4, **kw)


def test_backward_rounding_is_validated_and_recorded():
    from myrtle_vision.utils.quantize import QuantPlan
    m = _vit(q_format="FP16_32", backward_format=(5, 2), backward_rounding="stochastic")
    assert m.quantizer.plan.grad == (5, 2) and m.quantizer.plan.grad_rounding == "stochastic"
    assert _vit(q_format="FP16_32", backward_format=(5, 2)).quantizer.plan.grad_rounding == "nearest"
    # without a gradient format the argument changes nothing, as in QPyTorch
    plain = _vit(q_format="FP16_32", backward_rounding="stochastic").quantizer.plan
    assert plain == _vit(q_format="FP16_32").quantizer.plan and plain.grad_rounding == "nearest"
    for bad in ("Stochastic", "round", "", None, 1):
        with pytest.raises(ValueError):
            _vit(q_format="FP16_32", backward_format=(5, 2), backward_rounding=bad)
    with pytest.raises(NotImplementedError):
        _vit(q_format="TF32", backward_format=(5, 2), backward_rounding="stochastic")
    # every existing QuantPlan(...) construction keeps its meaning
    assert QuantPlan((5, 10), None, None, None).grad_rounding == "nearest"
    assert QuantPlan((5, 10), None, None, None, (5, 2)) == ((5, 10), None, None, None, (5, 2), "nearest")


def test_engine_switch_follows_the_plan():
    import mv_engine
    from myrtle_vision.utils.quantize import QuantPlan
    params = [torch.zeros(1) for _ in range(2 + mv_engine.PER_LAYER)]

    def engine(plan):
        cfg = mv_engine.EngineConfig(128, 2, 256, 1, 16, plan)
        return mv_engine.EncoderEngine(cfg, params)
    e = engine(QuantPlan((5, 10), None, None, None, (5, 2), "stochastic"))
    assert e.grad_round and e.rank == 0 and e.last_grad_round_seed is None and e.fixed_grad_round_seed is None
    assert not engine(QuantPlan((5, 10), None, None, None, (5, 2))).grad_round
    assert not engine(QuantPlan((5, 10), None, None, None, None, "stochastic")).grad_round
    # no draw without a backward to follow, or with the mode off: torch's generator is left alone
    assert e._draw_grad_round(False) is None


@pytest.mark.parametrize("decoder,names", [
    ("classification", ["norm in", "linear in", "linear w"]),
    ("segmentation", ["norm in", "linear in", "linear w"]),
    ("detection", ["class_embed in", "class_embed w", "bbox_embed in", "bbox_embed w"]),
])
def test_decoder_sites_follow_its_forward(decoder, names, monkeypatch):
    """The decoder's stubs take sites 10 depth + 1 + j in the order its forward applies them (LayerNorm input first,
    then input and weight of each Linear), each with the rank in the high word."""
    import myrtle_vision.models.vit as vit
    m = _vit(decoder, q_format="FP16_32", backward_format=(5, 2), backward_rounding="stochastic")
    seen = []

    def fake_fq(x, fmt, gfmt=None):
        if gfmt is not None:
            seen.append((tuple(x.shape), gfmt))
        return x
    monkeypatch.setattr(vit, "_fq", fake_fq)

    class Eng:
        rank = 3
    seed = torch.tensor([12345], dtype=torch.int64)
    m._engine, m._grad_round_seed = Eng(), seed
    m.train()
    x = torch.randn(2, 26, 128)
    m._decode(x, (80, 80))
    lin = None if decoder == "detection" else m.decoder.linear
    assert len(seen) == len(names)
    for j, ((shape, g), name) in enumerate(zip(seen, names)):
        assert g[:2] == (5, 2) and g[2] is seed
        assert g[3] == 10 * 2 + 1 + j + (3 << 32), name
        if name.endswith(" w"):
            assert len(shape) == 2 and shape[1] == 128
    if lin is not None:
        assert seen[2][0] == tuple(vit._unwrap(lin).weight.shape)
    # nearest rounding, or no seed drawn: the plain gradient format
    m._grad_round_seed = None
    seen.clear()
    m._decode(x, (80, 80))
    assert all(g == (5, 2) for _, g in seen)


def test_offsets_carry_the_rank_in_the_high_word():
    import mv_engine
    assert mv_engine.grad_round_offset(7) == 7
    assert mv_engine.grad_round_offset(7, 1) == 7 + 2 ** 32
    assert mv_engine.grad_round_offset(10 * 12 + 3, 5) == (5 << 32) | 123
    seed = 0x0123456789ABCDEF
    for man, half in ((2, False), (3, False), (7, True), (10, True)):
        bits = grad_round_oracle.round_bits(40, 5, man, seed, mv_engine.grad_round_offset(9, 2))
        assert np.array_equal(bits, quant_oracle.philox_bits(40, seed, 9 + (2 << 32), half=half))
        other = quant_oracle.philox_bits(40, seed, 9 + (1 << 32), half=half)
        assert not np.array_equal(bits, other)          # ranks draw different bits for the same site


def test_oracle_rounding_is_the_stream_and_is_unbiased():
    seed, off = -5, 17
    g = torch.linspace(-3.0, 3.0, 1000)
    for e, m in ((5, 2), (4, 3), (5, 7), (5, 10)):
        q = grad_round_oracle.stochastic_round(g, e, m, seed, off)
        bits = quant_oracle.philox_bits(1000, seed & (2 ** 64 - 1), off, half=m >= 7)
        ref = quant_oracle.float_quantize(g.numpy(), e, m, rounding="stochastic", rbits=bits)
        assert np.array_equal(q.numpy(), ref)
        assert torch.equal(vit_oracle._fq_np(q, e, m), q)              # on the grid
    # E[q(x)] = x: mean over seeds of one value between two E5M2 grid points
    x = torch.full((4096,), 1.1)
    means = torch.stack([grad_round_oracle.stochastic_round(x, 5, 2, s, 0) for s in range(8)]).mean()
    assert abs(float(means) - 1.1) < 0.01


def test_oracle_step_rounds_weight_gradients_onto_the_grid():
    case = CASES["classification"]
    arch = dict(ARCH, depth=1)
    P = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], dim=arch["dim"],
                               depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], seed=5)
    img, tgt = make_inputs("classification", case, 5)
    img, tgt = img[:2], tgt[:2]
    kw = dict(decoder="classification", heads=arch["heads"], grad_format=(5, 2), loss_scale=65536.0)
    _, _, g1 = grad_round_oracle.train_step(P, img, tgt, seed=1, **kw)
    _, _, g1b = grad_round_oracle.train_step(P, img, tgt, seed=1, **kw)
    _, _, g2 = grad_round_oracle.train_step(P, img, tgt, seed=2, **kw)
    w = "transformer.layers.0.1.fn.fn.net.0.weight"
    assert torch.equal(g1[w], g1b[w]) and not torch.equal(g1[w], g2[w])
    for k, v in g1.items():
        if k.endswith(".weight") and v is not None and v.dim() == 2:
            assert torch.equal(vit_oracle._fq_np(v, 5, 2), v), k
