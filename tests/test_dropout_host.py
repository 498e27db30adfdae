"""Host side of dropout (no GPU): the probability checks, the (thr, scale) of the declared mask stream, the masks and
the training step of the CPU dropout reference (tests/dropout_oracle.py), and the ABI struct the GEMM's dropout fields
travel in."""
import numpy as np
import pytest
import torch

import dropout_oracle
from oracle import quant_oracle, vit_oracle
from oracle.golden_cases import ARCH, CASES, make_inputs


def test_probability_range_and_stream_parameters():
    import mv_native as mv
    import mv_engine
    assert mv.drop_params(0.0) == (0, 1.0)
    assert mv.drop_params(1.0) == (65536, 0.0)
    thr, scale = mv.drop_params(0.1)
    assert thr == 6554 and scale == float(np.float32(1.0) / np.float32(0.9))
    assert abs(thr / 65536 - 0.1) <= 2.0 ** -17
    for bad in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            mv.drop_params(bad)
        with pytest.raises(ValueError):
            mv_engine.EngineConfig(128, 2, 256, 2, 16, None, dropout=bad)


def test_gemm_args_end_with_the_dropout_and_rounding_fields():
    import mv_native as mv
    names = [f[0] for f in mv.GemmArgs._fields_]
    assert names[-6:] == ["drop_seed", "drop_thr", "drop_scale", "drop_site", "round_seed", "round_offset"]
    assert mv.GemmArgs().drop_seed is None                      # zero-initialised: off
    assert mv.GemmArgs().round_seed is None                     # zero-initialised: nearest


def test_oracle_mask_is_the_declared_stream():
    seed, site = 0xDEADBEEF12345678, 7
    m = dropout_oracle.dropout_mask((5, 24), 0.25, seed, site).flatten().numpy()
    bits = quant_oracle.philox_bits(120, seed, site, half=True)
    scale = np.float32(1.0) / np.float32(0.75)
    assert np.array_equal(m, np.where(bits >= 16384, scale, np.float32(0.0)).astype(np.float32))
    # negative int64 seeds (what a device int64 holds) mean their two's-complement 64 bits
    assert torch.equal(dropout_oracle.dropout_mask((3, 8), 0.5, -1, 1), dropout_oracle.dropout_mask((3, 8), 0.5, 2 ** 64 - 1, 1))
    assert not dropout_oracle.dropout_mask((64,), 1.0, 3, 0).any()
    assert bool((dropout_oracle.dropout_mask((64,), 0.0, 3, 0) == 1).all())


def test_reference_step_with_dropout():
    """At p = 0 the dropout reference is vit_oracle's step bit for bit; p > 0 changes the result as a pure function of
    the seed, and p = 1 on the blocks leaves nothing of their branches (zero gradients for their Linears)."""
    case = CASES["classification"]
    P = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], seed=4, **{
        k: ARCH[k] for k in ("dim", "depth", "heads", "mlp_dim")})
    img, tgt = make_inputs("classification", case, 5)
    kw = dict(decoder="classification", heads=ARCH["heads"], q_format="FP16_32")
    o0, l0, g0 = vit_oracle.train_step(P, img, tgt, **kw)
    o1, l1, g1 = dropout_oracle.train_step(P, img, tgt, dropout=(0.0, 0.0, 9), **kw)
    assert torch.equal(o0, o1) and torch.equal(l0, l1)
    assert all(torch.equal(g0[k], g1[k]) for k in g0 if g0[k] is not None)
    o2, _, _ = dropout_oracle.train_step(P, img, tgt, dropout=(0.1, 0.1, 9), **kw)
    assert not torch.equal(o0, o2)
    o3, _, _ = dropout_oracle.train_step(P, img, tgt, dropout=(0.1, 0.1, 9), **kw)
    assert torch.equal(o2, o3)
    _, _, g4 = dropout_oracle.train_step(P, img, tgt, dropout=(1.0, 0.0, 9), **kw)
    assert float(g4["transformer.layers.0.1.fn.fn.net.3.weight"].abs().max()) == 0.0
    assert float(g4["transformer.layers.1.0.fn.fn.to_qkv.weight"].abs().max()) == 0.0


def test_model_accepts_dropout_and_checks_it():
    from myrtle_vision.models.vit import ViT
    m = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2,
            mlp_dim=256, dropout=0.1, emb_dropout=0.1)
    assert (m.dropout_p, m.emb_dropout_p) == (0.1, 0.1)
    with pytest.raises(ValueError):
        ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2,
            mlp_dim=256, dropout=1.5)
