"""Stochastic rounding of the gradient quantiser (ViT(backward_format=..., backward_rounding="stochastic")) on the fused
path: the device-seed quantiser against mv_float_quantize, each fused site (dgrad GEMM epilogues, LayerNorm backward)
against the unfused value passed through that quantiser, unbiasedness, the model step against the CPU reference
(tests/grad_round_oracle.py), and seeds across steps, CUDA-graph replays and data-parallel ranks.  Formats (5, 2) and
(4, 3) take the 32-bit stream, (5, 7) and (5, 10) the 16-bit one."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import grad_round_oracle
import dropout_oracle
from oracle import vit_oracle
from oracle.golden_cases import ARCH, CASES, make_inputs

pytestmark = pytest.mark.gpu
dev = "cuda"
FORMATS = [(5, 2), (4, 3), (5, 7), (5, 10)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# repeated steps agree up to the summation order of the split-K / column-sum / dQ red.adds, which varies from run to run;
# a rounding whose input moved by an ulp across a threshold flips by a whole step, so the bar is relative L2 (two seeds
# differ by 10 % and more on E5M2)
REPEAT_TOL = 5e-3


def seed_tensor(s):
    return torch.tensor([s], dtype=torch.int64, device=dev)


# ------------------------------------------------------------------------------------------- device-seed quantiser
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("n", [1, 7, 1003, 65541])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_device_seed_quantiser_equals_host_seed(fmt, n, out_dtype):
    import mv_native as mv
    torch.manual_seed(n)
    x = torch.randn(n + 1, device=dev) * 3
    x[::97] = 0.0
    x[5::101] *= 1e-6                                    # below the lowest normal binade of the small formats
    for seed, offset in ((0x0123456789ABCDEF, 3), (-7, 5 + (1 << 32)), (42, 123 + (7 << 32))):
        for src in (x[:n], x[1:]):                       # aligned and unaligned (the scalar kernels)
            ref = mv.float_quantize(src, fmt[0], fmt[1], "stochastic", seed=seed & (2 ** 64 - 1), offset=offset,
                                    out_dtype=out_dtype)
            got = mv.float_quantize_dev(src, fmt[0], fmt[1], (seed_tensor(seed), offset), out_dtype=out_dtype)
            assert torch.equal(got.view(torch.int16 if out_dtype == torch.float16 else torch.int32),
                               ref.view(torch.int16 if out_dtype == torch.float16 else torch.int32))


# ---------------------------------------------------------------------------------------------------- GEMM sites
def _operands(M, N, K, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    A = (torch.randn(M, K, device=dev, generator=g) * 0.5).half()
    B = (torch.randn(N, K, device=dev, generator=g) * 0.5).half()
    return A, B


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("M,N,K,tile_n", [(514, 384, 384, 0),       # ragged M (2 x 257 tokens), compile-time epilogue
                                          (514, 100, 384, 0),       # N % 8 != 0: the generic epilogue
                                          (16448, 384, 1536, 192),  # 65 x 2 tiles: tiles late in a CTA's walk
                                          (16448, 1536, 384, 256)])
def test_plain_dgrad_site(fmt, M, N, K, tile_n):
    import mv_native as mv
    A, B = _operands(M, N, K, M + N)
    ref32 = torch.empty(M, N, device=dev)
    mv.gemm(A, B, ref32, tile_n=tile_n)
    for seed, offset in ((11, 3), (-2, 7 + (3 << 32))):
        gr = (seed_tensor(seed), offset)
        out = torch.empty(M, N, dtype=torch.float16, device=dev)
        mv.gemm(A, B, out, q_out=fmt, tile_n=tile_n, grad_round=gr, tag="dgrad")
        want = mv.float_quantize_dev(ref32, fmt[0], fmt[1], gr, out_dtype=torch.float16)
        assert torch.equal(out.view(torch.int16), want.view(torch.int16)), (seed, offset)
    # a different seed or rank rounds differently
    o2 = torch.empty(M, N, dtype=torch.float16, device=dev)
    mv.gemm(A, B, o2, q_out=fmt, tile_n=tile_n, grad_round=(seed_tensor(11), 3 + (1 << 32)), tag="dgrad")
    assert not torch.equal(o2, out)


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("colsum", [True, False])
@pytest.mark.parametrize("M,N,tile_n", [(514, 1536, 0), (16448, 1536, 0),   # 256-wide tiles, aux by TMA
                                        (514, 100, 0),                      # N % 8 != 0
                                        (16448, 384, 0),                    # mlp_dim 384: 192-wide tiles, no aux TMA
                                        (16448, 1536, 128)])                # forced narrow tiles
def test_gelu_dgrad_site(fmt, colsum, M, N, tile_n):
    """fc2's input stub: q_out rounds before the gelu' multiply; colsum sums the stored (fp32) values."""
    import mv_native as mv
    K = 384
    A, B = _operands(M, N, K, 5 * M + N)
    aux = (torch.rand(M, N, device=dev) * 1.1).half()
    ref32 = torch.empty(M, N, device=dev)
    mv.gemm(A, B, ref32, tile_n=tile_n)
    gr = (seed_tensor(1234), 8 + (2 << 32))
    out = torch.empty(M, N, dtype=torch.float16, device=dev)
    cs = torch.zeros(N, device=dev) if colsum else None
    mv.gemm(A, B, out, aux=aux, epilogue=mv.EPI_DGELU, colsum=cs, q_out=fmt, grad_round=gr, tile_n=tile_n)
    q = mv.float_quantize_dev(ref32, fmt[0], fmt[1], gr) * aux.float()
    assert torch.equal(out.view(torch.int16), q.half().view(torch.int16))
    if colsum:
        want = q.double().sum(0)
        assert float((cs.double() - want).abs().max()) <= 1e-5 * float(want.abs().max())


def test_fused_site_raises_the_overflow_flag_on_saturation():
    import mv_native as mv
    M, N, K = 514, 384, 384
    A, B = _operands(M, N, K, 9)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    out = torch.empty(M, N, dtype=torch.float16, device=dev)
    mv.set_overflow_flag(flag)
    try:
        mv.gemm(A, B, out, q_out=(5, 2), grad_round=(seed_tensor(1), 0), tag="dgrad")
        torch.cuda.synchronize()
        assert int(flag) == 0
        mv.gemm((A.float() * 4096).half(), B, out, q_out=(5, 2), grad_round=(seed_tensor(1), 0), tag="dgrad")
        torch.cuda.synchronize()
        assert int(flag) == 1                      # values beyond fp16 saturate (to E5M2's 57344) and report
    finally:
        mv.set_overflow_flag(None)


# ------------------------------------------------------------------------------------- LayerNorm backward site
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("D", [384, 200])
@pytest.mark.parametrize("dropout", [False, True])
def test_layernorm_backward_site_with_q_grad(fmt, D, dropout):
    """The LN-input stub rounds LN'(dy) before dres is added: dx = q(LN'(dy)) + dres, dx_f16 its (masked) copy."""
    import mv_native as mv
    torch.manual_seed(D)
    rows = 2056
    x = torch.randn(rows, D, device=dev) * 2
    g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    _, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    dy = torch.randn(rows, D, device=dev).half(); dres = torch.randn(rows, D, device=dev)
    ln, _ = mv.layernorm_q_bwd(dy, x, g, mean, rstd, q_in=(5, 10), want_f16=False)       # unrounded, no dres
    gr = (seed_tensor(77), 5 + (1 << 32))
    q = mv.float_quantize_dev(ln, fmt[0], fmt[1], gr)
    drop = (seed_tensor(55), 0.1, 9) if dropout else None
    bp = torch.zeros(D, device=dev)
    dx, h = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dbias_prev=bp, q_grad=fmt, drop=drop,
                               grad_round=gr)
    want = q + dres
    assert torch.equal(dx, want)
    m = dropout_oracle.dropout_mask((rows, D), 0.1, 55, 9).to(dev) if dropout else torch.ones_like(want)
    assert torch.equal(h, (want * m).half())
    ws = (want.double() * m.double()).sum(0)
    assert float((bp.double() - ws).abs().max()) <= 1e-5 * float(ws.abs().max())


def test_a_failed_backward_leaves_no_gradient_format_behind(monkeypatch):
    """The gradient format is an argument of each LayerNorm-backward call, not process state: after a backward with
    backward_format raises part-way, a LayerNorm backward without q_grad, on fp32 dy, runs and is unrounded."""
    import mv_native as mv
    case = CASES["classification"]
    m, _ = build(case, 3, rounding="nearest")
    img, tgt = make_inputs("classification", case, 3)
    loss = F.cross_entropy(m(img.to(dev)), tgt.to(dev)) * 65536.0
    gemm, calls = mv.gemm, []

    def failing_gemm(*args, **kwargs):
        calls.append(kwargs.get("tag"))
        if len(calls) == 5:                              # to_out's dgrad: after the last block's LN2 backward
            raise mv.MvError("injected failure")
        return gemm(*args, **kwargs)

    monkeypatch.setattr(mv, "gemm", failing_gemm)
    with pytest.raises(mv.MvError, match="injected failure"):
        loss.backward()
    monkeypatch.undo()
    assert len(calls) == 5
    torch.manual_seed(4)
    rows, D = 1003, 192
    x = torch.randn(rows, D, device=dev) * 2
    g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    _, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    dy = torch.randn(rows, D, device=dev)
    dx, _ = mv.layernorm_q_bwd(dy, x, g, mean, rstd, q_in=(5, 10), want_f16=False)
    xr = mv.float_quantize(x, 5, 10).double().requires_grad_(True)
    F.layer_norm(xr, (D,), g.double(), b.double(), 1e-5).backward(dy.double())
    assert float((dx.double() - xr.grad).abs().max()) <= 1e-6 * float(xr.grad.abs().max())


# ------------------------------------------------------------------------------------------------ unbiasedness
def test_fused_dgrad_is_unbiased():
    """Mean over 256 seeds of each element within a quarter step of the fp32 value (Hoeffding: a false failure below
    2 exp(-32) per element)."""
    import mv_native as mv
    M, N, K = 256, 384, 128
    A, B = _operands(M, N, K, 3)
    ref32 = torch.empty(M, N, device=dev)
    mv.gemm(A, B, ref32)
    for fmt in ((5, 2), (5, 7)):
        acc = torch.zeros(M, N, dtype=torch.float64, device=dev)
        out = torch.empty(M, N, dtype=torch.float16, device=dev)
        for s in range(256):
            mv.gemm(A, B, out, q_out=fmt, grad_round=(seed_tensor(1000 + s), 1), tag="dgrad")
            acc += out.double()
        mean = acc / 256
        e = torch.floor(torch.log2(ref32.abs().clamp_min(2.0 ** -14))).clamp_min(-14)
        step = torch.exp2(e - fmt[1]).double()
        assert bool(((mean - ref32.double()).abs() <= 0.25 * step).all()), fmt
        near = torch.empty(M, N, dtype=torch.float16, device=dev)
        mv.gemm(A, B, near, q_out=fmt, tag="dgrad")
        assert float((mean - ref32.double()).abs().mean()) < float((near.double() - ref32.double()).abs().mean())


# ------------------------------------------------------------------------------------------------------- model
def build(case, seed, rounding="stochastic", dropout=0.0, gfmt=(5, 2)):
    from myrtle_vision.models.vit import ViT
    m = ViT(decoder="classification", image_size=case["image_size"], patch_size=16, num_classes=case["num_classes"],
            dim=ARCH["dim"], depth=ARCH["depth"], heads=ARCH["heads"], mlp_dim=ARCH["mlp_dim"], q_format="FP16_32",
            backward_format=gfmt, backward_rounding=rounding, dropout=dropout, emb_dropout=dropout)
    P = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], dim=ARCH["dim"],
                               depth=ARCH["depth"], heads=ARCH["heads"], mlp_dim=ARCH["mlp_dim"], seed=seed)
    m.load_state_dict({k: P[vit_oracle.canonical_key(k)] for k in m.state_dict()})
    return m.to(dev).train(), P


def _grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_model_step_matches_the_oracle(p_drop):
    """E5M2 gradients, loss x 65536 (the reference's GradScaler), the seed fixed: every parameter's error below 0.75 of
    the oracle's distance to the straight-through backward (the bar of tests/test_gpu_model.py's nearest test), Linear
    weight gradients on the E5M2 grid, and not the nearest-rounding result."""
    import mv_native as mv
    gfmt, scale, gseed = (5, 2), 65536.0, 0x5EED1234
    case = CASES["classification"]
    m, P = build(case, 77, dropout=p_drop)
    eng = m.engine()
    eng.fixed_grad_round_seed = seed_tensor(gseed)
    if p_drop:
        eng.fixed_dropout_seed = seed_tensor(99)
    img, tgt = make_inputs("classification", case, 77)
    out = m(img.to(dev))
    (F.cross_entropy(out, tgt.to(dev)) * scale).backward()
    assert int(eng.last_grad_round_seed.item()) == gseed
    kw = dict(decoder="classification", heads=ARCH["heads"], q_format="FP16_32", loss_scale=scale)
    drop = (p_drop, p_drop, 99)
    _, _, og = grad_round_oracle.train_step(P, img, tgt, grad_format=gfmt, seed=gseed, dropout=drop, **kw)
    _, _, ste = dropout_oracle.train_step(P, img, tgt, dropout=drop, **kw)
    got = _grads(m)
    for n, p in m.named_parameters():
        k = vit_oracle.canonical_key(n)
        if og[k] is None:
            continue
        ref = og[k].double()
        err = float((got[n].cpu().double() - ref).norm() / (ref.norm() + 1e-30))
        d = float((ste[k].double() - ref).norm() / (ref.norm() + 1e-30))
        assert err < 0.75 * d + 1e-4, (k, err, d)
        if k.endswith(".weight") and p.dim() == 2:
            assert torch.equal(mv.float_quantize(got[n], *gfmt), got[n]), k
    near, _ = build(case, 77, rounding="nearest", dropout=p_drop)
    if p_drop:
        near.engine().fixed_dropout_seed = seed_tensor(99)
    (F.cross_entropy(near(img.to(dev)), tgt.to(dev)) * scale).backward()
    gn = _grads(near)
    assert all(not torch.equal(gn[k], got[k]) for k in got if got[k].dim() == 2), "stochastic equals nearest"


def test_seed_draws_replays_and_the_nearest_mode():
    """torch.manual_seed repeats a step; a graphed step draws a new seed per replay and each replay equals an eager step
    with that seed fixed; nearest rounding draws nothing."""
    from myrtle_vision.utils.graph import GraphedTrainStep
    case = CASES["classification"]
    img, tgt = make_inputs("classification", case, 6)
    img, tgt = img.to(dev), tgt.to(dev)
    runs = []
    for _ in range(2):
        m, _ = build(case, 5)
        torch.manual_seed(321)
        m.zero_grad(set_to_none=True)
        (F.cross_entropy(m(img), tgt) * 65536.0).backward()
        runs.append((int(m.engine().last_grad_round_seed.item()), _grads(m)))
    assert runs[0][0] == runs[1][0]
    for k in runs[0][1]:
        a, b = runs[0][1][k], runs[1][1][k]
        assert float((a - b).double().norm()) <= REPEAT_TOL * float(a.double().norm()) + 1e-12, k
    # nearest: no generator draw
    n, _ = build(case, 5, rounding="nearest")
    state = torch.cuda.get_rng_state()
    (F.cross_entropy(n(img), tgt) * 65536.0).backward()
    assert torch.equal(torch.cuda.get_rng_state(), state) and n.engine().last_grad_round_seed is None

    m, _ = build(case, 5)
    loss = lambda out, t: F.cross_entropy(out, t) * 65536.0
    step = GraphedTrainStep(m, loss, img, tgt)
    eng = m.engine()
    step(img, tgt)
    s1, g1 = eng.last_grad_round_seed.clone(), _grads(m)
    step(img, tgt)
    s2, g2 = eng.last_grad_round_seed.clone(), _grads(m)
    assert not torch.equal(s1, s2)
    for s, g in ((s1, g1), (s2, g2)):
        eng.fixed_grad_round_seed = s
        try:
            m.zero_grad(set_to_none=True)
            loss(m(img), tgt).backward()
        finally:
            eng.fixed_grad_round_seed = None
        for k, v in _grads(m).items():
            assert float((v - g[k]).double().norm()) <= REPEAT_TOL * float(g[k].double().norm()) + 1e-12, k


def _dp_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200"))
    import torch.distributed as dist
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.parallel import DataParallel
    import mv_native as mv
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, world_size=world, rank=rank)
    try:
        d = torch.device("cuda", rank)
        torch.manual_seed(11)
        model = ViT(decoder="classification", image_size=96, patch_size=16, num_classes=7, dim=128, depth=2, heads=2,
                    mlp_dim=256, q_format="FP16_32", backward_format=(5, 2), backward_rounding="stochastic").to(d).train()
        dp = DataParallel(model)
        eng = model.engine()
        eng.fixed_grad_round_seed = torch.tensor([777], dtype=torch.int64, device=d)    # one seed on both ranks
        g = torch.Generator().manual_seed(5)
        img = torch.randn(4, 3, 96, 96, generator=g).clamp(-1, 1)          # the same batch on both ranks
        y = torch.randint(0, 7, (4,), generator=g)
        (F.cross_entropy(dp(img.to(d)), y.to(d)) * 65536.0).backward()
        torch.cuda.synchronize()
        ret["rank_%d" % rank] = eng.rank
        w = model.transformer.layers[0][1].fn.fn.net[0]
        w = w[1] if isinstance(w, torch.nn.Sequential) else w
        gw = w.weight.grad
        # identical local gradients, rounded with different offsets: their mean leaves the E5M2 grid
        ret["off_grid_%d" % rank] = float((mv.float_quantize(gw, 5, 2) != gw).float().mean())
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ranks_round_with_different_offsets():
    import random
    import torch.multiprocessing as mp
    port = 29500 + random.randint(0, 2000)
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret["rank_0"] == 0 and ret["rank_1"] == 1, dict(ret)
    assert ret["off_grid_0"] > 0.05 and ret["off_grid_1"] > 0.05, dict(ret)
