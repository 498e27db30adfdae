"""Dropout on the fused path (ViT(dropout=..., emb_dropout=...) in training mode): the mask stream of
include/mv_b200.h ("dropout mask") against the oracle's restatement, the fused GEMM / LayerNorm-backward sites against
the same kernels without dropout masked on the host, the model step against the CPU reference (tests/dropout_oracle.py) with the seed the
engine drew, and the behaviour a training loop relies on (reproducibility, fresh masks per step and per graph replay,
eval and p = 0 untouched)."""
import copy
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dropout_oracle
from oracle import vit_oracle
from oracle.golden_cases import ARCH, CASES, make_inputs

pytestmark = pytest.mark.gpu
dev = "cuda"
TOL = (1e-3, 2e-3, 5e-3)            # the bars of tests/test_gpu_model.py
P_DROP = 0.1


def seed_tensor(s):
    return torch.tensor([s], dtype=torch.int64, device=dev)


def mask(shape, p, seed, site):
    return dropout_oracle.dropout_mask(shape, p, seed, site).to(dev)


# ------------------------------------------------------------------------------------------------ mask stream
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("rows,cols,pitch", [(257, 384, 384), (33, 13, 13), (7, 40, 56), (1000, 1536, 1536)])
def test_mask_stream_matches_the_oracle(dtype, rows, cols, pitch):
    import mv_native as mv
    for seed, site in [(1, 0), (0x9234_5678_9ABC_DEF0 - 2 ** 64, 37), (-1, 36), (42, 5)]:
        base = torch.ones(rows, pitch, dtype=dtype, device=dev)
        x = base[:, :cols]
        got = mv.dropout(x, (seed_tensor(seed), P_DROP, site))
        want = dropout_oracle.dropout_mask((rows, cols), P_DROP, seed, site)
        assert torch.equal(got.float().cpu(), want.to(dtype).float()), (seed, site)
        # in place, through the row pitch: the padding columns are not touched
        mv.dropout(x, (seed_tensor(seed), P_DROP, site), out=x)
        assert torch.equal(x.float().cpu(), want.to(dtype).float())
        assert bool((base[:, cols:] == 1).all())


def test_kept_fraction_and_the_end_points():
    import mv_native as mv
    n = 1 << 24
    x = torch.ones(n // 1024, 1024, device=dev)
    for p in (0.1, 0.5, 0.9):
        thr, scale = mv.drop_params(p)
        y = mv.dropout(x, (seed_tensor(99), p, 3))
        kept = float((y != 0).float().mean())
        q = 1.0 - thr / 65536.0
        assert abs(kept - q) < 5 * (q * (1 - q) / n) ** 0.5, (p, kept, q)
        assert float(y.max()) == scale
    r = torch.randn(123, 77, device=dev)
    assert torch.equal(mv.dropout(r, (seed_tensor(5), 0.0, 1)), r)                  # p = 0: a bit-exact copy
    assert not mv.dropout(r, (seed_tensor(5), 1.0, 1)).any()                         # p = 1: zeros
    with pytest.raises(ValueError):
        mv.dropout(r, (seed_tensor(5), 1.5, 1))


# ------------------------------------------------------------------------------------------------ kernel sites
def _ulps16(a, b):
    """|a - b| in units of half an fp16 ulp of b (0 where both are 0)."""
    a, b = a.double(), b.double()
    e = torch.floor(torch.log2(b.abs().clamp_min(2.0 ** -14)))
    return (a - b).abs() / torch.exp2(e - 11)


@pytest.mark.parametrize("fmt", ["FP16_32", "FP16_16"])
@pytest.mark.parametrize("N,K", [(384, 384), (384, 1536), (132, 384)])
def test_residual_gemm_site(fmt, N, K):
    """x + D(o(a W^T + b)) then q_res: the proj (K = 384, residual by TMA) and fc2 (K = 1536) epilogues, and the generic
    path (N % 8 != 0), against the GEMM without dropout masked on the host."""
    import mv_native as mv
    torch.manual_seed(1)
    qo = (5, 10) if fmt == "FP16_16" else None
    M = 2056                                                      # 8 x 257 tokens: a partial last tile
    A = (torch.randn(M, K, device=dev) * 0.5).half()
    B = (torch.randn(N, K, device=dev) * 0.1).half()
    bias = 0.1 * torch.randn(N, device=dev)
    res = torch.randn(M, N, device=dev)
    drop = (seed_tensor(777), P_DROP, 4)
    y0 = torch.empty(M, N, device=dev)
    mv.gemm(A, B, y0, bias=bias, q_out=qo)
    got = torch.empty(M, N, device=dev)
    mv.gemm(A, B, got, bias=bias, q_out=qo, residual=res, q_res=qo, drop=drop)
    want = y0.double() * mask((M, N), P_DROP, 777, 4).double() + res.double()
    if qo is None:
        assert float((got.double() - want).abs().max()) <= 1e-6 * float(want.abs().max())
    else:
        want = mv.float_quantize(want.float(), *qo)
        flips = _ulps16(got, want) > 0
        assert float(flips.float().mean()) < 1e-3 and float(_ulps16(got, want).max()) <= 2.0


@pytest.mark.parametrize("fmt", ["FP16_32", "FP16_16"])
@pytest.mark.parametrize("N", [1536, 132])
def test_gelu_gemm_site(fmt, N):
    """h = H(D(gelu(o(u)))) and aux = fp16(keep * s * gelu'(u)): both multiplied before they are rounded.  Against the
    outputs without dropout times the mask: they differ by one more rounding, at most an fp16 ulp, and are exactly
    zero where the mask drops."""
    import mv_native as mv
    torch.manual_seed(2)
    qo = (5, 10) if fmt == "FP16_16" else None
    M, K = 2056, 384
    A = (torch.randn(M, K, device=dev) * 0.5).half()
    B = (torch.randn(N, K, device=dev) * 0.1).half()
    bias = 0.1 * torch.randn(N, device=dev)
    h0, a0 = (torch.empty(M, N, dtype=torch.float16, device=dev) for _ in range(2))
    h1, a1 = (torch.empty(M, N, dtype=torch.float16, device=dev) for _ in range(2))
    mv.gemm(A, B, h0, bias=bias, q_out=qo, aux=a0, epilogue=mv.EPI_GELU, q_res=(5, 10))
    mv.gemm(A, B, h1, bias=bias, q_out=qo, aux=a1, epilogue=mv.EPI_GELU, q_res=(5, 10),
            drop=(seed_tensor(31337), P_DROP, 7))
    m = mask((M, N), P_DROP, 31337, 7).double()
    for got, plain in ((h1, h0), (a1, a0)):
        want = plain.double() * m
        assert torch.equal(got[m == 0].double(), want[m == 0])
        # the plain value's rounding error (half an ulp) scaled by s, plus the masked value's own: 0.5 + 0.5 s ulps
        assert float(_ulps16(got, want).max()) <= 1.0 + 1.0 / (1.0 - P_DROP) + 1e-3
    # the backward needs nothing new: the gelu' dgrad multiplies by the stored (masked) derivative
    d = torch.randn(M, K, device=dev).half()
    W = (torch.randn(N, K, device=dev) * 0.1).half()
    du = torch.empty(M, N, dtype=torch.float16, device=dev)
    mv.gemm(d, W, du, aux=a1, epilogue=mv.EPI_DGELU)
    assert not du[m == 0].any()


@pytest.mark.parametrize("D", [384, 196])
def test_layernorm_backward_site(D):
    """dx_f16 and dbias_prev carry keep * s * dx; the fp32 residual dx is bit-identical to the unmasked kernel's
    (mask_dx off) or exactly its masked value (mask_dx on, the embedding site)."""
    import mv_native as mv
    torch.manual_seed(3)
    rows = 2056
    x = torch.randn(rows, D, device=dev) * 2
    g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    _, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    dy = torch.randn(rows, D, device=dev).half(); dres = torch.randn(rows, D, device=dev)
    m = mask((rows, D), P_DROP, 55, 9)
    drop = (seed_tensor(55), P_DROP, 9)
    bp0, bp1 = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    dx0, h0 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dbias_prev=bp0)
    dx1, h1 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dbias_prev=bp1, drop=drop)
    assert torch.equal(dx1, dx0)
    assert torch.equal(h1, (dx0 * m).half())
    want = (dx0.double() * m.double()).sum(0)
    assert float((bp1.double() - want).abs().max()) < 1e-5 * float(want.abs().max())
    dx2, h2 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), drop=drop, mask_dx=True)
    assert torch.equal(dx2, dx0 * m) and torch.equal(h2, h1)


# ------------------------------------------------------------------------------------------------ model
def build(decoder, case, fmt, seed, arch=ARCH, dropout=P_DROP, emb_dropout=P_DROP, **kw):
    from myrtle_vision.models.vit import ViT
    m = ViT(decoder=decoder, image_size=case["image_size"], patch_size=16, num_classes=case["num_classes"],
            dim=arch["dim"], depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], q_format=fmt,
            dropout=dropout, emb_dropout=emb_dropout, **kw)
    P = vit_oracle.init_params(decoder=decoder, num_classes=case["num_classes"], dim=arch["dim"],
                               depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], seed=seed)
    m.load_state_dict({k: P[vit_oracle.canonical_key(k)] for k in m.state_dict()})
    return m.to(dev).train(), P


def loss_fn(decoder, out, tgt):
    if decoder == "detection":
        return (F.cross_entropy(out["pred_logits"].flatten(0, 1), tgt["labels"].flatten())
                + (out["pred_boxes"] - tgt["boxes"]).abs().mean())
    return F.cross_entropy(out, tgt)


def todev(t):
    return {k: v.to(dev) for k, v in t.items()} if isinstance(t, dict) else t.to(dev)


def check_against_oracle(m, P, img, tgt, decoder, heads, fmt, out, loss, seed, tol=TOL):
    tol_loss, tol_out, tol_grad = tol
    oo, ol, og = dropout_oracle.train_step(P, img, tgt, decoder=decoder, heads=heads, q_format=fmt,
                                           dropout=(P_DROP, P_DROP, seed))
    assert abs(loss.item() - float(ol)) < tol_loss * abs(float(ol)), (loss.item(), float(ol))
    outs = out if isinstance(out, dict) else {"out": out}
    refs = oo if isinstance(oo, dict) else {"out": oo}
    for k in outs:
        ref = refs[k].detach()
        o = outs[k].detach().cpu()
        assert float((o - ref).abs().max()) < tol_out * float(ref.abs().max()), k
    grads = {vit_oracle.canonical_key(n): p.grad for n, p in m.named_parameters()}
    for k, ref in og.items():
        if ref is None:
            assert grads[k] is None, k
            continue
        g = grads[k].detach().cpu().double()
        err = float((g - ref.double()).norm() / (ref.double().norm() + 1e-30))
        assert err < tol_grad, (k, err)


@pytest.mark.parametrize("decoder", list(CASES))
@pytest.mark.parametrize("fmt", ["FP16_32", "FP16_16", "TF32", "FP32"])
def test_model_step_matches_the_oracle(decoder, fmt):
    tol = (1e-5, 5e-5, 1e-4) if fmt == "FP32" else TOL
    case = CASES[decoder]
    m, P = build(decoder, case, fmt, 11)
    img, tgt = make_inputs(decoder, case, 12)
    out = m(img.to(dev))
    loss = loss_fn(decoder, out, todev(tgt))
    loss.backward()
    seed = int(m.engine().last_dropout_seed.item())
    check_against_oracle(m, P, img, tgt, decoder, ARCH["heads"], fmt, out, loss, seed, tol)


def test_model_step_at_benchmark_shape():
    """ViT-Small, 256 x 256, N = 257, FP16_32, batch 8: the fused epilogues at the shapes the benchmark runs."""
    case = dict(image_size=256, num_classes=45, batch=8)
    m, P = build("classification", case, "FP16_32", 1234, arch=dict(dim=384, depth=12, heads=6, mlp_dim=1536))
    img, tgt = make_inputs("classification", case, 1234)
    out = m(img.to(dev))
    loss = F.cross_entropy(out, tgt.to(dev))
    loss.backward()
    check_against_oracle(m, P, img, tgt, "classification", 6, "FP16_32", out, loss,
                         int(m.engine().last_dropout_seed.item()))


def test_model_step_with_the_gradient_quantiser():
    """backward_format on: the stub's rounding (the dgrad q_out) comes before the mask.  Bounded as in
    tests/test_gpu_model.py's gradient-quantiser test: by a fraction of what the straight-through backward differs."""
    gfmt, scale = (5, 2), 65536.0
    case = CASES["classification"]
    m, P = build("classification", case, "FP16_32", 77, backward_format=gfmt)
    img, tgt = make_inputs("classification", case, 77)
    out = m(img.to(dev))
    (F.cross_entropy(out, tgt.to(dev)) * scale).backward()
    seed = int(m.engine().last_dropout_seed.item())
    kw = dict(decoder="classification", heads=ARCH["heads"], q_format="FP16_32", loss_scale=scale,
              dropout=(P_DROP, P_DROP, seed))
    _, _, og = dropout_oracle.train_step(P, img, tgt, grad_format=gfmt, **kw)
    _, _, ste = dropout_oracle.train_step(P, img, tgt, **kw)
    for n, p in m.named_parameters():
        k = vit_oracle.canonical_key(n)
        if og[k] is None:
            continue
        ref = og[k].double()
        err = float((p.grad.detach().cpu().double() - ref).norm() / (ref.norm() + 1e-30))
        d = float((ste[k].double() - ref).norm() / (ref.norm() + 1e-30))
        assert err < 0.75 * d + 1e-4, (k, err, d)


def _grads(m):
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


def test_reproducible_under_manual_seed_and_fresh_masks_per_step():
    """Same torch.manual_seed: the same seeds, masks and losses bit for bit; the gradients up to the summation order of the
    split-K / column-sum red.adds, which varies from run to run with or without dropout."""
    case = CASES["classification"]
    img, tgt = make_inputs("classification", case, 6)
    img, tgt = img.to(dev), tgt.to(dev)
    runs = []
    for _ in range(2):
        m, _ = build("classification", case, "FP16_32", 5)
        torch.manual_seed(123)
        losses, grads, seeds = [], [], []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            loss = F.cross_entropy(m(img), tgt)
            loss.backward()
            losses.append(loss.item()); grads.append(_grads(m)); seeds.append(int(m.engine().last_dropout_seed.item()))
        runs.append((losses, grads, seeds))
    (l0, g0, s0), (l1, g1, s1) = runs
    assert l0 == l1 and s0 == s1
    for a, b in zip(g0, g1):
        for k in a:
            assert float((a[k] - b[k]).double().norm()) <= 1e-5 * float(a[k].double().norm()) + 1e-12, k
    assert s0[0] != s0[1] and l0[0] != l0[1]                     # consecutive steps: new masks


def test_eval_and_zero_probability_are_untouched():
    """model.eval() output is bit-identical to a dropout = 0 model's; p = 0 in training draws nothing and matches too."""
    case = CASES["classification"]
    img, _ = make_inputs("classification", case, 6)
    img = img.to(dev)
    m, _ = build("classification", case, "FP16_32", 5)
    z, _ = build("classification", case, "FP16_32", 5, dropout=0.0, emb_dropout=0.0)
    with torch.no_grad():
        ref = z.eval()(img)
        assert torch.equal(m.eval()(img), ref)
        state = torch.cuda.get_rng_state()
        out = z.train()(img)
        assert torch.equal(torch.cuda.get_rng_state(), state) and z.engine().last_dropout_seed is None
        assert torch.equal(out, ref)
        assert not torch.equal(m.train()(img), ref)              # training mode drops


def test_graph_replays_draw_new_masks_and_match_eager():
    from myrtle_vision.utils.graph import GraphedTrainStep
    case = CASES["classification"]
    m, _ = build("classification", case, "FP16_32", 5)
    img, tgt = make_inputs("classification", case, 6)
    img, tgt = img.to(dev), tgt.to(dev)
    step = GraphedTrainStep(m, F.cross_entropy, img, tgt)
    eng = m.engine()
    l1 = step(img, tgt).item()
    s1 = eng.last_dropout_seed.clone()
    g1 = _grads(m)
    l2 = step(img, tgt).item()
    s2 = eng.last_dropout_seed.clone()
    assert l1 != l2 and not torch.equal(s1, s2)
    # the second replay again, eagerly with its seed
    m.zero_grad(set_to_none=True)
    eng.fixed_dropout_seed = s2
    try:
        le = F.cross_entropy(m(img), tgt)
        le.backward()
    finally:
        eng.fixed_dropout_seed = None
    assert abs(le.item() - l2) < 1e-6 * abs(l2) + 1e-7
    eng.fixed_dropout_seed = s1
    try:
        m.zero_grad(set_to_none=True)
        F.cross_entropy(m(img), tgt).backward()
    finally:
        eng.fixed_dropout_seed = None
    for n, g in _grads(m).items():
        assert torch.allclose(g, g1[n], rtol=1e-3, atol=1e-7), n


def test_classification_entry_point_trains_with_dropout(tmp_path):
    import importlib.util
    from test_gpu_train import config
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("train_classification_dropout",
                                                  os.path.join(root, "myrtle-vision_b200", "classification", "train.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    cfg = config("classification", tmp_path, "FP16_32", 80, 5)
    cfg["vit_config"].update(dropout=P_DROP, emb_dropout=P_DROP)
    cfg["train_config"]["epochs"] = 6
    history = mod.train_deit(0, 1, copy.deepcopy(cfg))
    assert len(history) == 6 and all(np.isfinite(history))
    assert sorted(os.listdir(cfg["train_config"]["output_directory"]))[:2] == ["vit_000000", "vit_000005"]
