"""Mixup / CutMix / label smoothing on the fused path (utils/mixup.py): the device draw against its distributions, the
mixing patch gather bit for bit against tests/mixup_oracle.py, the soft-target loss kernel against float64, the step on
the mixed batch against the CPU oracle, graph replays, seeding and train_deit with DeiT's settings."""
import copy
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from scipy import stats

import mixup_oracle
from oracle import quant_oracle, vit_oracle
from oracle.golden_cases import ARCH, CASES

pytestmark = pytest.mark.gpu
dev = "cuda"
TOL = (1e-3, 2e-3, 5e-3)             # the bars of tests/test_gpu_model.py: loss, outputs, parameter gradients
TOL_FP32 = (1e-5, 5e-5, 1e-4)


def _spec(mixup=1.0, cutmix=0.0, prob=1.0, switch=0.5, mode="batch"):
    import mv_native as mv
    return mv.MixSpec(mixup, cutmix, prob, switch, mv.MIX_MODES[mode])


def _draw_many(spec, n_seeds, B, H=256, W=256, rank=0):
    """Records of n_seeds fixed seeds -> dict of CPU tensors [n_seeds, B]."""
    import mv_native as mv
    seeds = torch.arange(1, n_seeds + 1, dtype=torch.int64, device=dev) * 0x9E3779B97F4A7C15 % (2 ** 62)
    out = [mixup_oracle.records(mv.mix_draw(seeds[i:i + 1], B, H, W, spec, rank=rank)) for i in range(n_seeds)]
    return {k: torch.stack([o[k] for o in out]) for k in out[0]}


# ------------------------------------------------------------------------------------------------ draw
@pytest.mark.parametrize("mode", ["batch", "pair", "elem"])
@pytest.mark.parametrize("alpha", [0.2, 0.8, 1.0, 2.0])
def test_mixup_lambda_is_beta(mode, alpha):
    B = 8
    r = _draw_many(_spec(mixup=alpha, mode=mode), 3000 if mode == "batch" else 400, B)
    lam = r["lam"][:, 0] if mode == "batch" else r["lam"][:, :B // 2].flatten() if mode == "pair" else r["lam"].flatten()
    assert stats.kstest(lam.double().numpy(), stats.beta(alpha, alpha).cdf).pvalue > 1e-3
    assert (r["cutmix"] == 0).all()
    assert torch.equal(r["w_self"], r["lam"])
    assert (r["w_other"].double() - (1.0 - r["lam"].double())).abs().max() < 1.2e-7     # fp32(1 - lam), fp64 difference
    if mode == "batch":
        assert (r["lam"] == r["lam"][:, :1]).all()
    if mode == "pair":
        assert torch.equal(r["lam"], r["lam"].flip(1))


@pytest.mark.parametrize("mode", ["batch", "pair", "elem"])
@pytest.mark.parametrize("alpha", [0.2, 0.8, 1.0, 2.0])
def test_cutmix_box_and_corrected_lambda(mode, alpha):
    H, W, B = 224, 160, 6
    r = _draw_many(_spec(mixup=0.0, cutmix=alpha, mode=mode), 1500 if mode == "batch" else 300, B, H, W)
    assert (r["cutmix"] == 1).all()
    area = ((r["y1"] - r["y0"]) * (r["x1"] - r["x0"])).double()
    assert torch.equal(r["lam"], (1.0 - area / (H * W)).float())
    assert ((0 <= r["y0"]) & (r["y0"] <= r["y1"]) & (r["y1"] <= H) & (0 <= r["x0"]) & (r["x0"] <= r["x1"])
            & (r["x1"] <= W)).all()
    for k in ("y0", "y1", "x0", "x1", "lam"):
        if mode == "batch":
            assert (r[k] == r[k][:, :1]).all()
        if mode == "pair":
            assert torch.equal(r[k], r[k].flip(1))


def test_cutmix_centres_are_uniform():
    # Beta(0.05, 0.05) puts lam near 1 often enough that cut_h, cut_w <= 1: then y0 = y1 = cy and x0 = x1 = cx
    H, W = 200, 120
    r = _draw_many(_spec(mixup=0.0, cutmix=0.05, mode="elem"), 200, 16, H, W)
    tiny = (r["y1"] == r["y0"]).flatten() & (r["x1"] == r["x0"]).flatten()
    cy, cx = r["y0"].flatten()[tiny], r["x0"].flatten()[tiny]
    assert tiny.sum() > 500
    # discrete uniform on {0 .. H-1}: chi-square over the values
    for v, n in ((cy, H), (cx, W)):
        counts = torch.bincount(v.long(), minlength=n)
        assert len(counts) == n
        assert stats.chisquare(counts.numpy()).pvalue > 1e-3


@pytest.mark.parametrize("prob,switch", [(0.3, 0.5), (1.0, 0.2), (0.7, 0.9)])
def test_mix_and_switch_probabilities(prob, switch):
    r = _draw_many(_spec(mixup=0.8, cutmix=1.0, prob=prob, switch=switch, mode="elem"), 100, 64)
    n = r["lam"].numel()
    mixed = (r["cutmix"] == 1) | (r["w_other"] != 0)
    cut = (r["cutmix"] == 1).sum().item()
    # binomial bounds at about 5 sigma
    assert abs(mixed.sum().item() / n - prob) < 5 * (prob * (1 - prob) / n) ** 0.5 + 1e-3
    k = mixed.sum().item()
    assert abs(cut / k - switch) < 5 * (switch * (1 - switch) / k) ** 0.5 + 1e-3
    un = ~mixed
    assert (r["lam"][un] == 1).all() and (r["w_self"][un] == 1).all() and (r["y0"][un] == r["y1"][un]).all()


def test_same_seed_same_records_and_ranks_differ():
    import mv_native as mv
    seed = torch.tensor([12345], dtype=torch.int64, device=dev)
    spec = _spec(mixup=0.8, cutmix=1.0, mode="elem")
    a, b = mv.mix_draw(seed, 32, 64, 64, spec), mv.mix_draw(seed, 32, 64, 64, spec)
    assert torch.equal(a, b)
    c = mv.mix_draw(seed, 32, 64, 64, spec, rank=1)
    assert not torch.equal(a, c)


# ------------------------------------------------------------------------------------------------ patchify
def _fixed_recs(B, H, W, kind):
    """Hand-made records: boxes at the edges, empty boxes, lam = 1, and Mixup weights."""
    rec = np.zeros((B, 8), dtype=np.int32)
    f = rec[:, :3].view(np.float32)
    f[:, 0] = f[:, 1] = 1.0
    boxes = [(0, H, 0, W), (0, 5, 0, 7), (H - 3, H, W - 9, W), (10, 10, 3, 30), (3, 17, 2, 6), (1, H - 1, 5, 6)]
    for b in range(B):
        if kind == "cutmix" and b % 7 != 6:
            y0, y1, x0, x1 = boxes[b % len(boxes)]
            rec[b, 3:] = (1, y0, y1, x0, x1)
            f[b, 0] = 1.0 - (y1 - y0) * (x1 - x0) / (H * W)
        elif kind == "mixup" and b % 5 != 4:
            lam = np.float64(0.1 + 0.8 * b / B)
            f[b] = (np.float32(lam), np.float32(lam), np.float32(1.0 - lam))
    return torch.from_numpy(rec).to(dev)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("q", [(5, 10), (8, 10), None])
@pytest.mark.parametrize("cls_slot", [0, 1, 2])
@pytest.mark.parametrize("P", [16, 8])
@pytest.mark.parametrize("kind", ["mixup", "cutmix", "none"])
def test_patchify_mix_bit_exact(kind, P, cls_slot, q, dtype):
    import mv_native as mv
    if dtype == torch.float16 and q == (8, 10):
        pytest.skip("fp16 containers hold formats with exp <= 5 only")
    B, C, H, W = 8, 3, 48, 64
    g = torch.Generator().manual_seed(P * 100 + cls_slot)
    img = torch.randn(B, C, H, W, generator=g) * 3
    recs = _fixed_recs(B, H, W, kind)
    mixed = mixup_oracle.apply(img, mixup_oracle.records(recs))
    got = mv.patchify_mix_q(img.to(dev), recs, P, q_in=q, out_dtype=dtype, cls_slot=cls_slot)
    want_dev = mv.patchify_q(mixed.to(dev), P, q_in=q, out_dtype=dtype, cls_slot=cls_slot)
    assert torch.equal(got.view(torch.int16 if dtype == torch.float16 else torch.int32),
                       want_dev.view(torch.int16 if dtype == torch.float16 else torch.int32))
    # against the CPU oracle too: unfold the mixed image and quantise
    x = mixed if q is None else torch.from_numpy(quant_oracle.float_quantize(mixed.numpy(), *q))
    pt = x.view(B, C, H // P, P, W // P, P).permute(0, 2, 4, 3, 5, 1).reshape(B, -1, P * P * C).to(dtype)
    z = torch.zeros(B, 1, P * P * C, dtype=dtype)
    pt = torch.cat([z, pt] if cls_slot == 1 else [z, pt, z] if cls_slot == 2 else [pt], dim=1).reshape(-1, P * P * C)
    assert torch.equal(got.cpu(), pt)


# ------------------------------------------------------------------------------------------------ loss kernel
@pytest.mark.parametrize("C", [2, 45, 1000])
@pytest.mark.parametrize("smoothing", [0.0, 0.1])
@pytest.mark.parametrize("mixed", [False, True])
def test_loss_kernel_against_float64(mixed, smoothing, C):
    import mv_native as mv
    B = 256
    g = torch.Generator().manual_seed(C + int(10 * smoothing))
    x = 4 * torch.randn(B, C, generator=g)
    x[::3, 1] = 40.0                                           # dominant classes keep their digits
    y = torch.randint(0, C, (B,), generator=g)
    recs = mv.mix_draw(torch.tensor([C], dtype=torch.int64, device=dev), B, 64, 64,
                       _spec(mixup=0.8, cutmix=1.0, mode="elem")) if mixed else None
    lam = mixup_oracle.records(recs)["lam"] if mixed else torch.ones(B)
    x64 = x.double().requires_grad_()
    ref = mixup_oracle.loss(x64, y, lam, smoothing)
    ref.backward()
    loss, dx = mv.mix_ce_loss(x.to(dev), y.to(dev), recs, smoothing)
    assert abs(float(loss) - float(ref)) <= 2e-6 * abs(float(ref)) + 1e-7
    assert (dx.cpu().double() - x64.grad).abs().max() <= 1e-5 * x64.grad.abs().max() + 1e-9
    again = mv.mix_ce_loss(x.to(dev), y.to(dev), recs, smoothing)
    assert torch.equal(again[0], loss) and torch.equal(again[1], dx)


@pytest.mark.parametrize("smoothing", [0.0, 0.1])
def test_unmixed_loss_is_cross_entropy(smoothing):
    from myrtle_vision.utils.mixup import mix_cross_entropy
    g = torch.Generator().manual_seed(4)
    x = (3 * torch.randn(64, 45, generator=g)).to(dev)
    y = torch.randint(0, 45, (64,), generator=g).to(dev)
    a, b = x.clone().requires_grad_(), x.clone().requires_grad_()
    ours = mix_cross_entropy(a, y, None, smoothing)
    ref = F.cross_entropy(b, y, label_smoothing=smoothing)
    ours.backward()
    ref.backward()
    assert torch.allclose(ours, ref, rtol=1e-6, atol=1e-7)
    assert torch.allclose(a.grad, b.grad, rtol=1e-5, atol=1e-8)


def test_bad_labels_give_nan_and_a_skipped_step():
    import mv_native as mv
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.mixup import MixupLoss
    from myrtle_vision.utils.optim import create_optimizer
    import argparse
    B, C = 8, 5
    x = torch.randn(B, C, device=dev)
    y = torch.randint(0, C, (B,), device=dev)
    recs = _fixed_recs(B, 32, 32, "mixup")            # images 4 are unmixed (lam = 1): their partner's label is unused
    y_bad = y.clone()
    y_bad[3] = C                                        # image 3 (lam < 1) and its partner 4 ... image 4 has lam = 1
    loss, dx = mv.mix_ce_loss(x, y_bad, recs, 0.1)
    rows = torch.isnan(dx).any(1).cpu()
    assert torch.isnan(loss)
    assert rows[3] and not rows[4] and not rows[0]
    # in a step: the overflow sink sees the NaN gradient and the optimizer skips the update
    torch.manual_seed(0)
    m = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=C, dim=128, depth=1, heads=2,
            mlp_dim=256, q_format="FP16_32").to(dev).train()
    args = argparse.Namespace(opt="adamw", weight_decay=0.05, lr=1e-3, opt_eps=1e-8, opt_betas=None, momentum=0.9)
    opt = create_optimizer(args, m)
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    img = torch.randn(B, 3, 80, 80, device=dev)
    MixupLoss(0.1)((m(img, mix=recs), recs), y_bad).backward()
    eng = m.engine()
    opt.step(found_inf=eng.found_inf)
    assert float(eng.found_inf) != 0
    assert all(torch.equal(p, before[n]) for n, p in m.named_parameters())


# ------------------------------------------------------------------------------------------------ model
def _model(fmt, case, seed, arch=ARCH):
    from myrtle_vision.models.vit import ViT
    m = ViT(decoder="classification", image_size=case["image_size"], patch_size=16, num_classes=case["num_classes"],
            dim=arch["dim"], depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], q_format=fmt)
    P = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], dim=arch["dim"],
                               depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], seed=seed)
    m.load_state_dict({k: P[vit_oracle.canonical_key(k)] for k in m.state_dict()})
    return m.to(dev).train(), P


@pytest.mark.parametrize("fmt", ["FP16_32", "FP16_16", "TF32", "FP32"])
def test_step_on_the_mixed_batch_matches_the_oracle(fmt):
    from myrtle_vision.utils.mixup import Mixup, MixupLoss, MixupWrapper
    case = CASES["classification"]
    m, P = _model(fmt, case, 11)
    g = torch.Generator().manual_seed(12)
    img = torch.randn(8, 3, case["image_size"], case["image_size"], generator=g)
    tgt = torch.randint(0, case["num_classes"], (8,), generator=g)
    w = MixupWrapper(m, Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, mode="elem", label_smoothing=0.1))
    torch.manual_seed(3)
    logits, recs = w(img.to(dev))
    loss = MixupLoss(0.1)((logits, recs), tgt.to(dev))
    loss.backward()
    rec = mixup_oracle.records(recs)
    assert (rec["lam"] < 1).any()
    mixed = mixup_oracle.apply(img, rec)
    tol_loss, tol_out, tol_grad = TOL_FP32 if fmt == "FP32" else TOL
    out, ol, og = mixup_oracle.train_step(P, mixed, tgt, rec["lam"], 0.1, heads=ARCH["heads"], q_format=fmt)
    assert abs(loss.item() - float(ol)) < tol_loss * abs(float(ol)), (loss.item(), float(ol))
    assert (logits.detach().cpu() - out.detach()).abs().max() < tol_out * out.detach().abs().max()
    grads = {vit_oracle.canonical_key(n): p.grad for n, p in m.named_parameters()}
    for k, ref in og.items():
        if ref is None:
            continue
        g = grads[k].detach().cpu().double()
        assert (g - ref.double()).norm() < tol_grad * ref.double().norm() + 1e-12, k


def test_wrapper_logits_equal_the_vit_on_the_mixed_image():
    from myrtle_vision.utils.mixup import Mixup, MixupWrapper
    case = CASES["classification"]
    m, _ = _model("FP16_32", case, 5)
    img = torch.randn(6, 3, case["image_size"], case["image_size"], generator=torch.Generator().manual_seed(6))
    w = MixupWrapper(m, Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, mode="pair"))
    with torch.no_grad():
        torch.manual_seed(9)
        logits, recs = w(img.to(dev))
        mixed = mixup_oracle.apply(img, mixup_oracle.records(recs)).to(dev)
        direct = m(mixed)
    assert torch.equal(logits, direct)
    assert w.last_mix is recs


# ------------------------------------------------------------------------------------------------ step behaviour
def _small_wrapper(seed=0):
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.mixup import Mixup, MixupWrapper
    torch.manual_seed(seed)
    m = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=1, heads=2,
            mlp_dim=256, q_format="FP16_32").to(dev).train()
    return MixupWrapper(m, Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, mode="elem"))


def test_graph_replays_draw_new_records_and_manual_seed_repeats_them():
    from myrtle_vision.utils.graph import GraphedTrainStep
    from myrtle_vision.utils.mixup import MixupLoss
    w = _small_wrapper()
    img = torch.randn(8, 3, 80, 80, device=dev)
    y = torch.randint(0, 5, (8,), device=dev)
    step = GraphedTrainStep(w, MixupLoss(0.1), img, y)
    seen = []
    torch.manual_seed(21)
    for _ in range(3):
        step(img, y)
        seen.append(w.last_mix.clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    torch.manual_seed(21)
    step(img, y)
    assert torch.equal(w.last_mix, seen[0])


def test_eval_draws_nothing():
    w = _small_wrapper().eval()
    img = torch.randn(8, 3, 80, 80, device=dev)
    state = torch.cuda.get_rng_state()
    with torch.no_grad():
        logits, recs = w(img)
    assert recs is None and torch.equal(torch.cuda.get_rng_state(), state)
    with torch.no_grad():
        assert torch.equal(logits, w.vit(img))


def test_without_mixing_the_step_launches_the_same_kernels():
    import mv_native as mv
    from myrtle_vision.utils.trainer import build_criterion
    w = _small_wrapper()
    m = w.vit
    img = torch.randn(8, 3, 80, 80, device=dev)
    y = torch.randint(0, 5, (8,), device=dev)
    crit = build_criterion("classification", {}, 5, dev)
    assert crit is F.cross_entropy
    crit(m(img), y).backward()                 # the first step also quantises the weight operands once
    counts = []
    for _ in range(2):
        mv.enable_timing(True)
        n0 = mv.launch_count()
        crit(m(img), y).backward()
        torch.cuda.synchronize()
        counts.append((mv.launch_count() - n0, sorted(mv.timing_summary())))
    mv.enable_timing(False)
    assert counts[0] == counts[1]
    assert "patchify" in counts[0][1] and "patchify_mix" not in counts[0][1] and "mix_ce_loss" not in counts[0][1]
    # with mixing: the same launches plus the draw, with the mixing gather in place of the plain one, plus the loss
    mv.enable_timing(True)
    n0 = mv.launch_count()
    from myrtle_vision.utils.mixup import MixupLoss
    MixupLoss(0.1)(w(img), y).backward()
    torch.cuda.synchronize()
    names = sorted(mv.timing_summary())
    mv.enable_timing(False)
    assert mv.launch_count() - n0 == counts[0][0] + 3
    assert "patchify_mix" in names and "patchify" not in names and "mix_ce_loss" in names


def test_train_deit_with_deit_settings_and_resume(tmp_path):
    from myrtle_vision.utils.trainer import train_deit
    vit = {"patch_size": 16, "embed_dim": 128, "depth": 2, "heads": 2, "mlp_dim": 256, "dropout": 0.0,
           "emb_dropout": 0.0, "decoder": "classification", "image_size": 80, "q_format": "FP16_32"}
    train = {"output_directory": str(tmp_path / "ckpt"), "checkpoint_path": "", "epochs": 8, "local_batch_size": 4,
             "global_batch_size": 4, "iters_per_checkpoint": 4, "iters_per_val": 4, "seed": 1234,
             "drop_last_batch": True, "optimizer": "adamw", "opt_eps": 1e-8, "opt_betas": None, "clip_grad": None,
             "momentum": 0.9, "weight_decay": 0.05, "scheduler": "cosine", "lr": 2e-3, "warmup_lr": 2e-3,
             "min_lr": 1e-4, "decay_epochs": 15, "warmup_epochs": 0, "cooldown_epochs": 0, "patience_epochs": 5,
             "decay_rate": 0.1, "distributed": False, "num_workers": 0,
             "mixup": 0.8, "cutmix": 1.0, "mixup_prob": 1.0, "mixup_switch_prob": 0.5, "mixup_mode": "batch",
             "smoothing": 0.1}
    cfg = {"train_config": train, "dist_config": {"dist_backend": "nccl", "dist_url": "tcp://127.0.0.1:54399"},
           "vit_config": vit,
           "data_config": {"number_of_classes": 5, "synthetic": {"train_length": 4, "val_length": 4, "seed": 7}}}
    history = train_deit(0, 1, copy.deepcopy(cfg))
    assert len(history) == 8 and all(torch.isfinite(torch.tensor(history)))
    out_dir = train["output_directory"]
    assert sorted(os.listdir(out_dir))[:2] == ["vit_000000", "vit_000004"]
    ck = torch.load(os.path.join(out_dir, "vit_000004"), map_location="cpu")
    assert "distiller" not in ck and not any(k.startswith("vit.") for k in ck["model"])
    cfg2 = copy.deepcopy(cfg)
    cfg2["train_config"]["checkpoint_path"] = os.path.join(out_dir, "vit_000004")
    more = train_deit(0, 1, cfg2, max_iterations=6)
    assert len(more) == 2 and all(torch.isfinite(torch.tensor(more)))
