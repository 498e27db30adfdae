"""Knowledge distillation on the fused path (models/distill.py): the loss kernel against float64 torch, the token rows
bit for bit, the student's step with the distillation token against the CPU restatement (tests/distill_oracle.py), the
graphed step, the overflow sink with a teacher inside the step, and train_deit with a distiller_config."""
import copy
import os

import pytest
import torch
import torch.nn.functional as F

import distill_oracle
from oracle import vit_oracle
from oracle.golden_cases import ARCH, CASES, make_inputs

pytestmark = pytest.mark.gpu
dev = "cuda"
TOL = (1e-3, 2e-3, 5e-3)             # the bars of tests/test_gpu_model.py: loss, outputs, parameter gradients
TOL_FP32 = (1e-5, 5e-5, 1e-4)
SMALL = dict(dim=384, depth=12, heads=6, mlp_dim=1536)


# ------------------------------------------------------------------------------------------------ loss kernel
@pytest.mark.parametrize("B", [1, 7, 256])
@pytest.mark.parametrize("C", [2, 45, 1000, 1001])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("T", [1.0, 4.0])
@pytest.mark.parametrize("hard", [False, True])
def test_loss_kernel_against_float64(hard, T, alpha, C, B):
    import mv_native as mv
    g = torch.Generator().manual_seed(C * 1000 + B)
    s, d, t = (3 * torch.randn(B, C, generator=g) for _ in range(3))
    t[::2, C - 1] = t[::2, 0] = t.max() + 1.0               # ties: torch.argmax takes the first index
    y = torch.randint(0, C, (B,), generator=g)
    s64, d64 = s.double().requires_grad_(), d.double().requires_grad_()
    ref = distill_oracle.loss(s64, d64, t.double(), y, T, alpha, hard)
    ref.backward()
    loss, ds, dd = mv.distill_loss(s.to(dev), d.to(dev), t.to(dev), y.to(dev), T, alpha, hard)
    assert abs(float(loss) - float(ref)) <= 2e-6 * abs(float(ref)) + 1e-7
    for got, want in ((ds, s64.grad), (dd, d64.grad)):
        assert (got.cpu().double() - want).abs().max() <= 1e-5 * want.abs().max() + 1e-9
    # deterministic: the batch sum has a fixed order
    again = mv.distill_loss(s.to(dev), d.to(dev), t.to(dev), y.to(dev), T, alpha, hard)
    assert torch.equal(again[0], loss) and torch.equal(again[1], ds) and torch.equal(again[2], dd)


def test_loss_autograd_scales_by_the_incoming_gradient_and_flags_bad_labels():
    from myrtle_vision.models.distill import distill_loss
    g = torch.Generator().manual_seed(3)
    s, d, t = (torch.randn(5, 10, generator=g).to(dev) for _ in range(3))
    y = torch.randint(0, 10, (5,), generator=g).to(dev)
    a, b = s.clone().requires_grad_(), d.clone().requires_grad_()
    distill_loss(a, b, t, y, 2.0, 0.3).backward()
    a2, b2 = s.clone().requires_grad_(), d.clone().requires_grad_()
    (3.0 * distill_loss(a2, b2, t, y, 2.0, 0.3)).backward()
    assert torch.allclose(a2.grad, 3 * a.grad, rtol=1e-6) and torch.allclose(b2.grad, 3 * b.grad, rtol=1e-6)
    y[2] = 10
    bad = distill_loss(s, d, t, y, 2.0, 0.3)
    assert torch.isnan(bad)


# ------------------------------------------------------------------------------------------------ token rows
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_patchify_token_slots_bit_exact(dtype):
    import mv_native as mv
    img = torch.randn(3, 3, 80, 96, device=dev)
    one = mv.patchify_q(img, 16, q_in=(5, 10), out_dtype=dtype, cls_slot=True).view(3, 31, 768)
    two = mv.patchify_q(img, 16, q_in=(5, 10), out_dtype=dtype, cls_slot=2).view(3, 32, 768)
    want = torch.cat((one, torch.zeros(3, 1, 768, dtype=dtype, device=dev)), dim=1)
    assert torch.equal(two, want)


@pytest.mark.parametrize("q_ff", [None, (5, 10)])
def test_token_row_bit_exact(q_ff):
    import mv_native as mv
    B, N, D = 4, 27, 128
    x = torch.randn(B * N, D, device=dev)
    tok = torch.randn(D, device=dev) * 100
    want = x.clone().view(B, N, D)
    want[:, N - 1] = mv.float_quantize(tok, *q_ff) if q_ff else tok
    mv.token_row(tok, x, B, N, D, N - 1, q_ff=q_ff)
    assert torch.equal(x.view(B, N, D), want)


# ------------------------------------------------------------------------------------------------ model step
def _key(name, fmt):
    """State-dict name -> oracle name.  FP32 names are unwrapped already (and distill_mlp.1.* is not a wrapper)."""
    return name if fmt == "FP32" else vit_oracle.canonical_key(name)


def _wrapper(fmt, arch, case, seed, emb_dropout=0.0, dropout=0.0, T=2.0, alpha=0.5, hard=False, teacher_fmt="FP32"):
    from myrtle_vision.models.distill import DistillWrapper
    from myrtle_vision.models.vit import ViT

    def vit(q, **kw):
        return ViT(decoder="classification", image_size=case["image_size"], patch_size=16,
                   num_classes=case["num_classes"], dim=arch["dim"], depth=arch["depth"], heads=arch["heads"],
                   mlp_dim=arch["mlp_dim"], q_format=q, **kw)
    student, teacher = vit(fmt, dropout=dropout, emb_dropout=emb_dropout), vit(teacher_fmt)
    P = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], dim=arch["dim"],
                               depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    P["distillation_token"] = torch.randn(1, 1, arch["dim"], generator=g)
    P["distill_mlp.0.weight"] = 1.0 + 0.1 * torch.randn(arch["dim"], generator=g)
    P["distill_mlp.0.bias"] = 0.1 * torch.randn(arch["dim"], generator=g)
    P["distill_mlp.1.weight"] = (torch.rand(case["num_classes"], arch["dim"], generator=g) * 2 - 1) * arch["dim"] ** -0.5
    P["distill_mlp.1.bias"] = (torch.rand(case["num_classes"], generator=g) * 2 - 1) * arch["dim"] ** -0.5
    student.load_state_dict({k: P[vit_oracle.canonical_key(k)] for k in student.state_dict()})
    PT = vit_oracle.init_params(decoder="classification", num_classes=case["num_classes"], dim=arch["dim"],
                                depth=arch["depth"], heads=arch["heads"], mlp_dim=arch["mlp_dim"], seed=seed + 2)
    teacher.load_state_dict({k: PT[vit_oracle.canonical_key(k)] for k in teacher.state_dict()})
    w = DistillWrapper(student=student, teacher=teacher, temperature=T, alpha=alpha, hard=hard)
    w.load_distiller_state_dict({k: P[_key(k, fmt)] for k in w.distiller_state_dict()})
    return w.to(dev).train(), P


def _check(w, P, img, tgt, fmt, heads, dropout=None):
    from myrtle_vision.models.distill import DistillLoss
    tol_loss, tol_out, tol_grad = TOL_FP32 if fmt == "FP32" else TOL
    crit = DistillLoss(w.temperature, w.alpha, w.hard)
    out = w(img.to(dev))
    loss = crit(out, tgt.to(dev))
    loss.backward()
    if dropout is not None:
        dropout = dropout + (int(w.engine().last_dropout_seed.item()),)
    s, d, ol, og = distill_oracle.train_step(P, img, tgt, out[2].cpu(), heads=heads, q_format=fmt,
                                             temperature=w.temperature, alpha=w.alpha, hard=w.hard, dropout=dropout)
    assert abs(loss.item() - float(ol)) < tol_loss * abs(float(ol)), (loss.item(), float(ol))
    for got, ref in ((out[0], s), (out[1], d)):
        assert (got.detach().cpu() - ref).abs().max() < tol_out * ref.abs().max()
    grads = {_key(n.replace("student.", "", 1), fmt): p.grad for n, p in w.named_parameters()}
    worst = 0.0
    for k, ref in og.items():
        if ref is None:
            assert grads.get(k) is None, k
            continue
        err = float((grads[k].detach().cpu().double() - ref.double()).norm() / (ref.double().norm() + 1e-30))
        worst = max(worst, err)
        assert err < tol_grad, (k, err)
    assert {"distillation_token", "distill_mlp.0.weight", "distill_mlp.1.weight"} <= set(og)
    return worst


@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("fmt", ["FP16_32", "FP16_16", "TF32", "FP32"])
def test_student_step_matches_the_oracle(fmt, hard):
    case = CASES["classification"]
    w, P = _wrapper(fmt, ARCH, case, 11, hard=hard)
    img, tgt = make_inputs("classification", case, 12)
    print(fmt, hard, _check(w, P, img, tgt, fmt, ARCH["heads"]))


def test_student_step_at_benchmark_shape():
    """ViT-Small 256 x 256, FP16_32: N = 258 tokens (the short-sequence attention kernels' odd-key path)."""
    case = dict(image_size=256, num_classes=45, batch=8)
    w, P = _wrapper("FP16_32", SMALL, case, 1234, T=4.0, alpha=0.5)
    img, tgt = make_inputs("classification", case, 1234)
    print(_check(w, P, img, tgt, "FP16_32", SMALL["heads"]))


def test_embedding_dropout_covers_the_token_row():
    """The oracle masks the whole sequence with the embedding site, the token row included: an unmasked token row would
    put a quarter of the distillation head's input off by the 1 / (1 - p) scale."""
    case = CASES["classification"]
    w, P = _wrapper("FP16_32", ARCH, case, 21, emb_dropout=0.25, dropout=0.1)
    img, tgt = make_inputs("classification", case, 22)
    print(_check(w, P, img, tgt, "FP16_32", ARCH["heads"], dropout=(0.1, 0.25)))


def test_without_a_token_the_forward_is_unchanged():
    case = CASES["classification"]
    w, _ = _wrapper("FP16_32", ARCH, case, 31)
    img, _ = make_inputs("classification", case, 32)
    img = img.to(dev)
    with torch.no_grad():
        a = w.student(img)
        s, _, _ = w(img)
    assert a.shape == s.shape and not torch.equal(a, s)     # the token takes part in attention
    with torch.no_grad():
        assert torch.equal(w.student(img), a)


# ------------------------------------------------------------------------------------------------ graphed step
def test_graphed_step_equals_eager_and_leaves_the_teacher_operands_alone():
    from myrtle_vision.models.distill import DistillLoss
    from myrtle_vision.utils.graph import GraphedTrainStep
    case = CASES["classification"]
    w, _ = _wrapper("FP16_32", ARCH, case, 41, teacher_fmt="FP16_32")
    img, tgt = make_inputs("classification", case, 42)
    img, tgt = img.to(dev), tgt.to(dev)
    crit = DistillLoss(w.temperature, w.alpha, w.hard)
    step = GraphedTrainStep(w, crit, img, tgt)
    teng = w.teacher.engine()
    assert teng.frozen_weights
    wq = teng._wq[teng._weight_indices()[1]][0]
    for r in range(3):
        keep = wq.clone()
        wq.fill_(0.5)                        # a replay that re-quantised the teacher would overwrite this
        loss_g = step(img, tgt).item()
        assert bool((wq == 0.5).all())
        wq.copy_(keep)
        loss_g = step(img, tgt).item()
        g_graph = {n: p.grad.clone() for n, p in w.named_parameters() if p.grad is not None}
        assert "distillation_token" in g_graph and "distill_mlp.1.1.weight" in g_graph
        w.zero_grad(set_to_none=True)
        loss_e = crit(w(img), tgt)
        loss_e.backward()
        assert abs(loss_g - loss_e.item()) < 1e-6 * abs(loss_e.item()) + 1e-7, r
        for n, p in w.named_parameters():
            if p.grad is not None:
                assert torch.allclose(p.grad, g_graph[n], rtol=1e-3, atol=1e-7), (r, n)
        with torch.no_grad():                # the student changes between steps, the teacher does not
            for p in w.parameters():
                p.add_(0.01 * torch.randn_like(p))


# ------------------------------------------------------------------------------------------------ overflow
@pytest.mark.parametrize("teacher_first", [True, False])
def test_overflow_skips_the_update_and_the_teacher_never_sets_found_inf(teacher_first):
    from myrtle_vision.models.distill import DistillLoss
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    case = CASES["classification"]
    w, _ = _wrapper("FP16_32", ARCH, case, 51, teacher_fmt="FP16_32")
    img, tgt = make_inputs("classification", case, 52)
    img, tgt = img.to(dev), tgt.to(dev)
    tw = dict(w.teacher.named_parameters())["transformer.layers.0.0.fn.fn.to_qkv.1.weight"]
    with torch.no_grad():
        tw.mul_(2.0 ** 17)                   # the teacher's qkv saturates fp16: would raise a registered flag
    crit = DistillLoss(w.temperature, w.alpha, w.hard)
    eng, teng = w.engine(), w.teacher.engine()

    def step():
        w.zero_grad(set_to_none=True)
        if teacher_first:
            out = w(img)
        else:
            s, row = w.student(img, distill_token=w.distillation_token)
            d = w.student._linear(w.distill_mlp[1], w.student._norm(w.distill_mlp[0], row, 3), 4)
            out = (s, d, w.teacher_logits(img))
        crit(out, tgt).backward()

    step()
    torch.cuda.synchronize()
    assert float(eng.found_inf) == 0.0 and int(eng.overflow.item()) == 0
    assert float(teng.found_inf) == 0.0 and int(teng.overflow.item()) == 0
    opt = FusedAdamW(list(w.parameters()), lr=1e-2, model=w)
    eng.scaler_state[1] = 2.0 ** 40        # the student's own backward overflows
    step()
    before = {n: p.detach().clone() for n, p in w.named_parameters()}
    opt.step(found_inf=eng.found_inf)
    torch.cuda.synchronize()
    assert float(eng.found_inf) == 1.0
    for n, p in w.named_parameters():
        assert torch.equal(p, before[n]), n
    eng.found_inf.zero_()
    eng.scaler_state[1] = 1024.0
    step()
    opt.step(found_inf=eng.found_inf)
    assert not torch.equal(w.distillation_token, before["distillation_token"])


# ------------------------------------------------------------------------------------------------ train_deit
def test_train_deit_with_a_vit_teacher_and_resume(tmp_path):
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.trainer import train_deit
    vit = {"patch_size": 16, "embed_dim": 128, "depth": 2, "heads": 2, "mlp_dim": 256, "dropout": 0.0,
           "emb_dropout": 0.0, "decoder": "classification", "image_size": 80}
    torch.manual_seed(5)
    teacher = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2,
                  mlp_dim=256, q_format="FP32")
    path = str(tmp_path / "teacher.pt")
    torch.save({"model": teacher.state_dict()}, path)
    train = {"output_directory": str(tmp_path / "ckpt"), "checkpoint_path": "", "epochs": 8, "local_batch_size": 4,
             "global_batch_size": 4, "iters_per_checkpoint": 4, "iters_per_val": 4, "seed": 1234,
             "drop_last_batch": True, "optimizer": "adamw", "opt_eps": 1e-8, "opt_betas": None, "clip_grad": None,
             "momentum": 0.9, "weight_decay": 0.05, "scheduler": "cosine", "lr": 2e-3, "warmup_lr": 2e-3,
             "min_lr": 1e-4, "decay_epochs": 15, "warmup_epochs": 0, "cooldown_epochs": 0, "patience_epochs": 5,
             "decay_rate": 0.1, "distributed": False, "num_workers": 0}
    cfg = {"train_config": train, "dist_config": {"dist_backend": "nccl", "dist_url": "tcp://127.0.0.1:54398"},
           "vit_config": dict(vit, q_format="FP16_32"),
           "data_config": {"number_of_classes": 5, "synthetic": {"train_length": 4, "val_length": 4, "seed": 7}},
           "distiller_config": {"teacher": {"kind": "vit", "vit_config": dict(vit, q_format="FP32"), "checkpoint": path},
                                "temperature": 2.0, "alpha": 0.5, "hard": False}}
    history = train_deit(0, 1, copy.deepcopy(cfg))
    assert len(history) == 8 and all(torch.isfinite(torch.tensor(history)))
    assert history[-1] < history[0], history
    out_dir = train["output_directory"]
    assert sorted(os.listdir(out_dir))[:2] == ["vit_000000", "vit_000004"]
    ck = torch.load(os.path.join(out_dir, "vit_000004"), map_location="cpu")
    assert set(ck["distiller"]) == {"distillation_token", "distill_mlp.0.1.weight", "distill_mlp.0.1.bias",
                                    "distill_mlp.1.1.weight", "distill_mlp.1.1.bias"}
    student = ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2,
                  mlp_dim=256, q_format="FP16_32")
    student.load_state_dict(ck["model"])              # the eval scripts load "model" unchanged
    cfg2 = copy.deepcopy(cfg)
    cfg2["train_config"]["checkpoint_path"] = os.path.join(out_dir, "vit_000004")
    more = train_deit(0, 1, cfg2, max_iterations=6)
    assert len(more) == 2 and all(torch.isfinite(torch.tensor(more)))
