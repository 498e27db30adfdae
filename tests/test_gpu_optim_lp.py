"""qtorch.optim.OptimLP on the GPU: the fused mv_adamw_lp_step against the composed path (standalone quantisers
around FusedAdamW.step), the optimizer rounding stream, overflow skips, the model's operands, resume, the trainer
and data-parallel ranks."""
import copy
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle.golden_cases import CASES, make_inputs

pytestmark = pytest.mark.gpu
dev = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(1,), (7,), (1024,), (1025,), (33, 65), (384, 1536), (3, 5, 7)]
FORMATS = {
    "float5_10_sr": ("float", 5, 10, "stochastic"),    # 16-bit stream
    "float8_7_sr": ("float", 8, 7, "stochastic"),      # 16-bit stream
    "float4_3_sr": ("float", 4, 3, "stochastic"),      # 32-bit stream
    "float5_2_rn": ("float", 5, 2, "nearest"),
    "fixed11_9_sr": ("fixed", 11, 9, True, False, "stochastic"),
    "fixed8_4_sym_rn": ("fixed", 8, 4, True, True, "nearest"),
}
SITES = ["grad", "momentum", "acc", "weight", "all"]


def quant(f):
    from qtorch import FixedPoint, FloatingPoint
    from qtorch.quant import quantizer
    num = FloatingPoint(f[1], f[2]) if f[0] == "float" else FixedPoint(f[1], f[2], clamp=f[3], symmetric=f[4])
    return quantizer(forward_number=num, forward_rounding=f[-1])


def nearest(x, f):
    import mv_native as mv
    if f[0] == "float":
        return mv.float_quantize(x, f[1], f[2], "nearest")
    return mv.fixed_point_quantize(x, f[1], f[2], f[3], f[4], "nearest")


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def lp_kwargs(site, f):
    q = quant(f)
    kw = {"grad": dict(grad_quant=q, grad_scaling=2.0), "momentum": dict(momentum_quant=q), "acc": dict(acc_quant=q),
          "weight": dict(weight_quant=q)}
    if site == "all":
        return dict(grad_quant=q, grad_scaling=0.5, momentum_quant=q, acc_quant=q, weight_quant=q)
    return kw[site]


def with_tiles(opt, params):
    """Route the 2-D parameters of a model-less FusedAdamW through the 32x32-tile path with (5, 10) fp16 operands."""
    ops = {id(p): (torch.empty(p.shape, dtype=torch.float16, device=dev),
                   torch.empty(p.shape[::-1], dtype=torch.float16, device=dev), (5, 10)) for p in params if p.dim() == 2}
    opt._operands = lambda: ops
    return ops


def make_pair(site, f, seed=1234, tiles=True):
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch.optim import OptimLP
    torch.manual_seed(0)
    ps = [(torch.randn(s, device=dev) * 0.5).requires_grad_(True) for s in SHAPES]
    qs = [p.detach().clone().requires_grad_(True) for p in ps]
    kw = dict(lr=3e-3, betas=(0.9, 0.95), eps=1e-8)
    groups = lambda t: [{"params": t[:3], "weight_decay": 0.0}, {"params": t[3:], "weight_decay": 0.05}]
    inner = FusedAdamW(groups(ps), **kw)
    ops = with_tiles(inner, ps) if tiles else {}
    fused = OptimLP(inner, seed=seed, **lp_kwargs(site, f))
    comp = OptimLP(FusedAdamW(groups(qs), **kw), seed=seed, fused=False, **lp_kwargs(site, f))
    assert fused.fused and not comp.fused
    return ps, qs, fused, comp, ops


def set_grads(ps, qs, it, scale):
    for p, q in zip(ps, qs):
        g = torch.randn_like(p) * (10.0 ** (it % 3 - 2)) * scale
        p.grad, q.grad = g.clone(), g.clone()


@pytest.mark.parametrize("fmt", list(FORMATS))
@pytest.mark.parametrize("site", SITES)
def test_fused_equals_composed(site, fmt):
    import mv_native as mv
    f = FORMATS[fmt]
    ps, qs, fused, comp, ops = make_pair(site, f)
    inv = torch.tensor(1.0 / 256.0, device=dev)
    for it in range(4):
        set_grads(ps, qs, it, 256.0)
        if it == 2:
            for grp in fused.param_groups + comp.param_groups:
                grp["lr"] = 1e-3
        fused.step(inv_scale=inv)
        comp.step(inv_scale=inv)
        for k, (p, q) in enumerate(zip(ps, qs)):
            assert torch.equal(bits(p), bits(q)), (it, k, p.shape)
            assert torch.equal(bits(p.grad), bits(q.grad)), (it, k, "grad")
            for name in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(bits(fused.state[p][name]), bits(comp.state[q][name])), (it, k, name)
            if fused.acc[k] is not None:
                assert torch.equal(bits(fused.acc[k]), bits(comp.acc[k])), (it, k, "acc")
    for p in ps:
        if id(p) in ops:
            q, qt, _ = ops[id(p)]
            want, want_t = mv.quantize_weight(p.detach(), 5, 10)
            assert torch.equal(q, want) and torch.equal(qt, want_t)


@pytest.mark.parametrize("fmt", list(FORMATS))
def test_values_stay_on_their_grids(fmt):
    f = FORMATS[fmt]
    ps, qs, opt, _, _ = make_pair("all", f)
    for it in range(3):
        set_grads(ps, qs, it, 1.0)
        opt.step()
        for k, p in enumerate(ps):
            for name, t in (("p", p), ("acc", opt.acc[k]), ("exp_avg", opt.state[p]["exp_avg"]),
                            ("exp_avg_sq", opt.state[p]["exp_avg_sq"]), ("grad", p.grad)):
                assert torch.equal(nearest(t, f), t), (it, k, name)        # +-0 alike: nearest maps -0 to +0


@pytest.mark.parametrize("fmt", ["float8_7_sr", "float4_3_sr", "fixed11_9_sr"])
def test_stream_is_pinned_to_the_standalone_quantiser(fmt):
    import mv_native as mv
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch.optim import OptimLP, lp_offset
    f = FORMATS[fmt]
    torch.manual_seed(1)
    ps = [(torch.randn(s, device=dev) * 0.5).requires_grad_(True) for s in SHAPES]
    p0 = [p.detach().clone() for p in ps]
    inner = FusedAdamW(ps, lr=0.0, weight_decay=0.0)
    with_tiles(inner, ps)
    seed = 0x0123456789ABCDEF
    opt = OptimLP(inner, weight_quant=quant(f), seed=seed)
    for p in ps:
        p.grad = torch.randn_like(p)
    opt.step()
    for k, (p, x) in enumerate(zip(ps, p0)):
        off = lp_offset(1, k, 4)
        if f[0] == "float":
            want = mv.float_quantize(x, f[1], f[2], "stochastic", seed=seed, offset=off)
        else:
            want = mv.fixed_point_quantize(x, f[1], f[2], f[3], f[4], "stochastic", seed=seed, offset=off)
        assert torch.equal(bits(p), bits(want)), (k, p.shape)


def test_overflow_skip_changes_nothing_and_keeps_the_stream():
    f = FORMATS["float8_7_sr"]
    ps, qs, a, b, _ = make_pair("all", f, tiles=False)
    set_grads(ps, qs, 1, 1.0)
    before = [(p.detach().clone(), p.grad.clone(), a.acc[k].clone()) for k, p in enumerate(ps)]
    a.step(found_inf=torch.tensor([1.0], device=dev))
    assert a.step_count() == 0
    for k, p in enumerate(ps):
        assert torch.equal(bits(p), bits(before[k][0])) and torch.equal(bits(p.grad), bits(before[k][1]))
        assert torch.equal(bits(a.acc[k]), bits(before[k][2]))
        assert not a.state[p] or (a.state[p]["exp_avg"] == 0).all()
    a.step(found_inf=torch.tensor([0.0], device=dev))
    b.step()                                           # composed, its first real step: step index 1
    assert a.step_count() == 1 and b.step_count() == 1
    for k, (p, q) in enumerate(zip(ps, qs)):
        assert torch.equal(bits(p), bits(q)), k
        assert torch.equal(bits(a.acc[k]), bits(b.acc[k])), k


def _vit(fmt="FP16_32", seed=3):
    from myrtle_vision.models.vit import ViT
    case = CASES["classification"]
    torch.manual_seed(seed)
    return ViT(decoder="classification", image_size=case["image_size"], patch_size=16, num_classes=5,
               dim=128, depth=2, heads=2, mlp_dim=256, q_format=fmt).to(dev).train()


def test_model_operands_come_from_the_lp_kernel():
    import mv_native as mv
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from myrtle_vision.utils.optim import add_weight_decay
    from qtorch.optim import OptimLP
    case = CASES["classification"]
    m = _vit()
    twin = copy.deepcopy(m)
    img, tgt = make_inputs("classification", case, 11)
    img, tgt = img.to(dev), tgt.to(dev)
    kw = lp_kwargs("all", FORMATS["float8_7_sr"])
    ours = OptimLP(FusedAdamW(add_weight_decay(m, 0.05), lr=1e-3, model=m), seed=5, **kw)
    ref = OptimLP(FusedAdamW(add_weight_decay(twin, 0.05), lr=1e-3, model=twin), seed=5, fused=False, **kw)
    assert ours.fused
    for it in range(3):
        m.zero_grad(set_to_none=True)
        F.cross_entropy(m(img), tgt).backward()
        for p, q in zip(m.parameters(), twin.parameters()):
            q.grad = None if p.grad is None else p.grad.clone()
        ours.step()
        ref.step()
        n0 = mv.launch_count()
        m.engine().quantised_weights()
        assert mv.launch_count() == n0                 # operands came from the LP kernel
        for (n, p), q in zip(m.named_parameters(), twin.parameters()):
            assert torch.equal(bits(p), bits(q)), (it, n)
    eng = m.engine()
    e, man = eng.fmt
    for i, (qw, qwt) in eng._wq.items():
        want, want_t = mv.quantize_weight(eng.params[i].detach(), e, man, out_dtype=qw.dtype)
        assert torch.equal(qw, want) and torch.equal(qwt, want_t)


def test_composed_callable_refreshes_the_engine_operands():
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch.optim import OptimLP
    case = CASES["classification"]
    m = _vit()
    img, tgt = make_inputs("classification", case, 11)
    img, tgt = img.to(dev), tgt.to(dev)
    opt = OptimLP(FusedAdamW(m.parameters(), lr=1e-2, model=m), weight_quant=lambda t: t.half().float())
    assert not opt.fused
    F.cross_entropy(m(img), tgt).backward()
    opt.step()
    twin = _vit(seed=9)
    twin.load_state_dict(m.state_dict())
    for p in m.parameters():
        if p.grad is not None:
            assert torch.equal(p, p.half().float())
    with torch.no_grad():
        assert torch.equal(m(img), twin(img))


def test_stochastic_rounding_follows_small_updates():
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch.optim import OptimLP
    lr, steps, n = 2.0 ** -9, 4, 1024                  # (8,7) on [1, 2): grid step 2^-7, updates of a quarter of it

    def run(weight_quant, seed=0):
        p = torch.full((n,), 1.5, device=dev, requires_grad=True)
        inner = FusedAdamW([p], lr=lr, weight_decay=0.0)
        opt = OptimLP(inner, weight_quant=weight_quant, seed=seed) if weight_quant is not None else inner
        for _ in range(steps):
            p.grad = torch.ones_like(p)
            opt.step()
        return p.detach()

    exact = run(None)
    assert (exact < 1.5 - 3.9 * lr).all()
    assert (run(quant(("float", 8, 7, "nearest"))) == 1.5).all()          # every update lost
    sr = torch.stack([run(quant(FORMATS["float8_7_sr"]), seed) for seed in range(256)])
    mean, sigma = sr.mean(), sr.std() / sr.numel() ** 0.5
    assert abs(float(mean) - float(exact.mean())) < 3 * float(sigma), (float(mean), float(exact.mean()), float(sigma))


@pytest.mark.parametrize("fused", [None, False])
def test_resume_continues_bit_for_bit(fused, tmp_path):
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch.optim import OptimLP
    kw = lp_kwargs("all", FORMATS["float8_7_sr"])

    def fresh():
        torch.manual_seed(4)
        ps = [(torch.randn(s, device=dev) * 0.5).requires_grad_(True) for s in SHAPES]
        return ps, OptimLP(FusedAdamW(ps, lr=2e-3), fused=fused, **kw)

    def step(ps, opt, it):
        g = torch.Generator(device=dev).manual_seed(100 + it)
        for p in ps:
            p.grad = torch.randn(p.shape, device=dev, generator=g)
        opt.step(found_inf=torch.tensor([1.0 if it == 1 else 0.0], device=dev))   # step 1 overflows

    ps, opt = fresh()
    for it in range(5):
        step(ps, opt, it)
    ps2, opt2 = fresh()
    for it in range(3):
        step(ps2, opt2, it)
    path = tmp_path / "ckpt.pt"
    torch.save({"params": [p.detach().cpu() for p in ps2], "optimizer": opt2.state_dict()}, path)
    ck = torch.load(path, map_location="cpu")
    ps3, opt3 = fresh()
    with torch.no_grad():
        for p, saved in zip(ps3, ck["params"]):
            p.copy_(saved)
    opt3.load_state_dict(ck["optimizer"])
    for it in range(3, 5):
        step(ps3, opt3, it)
    assert opt3.step_count() == opt.step_count() == 4
    for k, (p, q) in enumerate(zip(ps, ps3)):
        assert torch.equal(bits(p), bits(q)), k
        assert torch.equal(bits(opt.acc[k]), bits(opt3.acc[k])), k


def test_trainer_with_optim_lp(tmp_path):
    from myrtle_vision.utils.models import get_models, get_optimizer_args
    from myrtle_vision.utils.optim import create_optimizer
    from myrtle_vision.utils.trainer import train_deit
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_train import config
    cfg = config("classification", tmp_path, "FP16_32", 80, 5)
    cfg["train_config"]["iters_per_checkpoint"] = 3
    lp = {"weight_quant": {"float": [8, 7]}, "grad_quant": {"float": [5, 10], "rounding": "nearest"},
          "momentum_quant": {"float": [8, 7]}, "acc_quant": None, "grad_scaling": 1.0, "seed": 17}
    cfg["train_config"]["optim_lp"] = lp
    history = train_deit(0, 1, copy.deepcopy(cfg), max_iterations=4)
    assert len(history) == 4 and all(torch.isfinite(torch.tensor(history)))
    ck = torch.load(os.path.join(cfg["train_config"]["output_directory"], "vit_000003"), map_location="cpu")
    assert ck["optimizer"]["seed"] == 17 and 1 <= ck["optimizer"]["step"] <= 3     # an overflow step does not count
    vit, _ = get_models(copy.deepcopy(cfg))
    vit = vit.to(dev)
    vit.load_state_dict(ck["model"])
    params = [p for g in create_optimizer(get_optimizer_args(cfg["train_config"]), vit).param_groups
              for p in g["params"]]
    stepped = list(ck["optimizer"]["optim"]["state"])
    assert stepped
    for k in stepped:
        p = params[k].detach()
        assert torch.equal(nearest(p, ("float", 8, 7)), p), k


def _rank_worker(rank, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "myrtle-vision_b200"))
    from myrtle_vision.utils.fused_adamw import FusedAdamW
    from qtorch import FloatingPoint
    from qtorch.optim import OptimLP
    from qtorch.quant import quantizer
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    torch.manual_seed(21)                              # ranks seeded alike
    ps = [(torch.randn(s) * 0.5).to(d).requires_grad_(True) for s in SHAPES]
    q = quantizer(FloatingPoint(8, 7), forward_rounding="stochastic")
    opt = OptimLP(FusedAdamW(ps, lr=1e-3), weight_quant=q, acc_quant=q)
    g = torch.Generator().manual_seed(3)
    for _ in range(3):
        for p in ps:
            p.grad = torch.randn(p.shape, generator=g).to(d)      # the same (all-reduced) gradients on every rank
        opt.step()
    ret[rank] = [p.detach().cpu().view(torch.int32).numpy().tobytes() for p in ps]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ranks_keep_bit_identical_parameters():
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_rank_worker, args=(ret,), nprocs=2, join=True)
    assert ret[0] == ret[1]
