"""The overflow sink (mv_set_overflow_flag, include/mv_b200.h) site by site, and its registration around the engine.

Every kernel that rounds an unquantised value into an fp16 container raises the flag when the largest |value| it stores
is at least 65520: from there round-to-nearest passes 65504 and the container saturates.  mv_scale_f32 also raises it on
a non-finite result.  A missed raise trains on gradients clamped to 65504 where GradScaler would have skipped the step; a
false raise skips steps and backs the operand scale off for ever.  The tests build inputs whose fp32 results are exact
(or, for attention, at least 10 % away from the threshold) and compare the flag and the stored values with a plain
reference: +-65504 where the container saturates, never inf."""
import gc
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"
f16 = torch.float16

LIMIT = 65520.0                 # the least |value| whose fp16 rounding passes 65504
BELOW = 65519.9921875           # the largest fp32 value below it: stored as 65504, no raise
F16_MAX = 65504.0
VALUES = (BELOW, LIMIT, -LIMIT)


def flag_after(fn):
    """Zero a local device int, register it, run fn, unregister it (whatever happens) and read it back."""
    import mv_native as mv
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    mv.set_overflow_flag(flag)
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        mv.set_overflow_flag(None)
    return int(flag.item())


def raises(value):
    return abs(value) >= LIMIT


def stored(value):
    """What the fp16 container must hold for an exact fp32 value."""
    return float(np.float16(np.clip(value, -F16_MAX, F16_MAX)))


def seed_tensor(s):
    return torch.tensor([s], dtype=torch.int64, device=dev)


def keep_mask(rows, cols, p, seed, site):
    """The dropout mask of include/mv_b200.h ("dropout mask") from the library's 16-bit stream dump."""
    import mv_native as mv
    thr, _ = mv.drop_params(p)
    return (mv.philox_bits(rows * cols, seed, offset=site, half=True) >= thr).view(rows, cols)


# --------------------------------------------------------------------------------------------------------- GEMM
K = 64


def exact_operands(M, N, m, n, value, mul=1.0):
    """A [M, K], B [N, K] fp16, all zero except A[m, 0:2] = (1, 1) and B[n, 0:2] = two fp16 values whose fp32 sum is
    value / mul exactly (mul a power of two): C = A B^T is zero except C[m, n], in any summation order."""
    big = float(np.sign(value)) * F16_MAX
    A = torch.zeros(M, K, dtype=f16, device=dev)
    B = torch.zeros(N, K, dtype=f16, device=dev)
    A[m, 0:2] = 1.0
    B[n, 0] = big / mul
    B[n, 1] = (value - big) / mul
    assert float(B[n, 0].float()) + float(B[n, 1].float()) == value / mul
    return A, B


def ceil8(n):
    return (n + 7) // 8 * 8


def gemm_path(name, A, B, drop=None):
    """Run one fp16-output path of mv_gemm (dispatch in gemm2_host / mv_gemm) -> (out [M, N] fp16, colsum or None)."""
    import mv_native as mv
    M, N = A.shape[0], B.shape[0]
    cs = None
    if name == "v1_256":                    # variant 1, fast epi_chunk on 256-wide tiles
        out = torch.empty(M, N, dtype=f16, device=dev)
        mv.gemm(A, B, out, tile_n=256)
    elif name in ("v1_192", "v1_128"):      # variant 1, TMA-store chunk (16-byte row pitch)
        out = torch.empty(M, ceil8(N), dtype=f16, device=dev)[:, :N]
        mv.gemm(A, B, out, tile_n=int(name[3:]))
    elif name in ("v6_aux_tma", "v6_aux_ld", "v11"):   # gelu' dgrad (aux = 1): aux by TMA / unaligned ld_aux / + colsum
        pitch = ceil8(N) + (4 if name == "v6_aux_ld" else 0)
        aux = torch.ones(M, pitch, dtype=f16, device=dev)[:, :N]
        out = torch.empty(M, N, dtype=f16, device=dev)
        if name == "v11":
            cs = torch.zeros(N, device=dev)
        mv.gemm(A, B, out, aux=aux, epilogue=mv.EPI_DGELU, colsum=cs, tile_n=256)
    elif name == "generic":                 # out one element off its 8-byte alignment: generic chunks everywhere
        out = torch.empty(M * N + 1, dtype=f16, device=dev)[1:].view(M, N)
        mv.gemm(A, B, out)
    elif name == "tf32":                    # single-CTA kind::tf32 gemm_kernel: the fp16 values are exact tf32 operands
        out = torch.empty(M, N, dtype=f16, device=dev)
        mv.gemm(A.float(), B.float(), out)
    elif name == "drop":                    # the dropout instantiation's generic chunk, fp16 output
        out = torch.empty(M, N, dtype=f16, device=dev)
        mv.gemm(A, B, out, drop=drop)
    else:
        raise ValueError(name)
    return out, cs


GEMM_PATHS = ["v1_256", "v1_192", "v1_128", "v6_aux_tma", "v6_aux_ld", "v11", "generic", "tf32", "drop"]
# (M, N, row, column of the value): an interior full chunk; the last row and column of ragged tails; a tile late in a
# persistent CTA's walk (64 x 6 cluster tiles of 256 x 256 over 74 clusters; 128 x 12 single-CTA tiles over 148 CTAs)
PLACES = {"interior": (1024, 1536, 300, 700), "tail": (1000, 1500, 999, 1499), "late": (16384, 1536, 16383, 1535)}
DROP_P, DROP_SITE = 0.5, 5


def drop_seed_keeping(M, N, m, n, kept=True):
    """A seed whose mask keeps (or drops) element (m, n) of an [M, N] site tensor."""
    for s in range(1, 64):
        if bool(keep_mask(M, N, DROP_P, s, DROP_SITE)[m, n]) == kept:
            return s
    raise AssertionError("no seed found")


@pytest.mark.parametrize("place", list(PLACES))
@pytest.mark.parametrize("path", GEMM_PATHS)
def test_gemm_exact_threshold(path, place):
    """65519.9921875 stores 65504 and does not raise; 65520 and -65520 raise and store +-65504; every other output 0."""
    M, N, m, n = PLACES[place]
    drop, mul = None, 1.0
    if path == "drop":
        drop, mul = (seed_tensor(drop_seed_keeping(M, N, m, n)), DROP_P, DROP_SITE), 2.0   # kept: x 1 / (1 - p)
    for value in VALUES:
        A, B = exact_operands(M, N, m, n, value, mul)
        res = {}
        flag = flag_after(lambda: res.update(zip(("out", "cs"), gemm_path(path, A, B, drop))))
        out = res["out"]
        assert flag == int(raises(value)), (path, place, value)
        assert float(out[m, n]) == stored(value), (path, place, value, float(out[m, n]))
        out[m, n] = 0.0
        assert int(torch.count_nonzero(out)) == 0, (path, place, value)
        if res["cs"] is not None:       # the fused bias gradient sums the fp32 values, before the container rounding
            want = torch.zeros(N, device=dev)
            want[n] = value
            assert torch.equal(res["cs"], want)


@pytest.mark.parametrize("path", GEMM_PATHS)
def test_gemm_no_false_positive(path):
    """Random operands scaled so that the fp64 max |C| is about 65000: no raise, values as the reference."""
    M, N, _, _ = PLACES["tail"]
    torch.manual_seed(11)
    A = torch.randn(M, K, device=dev).half()
    Bf = torch.randn(N, K, device=dev)
    drop, mask = None, torch.ones(M, N, device=dev, dtype=torch.float64)
    if path == "drop":
        drop = (seed_tensor(3), DROP_P, DROP_SITE)
        mask = keep_mask(M, N, DROP_P, 3, DROP_SITE).double() * 2.0
    ref = (A.double() @ Bf.double().t()) * mask
    B = (Bf * (65000.0 / float(ref.abs().max()))).half()
    ref = (A.double() @ B.double().t()) * mask
    assert 64000.0 < float(ref.abs().max()) < 65400.0
    res = {}
    assert flag_after(lambda: res.update(out=gemm_path(path, A, B, drop)[0])) == 0, path
    err = (res["out"].double() - ref).abs()
    assert bool((err <= ref.abs() * 2 ** -11 + 0.05).all())          # half an fp16 ulp + fp32 summation order


@pytest.mark.parametrize("place", ["interior", "tail"])
def test_gemm_outputs_that_never_raise(place):
    """Accumulators far past 65520 that do not land unquantised in an fp16 container: the output quantisers clamp,
    GELU outputs are activations, fp32 outputs and split-K accumulation do not saturate."""
    import mv_native as mv
    M, N, m, n = PLACES[place]
    A, B = exact_operands(M, N, m, n, 2 * F16_MAX)       # C[m, n] = 131008
    h = lambda: torch.empty(M, N, dtype=f16, device=dev)
    cases = {
        "q_out": lambda: mv.gemm(A, B, h(), q_out=(5, 10)),
        "q_res": lambda: mv.gemm(A, B, h(), q_res=(5, 10)),
        "q_out_tf32": lambda: mv.gemm(A.float(), B.float(), h(), q_out=(5, 10)),
        "gelu": lambda: mv.gemm(A, B, h(), aux=h(), epilogue=mv.EPI_GELU),
        "gelu_q_res": lambda: mv.gemm(A, B, h(), aux=h(), epilogue=mv.EPI_GELU, q_res=(5, 10)),
        "fp32": lambda: mv.gemm(A, B, torch.empty(M, N, device=dev)),
        "fp32_tf32": lambda: mv.gemm(A.float(), B.float(), torch.empty(M, N, device=dev)),
        "accumulate": lambda: mv.gemm(A, B, torch.zeros(M, N, device=dev), accumulate=True),
    }
    for name, fn in cases.items():
        assert flag_after(fn) == 0, name
    o = torch.empty(M, N, device=dev)
    mv.gemm(A, B, o)
    assert float(o[m, n]) == 2 * F16_MAX


# -------------------------------------------------------------------------------------------- LayerNorm backward
@pytest.mark.parametrize("kind", ["f16", "f32", "grad_fmt", "drop"])
@pytest.mark.parametrize("D", [128, 192, 384, 768])
def test_layernorm_bwd_sites(D, kind):
    """dy = 0 makes dx = dres exactly; the value sits in the last row of a row count that is not a multiple of the eight
    rows a CTA takes.  Plain (fp16 / fp32 dy), with the gradient quantiser (q_grad), and the dropout variant,
    whose fp16 copy is the masked gradient: 40000 raises at a kept element (x 2) and not at a dropped one."""
    import mv_native as mv
    torch.manual_seed(D)
    rows = 1003
    x = torch.randn(rows, D, device=dev)
    g = 1 + 0.1 * torch.randn(D, device=dev)
    _, mean, rstd = mv.layernorm_q_fwd(x, g, torch.zeros(D, device=dev), q_in=(5, 10), q_post=(5, 10))
    dy = torch.zeros(rows, D, device=dev, dtype=torch.float32 if kind == "f32" else f16)
    seed = 77
    drop = (seed_tensor(seed), DROP_P, DROP_SITE) if kind == "drop" else None
    mul = torch.ones(rows, D, device=dev)
    if kind == "drop":
        mul = keep_mask(rows, D, DROP_P, seed, DROP_SITE).float() * 2.0
    kept_cols = torch.nonzero(mul[-1] > 0).flatten()
    col = int(kept_cols[-1])                                  # a kept column of the last row (every column without dropout)

    def run(dres, want_f16=True):
        out = {}

        def call():
            out["dx"], out["dx16"] = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), want_f16=want_f16,
                                                        q_grad=(5, 2) if kind == "grad_fmt" else None, drop=drop)
        return flag_after(call), out["dx"], out["dx16"]

    cases = [(col, v / float(mul[-1, col])) for v in VALUES]  # exact thresholds of the stored (masked) value
    if kind == "drop":
        dropped = int(torch.nonzero(mul[-1] == 0).flatten()[-1])
        cases += [(col, 40000.0), (dropped, 40000.0)]
    for c, v in cases:
        dres = torch.zeros(rows, D, device=dev)
        dres[-1, c] = v
        flag, dx, dx16 = run(dres)
        s = v * float(mul[-1, c])
        assert flag == int(raises(s)), (kind, D, c, v)
        assert torch.equal(dx, dres)                                   # the fp32 residual gradient is never masked
        want16 = torch.zeros(rows, D, device=dev)
        want16[-1, c] = stored(s)
        assert torch.equal(dx16.float(), want16), (kind, D, c, v)
    dres = torch.zeros(rows, D, device=dev)
    dres[-1, col] = 1e6
    assert run(dres, want_f16=False)[0] == 0                           # no fp16 copy: nothing to saturate


# ------------------------------------------------------------------------------------------------------ mv_dropout
@pytest.mark.parametrize("in_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("rows,cols", [(257, 384), (33, 13)])          # 16-byte vectors / element by element
def test_dropout(rows, cols, in_dtype):
    import mv_native as mv
    seed = 4242
    mask = keep_mask(rows, cols, DROP_P, seed, DROP_SITE)
    kept = int(torch.nonzero(mask[-1]).flatten()[-1])
    dropped = int(torch.nonzero(~mask[-1]).flatten()[-1])
    drop = (seed_tensor(seed), DROP_P, DROP_SITE)
    cases = [(kept, v / 2.0) for v in VALUES] + [(kept, 40000.0), (dropped, 40000.0)]
    for c, v in cases:
        x = torch.zeros(rows, cols, device=dev)
        x[-1, c] = v
        x = x.to(in_dtype)
        s = float(x[-1, c]) * (2.0 if c == kept else 0.0)
        res = {}
        flag = flag_after(lambda: res.update(out=mv.dropout(x, drop, out_dtype=f16)))
        assert flag == int(raises(s)), (c, v)
        want = torch.zeros(rows, cols, device=dev)
        want[-1, c] = stored(s)
        assert torch.equal(res["out"].float(), want)
        if in_dtype == torch.float32:                                  # fp32 output: never raises
            assert flag_after(lambda: res.update(out=mv.dropout(x, drop))) == 0
            assert float(res["out"][-1, c]) == s


# ------------------------------------------------------------------------------------------------------ scale_f32
N_SCALE = 1 << 22                  # more than one grid stride (148 * 8 CTAs x 256 threads x 4 elements)


@pytest.mark.parametrize("invert", [False, True])
def test_scale_f32_fp16_copy_threshold(invert):
    import mv_native as mv
    k = 9
    S = torch.tensor([2.0 ** (-k if invert else k)], device=dev)
    for idx in (0, N_SCALE - 1):
        for v in VALUES:
            x = torch.zeros(N_SCALE, device=dev)
            x[idx] = v * 2.0 ** -k
            res = {}
            flag = flag_after(lambda: res.update(zip(("o", "h"), mv.scale_f32(x, S, invert=invert, want_f16=True))))
            assert flag == int(raises(v)), (invert, idx, v)
            assert float(res["o"][idx]) == v and float(res["h"][idx].float()) == stored(v)
            assert int(torch.count_nonzero(res["h"])) == 1
        x = torch.zeros(N_SCALE, device=dev)
        x[idx] = float("nan")
        assert flag_after(lambda: mv.scale_f32(x, S, invert=invert, want_f16=True)) == 1


def test_scale_f32_fp32_nonfinite():
    """fp32 only: inf and NaN raise, wherever they are; finite values up to FLT_MAX never do, also when a float4 holds
    large values of both signs (their partial sums overflow to +inf and -inf)."""
    import mv_native as mv
    one = torch.ones(1, device=dev)
    for idx in (0, N_SCALE - 1):
        for bad in (float("inf"), float("-inf"), float("nan")):
            x = torch.zeros(N_SCALE, device=dev)
            x[idx] = bad
            assert flag_after(lambda: mv.scale_f32(x, one)) == 1, (idx, bad)
            assert flag_after(lambda: mv.scale_f32(x, one, invert=True)) == 1, (idx, bad)
    fmax = float(np.finfo(np.float32).max)
    x = torch.zeros(N_SCALE, device=dev)
    x[0], x[-1] = fmax, -fmax
    x[8:12] = torch.tensor([3e38, 3e38, -3e38, -3e38])
    x[16:20] = torch.tensor([3e38, -3e38, 3e38, -3e38])
    res = {}
    assert flag_after(lambda: res.update(o=mv.scale_f32(x, one)[0])) == 0
    assert torch.equal(res["o"], x)
    assert flag_after(lambda: mv.scale_f32(x, one, invert=True)) == 0


# ------------------------------------------------------------------------------------------------ attention backward
def attention_case(B, H, N, which, sel, gamma):
    """qkv fp16 [B*N, 3*H*64] and dO fp16 [B*N, H*64], zero except in the last image and head, built so that one
    gradient grows with gamma (the dO magnitude) and only at row / key `sel`:
      dv: every query attends to key sel (score 16), dO constant    -> dV[sel] ~ N * gamma
      dq: q = 0 (uniform P), K[sel] = 256 e1, V[sel] = 256 e0, dO[sel] = gamma e0     -> dQ[sel, 1]
      dk: q = 256 e1 everywhere, K = 0, V[sel] = 256 e0, dO = gamma e0                 -> dK[sel, 1]"""
    qkv = torch.zeros(B, N, 3, H, 64, device=dev)
    do = torch.zeros(B, N, H, 64, device=dev)
    q, k, v = qkv[-1, :, 0, -1], qkv[-1, :, 1, -1], qkv[-1, :, 2, -1]
    if which == "dv":
        q[:] = 2.0
        k[sel] = 1.0
        do[-1, :, -1] = gamma
    elif which == "dq":
        k[sel, 1] = 256.0
        v[sel, 0] = 256.0
        do[-1, sel, -1, 0] = gamma
    else:
        q[:, 1] = 256.0
        v[sel, 0] = 256.0
        do[-1, :, -1, 0] = gamma
    return qkv.reshape(B * N, 3 * H * 64).half(), do.reshape(B * N, H * 64).half()


def attention_ref(qkv, do, B, H, N):
    x = qkv.double().reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    q, k, v = [t.clone().requires_grad_(True) for t in (x[0], x[1], x[2])]
    o = ((q @ k.transpose(-2, -1)) * 0.125).softmax(-1) @ v
    o.transpose(1, 2).reshape(B * N, H * 64).backward(do.double())
    return torch.stack([q.grad, k.grad, v.grad]).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * H * 64)


@pytest.mark.parametrize("which", ["dq", "dk", "dv"])
@pytest.mark.parametrize("N", [257,        # short-sequence kernel: parked dQ / dK / dV slices
                               259,        # odd-key rows
                               272,        # rows >= 256
                               300,        # blocked: dQ by red.add, then dq_convert_kernel
                               2501])
def test_attention_bwd(N, which):
    """The flag equals (fp64 max |dq|, |dk|, |dv| >= 65520), with that max at most 0.9 or at least 1.1 times 65520."""
    import mv_native as mv
    B, H, sel = 2, 2, N - 1
    qkv, do = attention_case(B, H, N, which, sel, 1.0)
    unit = float(attention_ref(qkv, do, B, H, N).abs().max())
    for target in (0.8 * LIMIT, 1.25 * LIMIT):
        qkv, do = attention_case(B, H, N, which, sel, target / unit)
        ref = attention_ref(qkv, do, B, H, N)
        big = float(ref.abs().max())
        assert big <= 0.9 * LIMIT or big >= 1.1 * LIMIT, big
        assert float(ref.abs().max(dim=1).values.argmax()) % N == sel     # the largest value sits at row / key sel
        out, lse = mv.attention_fwd(qkv, B, H, N)
        res = {}
        flag = flag_after(lambda: res.update(d=mv.attention_bwd(qkv, out, do, lse, B, H, N)))
        assert flag == int(big >= LIMIT), (N, which, big)
        got = res["d"].double()
        assert torch.isfinite(got).all()
        assert float((got - ref.clamp(-F16_MAX, F16_MAX)).abs().max()) < 3e-3 * min(big, F16_MAX)


# ------------------------------------------------------------------------------------------------ overflow_update
def overflow_update_ref(flag, slot, state, backoff, growth, interval, min_target, max_target):
    """overflow_update_kernel (csrc/norm.cu) restated in fp32."""
    f32 = np.float32
    found = flag != 0
    if slot is not None:
        found = found or not (slot == 0.0)                  # NaN counts
    target, good = f32(state[1]), f32(state[2])
    if found:
        target, good = max(f32(target * f32(backoff)), f32(min_target)), f32(0.0)
    else:
        good = f32(good + f32(1.0))
        if good >= f32(interval):
            target, good = min(f32(target * f32(growth)), f32(max_target)), f32(0.0)
    return np.array([1.0 if (found or state[0] != 0.0) else 0.0, target, good], dtype=np.float32)


@pytest.mark.parametrize("with_slot", [False, True])
def test_overflow_update_sequence(with_slot):
    import mv_native as mv
    rng = random.Random(7 + with_slot)
    kw = dict(backoff=1.0 / 16, growth=2.0, growth_interval=3, min_target=2.0 ** -6, max_target=2.0 ** 6)
    state = torch.tensor([0.0, 1.0, 0.0], device=dev)
    ref = state.cpu().numpy()
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    slot = torch.zeros(1, device=dev) if with_slot else None
    hit_min = hit_max = sticky = 0
    for step in range(200):
        p_bad = (0.0, 0.05, 0.7)[(step // 20) % 3]
        f = rng.choice((1, 2, -1)) if rng.random() < p_bad else 0
        s = None
        if with_slot:
            s = rng.choice((1.0, float("nan"), 2.0 ** -70)) if rng.random() < p_bad else rng.choice((0.0, -0.0))
            slot.fill_(s)
        flag.fill_(f)
        if rng.random() < 0.5:                             # consumers clear found_inf; otherwise it stays sticky
            state[0] = 0.0
            ref[0] = 0.0
        elif ref[0] != 0.0:
            sticky += 1
        mv.overflow_update(flag, state, shared_slot=slot, **kw)
        want = overflow_update_ref(f, s, ref, kw["backoff"], kw["growth"], kw["growth_interval"], kw["min_target"],
                                   kw["max_target"])
        hit_min += bool(want[1] == kw["min_target"] and ref[1] * kw["backoff"] < kw["min_target"])
        hit_max += bool(want[1] == kw["max_target"] and ref[1] * kw["growth"] > kw["max_target"])
        ref = want
        got = state.cpu().numpy()
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (step, got, ref)
    assert hit_min and hit_max and sticky, (hit_min, hit_max, sticky)


# ------------------------------------------------------------------------------------------------ engine lifecycle
def small_vit(seed=2, fmt="FP16_32"):
    from myrtle_vision.models.vit import ViT
    torch.manual_seed(seed)
    return ViT(decoder="classification", image_size=80, patch_size=16, num_classes=5, dim=128, depth=2, heads=2,
               mlp_dim=256, q_format=fmt).to(dev).train()


def batch(seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.randn(4, 3, 80, 80, device=dev, generator=g).clamp(-1, 1),
            torch.randint(0, 5, (4,), device=dev, generator=g))


def train_step(model, img, tgt):
    import torch.nn.functional as F
    model.zero_grad(set_to_none=True)
    F.cross_entropy(model(img), tgt).backward()


def saturating_gemm():
    """A standalone call that saturates: fp16 output, no quantiser, accumulator 65520."""
    import mv_native as mv
    A, B = exact_operands(256, 256, 3, 5, LIMIT)
    out = torch.empty(256, 256, dtype=f16, device=dev)
    mv.gemm(A, B, out)
    return out


def test_engine_unregisters_its_flag():
    """The engine's flag is registered only while its own kernels run.  Each engine's `overflow` tensor stays alive
    here, so a stray write would land in memory this test owns."""
    img, tgt = batch()
    model = small_vit()
    held = []

    def check(what):
        for flag in held:
            flag.zero_()
        saturating_gemm()
        torch.cuda.synchronize()
        assert all(int(f.item()) == 0 for f in held), what

    def step(what):
        train_step(model, img, tgt)
        held.append(model.engine().overflow)
        check("after a training step " + what)

    step("")
    model.to(dev)                                  # rebuilds the engine on the next use
    check("after model.to(dev)")
    step("of the rebuilt engine")
    assert held[1] is not held[0]
    model.convert()                                # ModelQuantizer.convert: a new engine on the fp32-grade path
    check("after convert()")
    step("after convert()")
    del model
    gc.collect()
    check("after the model is deleted")
    # the standalone call itself still reports into a flag registered around it
    assert flag_after(saturating_gemm) == 1


def test_two_models_report_into_their_own_flags():
    """A and B interleaved, with a standalone saturating call between the forwards and the backwards (say, a caller's
    own projection): A's saturating backward raises A's found_inf only; B's stays 0."""
    import torch.nn.functional as F
    img, tgt = batch()
    a, b = small_vit(2), small_vit(3)
    ea, eb = a.engine(), b.engine()
    for m in (a, b):
        m.zero_grad(set_to_none=True)
    la = F.cross_entropy(a(img), tgt)
    lb = F.cross_entropy(b(img), tgt)
    saturating_gemm()
    ea.scaler_state[1] = 2.0 ** 40                 # A's fp16 gradient operands saturate
    la.backward()
    lb.backward()
    assert float(ea.found_inf) == 1.0 and float(eb.found_inf) == 0.0
    assert float(eb.scaler_state[1]) == 1024.0


def test_forward_qkv_saturation_skips_the_step():
    """FP16_32 stores qkv unquantised in fp16: a training forward whose qkv passes 65520 raises found_inf (the step is
    skipped; backing the gradient scale off does not cure it, so every later step is skipped as well).  An eval forward
    of the same input writes into no flag."""
    import mv_native as mv
    img, tgt = batch()
    model = small_vit()
    w = dict(model.named_parameters())["transformer.layers.0.0.fn.fn.to_qkv.1.weight"]
    with torch.no_grad():
        w.mul_(2.0 ** 17)
    eng = model.engine()
    train_step(model, img, tgt)
    assert float(eng.found_inf) == 1.0
    eng.found_inf.zero_()
    eng.overflow.zero_()
    user = torch.zeros(1, dtype=torch.int32, device=dev)
    model.eval()
    mv.set_overflow_flag(user)
    try:
        with torch.no_grad():
            model(img)
        torch.cuda.synchronize()
    finally:
        mv.set_overflow_flag(None)
    assert int(user.item()) == 0 and int(eng.overflow.item()) == 0 and float(eng.found_inf) == 0.0


def test_graphed_step_keeps_reporting():
    """A captured step keeps the flag pointer its kernels were captured with: scoping the registration to the engine's
    launches does not switch reporting off in replays."""
    import torch.nn.functional as F
    from myrtle_vision.utils.graph import GraphedTrainStep
    img, tgt = batch()
    model = small_vit()
    step = GraphedTrainStep(model, F.cross_entropy, img, tgt, warmup=2)
    eng = model.engine()
    eng.found_inf.zero_()
    eng.scaler_state[1] = 1024.0
    step()
    torch.cuda.synchronize()
    assert float(eng.found_inf) == 0.0
    eng.scaler_state[1] = 2.0 ** 40
    step()
    torch.cuda.synchronize()
    assert float(eng.found_inf) == 1.0 and float(eng.scaler_state[1]) == 2.0 ** 36
    eng.found_inf.zero_()
    eng.scaler_state[1] = 1024.0
    step()
    torch.cuda.synchronize()
    assert float(eng.found_inf) == 0.0
