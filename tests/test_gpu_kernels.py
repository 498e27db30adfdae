"""Floating-point kernels (tcgen05 GEMM + epilogues, LayerNorm, attention) vs a torch fp64
reference of the same op on the same inputs.  Tolerances are written at each assert."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
dev = "cuda"


def relmax(a, b):
    return ((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30)).item()


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 384, 512), (200, 45, 384), (1000, 384, 1536),
                                   (2501 * 2, 1152, 384), (520, 1536, 384), (384, 256, 8192)])
@pytest.mark.parametrize("a_major,b_major", [(0, 0), (1, 1), (1, 0), (0, 1)])
def test_gemm_layouts(M, N, K, a_major, b_major):
    import mv_native as mv
    if (a_major and M % 8) or (b_major and N % 8):
        pytest.skip("MN-major operands need a 16-byte row pitch")
    torch.manual_seed(0)
    A = torch.randn((K, M) if a_major else (M, K), device=dev).half()
    B = torch.randn((K, N) if b_major else (N, K), device=dev).half()
    out = torch.full((M, N), float("nan"), device=dev)
    mv.gemm(A, B, out, a_major=a_major, b_major=b_major)
    Af = A.double().t() if a_major else A.double()
    Bf = B.double().t() if b_major else B.double()
    # exact products, fp32 accumulation: 1e-5 of the largest entry (3e-5 for K = 8192)
    assert relmax(out, Af @ Bf.t()) < (1e-5 if K <= 2048 else 3e-5)


def test_gemm_tf32_kmajor():
    import mv_native as mv
    torch.manual_seed(0)
    A = torch.randn(256, 256, device=dev); B = torch.randn(128, 256, device=dev)
    out = torch.empty(256, 128, device=dev)
    mv.gemm(A, B, out)
    assert relmax(out, A.double() @ B.double().t()) < 2e-3        # tf32 operand truncation


def test_gemm_splitk_accumulate_and_epilogues():
    import mv_native as mv
    torch.manual_seed(1)
    T, No, Ki = 8192, 384, 1536
    dY = torch.randn(T, No, device=dev).half(); X = torch.randn(T, Ki, device=dev).half()
    out = torch.zeros(No, Ki, device=dev)
    mv.gemm(dY, X, out, a_major=1, b_major=1, accumulate=True)
    assert relmax(out, dY.double().t() @ X.double()) < 1e-5
    M, N, K = 514, 384, 384
    A = torch.randn(M, K, device=dev).half(); B = (torch.randn(N, K, device=dev) * 0.05).half()
    bias = torch.randn(N, device=dev); res = torch.randn(M, N, device=dev)
    lin = A.double() @ B.double().t() + bias.double()
    out = torch.empty(M, N, device=dev)
    mv.gemm(A, B, out, bias=bias, residual=res)
    assert relmax(out, lin + res.double()) < 1e-5
    # q_out: quantise in the epilogue == standalone quant of the fp32 result (up to fp32 sum order)
    outq = torch.empty(M, N, device=dev, dtype=torch.float16)
    mv.gemm(A, B, outq, bias=bias, q_out=(5, 10))
    want = mv.float_quantize(lin.float(), 5, 10)
    assert ((outq.float() - want).abs() > 0).float().mean().item() < 6e-3      # rare 1-ulp flips only
    assert relmax(outq, want) < 1e-3
    gp = torch.empty(M, N, device=dev, dtype=torch.float16); h = torch.empty_like(gp)
    mv.gemm(A, B, h, bias=bias, aux=gp, epilogue=mv.EPI_GELU, q_res=(5, 10))
    uu = lin.clone().requires_grad_(True)
    F.gelu(uu).sum().backward()
    # GELU epilogue: out = q(gelu(u)), aux = gelu'(u) saved for the backward
    assert relmax(h, F.gelu(lin)) < 1e-3 and relmax(gp, uu.grad) < 1e-3
    # DGELU epilogue: out = (A B^T) * aux
    d = torch.empty(M, N, device=dev, dtype=torch.float16)
    mv.gemm(A, B, d, aux=gp, epilogue=mv.EPI_DGELU)
    assert relmax(d, (A.double() @ B.double().t()) * uu.grad) < 2e-3
    # ... with the fused bias gradient: colsum += column sums of the stored values.  M = 514 has full tiles
    # (fast epilogue, red.add.v4 per 32-row group) and a 2-row tail (generic epilogue)
    for rows in (514, 512, 130):
        cs = torch.full((N,), 2.0, device=dev)
        d2 = torch.empty(rows, N, device=dev, dtype=torch.float16)
        mv.gemm(A[:rows], B, d2, aux=gp[:rows], epilogue=mv.EPI_DGELU, colsum=cs)
        assert torch.equal(d2, d[:rows])
        assert relmax(cs - 2.0, ((A[:rows].double() @ B.double().t()) * gp[:rows].double()).sum(0)) < 1e-4
    cs = torch.zeros(N, device=dev)
    o3 = torch.empty(M, N, device=dev)
    mv.gemm(A, B, o3, bias=bias, colsum=cs)              # no compile-time variant: generic epilogue
    assert relmax(cs, lin.sum(0)) < 1e-5
    # residual broadcast over images (positional embedding)
    pos = torch.randn(257, N, device=dev)
    A2 = torch.randn(2 * 257, K, device=dev).half()
    o2 = torch.empty(2 * 257, N, device=dev)
    mv.gemm(A2, B, o2, bias=bias, residual=pos, rows_per_img=257)
    assert relmax(o2, A2.double() @ B.double().t() + bias.double() + pos.double().repeat(2, 1)) < 1e-5


@pytest.mark.parametrize("T,No,Ki", [(8192, 1536, 384), (8200, 1152, 384), (4097, 384, 384), (8192, 384, 768),
                                     (65792, 200, 384)])
def test_gemm_wgrad_384_wide_tiles(T, No, Ki):
    """Split-K wgrad into outputs 384 (or a multiple) wide: 256 x 384 cluster tiles, two MMAs (N = 256, N = 128)
    per k step into one accumulator.  Against fp64 and against the 128-wide tiling, row tails included."""
    import mv_native as mv
    torch.manual_seed(T + No)
    dY = torch.randn(T, No, device=dev).half(); X = torch.randn(T, Ki, device=dev).half()
    ref = dY.double().t() @ X.double()
    for tile_n in (0, 384, 128):
        out = torch.full((No, Ki), 1.0, device=dev)
        mv.gemm(dY, X, out, a_major=1, b_major=1, accumulate=True, tile_n=tile_n)
        assert relmax(out - 1.0, ref) < 1e-5, tile_n
    # the same product accumulated into the transposed output: out_t[n, m] += acc[m, n]
    out_t = torch.full((Ki, No), 1.0, device=dev)
    mv.gemm(dY, X, out_t, a_major=1, b_major=1, accumulate=True, transpose_out=True)
    assert relmax(out_t - 1.0, ref.t()) < 1e-5


@pytest.mark.parametrize("M", [16384, 8192 + 40])
def test_gemm_epilogue_operands_and_outputs_by_tma(M):
    """The epilogue paths that move their operand / result by TMA (gemm2_kernel AUX = 1, 2, 3), at sizes where every
    cluster walks several tiles (the aux buffers are re-filled while the previous chunk is still in registers: a missing
    proxy fence showed up as a few hundred wrong values only from M ~ 8k upwards), with a ragged row tail.
      gelu' dgrad (fp16 aux chunk prefetched), with and without the fused bias gradient;
      x + Linear at K = 384 (fp32 residual chunk prefetched), FP16_32 and FP16_16 flags;
      plain fp16 outputs (TMA-store epilogue), with bias / with the (5,10) output quantiser."""
    import mv_native as mv
    torch.manual_seed(M)
    K = 384
    A = (torch.randn(M, K, device=dev) * 0.5).half()
    for _ in range(2):                                   # twice: different timing, same answer
        B = (torch.randn(1536, K, device=dev) * 0.1).half()
        aux = torch.rand(M, 1536, device=dev).half()
        want = (A.double() @ B.double().t()) * aux.double()
        for colsum in (False, True):
            d = torch.full((M, 1536), float("nan"), device=dev, dtype=torch.float16)
            cs = torch.zeros(1536, device=dev) if colsum else None
            mv.gemm(A, B, d, aux=aux, epilogue=mv.EPI_DGELU, colsum=cs)
            assert relmax(d, want) < 2e-3
            if colsum:
                assert relmax(cs, want.sum(0)) < 1e-4        # fp32 sums of the values before their fp16 rounding
        B = (torch.randn(384, K, device=dev) * 0.1).half()
        bias = torch.randn(384, device=dev); res = torch.randn(M, 384, device=dev)
        lin = A.double() @ B.double().t() + bias.double()
        o = torch.full((M, 384), float("nan"), device=dev)
        mv.gemm(A, B, o, bias=bias, residual=res)
        assert relmax(o, lin + res.double()) < 1e-5
        mv.gemm(A, B, o, bias=bias, residual=res, q_out=(5, 10), q_res=(5, 10))
        wantq = mv.float_quantize(mv.float_quantize(lin.float(), 5, 10) + res, 5, 10)
        assert ((o - wantq).abs() > 0).float().mean().item() < 6e-3 and relmax(o, wantq) < 1e-3
        B = (torch.randn(1152, K, device=dev) * 0.1).half()
        bias = torch.randn(1152, device=dev)
        lin = (A.double() @ B.double().t() + bias.double()).float()
        h = torch.full((M, 1152), float("nan"), device=dev, dtype=torch.float16)
        mv.gemm(A, B, h, bias=bias)
        assert relmax(h, lin) < 1e-3 and not torch.isnan(h.float()).any()
        mv.gemm(A, B, h, bias=bias, q_out=(5, 10))
        wantq = mv.float_quantize(lin, 5, 10)
        assert ((h.float() - wantq).abs() > 0).float().mean().item() < 6e-3 and relmax(h, wantq) < 1e-3


def test_gemm_rejects_mixed_operand_types():
    import mv_native as mv
    A = torch.zeros(128, 64, device=dev).half()
    for B in (torch.zeros(128, 64, device=dev).bfloat16(), torch.zeros(128, 64, device=dev)):
        with pytest.raises(mv.MvError, match="share one element type"):
            mv.gemm(A, B, torch.empty(128, 128, device=dev))


@pytest.mark.parametrize("D", [128, 192, 384, 768])
def test_layernorm_q(D):
    import mv_native as mv
    torch.manual_seed(D)
    rows = 1000
    x = torch.randn(rows, D, device=dev) * 3
    g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    y, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    xq = mv.float_quantize(x, 5, 10)
    ref = mv.float_quantize(F.layer_norm(xq.double(), (D,), g.double(), b.double(), 1e-5).float(), 5, 10)
    assert (y.float() - ref).abs().max().item() <= 2 ** -9 * ref.abs().max().item()   # <= 1 fp16 ulp
    assert ((y.float() != ref).float().mean().item()) < 2e-3
    y32, _, _ = mv.layernorm_q_fwd(x, g, b, out_dtype=torch.float32)
    assert (y32 - F.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-5).float()).abs().max() < 5e-6
    dy = torch.randn(rows, D, device=dev); dres = torch.randn(rows, D, device=dev)
    xr = xq.double().requires_grad_(True); gr = g.double().requires_grad_(True); br = b.double().requires_grad_(True)
    F.layer_norm(xr, (D,), gr, br, 1e-5).backward(dy.double())
    dg = torch.zeros(D, device=dev); db = torch.zeros(D, device=dev); dp = torch.zeros(D, device=dev)
    dx, dx16 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dgamma=dg, dbeta=db,
                                  dbias_prev=dp)
    want = xr.grad + dres.double()
    assert relmax(dx, want) < 1e-6 and relmax(dx16, want) < 1e-3
    assert relmax(dg, gr.grad) < 1e-5 and relmax(db, br.grad) < 1e-5 and relmax(dp, want.sum(0)) < 1e-5


def test_gradient_quantiser_sites_per_call():
    """QPyTorch's backward_number at the QuantStubs (mv_layernorm_q_bwd's q_grad / the dgrad GEMM's q_out), kernel by kernel
    against fp64 references: the fp32 arithmetic is within 1e-6 of them, so apart from a handful of near-tie flips the
    quantised values must be EQUAL (the model-level test can only bound the flips that fp16 containers add)."""
    import mv_native as mv
    torch.manual_seed(5)
    G = (5, 2)                                                   # E5M2 gradients
    rows, D = 2000, 384
    x = torch.randn(rows, D, device=dev) * 2
    g = 1 + 0.1 * torch.randn(D, device=dev); b = 0.1 * torch.randn(D, device=dev)
    _, mean, rstd = mv.layernorm_q_fwd(x, g, b, q_in=(5, 10), q_post=(5, 10))
    xq = mv.float_quantize(x, 5, 10)
    dy = torch.randn(rows, D, device=dev).half(); dres = torch.randn(rows, D, device=dev)
    xr = xq.double().requires_grad_(True)
    F.layer_norm(xr, (D,), g.double(), b.double(), 1e-5).backward(dy.double())
    dp = torch.zeros(D, device=dev)
    dx, dx16 = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10), dbias_prev=dp, q_grad=G)
    want = mv.float_quantize(xr.grad.float(), *G).double() + dres.double()       # the stub rounds BEFORE the residual add
    assert ((dx.double() - want).abs() > 1e-6 * want.abs().max()).float().mean().item() < 1e-3
    assert relmax(dp, want.sum(0)) < 1e-3
    plain, _ = mv.layernorm_q_bwd(dy, x, g, mean, rstd, dres=dres, q_in=(5, 10))  # and without q_grad, unrounded
    assert relmax(plain, xr.grad + dres.double()) < 1e-6
    # dgrad GEMMs: plain (stub in front of qkv / proj / fc1) and gelu' (stub in front of fc2: rounded BEFORE the multiply)
    M, N, K = 1000, 1536, 384
    A = (torch.randn(M, K, device=dev) * 0.5).half(); B = (torch.randn(N, K, device=dev) * 0.1).half()
    aux = torch.rand(M, N, device=dev).half()
    lin = (A.double() @ B.double().t())
    q = mv.float_quantize(lin.float(), *G).double()
    d = torch.empty(M, N, device=dev, dtype=torch.float16)
    mv.gemm(A, B, d, q_out=G)
    assert ((d.double() - q).abs() > 0).float().mean().item() < 1e-3
    cs = torch.zeros(N, device=dev)
    mv.gemm(A, B, d, aux=aux, epilogue=mv.EPI_DGELU, colsum=cs, q_out=G)
    want = q * aux.double()
    assert ((d.double() - want).abs() > 1e-3 * want.abs().max()).float().mean().item() < 1e-3
    assert relmax(cs, want.sum(0)) < 3e-2          # a flipped rounding moves a column sum by a whole E5M2 step


@pytest.mark.parametrize("B,H,N", [(1, 1, 64), (1, 1, 128), (2, 2, 257), (2, 3, 197), (1, 2, 1000), (1, 1, 17),
                                   (2, 1, 130), (2, 1, 131), (2, 1, 256), (1, 2, 272), (1, 1, 273), (40, 6, 257),
                                   (3, 2, 258), (2, 1, 259),      # odd keys: 2 (warp-MMA phase of the backward), 3 (third pass)
                                   (1, 6, 2501)])      # last: BASELINE config 5 (800 x 800 -> N = 2501), both det settings
def test_attention_fwd_bwd(B, H, N):
    """The sequence length picks the kernels: the short-sequence ones (attention_sn.cu) where they take N (backward:
    N <= 272; forward: mv_attention_sn_supported, which leaves N = 259 to the blocked forward), the blocked ones beyond."""
    import mv_native as mv
    torch.manual_seed(N)
    D = H * 64
    qkv = torch.randn(B * N, 3 * D, device=dev).half()
    out, lse = mv.attention_fwd(qkv, B, H, N)
    x = qkv.double().reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    q, k, v = [t.clone().requires_grad_(True) for t in (x[0], x[1], x[2])]
    s = (q @ k.transpose(-2, -1)) * 0.125
    o = (s.softmax(-1) @ v).transpose(1, 2).reshape(B * N, D)
    # fp16 probabilities on the tensor core: 2e-3 of the largest output
    assert relmax(out, o) < 2e-3
    assert (lse.double() - torch.logsumexp(s, -1) * 1.4426950408889634).abs().max() < 1e-3
    do = torch.randn(B * N, D, device=dev).half()
    o.backward(do.double())
    dbias = torch.full((3 * D,), 0.5, device=dev)
    dqkv = mv.attention_bwd(qkv, out, do, lse, B, H, N, dbias=dbias)
    # fused to_qkv bias gradient (+=): q from the stored dQ rows, v from the column sums of dO, k identically
    # zero in exact arithmetic (short-sequence kernel); column sums of dqkv otherwise
    ref_b = torch.stack([q.grad, k.grad, v.grad]).sum(dim=(1, 3)).reshape(3 * D)
    assert relmax(dbias - 0.5, ref_b) < 3e-3
    gq = dqkv.double().reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    for got, ref in zip(gq, (q.grad, k.grad, v.grad)):
        assert relmax(got, ref) < 3e-3
    # quantised output variant is exactly the quantisation of the plain one (same accumulators)
    outq, _ = mv.attention_fwd(qkv, B, H, N, q_out=(5, 10))
    assert relmax(outq, o) < 2e-3


def test_scale_f32():
    import mv_native as mv
    x = torch.randn(1000, 384, device=dev) * 300
    S = torch.tensor(2.0 ** 9, device=dev)
    y, yh = mv.scale_f32(x, S, want_f16=True)
    assert torch.equal(y, x * 512) and torch.equal(yh, (x * 512).clamp(-65504, 65504).half())
    z, none = mv.scale_f32(y, S, invert=True)
    assert torch.equal(z, x) and none is None
    mv.scale_f32(y, S.reshape(1), invert=True, out=y)                  # in place
    assert torch.equal(y, x)


def test_patchify_and_colsum():
    import mv_native as mv
    img = torch.randn(4, 3, 64, 96, device=dev)
    pt = mv.patchify_q(img, 16, q_in=(5, 10))
    ref = img.reshape(4, 3, 4, 16, 6, 16).permute(0, 2, 4, 3, 5, 1).reshape(4 * 24, 768).contiguous()
    assert torch.equal(pt.float(), mv.float_quantize(ref, 5, 10))
    pc = mv.patchify_q(img, 16, q_in=(5, 10), cls_slot=True).reshape(4, 25, 768)
    assert torch.equal(pc[:, 1:].reshape(-1, 768), pt) and pc[:, 0].abs().max() == 0
    for (C, Hh, Ww, P, fmt, dt) in [(3, 32, 48, 8, (5, 10), torch.float16), (1, 12, 24, 6, (8, 10), torch.float32),
                                    (4, 256, 256, 16, None, torch.float32)]:
        im = torch.randn(2, C, Hh, Ww, device=dev)
        got = mv.patchify_q(im, P, q_in=fmt, out_dtype=dt)
        want = im.reshape(2, C, Hh // P, P, Ww // P, P).permute(0, 2, 4, 3, 5, 1).reshape(-1, P * P * C)
        want = mv.float_quantize(want.contiguous(), *fmt) if fmt else want
        assert torch.equal(got.float(), want)
    a = torch.randn(8000, 1152, device=dev).half(); o = torch.zeros(1152, device=dev)
    mv.colsum(a, o)
    assert relmax(o, a.double().sum(0)) < 1e-5


@pytest.mark.parametrize("B,C,g,S", [(2, 17, 16, 256), (3, 4, 5, 80), (1, 24, 3, 48), (2, 32, 2, 32), (2, 7, 14, 224),
                                     (2, 19, 8, 64)])       # last: 8 pixels per cell (a warp spans six coarse cells), the 20-class tier
def test_fused_upsample_cross_entropy(B, C, g, S):
    """mv_upsample_ce against nn.Upsample(bilinear) + CrossEntropyLoss in fp64, incl. ignore_index."""
    from myrtle_vision.models.losses import upsampled_cross_entropy
    torch.manual_seed(C)
    y = (torch.randn(B, g * g, C, device=dev) * 3).requires_grad_(True)
    labels = torch.randint(0, C, (B, S, S), device=dev)
    labels[0, : S // 3, S // 2:] = -100
    loss = upsampled_cross_entropy(y, labels)
    (loss * 1.7).backward()
    yr = y.detach().double().requires_grad_(True)
    up = torch.nn.Upsample(size=S, mode="bilinear")(yr.transpose(1, 2).reshape(B, C, g, g))
    ref = F.cross_entropy(up, labels)
    (ref * 1.7).backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * abs(ref.item())
    assert relmax(y.grad, yr.grad) < 1e-4
    # all pixels ignored: zero loss, zero gradient, no NaN
    labels[:] = -100
    y.grad = None
    l0 = upsampled_cross_entropy(y, labels)
    l0.backward()
    assert l0.item() == 0.0 and float(y.grad.abs().max()) == 0.0


def test_persistent_kernels_repeat_bit_identically():
    """The CTA-pair GEMM and the short-sequence attention forward / backward stride a fixed share of the work per CTA
    in a fixed order: two identical calls give identical results."""
    import mv_native as mv
    torch.manual_seed(3)
    M, N, K = 4096, 1152, 384
    A = torch.randn(M, K, device=dev).half(); B = (torch.randn(N, K, device=dev) * 0.1).half()
    bias = torch.randn(N, device=dev)
    Bh, H, Nt = 5, 6, 257
    qkv = torch.randn(Bh * Nt, 3 * H * 64, device=dev).half()
    do = torch.randn(Bh * Nt, H * 64, device=dev).half()

    def run():
        out = torch.empty(M, N, device=dev, dtype=torch.float16)
        mv.gemm(A, B, out, bias=bias)
        o, lse = mv.attention_fwd(qkv, Bh, H, Nt, q_out=(5, 10))
        dbias = torch.zeros(3 * H * 64, device=dev)
        dqkv = mv.attention_bwd(qkv, o, do, lse, Bh, H, Nt, dbias=dbias)
        return out, o, lse, dqkv, dbias

    want = run()
    again = run()
    for w, g in zip(want[:4], again[:4]):
        assert torch.equal(w, g)
    assert relmax(again[4], want[4]) < 1e-5             # the fused bias gradient: CTAs of one head add in any order
