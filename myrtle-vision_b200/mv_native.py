"""ctypes binding of the C-ABI CUDA library (include/mv_b200.h).

There is no CPU fallback: every wrapper requires CUDA tensors and raises if the library is
missing or a call fails.  PyTorch is used only for device memory and streams.
"""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "csrc", os.environ.get("MV_ALT_LIB") or "libmv_b200.so")   # MV_ALT_LIB: an experiment build (tools/build_variant.sh)
_lib = None

F32, F16 = 0, 1
ROUND_NEAREST, ROUND_STOCHASTIC = 0, 1
EPI_NONE, EPI_GELU, EPI_DGELU = 0, 1, 2

_DT = {torch.float32: F32, torch.float16: F16}


class MvError(RuntimeError):
    pass


class GemmArgs(ctypes.Structure):
    _fields_ = [
        ("M", ctypes.c_int), ("N", ctypes.c_int), ("K", ctypes.c_int),
        ("A", ctypes.c_void_p), ("lda", ctypes.c_int), ("a_dtype", ctypes.c_int), ("a_major", ctypes.c_int),
        ("B", ctypes.c_void_p), ("ldb", ctypes.c_int), ("b_dtype", ctypes.c_int), ("b_major", ctypes.c_int),
        ("bias", ctypes.c_void_p),
        ("residual", ctypes.c_void_p), ("ld_res", ctypes.c_int),
        ("aux", ctypes.c_void_p), ("ld_aux", ctypes.c_int),
        ("out", ctypes.c_void_p), ("ld_out", ctypes.c_int), ("out_dtype", ctypes.c_int),
        ("epilogue", ctypes.c_int),
        ("q_out_exp", ctypes.c_int), ("q_out_man", ctypes.c_int),
        ("q_res_exp", ctypes.c_int), ("q_res_man", ctypes.c_int),
        ("accumulate", ctypes.c_int),
        ("rows_per_img", ctypes.c_int),
        ("tile_n", ctypes.c_int),
        ("colsum", ctypes.c_void_p),
        ("transpose_out", ctypes.c_int),
        ("drop_seed", ctypes.c_void_p), ("drop_thr", ctypes.c_uint32), ("drop_scale", ctypes.c_float),
        ("drop_site", ctypes.c_int),
        ("round_seed", ctypes.c_void_p), ("round_offset", ctypes.c_uint64),
    ]


class LayerNormBwdArgs(ctypes.Structure):
    _fields_ = [
        ("dy", ctypes.c_void_p), ("dy_dtype", ctypes.c_int), ("ld_dy", ctypes.c_int64),
        ("x", ctypes.c_void_p), ("ld_x", ctypes.c_int64),
        ("dres", ctypes.c_void_p), ("ld_dres", ctypes.c_int64),
        ("gamma", ctypes.c_void_p), ("mean", ctypes.c_void_p), ("rstd", ctypes.c_void_p),
        ("dx", ctypes.c_void_p), ("ld_dx", ctypes.c_int64),
        ("dx_f16", ctypes.c_void_p), ("ld_lp", ctypes.c_int64),
        ("dgamma", ctypes.c_void_p), ("dbeta", ctypes.c_void_p), ("dbias_prev", ctypes.c_void_p),
        ("rows", ctypes.c_int), ("D", ctypes.c_int),
        ("q_in_exp", ctypes.c_int), ("q_in_man", ctypes.c_int),
        ("q_grad_exp", ctypes.c_int), ("q_grad_man", ctypes.c_int),
        ("round_seed", ctypes.c_void_p), ("round_offset", ctypes.c_uint64),
        ("drop_seed", ctypes.c_void_p), ("drop_thr", ctypes.c_uint32), ("drop_scale", ctypes.c_float),
        ("drop_site", ctypes.c_int), ("mask_dx", ctypes.c_int),
    ]


MIX_MODES = {"batch": 0, "pair": 1, "elem": 2}       # MV_MIX_BATCH / MV_MIX_PAIR / MV_MIX_ELEM


class MixSpec(ctypes.Structure):
    _fields_ = [("mixup_alpha", ctypes.c_float), ("cutmix_alpha", ctypes.c_float), ("prob", ctypes.c_float),
                ("switch_prob", ctypes.c_float), ("mode", ctypes.c_int)]


class MixRec(ctypes.Structure):
    """One mv_mix_rec; on the device the records of a batch are an int32 [B, 8] tensor (mix_records reads it)."""
    _fields_ = [("lam", ctypes.c_float), ("w_self", ctypes.c_float), ("w_other", ctypes.c_float),
                ("cutmix", ctypes.c_int), ("y0", ctypes.c_int), ("y1", ctypes.c_int), ("x0", ctypes.c_int),
                ("x1", ctypes.c_int)]


# ctypes signatures of entry points declared with full argument types (tests/test_distill_host.py and
# tests/test_mixup_host.py hold them to the header's prototypes)
_P, _I, _F = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
SIGNATURES = {
    "mv_token_row": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mv_distill_loss": [_P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _P],
    "mv_mix_draw": [_P, _I, _I, _I, _I, MixSpec, _P, _P],
    "mv_patchify_mix_q": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "mv_mix_ce_loss": [_P, _P, _P, _I, _I, _F, _P, _P, _P, _P],
}


def so_path():
    return _SO


def lib():
    """Load libmv_b200.so (built in-tree by csrc/build.py).  Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise MvError(
                "CUDA extension %s is missing: run `python -c 'import __graft_entry__ as g; "
                "g.build()'` (there is no CPU fallback)" % _SO)
        _lib = ctypes.CDLL(_SO)
        _lib.mv_last_error.restype = ctypes.c_char_p
        _lib.mv_launch_count.restype = ctypes.c_int64
        for name, args in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.argtypes, fn.restype = args, ctypes.c_int
    return _lib


def _check(rc, what):
    if rc != 0:
        raise MvError("%s failed: %s" % (what, lib().mv_last_error().decode()))


# Optional per-kernel-class CUDA-event timing (bench.py's roofline leg).  Off by default.
_TIMERS = None
_WORK = {}      # class -> (algorithmic flop, algorithmic HBM bytes) of ONE launch (DESIGN.md section 4 figures)


def enable_timing(on=True):
    global _TIMERS
    _TIMERS = {} if on else None
    if on:
        _WORK.clear()


def work_summary():
    """{class: (flop per launch, bytes per launch)} for the classes timed since enable_timing(True)."""
    return dict(_WORK)


def timing_summary():
    """{class: (launches, total_ms)} — call after torch.cuda.synchronize()."""
    out = {}
    for name, evs in (_TIMERS or {}).items():
        out[name] = (len(evs), sum(a.elapsed_time(b) for a, b in evs))
    return out


class _timed:
    def __init__(self, name, flop=0.0, nbytes=0.0):
        self.name = name
        if _TIMERS is not None:
            _WORK[name] = (float(flop), float(nbytes))

    def __enter__(self):
        if _TIMERS is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if _TIMERS is not None:
            self.e1.record()
            _TIMERS.setdefault(self.name, []).append((self.e0, self.e1))
        return False


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise MvError("myrtle-vision_b200 kernels need CUDA tensors (there is no CPU fallback)")


def set_overflow_flag(flag):
    """Register the device int32 the backward kernels raise on fp16 saturation / non-finite gradients (None: off)."""
    if flag is not None:
        _need_cuda(flag)
        assert flag.dtype == torch.int32 and flag.numel() >= 1
    _check(lib().mv_set_overflow_flag(_ptr(flag)), "mv_set_overflow_flag")


def overflow_update(flag, state, shared_slot=None, backoff=1.0 / 16, growth=2.0, growth_interval=2000,
                    min_target=2.0 ** -10, max_target=1024.0):
    """state fp32 [3] = {found_inf, scale_target, good_steps} (mv_overflow_update in include/mv_b200.h)."""
    _need_cuda(flag, state)
    assert state.dtype == torch.float32 and state.numel() == 3 and flag.dtype == torch.int32
    _check(lib().mv_overflow_update(_ptr(flag), _ptr(shared_slot), _ptr(state), ctypes.c_float(backoff),
                                    ctypes.c_float(growth), int(growth_interval), ctypes.c_float(min_target),
                                    ctypes.c_float(max_target), _stream()), "mv_overflow_update")


def launch_count():
    return int(lib().mv_launch_count())


# ------------------------------------------------------------------ dropout
def drop_params(p):
    """(thr, scale) of nn.Dropout(p) in the mask stream of include/mv_b200.h: keep = bits16 >= thr with
    thr = nearbyint(p * 65536), scale = 1 / (1 - p) in fp32 (0 for p == 1)."""
    p = float(p)
    if not 0.0 <= p <= 1.0:
        raise ValueError("dropout probability has to be between 0 and 1, but got %r" % (p,))
    thr = int(round(p * 65536.0))                  # round half to even, as nearbyint
    scale = 0.0 if p == 1.0 else float(np.float32(1.0) / np.float32(1.0 - p))
    return thr, scale


def _drop_args(drop):
    """drop = (seed, p, site): seed a 1-element int64 CUDA tensor holding the 64-bit seed."""
    seed, p, site = drop
    _need_cuda(seed)
    assert seed.dtype == torch.int64 and seed.numel() == 1
    thr, scale = drop_params(p)
    return ctypes.c_void_p(seed.data_ptr()), int(site), ctypes.c_uint32(thr), ctypes.c_float(scale)   # C argument order


def dropout(x, drop, *, out=None, out_dtype=None, tag="dropout"):
    """mv_dropout: out = x * keep * scale over a 2-D fp32 / fp16 tensor (row pitch honoured); out may be x."""
    _need_cuda(x)
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype in (torch.float32, torch.float16)
    if out is None:
        out = torch.empty(x.shape, dtype=out_dtype or x.dtype, device=x.device)
    assert out.dim() == 2 and out.stride(1) == 1 and out.shape == x.shape
    seed, site, thr, scale = _drop_args(drop)
    with _timed(tag, 0.0, x.numel() * (x.element_size() + out.element_size())):
        _check(lib().mv_dropout(_ptr(x), _DT[x.dtype], ctypes.c_int64(x.stride(0)), _ptr(out), _DT[out.dtype],
                                ctypes.c_int64(out.stride(0)), x.shape[0], x.shape[1], seed, site, thr, scale,
                                _stream()), "mv_dropout")
    return out


# ------------------------------------------------------------------ gradient rounding
def _round_args(grad_round):
    """grad_round = (seed, offset): seed a 1-element int64 CUDA tensor holding the 64-bit seed, offset the stream's
    site + (rank << 32) (include/mv_b200.h "gradient rounding stream")."""
    seed, offset = grad_round
    _need_cuda(seed)
    assert seed.dtype == torch.int64 and seed.numel() == 1
    return ctypes.c_void_p(seed.data_ptr()), ctypes.c_uint64(int(offset))


def float_quantize_dev(x, exp, man, grad_round, out=None, out_dtype=torch.float32):
    """mv_float_quantize_dev: stochastic float_quantize with the seed read from device memory."""
    _need_cuda(x)
    x = x.contiguous()
    if x.dtype != torch.float32:
        x = x.float()
    if out is None:
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    assert out.is_contiguous() and out.numel() == x.numel()
    seed, offset = _round_args(grad_round)
    with _timed("quant_grad", 0.0, x.numel() * (4 + out.element_size())):
        _check(lib().mv_float_quantize_dev(_ptr(x), _ptr(out), _DT[out.dtype], ctypes.c_int64(x.numel()), int(exp),
                                           int(man), seed, offset, _stream()), "mv_float_quantize_dev")
    return out


# ------------------------------------------------------------------ fake-quant
def float_quantize(x, exp, man, rounding="nearest", seed=0, offset=0, out=None,
                   out_dtype=torch.float32):
    _need_cuda(x)
    x = x.contiguous()
    if x.dtype != torch.float32:
        x = x.float()
    if out is None:
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    rc = lib().mv_float_quantize(_ptr(x), _ptr(out), _DT[out.dtype], ctypes.c_int64(x.numel()),
                                 int(exp), int(man),
                                 ROUND_STOCHASTIC if rounding == "stochastic" else ROUND_NEAREST,
                                 ctypes.c_uint64(seed), ctypes.c_uint64(offset), _stream())
    _check(rc, "mv_float_quantize")
    return out


def fixed_point_quantize(x, wl, fl, clamp=True, symmetric=False, rounding="nearest", seed=0,
                         offset=0, with_mask=False, out=None):
    _need_cuda(x)
    x = x.contiguous().float()
    if out is None:
        out = torch.empty_like(x)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == x.numel()
    mask = torch.empty(x.shape, dtype=torch.uint8, device=x.device) if with_mask else None
    rc = lib().mv_fixed_point_quantize(_ptr(x), _ptr(out), _ptr(mask), ctypes.c_int64(x.numel()),
                                       int(wl), int(fl), int(bool(clamp)), int(bool(symmetric)),
                                       ROUND_STOCHASTIC if rounding == "stochastic" else ROUND_NEAREST,
                                       ctypes.c_uint64(seed), ctypes.c_uint64(offset), _stream())
    _check(rc, "mv_fixed_point_quantize")
    return (out, mask) if with_mask else out


def block_quantize(x, wl, dim=-1, rounding="nearest", seed=0, offset=0, out=None):
    _need_cuda(x)
    x = x.contiguous().float()
    if out is None:
        out = torch.empty_like(x)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == x.numel()
    if dim is None or dim < 0:
        outer, dsize, inner, whole = 1, 1, x.numel(), 1
    else:
        shape = list(x.shape)
        outer = 1
        for s in shape[:dim]:
            outer *= s
        dsize = shape[dim]
        inner = 1
        for s in shape[dim + 1:]:
            inner *= s
        whole = 0
    ws = torch.empty(max(dsize, 1), dtype=torch.float32, device=x.device)
    rc = lib().mv_block_quantize(_ptr(x), _ptr(out), _ptr(ws), ctypes.c_int64(outer),
                                 ctypes.c_int64(dsize), ctypes.c_int64(inner), whole, int(wl),
                                 ROUND_STOCHASTIC if rounding == "stochastic" else ROUND_NEAREST,
                                 ctypes.c_uint64(seed), ctypes.c_uint64(offset), _stream())
    _check(rc, "mv_block_quantize")
    return out


def philox_bits(n, seed, offset=0, device="cuda", half=False):
    """The random stream of the stochastic kernels; half=True: the 16-bit stream of float_quantize for man >= 7."""
    out = torch.empty(n, dtype=torch.int32, device=device)
    fn = lib().mv_philox_bits16 if half else lib().mv_philox_bits
    _check(fn(_ptr(out), ctypes.c_int64(n), ctypes.c_uint64(seed), ctypes.c_uint64(offset), _stream()), "mv_philox_bits")
    return out


def quantize_weight(w, exp, man, out_dtype=torch.float16, transpose=True, out=None, out_t=None):
    _need_cuda(w)
    assert w.dim() == 2 and w.dtype == torch.float32 and w.is_contiguous()
    rows, cols = w.shape
    if out is None:
        out = torch.empty(rows, cols, dtype=out_dtype, device=w.device)
    if transpose and out_t is None:
        out_t = torch.empty(cols, rows, dtype=out_dtype, device=w.device)
    rc = lib().mv_quantize_weight(_ptr(w), _ptr(out), _ptr(out_t) if transpose else None,
                                  _DT[out.dtype], rows, cols, int(exp), int(man), _stream())
    _check(rc, "mv_quantize_weight")
    return out, out_t


# ------------------------------------------------------------------------ GEMM
def gemm(A, B, out, *, a_major=0, b_major=0, bias=None, residual=None, aux=None,
         epilogue=EPI_NONE, q_out=None, q_res=None, accumulate=False, rows_per_img=0,
         M=None, N=None, K=None, tag=None, tile_n=0, colsum=None, transpose_out=False, drop=None,
         grad_round=None):
    """out[M,N] = A . B^T over K with the fused epilogue of mv_gemm (include/mv_b200.h).
    a_major/b_major = 0: operand is [M|N, K] (K contiguous); 1: operand is [K, M|N].
    fp16 operands run on the CTA-pair kernel, fp32 operands (tf32) on the single-CTA kernel.
    drop = (seed, p, site): dropout of the output after q_out (seed: int64 [1] CUDA tensor), None: off.
    grad_round = (seed, offset): q_out rounds stochastically, None: nearest."""
    _need_cuda(A, B, out)
    assert A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1
    if M is None:
        M = A.shape[0] if a_major == 0 else A.shape[1]
    if K is None:
        K = A.shape[1] if a_major == 0 else A.shape[0]
    if N is None:
        N = B.shape[0] if b_major == 0 else B.shape[1]
    a = GemmArgs()
    a.M, a.N, a.K = M, N, K
    # an element type without a code (e.g. bf16) goes in as -1: mv_gemm rejects it with the reason, before any launch
    a.A, a.lda, a.a_dtype, a.a_major = A.data_ptr(), A.stride(0), _DT.get(A.dtype, -1), a_major
    a.B, a.ldb, a.b_dtype, a.b_major = B.data_ptr(), B.stride(0), _DT.get(B.dtype, -1), b_major
    a.bias = bias.data_ptr() if bias is not None else None
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.stride(-1) == 1
        a.residual, a.ld_res = residual.data_ptr(), residual.stride(-2)
    if aux is not None:
        assert aux.dtype == torch.float16
        a.aux, a.ld_aux = aux.data_ptr(), aux.stride(-2)
    a.out, a.ld_out, a.out_dtype = out.data_ptr(), out.stride(-2), _DT.get(out.dtype, -1)
    a.epilogue = epilogue
    if q_out:
        a.q_out_exp, a.q_out_man = q_out
    if q_res:
        a.q_res_exp, a.q_res_man = q_res
    a.accumulate = int(bool(accumulate))
    a.rows_per_img = rows_per_img
    a.tile_n = tile_n
    a.transpose_out = int(bool(transpose_out))
    if colsum is not None:
        assert colsum.dtype == torch.float32 and colsum.is_contiguous() and colsum.numel() == N
        a.colsum = colsum.data_ptr()
    if drop is not None:
        seed, site, thr, scale = _drop_args(drop)
        a.drop_seed, a.drop_thr, a.drop_scale, a.drop_site = seed.value, thr.value, scale.value, site
    if grad_round is not None:
        seed, offset = _round_args(grad_round)
        a.round_seed, a.round_offset = seed.value, offset.value
    kind = "gemm_wgrad" if accumulate else ("gemm_dgrad" if epilogue == EPI_DGELU or tag == "dgrad"
                                            else "gemm_fwd")
    flop = nbytes = 0.0
    if _TIMERS is not None:
        kind = "%s_%dx%dx%d" % (kind, M, N, K)    # one roofline line per GEMM shape (M x N x K)
        # algorithmic traffic: both operands once, every output once, epilogue operands once
        flop = 2.0 * M * N * K
        nbytes = (M * K * A.element_size() + N * K * B.element_size() + M * N * out.element_size()
                  * (2 if accumulate else 1))
        if residual is not None:
            nbytes += (rows_per_img if rows_per_img else M) * N * 4
        if aux is not None:
            nbytes += M * N * 2
    with _timed(kind, flop, nbytes):
        _check(lib().mv_gemm(ctypes.byref(a), _stream()), "mv_gemm")
    return out


# ------------------------------------------------------------- LayerNorm & helpers
def _fmt(f):
    return (int(f[0]), int(f[1])) if f else (0, 0)


def layernorm_q_fwd(x, gamma, beta, *, q_in=None, q_post=None, out_dtype=torch.float16, eps=1e-5,
                    save_stats=True, tag=None):
    _need_cuda(x, gamma, beta)
    D = x.shape[-1]
    x2 = x.reshape(-1, D)
    assert x2.dtype == torch.float32 and x2.stride(1) == 1
    rows = x2.shape[0]
    y = torch.empty(rows, D, dtype=out_dtype, device=x.device)
    mean = torch.empty(rows, dtype=torch.float32, device=x.device) if save_stats else None
    rstd = torch.empty(rows, dtype=torch.float32, device=x.device) if save_stats else None
    qi, qp = _fmt(q_in), _fmt(q_post)
    with _timed(tag or "ln_fwd", 0.0, rows * D * (4 + y.element_size())):
        rc = lib().mv_layernorm_q_fwd(_ptr(x2), ctypes.c_int64(x2.stride(0)), _ptr(gamma), _ptr(beta),
                                      _ptr(y), ctypes.c_int64(D), _DT[out_dtype], _ptr(mean), _ptr(rstd),
                                      rows, D, ctypes.c_float(eps), qi[0], qi[1], qp[0], qp[1], _stream())
    _check(rc, "mv_layernorm_q_fwd")
    return y.reshape(x.shape), mean, rstd


def layernorm_q_bwd(dy, x, gamma, mean, rstd, *, dres=None, q_in=None, dgamma=None, dbeta=None,
                    dbias_prev=None, want_f16=True, dx=None, dx_f16=None, tag=None, q_grad=None, drop=None, mask_dx=False,
                    grad_round=None):
    """mv_layernorm_q_bwd (include/mv_b200.h).  q_grad = (exp, man): the gradient quantiser rounds the LayerNorm-input
    gradient, None: off.  drop = (seed, p, site): dx_f16 and dbias_prev see the masked gradient, dx too when mask_dx.
    grad_round = (seed, offset): q_grad rounds stochastically, None: nearest.  q_grad and drop take fp16 dy."""
    _need_cuda(dy, x)
    D = x.shape[-1]
    x2, dy2 = x.reshape(-1, D), dy.reshape(-1, D)
    rows = x2.shape[0]
    assert dy2.dtype in (torch.float32, torch.float16) and x2.dtype == torch.float32
    if dx is None:
        dx = torch.empty(rows, D, dtype=torch.float32, device=x.device)
    if want_f16 and dx_f16 is None:
        dx_f16 = torch.empty(rows, D, dtype=torch.float16, device=x.device)
    dres2 = dres.reshape(-1, D) if dres is not None else None
    # x 4 + dy + dres 4 read, dx 4 + fp16 copy 2 written
    with _timed(tag or "ln_bwd", 0.0, rows * D * (4 + dy2.element_size() + (4 if dres is not None else 0) + 4
                                            + (2 if dx_f16 is not None else 0))):
        a = LayerNormBwdArgs(
            dy=dy2.data_ptr(), dy_dtype=_DT[dy2.dtype], ld_dy=dy2.stride(0), x=x2.data_ptr(), ld_x=x2.stride(0),
            dres=_ptr(dres2), ld_dres=dres2.stride(0) if dres2 is not None else D,
            gamma=_ptr(gamma), mean=_ptr(mean), rstd=_ptr(rstd), dx=dx.data_ptr(), ld_dx=dx.stride(0),
            dx_f16=_ptr(dx_f16), ld_lp=D, dgamma=_ptr(dgamma), dbeta=_ptr(dbeta), dbias_prev=_ptr(dbias_prev),
            rows=rows, D=D, mask_dx=int(bool(mask_dx)))
        a.q_in_exp, a.q_in_man = _fmt(q_in)
        a.q_grad_exp, a.q_grad_man = _fmt(q_grad)
        if grad_round is not None:
            seed, offset = _round_args(grad_round)
            a.round_seed, a.round_offset = seed.value, offset.value
        if drop is not None:
            seed, site, thr, scale = _drop_args(drop)
            a.drop_seed, a.drop_thr, a.drop_scale, a.drop_site = seed.value, thr.value, scale.value, site
        rc = lib().mv_layernorm_q_bwd(ctypes.byref(a), _stream())
    _check(rc, "mv_layernorm_q_bwd")
    return dx, dx_f16


def colsum(x2d, out):
    _need_cuda(x2d, out)
    assert x2d.dim() == 2 and x2d.stride(1) == 1 and out.dtype == torch.float32
    with _timed("colsum", 0.0, x2d.numel() * x2d.element_size()):
        rc = lib().mv_colsum(_ptr(x2d), _DT[x2d.dtype], ctypes.c_int64(x2d.stride(0)), x2d.shape[0],
                             x2d.shape[1], _ptr(out), _stream())
    _check(rc, "mv_colsum")
    return out


def patchify_q(img, patch, q_in=None, out_dtype=torch.float16, cls_slot=False):
    """cls_slot: False / 0 (patch rows only), True / 1 (a zero class-token row first per image) or 2 (a zero row first
    and a zero row last per image: the class- and distillation-token slots)."""
    _need_cuda(img)
    img = img.contiguous().float()
    B, C, H, W = img.shape
    cls_slot = int(cls_slot)
    rows = B * ((H // patch) * (W // patch) + cls_slot)
    out = torch.empty(rows, patch * patch * C, dtype=out_dtype, device=img.device)
    q = _fmt(q_in)
    with _timed("patchify", 0.0, img.numel() * 4 + out.numel() * out.element_size()):
        _check(lib().mv_patchify_q(_ptr(img), _ptr(out), _DT[out_dtype], B, C, H, W, patch, q[0], q[1],
                                   cls_slot, _stream()), "mv_patchify_q")
    return out


def mix_draw(seed, B, H, W, spec, rank=0, recs=None):
    """mv_mix_draw: -> the records of one mixed batch, int32 [B, 8] on the device (mv_mix_rec each: use mix_records to
    read them).  seed: a 1-element int64 CUDA tensor; spec: a MixSpec."""
    _need_cuda(seed)
    assert seed.dtype == torch.int64 and seed.numel() == 1
    if recs is None:
        recs = torch.empty(B, 8, dtype=torch.int32, device=seed.device)
    assert recs.dtype == torch.int32 and recs.shape == (B, 8) and recs.is_contiguous()
    _check(lib().mv_mix_draw(_ptr(seed), int(rank), int(B), int(H), int(W), spec, _ptr(recs), _stream()),
           "mv_mix_draw")
    return recs


def mix_records(recs):
    """int32 [B, 8] records -> {"lam", "w_self", "w_other": fp32 [B]; "cutmix", "y0", "y1", "x0", "x1": int32 [B]}."""
    f = recs[:, :3].view(torch.float32)
    out = {"lam": f[:, 0], "w_self": f[:, 1], "w_other": f[:, 2]}
    out.update({k: recs[:, 3 + i] for i, k in enumerate(("cutmix", "y0", "y1", "x0", "x1"))})
    return out


def _check_recs(recs, B):
    _need_cuda(recs)
    assert recs.dtype == torch.int32 and recs.shape == (B, 8) and recs.is_contiguous(), "records must be int32 [B, 8]"


def patchify_mix_q(img, recs, patch, q_in=None, out_dtype=torch.float16, cls_slot=False):
    """patchify_q of the batch mixed as the records (mix_draw) say, in one pass (mv_patchify_mix_q)."""
    _need_cuda(img)
    img = img.contiguous().float()
    B, C, H, W = img.shape
    _check_recs(recs, B)
    cls_slot = int(cls_slot)
    rows = B * ((H // patch) * (W // patch) + cls_slot)
    out = torch.empty(rows, patch * patch * C, dtype=out_dtype, device=img.device)
    q = _fmt(q_in)
    with _timed("patchify_mix", 0.0, img.numel() * 8 + out.numel() * out.element_size()):
        _check(lib().mv_patchify_mix_q(_ptr(img), _ptr(recs), _ptr(out), _DT[out_dtype], B, C, H, W, patch, q[0], q[1],
                                       cls_slot, _stream()), "mv_patchify_mix_q")
    return out


def mix_ce_loss(logits, labels, recs, smoothing):
    """mv_mix_ce_loss: -> (loss fp32 [1], d loss / d logits), on the device.  logits fp32 [B, C], labels int64 [B],
    recs the records of the mixed batch or None (unmixed: label-smoothed cross-entropy)."""
    _need_cuda(logits, labels)
    logits = logits.detach().float().contiguous()
    labels = labels.contiguous()
    assert logits.dim() == 2, "logits must be [B, C]"
    assert labels.dtype == torch.int64 and labels.shape == logits.shape[:1], "labels must be int64 [B]"
    B, C = logits.shape
    if recs is not None:
        _check_recs(recs, B)
    loss = torch.empty(1, dtype=torch.float32, device=logits.device)
    rows = torch.empty(B, dtype=torch.float32, device=logits.device)
    dx = torch.empty_like(logits)
    with _timed("mix_ce_loss", 0.0, B * C * 4 * 3):
        _check(lib().mv_mix_ce_loss(_ptr(logits), _ptr(labels), _ptr(recs), B, C, ctypes.c_float(smoothing),
                                    _ptr(loss), _ptr(rows), _ptr(dx), _stream()), "mv_mix_ce_loss")
    return loss, dx


def cls_rows(cls, pos_q, x, B, n_tokens, D, q_ff=None):
    q = _fmt(q_ff)
    _check(lib().mv_cls_rows(_ptr(cls), _ptr(pos_q), _ptr(x), B, n_tokens, D, q[0], q[1], _stream()),
           "mv_cls_rows")


def token_row(tok, x, B, n_tokens, D, row, q_ff=None):
    """mv_token_row: x[b, row, :] = q_ff(tok) for every image of the token-major fp32 x [B * n_tokens, D]."""
    _need_cuda(tok, x)
    assert tok.dtype == torch.float32 and tok.is_contiguous() and tok.numel() == D
    assert x.dtype == torch.float32 and x.is_contiguous() and x.numel() == B * n_tokens * D
    q = _fmt(q_ff)
    _check(lib().mv_token_row(_ptr(tok), _ptr(x), B, n_tokens, D, int(row), q[0], q[1], _stream()), "mv_token_row")


def distill_loss(student, distill, teacher, labels, temperature, alpha, hard):
    """mv_distill_loss: -> (loss fp32 [1], d loss / d student, d loss / d distill), all on the device.  student,
    distill, teacher: fp32 [B, C]; labels: int64 [B]."""
    _need_cuda(student, distill, teacher, labels)
    student, distill, teacher = (t.detach().float().contiguous() for t in (student, distill, teacher))
    labels = labels.contiguous()
    assert student.dim() == 2 and student.shape == distill.shape == teacher.shape, "logits must all be [B, C]"
    assert labels.dtype == torch.int64 and labels.shape == student.shape[:1], "labels must be int64 [B]"
    B, C = student.shape
    loss = torch.empty(1, dtype=torch.float32, device=student.device)
    rows = torch.empty(B, dtype=torch.float32, device=student.device)
    ds, dd = torch.empty_like(student), torch.empty_like(distill)
    with _timed("distill_loss", 0.0, B * C * 4 * 5):
        _check(lib().mv_distill_loss(_ptr(student), _ptr(distill), _ptr(teacher), _ptr(labels), B, C,
                                     ctypes.c_float(temperature), ctypes.c_float(alpha), int(bool(hard)), _ptr(loss),
                                     _ptr(rows), _ptr(ds), _ptr(dd), _stream()), "mv_distill_loss")
    return loss, ds, dd


def scale_f32(x, scale, *, invert=False, out=None, out_h=None, want_f32=True, want_f16=False):
    """(x * scale [or / scale]) as fp32 and / or saturating fp16, `scale` a 0-dim / 1-element device tensor."""
    _need_cuda(x, scale)
    assert x.dtype == torch.float32 and scale.dtype == torch.float32 and scale.numel() == 1
    x = x.contiguous()
    if out is None and want_f32:
        out = torch.empty_like(x)
    if out_h is None and want_f16:
        out_h = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    _check(lib().mv_scale_f32(_ptr(x), _ptr(scale), int(bool(invert)), _ptr(out), _ptr(out_h),
                              ctypes.c_int64(x.numel()), _stream()), "mv_scale_f32")
    return out, out_h


def widen_transpose(x2d, *, want_copy=False, want_t=True, mul=1.0, padded=False):
    """fp16/fp32 [rows, cols] -> (fp32 copy or None, fp32 transpose [cols, rows] or None).  The
    transpose is a view of a buffer whose row pitch is padded to 16 bytes (TMA global stride rule)."""
    _need_cuda(x2d)
    assert x2d.dim() == 2 and x2d.stride(1) == 1 and x2d.dtype in (torch.float16, torch.float32)
    rows, cols = x2d.shape
    out = torch.empty(rows, cols, dtype=torch.float32, device=x2d.device) if want_copy else None
    pitch = (rows + 3) // 4 * 4
    alloc = torch.empty if pitch == rows else torch.zeros      # pad columns may be read as K (3xTF32 split)
    base_t = alloc(cols, pitch, dtype=torch.float32, device=x2d.device) if want_t else None
    out_t = base_t[:, :rows] if want_t else None
    _check(lib().mv_widen_transpose(_ptr(x2d), _DT[x2d.dtype], ctypes.c_int64(x2d.stride(0)), rows, cols,
                                    _ptr(out), _ptr(out_t), ctypes.c_int64(pitch), ctypes.c_float(mul),
                                    _stream()),
           "mv_widen_transpose")
    return out, (base_t if padded else out_t)


def split_tf32(x2d, mode):
    """fp32 [rows, cols] -> fp32 [rows, 3*cols]: [hi|lo|hi] (mode 0, A operand) or [hi|hi|lo] (mode 1, B)."""
    _need_cuda(x2d)
    assert x2d.dim() == 2 and x2d.stride(1) == 1 and x2d.dtype == torch.float32
    rows, cols = x2d.shape
    out = torch.empty(rows, 3 * cols, dtype=torch.float32, device=x2d.device)
    _check(lib().mv_split_tf32(_ptr(x2d), ctypes.c_int64(x2d.stride(0)), rows, cols, _ptr(out), int(mode),
                               _stream()), "mv_split_tf32")
    return out


def upsample_ce(y, labels, ignore_index=-100):
    """Fused bilinear upsample + cross entropy (mv_upsample_ce).  y fp32 [B, gh*gw, C] patch logits,
    labels int64 [B, H, W] -> (acc fp32 [2] = (sum of pixel losses, valid pixels), dy = d sum / dy)."""
    _need_cuda(y, labels)
    assert y.dtype == torch.float32 and labels.dtype == torch.int64 and y.dim() == 3 and labels.dim() == 3
    y, labels = y.contiguous(), labels.contiguous()
    B, hw, C = y.shape
    H, W = labels.shape[1:]
    gh = int(round((hw * H / W) ** 0.5))
    gw = hw // max(gh, 1)
    if gh * gw != hw or labels.shape[0] != B:
        raise MvError("upsample_ce: %d patches do not form a grid matching labels %s" % (hw, tuple(labels.shape)))
    dy = torch.zeros_like(y)
    acc = torch.zeros(2, dtype=torch.float32, device=y.device)
    _check(lib().mv_upsample_ce(_ptr(y), _ptr(labels), _ptr(dy), _ptr(acc), B, C, gh, gw, H, W,
                                ctypes.c_int64(ignore_index), _stream()), "mv_upsample_ce")
    return acc, dy


def linear_sum_assignment(cost, sizes, match=None, flag=None):
    """Batched scipy.optimize.linear_sum_assignment on the device (mv_linear_sum_assignment).
    cost fp32 [B, Q, Tmax], sizes int32 [B] (valid columns per image) -> match int32 [B, Tmax]:
    prediction matched to every target, -1 for padding.  flag int32 [1] (optional) is set to 1
    when a block has no finite matching.  No host synchronisation."""
    _need_cuda(cost, sizes)
    assert cost.dtype == torch.float32 and cost.dim() == 3 and sizes.dtype == torch.int32
    cost, sizes = cost.contiguous(), sizes.contiguous()
    B, Q, T = cost.shape
    assert sizes.numel() == B
    if match is None:
        match = torch.empty(B, T, dtype=torch.int32, device=cost.device)
    assert match.dtype == torch.int32 and match.shape == (B, T) and match.is_contiguous()
    _check(lib().mv_linear_sum_assignment(_ptr(cost), _ptr(sizes), B, Q, T, _ptr(match),
                                          _ptr(flag) if flag is not None else None, _stream()),
           "mv_linear_sum_assignment")
    return match


# ------------------------------------------------------------------- attention
def attention_fwd(qkv, B, H, N, *, scale=0.125, q_out=None, out_dtype=torch.float16, out=None,
                  lse=None):
    """qkv fp16 [B*N, 3*H*64] -> out [B*N, H*64] = q_out(softmax(q k^T * scale) v), lse [B,H,N]."""
    _need_cuda(qkv)
    assert qkv.dtype == torch.float16 and qkv.is_contiguous() and qkv.shape == (B * N, 3 * H * 64)
    if out is None:
        out = torch.empty(B * N, H * 64, dtype=out_dtype, device=qkv.device)
    if lse is None:
        lse = torch.empty(B, H, N, dtype=torch.float32, device=qkv.device)
    q = _fmt(q_out)
    with _timed("attn_fwd", 4.0 * B * H * N * N * 64, B * N * H * 64 * (3 * 2 + out.element_size())):
        rc = lib().mv_attention_fwd(_ptr(qkv), _ptr(out), _DT[out.dtype], _ptr(lse), B, H, N,
                                    ctypes.c_float(scale), q[0], q[1], _stream())
    _check(rc, "mv_attention_fwd")
    return out, lse


def attention_bwd(qkv, o, d_o, lse, B, H, N, *, scale=0.125, dqkv=None, delta=None,
                  dq_accum=None, dbias=None):
    """d_o fp16 [B*N, D] -> dqkv fp16 [B*N, 3D] (dq | dk | dv).  dbias fp32 [3D] (optional) += column sums
    of dqkv, the to_qkv bias gradient."""
    _need_cuda(qkv, o, d_o, lse)
    assert qkv.dtype == torch.float16 and o.dtype == torch.float16 and d_o.dtype == torch.float16
    assert o.is_contiguous() and d_o.is_contiguous() and qkv.is_contiguous()
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    if delta is None:
        delta = torch.empty(B, H, N, dtype=torch.float32, device=qkv.device)
    if dbias is not None:
        assert dbias.dtype == torch.float32 and dbias.is_contiguous() and dbias.numel() == 3 * H * 64
    if dq_accum is None:
        dq_accum = torch.empty(B * N, H * 64, dtype=torch.float32, device=qkv.device)
    with _timed("attn_bwd", 10.0 * B * H * N * N * 64, B * N * H * 64 * 2 * (3 + 1 + 1 + 3)):
        rc = lib().mv_attention_bwd(_ptr(qkv), _ptr(o), _ptr(d_o), _ptr(lse), _ptr(delta),
                                    _ptr(dq_accum), _ptr(dqkv), _ptr(dbias), B,
                                    H, N, ctypes.c_float(scale), _stream())
    _check(rc, "mv_attention_bwd")
    return dqkv
