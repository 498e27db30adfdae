"""B200-native Vision Transformer with myrtle-vision's constructor and outputs.

Drop-in for src/myrtle_vision/models/vit.py of the reference: `ViT(decoder=..., image_size=...,
patch_size=..., num_classes=..., dim=..., depth=..., heads=..., mlp_dim=..., q_format=...)`,
`.forward(img[B,3,H,W])`, `.convert()`, `.quantizer.prepare_qat(...)`; identical parameter names,
shapes, initial values for a given torch seed, and state_dict keys per q_format.

The modules below only *hold parameters* under the reference's names.  forward() does not call
them: the patch embedding and the transformer blocks run as fused sm_100a kernels through
mv_engine.EncoderFunction (C ABI: include/mv_b200.h), and only the tiny decoder heads, the
positional-embedding resize and the loss stay in PyTorch.  There is no CPU execution path.
"""
from typing import Optional, Union

import torch
import torch.nn.functional as F
from torch import nn

import mv_engine
import mv_native
from myrtle_vision.utils.quantize import ModelQuantizer, QFormat

MIN_NUM_PATCHES = 16


class Residual(nn.Module):
    def __init__(self, fn):
        super().__init__()
        self.fn = fn


class PreNorm(nn.Module):
    def __init__(self, dim, fn):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn


class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim, dropout=0.0):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden_dim), nn.GELU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, dim), nn.Dropout(dropout))


class Attention(nn.Module):
    def __init__(self, dim, heads=8, dim_head=64, dropout=0.0):
        super().__init__()
        inner_dim = dim_head * heads
        self.heads = heads
        self.scale = dim_head ** -0.5
        self.to_qkv = nn.Linear(dim, inner_dim * 3, bias=True)
        self.to_out = nn.Sequential(nn.Linear(inner_dim, dim), nn.Dropout(dropout))
        # the reference passes the softmax probabilities through this module so that forward hooks can read the
        # attention maps (models/vit.py:80-82, 94); a hook registered here switches that block's probabilities on
        # (mv_engine.EncoderEngine._probe_attention, debug only)
        self.attn_output = nn.Identity()


class Transformer(nn.Module):
    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout):
        super().__init__()
        self.layers = nn.ModuleList()
        for _ in range(depth):
            # construction order (Attention, LayerNorm, FeedForward, LayerNorm) fixes the RNG
            # stream so that a torch seed yields the reference's initial weights
            attn = Attention(dim, heads=heads, dim_head=dim_head, dropout=dropout)
            first = Residual(PreNorm(dim, attn))
            ff = FeedForward(dim, mlp_dim, dropout=dropout)
            second = Residual(PreNorm(dim, ff))
            self.layers.append(nn.Sequential(first, second))


class ClassificationDecoder(nn.Module):
    def __init__(self, dim, num_classes):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.linear = nn.Linear(dim, num_classes)


class SegmentationDecoder(nn.Module):
    def __init__(self, dim, num_classes, image_size, patch_size):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.linear = nn.Linear(dim, num_classes)
        self.upsample = nn.Upsample(size=image_size, mode="bilinear")
        self.image_size_in_patches = image_size // patch_size


class DetectionDecoder(nn.Module):
    def __init__(self, in_dim, num_classes, num_det_tokens):
        super().__init__()
        self.class_embed = nn.Linear(in_dim, num_classes + 1)   # +1 for no-class
        self.bbox_embed = nn.Linear(in_dim, 4)
        self.num_det_tokens = num_det_tokens


class _STEQuant(torch.autograd.Function):
    """float_quantize (nearest) on the GPU; backward straight-through, or float_quantize of the incoming gradient with
    the plan's gradient format (QPyTorch's backward_number; utils.quantize.QuantPlan.grad): gfmt = (exp, man) rounds to
    nearest, (exp, man, seed, offset) stochastically with the gradient rounding stream (mv_float_quantize_dev)."""

    @staticmethod
    def forward(ctx, x, exp, man, gfmt):
        ctx.gfmt = gfmt
        return mv_native.float_quantize(x.detach(), exp, man).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        if ctx.gfmt is not None and len(ctx.gfmt) == 4:
            e, m, seed, offset = ctx.gfmt
            g = mv_native.float_quantize_dev(g, e, m, (seed, offset)).to(g.dtype).view(g.shape)
        elif ctx.gfmt is not None:
            g = mv_native.float_quantize(g, ctx.gfmt[0], ctx.gfmt[1]).to(g.dtype)
        return g, None, None, None


class _FusedNorm(torch.autograd.Function):
    """Decoder LayerNorm with its quantisers on the library's kernels: y = q_out(LN(q_in(x))) in one pass
    (mv_layernorm_q_fwd, fp32 output) and dx, dgamma, dbeta in one pass (mv_layernorm_q_bwd) — in place of ATen's
    layer_norm + three standalone quantiser passes + GammaBetaBackward (0.85 ms per step on the segmentation head's
    [65 536, 384] input).  Straight-through quantisers, as everywhere (utils/quantize.py:87-89)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, q_in, q_out, eps):
        x2 = x.detach().reshape(-1, x.shape[-1]).contiguous()
        y, mean, rstd = mv_native.layernorm_q_fwd(x2, gamma.detach(), beta.detach(), q_in=q_in, q_post=q_out,
                                                  out_dtype=torch.float32, eps=eps, tag="ln_fwd_head")
        ctx.save_for_backward(x2, gamma, mean, rstd)
        ctx.q_in, ctx.shape = q_in, x.shape
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, gamma, mean, rstd = ctx.saved_tensors
        D = x2.shape[-1]
        dy2 = dy.reshape(-1, D).contiguous().float()
        dgamma = torch.zeros(D, dtype=torch.float32, device=dy.device)
        dbeta = torch.zeros(D, dtype=torch.float32, device=dy.device)
        dx, _ = mv_native.layernorm_q_bwd(dy2, x2, gamma.detach(), mean, rstd, q_in=ctx.q_in, dgamma=dgamma, dbeta=dbeta,
                                          want_f16=False, tag="ln_bwd_head")
        return dx.view(ctx.shape), dgamma, dbeta, None, None, None


def _fq(x, fmt, gfmt=None):
    return x if fmt is None else _STEQuant.apply(x, fmt[0], fmt[1], gfmt)


def _unwrap(module):
    """The parameter-holding module behind an optional Sequential(QuantStubSlot, module)."""
    if isinstance(module, nn.Sequential) and len(module) == 2 and not isinstance(
            module[1], (nn.Dropout,)):
        return module[1]
    return module


class ViT(nn.Module):
    def __init__(
        self,
        *,
        decoder: str,
        image_size: int,
        patch_size: int,
        num_classes: int,
        dim: int,
        depth: int,
        heads: int,
        mlp_dim: int,
        pool: str = "cls",
        channels: int = 3,
        dim_head: int = 64,
        dropout: float = 0.0,
        emb_dropout: float = 0.0,
        num_det_tokens: int = 100,
        profile: bool = False,
        q_format: Optional[Union[str, QFormat]] = None,
        backward_format=None,      # extension: (exp, man) gradient format, see ModelQuantizer.prepare_qat
        backward_rounding: str = "nearest",    # its rounding, "nearest" or "stochastic" (QPyTorch's backward_rounding)
    ):
        super().__init__()
        assert image_size % patch_size == 0, "Image dimensions must be divisible by the patch size."
        num_patches = (image_size // patch_size) ** 2
        patch_dim = channels * patch_size ** 2
        assert num_patches > MIN_NUM_PATCHES, (
            f"your number of patches ({num_patches}) is way too small for attention to be "
            f"effective (at least 16). Try decreasing your patch size")
        assert decoder in {"classification", "segmentation", "detection"}, \
            "decoder must be either classification, segmentation, or detection"
        self.patch_size = patch_size
        self.task = decoder
        self.profile = profile
        self.heads, self.dim, self.mlp_dim, self.depth = heads, dim, mlp_dim, depth
        self.dim_head = dim_head
        self.dropout_p, self.emb_dropout_p = dropout, emb_dropout

        # the positional embedding is stored at 14x14 and resized on the fly (vit.py:216-218)
        self.pos_embedding = nn.Parameter(torch.randn(1, 14 * 14 + 1, dim))
        self.pos_embedding_det = nn.Parameter(torch.randn(1, num_det_tokens, dim))
        self.patch_to_embedding = nn.Linear(patch_dim, dim)
        self.cls_token = nn.Parameter(torch.randn(1, 1, dim))
        self.det_tokens = nn.Parameter(torch.randn(1, num_det_tokens, dim))
        self.dropout = nn.Dropout(emb_dropout)
        self.transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)
        if decoder == "classification":
            self.decoder = ClassificationDecoder(dim, num_classes)
        elif decoder == "segmentation":
            self.decoder = SegmentationDecoder(dim, num_classes, image_size, patch_size)
        else:
            self.decoder = DetectionDecoder(dim, num_classes, num_det_tokens)

        self._engine = None
        self._grad_round_seed = None     # stochastic gradient rounding: the seed of the last encoder forward that drew one
        self.quantizer = ModelQuantizer(self)
        self.quantizer.prepare_qat(q_format if q_format is not None else QFormat.FP32, backward_format=backward_format,
                                   backward_rounding=backward_rounding)

    # ------------------------------------------------------------------ plumbing
    def _invalidate_engine(self):
        self._engine = None

    def _apply(self, fn, *args, **kwargs):
        self._engine = None              # parameters may move (.to / .cuda / .half)
        return super()._apply(fn, *args, **kwargs)

    def _engine_params(self):
        pe = _unwrap(self.patch_to_embedding)
        params = [pe.weight, pe.bias]
        for block in self.transformer.layers:
            pre1, pre2 = block[0].fn, block[1].fn
            ln1, ln2 = _unwrap(pre1.norm), _unwrap(pre2.norm)
            qkv = _unwrap(pre1.fn.to_qkv)
            out = _unwrap(pre1.fn.to_out[0])
            fc1, fc2 = _unwrap(pre2.fn.net[0]), _unwrap(pre2.fn.net[3])
            params += [ln1.weight, ln1.bias, qkv.weight, qkv.bias, out.weight, out.bias,
                       ln2.weight, ln2.bias, fc1.weight, fc1.bias, fc2.weight, fc2.bias]
        return params

    def engine(self):
        if self._engine is None:
            cfg = mv_engine.EngineConfig(self.dim, self.heads, self.mlp_dim, self.depth,
                                         self.patch_size, self.quantizer.plan, dropout=self.dropout_p,
                                         emb_dropout=self.emb_dropout_p)
            self._engine = mv_engine.EncoderEngine(cfg, self._engine_params())
            self._engine.profile = self.profile
            self._engine.probes = [block[0].fn.fn.attn_output for block in self.transformer.layers]
        return self._engine

    # ------------------------------------------------------------------- forward
    def _pos_full(self, gh, gw):
        """cls position + bicubic resize of the 14x14 grid (vit.py:292-302); FP16_16 quantises
        the concatenation (FloatFunctional output)."""
        ff = self.quantizer.plan.ff
        pos_cls, pos = self.pos_embedding[:, 0:1, :], self.pos_embedding[:, 1:, :]
        # bicubic interpolation is linear in the grid values: apply it as a cached
        # [gh*gw, 196] matrix (ATen's upsample_bicubic2d launches a single thread block here)
        pos = torch.matmul(self._resize_matrix(gh, gw, pos.device), pos)
        return _fq(torch.cat((pos_cls, pos), dim=1), ff)

    def _resize_matrix(self, gh, gw, device):
        key = (gh, gw, str(device))
        cache = self.__dict__.setdefault("_resize_cache", {})
        if key not in cache:
            basis = torch.eye(14 * 14).view(14 * 14, 1, 14, 14)
            w = F.interpolate(basis, size=(gh, gw), mode="bicubic", align_corners=False)
            cache[key] = w.view(14 * 14, gh * gw).t().contiguous().to(device)
        return cache[key]

    def _gfmt(self, j):
        """Gradient format of the decoder's j-th gradient-quantiser site (DECODER_GRAD_SITES): (exp, man), or with
        stochastic rounding (exp, man, seed, offset) — the seed of this forward, offset = the stream's site of stub j."""
        plan = self.quantizer.plan
        seed = self._grad_round_seed
        if plan.grad is None or seed is None:
            return plan.grad
        engine = self._engine
        return plan.grad + (seed, mv_engine.grad_round_offset(10 * self.depth + 1 + j, engine.rank))

    def _linear(self, holder, x, j=0):
        """j: gradient-quantiser site of the input stub; the weight's is j + 1."""
        plan = self.quantizer.plan
        lin = _unwrap(holder)
        y = F.linear(_fq(x, plan.inp, self._gfmt(j)), _fq(lin.weight, plan.inp, self._gfmt(j + 1)), lin.bias)
        return _fq(y, plan.out)

    def _norm(self, holder, x, j=0):
        plan = self.quantizer.plan
        ln = _unwrap(holder)
        d = x.shape[-1]
        if (x.is_cuda and x.dtype == torch.float32 and plan.grad is None and ln.elementwise_affine and d % 4 == 0
                and d <= 1024 and len(ln.normalized_shape) == 1):
            return _FusedNorm.apply(x, ln.weight, ln.bias, plan.inp, plan.out, ln.eps)
        y = F.layer_norm(_fq(x, plan.inp, self._gfmt(j)), ln.normalized_shape, ln.weight, ln.bias, ln.eps)
        return _fq(y, plan.out)

    def _decode(self, x, img_hw):
        dec = self.decoder
        if self.task == "classification":                               # vit.py:335-342
            return self._linear(dec.linear, self._norm(dec.norm, x[:, 0], 0), 1)
        if self.task == "segmentation":                                 # vit.py:359-374
            y = self._linear(dec.linear, self._norm(dec.norm, x[:, 1:], 0), 1)
            if self.training and getattr(dec, "fused_loss", False):
                return y                 # [B, gh*gw, C] for models.losses.upsampled_cross_entropy
            b, hw, c = y.size()
            y = y.transpose(1, 2).reshape(b, c, dec.image_size_in_patches, dec.image_size_in_patches)
            return dec.upsample(y)
        # detection (vit.py:389-396).  The reference's `self.decoder == "detection"` test is
        # always False (the attribute holds a Module), so det tokens never enter the sequence and
        # the heads read the last num_det_tokens *patch* tokens; reproduced here for parity.
        t = x[:, -dec.num_det_tokens:, :]
        return {"pred_logits": self._linear(dec.class_embed, t, 0),
                "pred_boxes": self._linear(dec.bbox_embed, t, 2).sigmoid()}

    def forward(self, img: torch.Tensor, distill_token: Optional[torch.Tensor] = None,
                mix: Optional[torch.Tensor] = None):
        """distill_token ([1, 1, dim], classification only): appended to the sequence as its last row, without a
        positional embedding (models/distill.py); the forward then returns (logits, encoder output of that row).
        mix (classification only): Mixup / CutMix records (utils/mixup.py): the encoder sees the batch mixed as they
        say, mixed inside the patch gather."""
        if not img.is_cuda:
            raise RuntimeError("myrtle-vision_b200 runs on CUDA (sm_100a) only; there is no CPU "
                               "fallback — move the model and the batch to a B200")
        if distill_token is not None:
            if self.task != "classification":
                raise ValueError("a distillation token needs decoder='classification', not %r" % (self.task,))
            if tuple(distill_token.shape) != (1, 1, self.dim):
                raise ValueError("distill_token must be [1, 1, %d], got %s" % (self.dim, tuple(distill_token.shape)))
        if mix is not None:
            if self.task != "classification":
                raise ValueError("Mixup / CutMix needs decoder='classification', not %r" % (self.task,))
            if distill_token is not None:
                raise ValueError("Mixup / CutMix together with a distillation token is not supported")
        b, c, h, w = img.shape
        p = self.patch_size
        engine = self.engine()
        engine.training = self.training          # dropout (self.dropout_p, self.emb_dropout_p) in training mode only
        pos_full = self._pos_full(h // p, w // p)
        x = mv_engine.EncoderFunction.apply(engine, img, pos_full, self.cls_token,
                                            *engine.params, token=distill_token, mix=mix)
        self._grad_round_seed = engine.step_grad_round_seed      # the decoder's stubs round with the encoder's seed
        with engine._range("mlp_head"):
            if distill_token is not None:
                return self._decode(x, (h, w)), x[:, -1]
            return self._decode(x, (h, w))

    def convert(self) -> None:
        self.quantizer.convert()
