"""CPU reference of the ViT training step with stochastically rounded gradient quantisers (not collected by pytest).

QPyTorch's Quantizer(forward_number, backward_number, backward_rounding="stochastic") at every quantiser that
vit_oracle.py gives a gradient format (the QuantStubs in front of Linear / LayerNorm and the weight fake-quant): the
backward rounds the incoming gradient with float_quantize(..., "stochastic") of oracle/quant_oracle.py, fed with the
random bits of the stream declared in include/mv_b200.h ("gradient rounding stream") — element i of site s takes the
bits the CUDA float_quantize uses for element i at offset s + (rank << 32): the 16-bit stream for man >= 7, the 32-bit
stream below.  The forward restates dropout_oracle.vit_forward (and so oracle/vit_oracle.py) with each stub's site.
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import quant_oracle
from oracle.vit_oracle import PLACEMENT, _fq_np
from dropout_oracle import _dropout


def round_bits(n, exp, man, seed, offset):
    """The random bits of elements 0 .. n-1 of a site: uint32 [n]."""
    del exp
    return quant_oracle.philox_bits(int(n), int(seed) & (2 ** 64 - 1), int(offset), half=man >= 7)


def stochastic_round(g, exp, man, seed, offset):
    """float_quantize(g, exp, man, "stochastic") with the stream's bits over g's flat (row-major) order."""
    a = g.detach().float().contiguous()
    bits = round_bits(a.numel(), exp, man, seed, offset)
    out = quant_oracle.float_quantize(a.numpy(), exp, man, rounding="stochastic", rbits=bits)
    return torch.from_numpy(np.asarray(out, dtype=np.float32)).view(g.shape).to(g.dtype)


class _SRQuant(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, exp, man, grad):
        ctx.grad = grad
        return _fq_np(x, exp, man)

    @staticmethod
    def backward(ctx, g):
        e, m, seed, offset = ctx.grad
        return stochastic_round(g, e, m, seed, offset), None, None, None


class _Sites:
    def __init__(self, grad_format, seed, rank):
        self.gf, self.seed, self.rank = grad_format, seed, rank

    def fq(self, x, fmt, site):
        if fmt is None:
            return x
        return _SRQuant.apply(x, fmt[0], fmt[1], self.gf + (self.seed, int(site) + (int(self.rank) << 32)))

    def linear(self, x, P, name, fin, fout, site):
        """Sequential(QuantStub, qat.Linear) with the input stub at `site` and the weight's at site + 1."""
        y = F.linear(self.fq(x, fin, site), self.fq(P[name + ".weight"], fin, site + 1), P[name + ".bias"])
        return _plain(y, fout)

    def layernorm(self, x, P, name, fin, fout, site):
        xq = self.fq(x, fin, site)
        y = F.layer_norm(xq, (xq.shape[-1],), P[name + ".weight"], P[name + ".bias"], 1e-5)
        return _plain(y, fout)


def _plain(x, fmt):
    from oracle.vit_oracle import fq
    return fq(x, fmt)


def vit_forward(P, img, *, decoder, grad_format, seed, rank=0, dropout=(0.0, 0.0, 0), patch_size=16, heads,
                q_format="FP16_32", num_det_tokens=100, image_size=None, dim_head=64):
    """dropout_oracle.vit_forward with the gradient quantisers rounding stochastically under `seed`."""
    fin, fout, ffn, fgelu = PLACEMENT[str(q_format)]
    S = _Sites(tuple(grad_format), seed, rank)
    fq = _plain
    dp, de, dseed = dropout
    b, c, h, w = img.shape
    p = patch_size
    gh, gw = h // p, w // p
    depth = 0
    while "transformer.layers.%d.0.fn.norm.weight" % depth in P:
        depth += 1
    x = img.reshape(b, c, gh, p, gw, p).permute(0, 2, 4, 3, 5, 1).reshape(b, gh * gw, p * p * c)
    # the patches need no gradient: the patch-embedding weight is site 10 * depth (its input stub would be 10 * depth - 1,
    # never reached)
    x = S.linear(x, P, "patch_to_embedding", fin, fout, 10 * depth - 1)
    dim = x.shape[-1]
    cls = P["cls_token"].repeat(b, 1, 1)
    x = fq(torch.cat((cls, x), dim=1), ffn)
    pos = P["pos_embedding"]
    pos_cls, pos_grid = pos[:, 0:1, :], pos[:, 1:, :]
    pos_grid = pos_grid.transpose(1, 2).view(1, -1, 14, 14)
    pos_grid = F.interpolate(pos_grid, size=(gh, gw), mode="bicubic", align_corners=False)
    pos_grid = pos_grid.view(1, -1, gh * gw).transpose(1, 2)
    pos_full = fq(torch.cat((pos_cls, pos_grid), dim=1), ffn)
    x = fq(x + pos_full.repeat(b, 1, 1), ffn)
    x = _dropout(x, de, dseed, 3 * depth)
    n = x.shape[1]
    dh = dim // heads
    for l in range(depth):
        pre, s0 = "transformer.layers.%d." % l, 10 * l
        y = S.layernorm(x, P, pre + "0.fn.norm", fin, fout, s0 + 0)
        qkv = S.linear(y, P, pre + "0.fn.fn.to_qkv", fin, fout, s0 + 1)
        qkv = qkv.reshape(b, n, 3, heads, dh).permute(2, 0, 3, 1, 4)
        attn = ((qkv[0] @ qkv[1].transpose(-2, -1)) * dim_head ** -0.5).softmax(dim=-1)
        o = (attn @ qkv[2]).transpose(1, 2).reshape(b, n, dim)
        o = S.linear(o, P, pre + "0.fn.fn.to_out.0", fin, fout, s0 + 3)
        x = fq(_dropout(o, dp, dseed, 3 * l) + x, ffn)
        y = S.layernorm(x, P, pre + "1.fn.norm", fin, fout, s0 + 5)
        u = S.linear(y, P, pre + "1.fn.fn.net.0", fin, fout, s0 + 6)
        g = _dropout(F.gelu(fq(u, fgelu)), dp, dseed, 3 * l + 1)
        o = S.linear(g, P, pre + "1.fn.fn.net.3", fin, fout, s0 + 8)
        x = fq(_dropout(o, dp, dseed, 3 * l + 2) + x, ffn)

    d0 = 10 * depth + 1
    if decoder == "classification":
        y = S.layernorm(x[:, 0], P, "decoder.norm", fin, fout, d0)
        return S.linear(y, P, "decoder.linear", fin, fout, d0 + 1)
    if decoder == "segmentation":
        y = S.layernorm(x[:, 1:], P, "decoder.norm", fin, fout, d0)
        y = S.linear(y, P, "decoder.linear", fin, fout, d0 + 1)
        bb, hw, cc = y.shape
        y = y.transpose(1, 2).view(bb, cc, gh, gw)
        return F.interpolate(y, size=image_size if image_size is not None else h, mode="bilinear")
    if decoder == "detection":
        t = x[:, -num_det_tokens:, :]
        return {"pred_logits": S.linear(t, P, "decoder.class_embed", fin, fout, d0),
                "pred_boxes": S.linear(t, P, "decoder.bbox_embed", fin, fout, d0 + 2).sigmoid()}
    raise ValueError(decoder)


def train_step(P, img, target, *, decoder, heads, grad_format, seed, rank=0, dropout=(0.0, 0.0, 0), q_format="FP16_32",
               patch_size=16, loss_scale=1.0):
    """(output, loss, grads dict) of one classification / segmentation step (cross entropy) times loss_scale."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    out = vit_forward(params, img, decoder=decoder, heads=heads, q_format=q_format, patch_size=patch_size,
                      grad_format=grad_format, seed=seed, rank=rank, dropout=dropout)
    loss = F.cross_entropy(out, target)
    (loss * loss_scale).backward()
    return out, loss.detach(), {k: v.grad for k, v in params.items()}
