"""CPU reference of the ViT training step with dropout, for the dropout tests (not collected by pytest itself).

oracle/vit_oracle.py restates the reference's forward without dropout; this module restates the same forward with the
model's nn.Dropout modules in training mode, built from that file's helpers (quantiser placement, fake-quant Linear and
LayerNorm), with the masks of the stream declared in include/mv_b200.h ("dropout mask"), so that autograd supplies the
masked backward.  Sites, as in the module tree of models/vit.py: after the positional add (3 * depth), on to_out's
output (3l), after GELU (3l + 1) and on fc2's output (3l + 2) of block l.
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import quant_oracle, vit_oracle
from oracle.vit_oracle import PLACEMENT, _layernorm, _linear, fq


def dropout_mask(shape, p, seed, site):
    """keep * scale of nn.Dropout(p) at dropout site `site` for a token-major tensor of `shape`: keep = bits16 >=
    nearbyint(p * 65536), bits16 = the 16-bit Philox stream with offset = site over the flat index, scale = 1 / (1 - p)
    in fp32 (0 for p == 1).  fp32 tensor of `shape`.  `seed` is taken as its 64-bit two's complement."""
    n = int(np.prod(shape))
    bits = quant_oracle.philox_bits(n, int(seed) & (2 ** 64 - 1), site, half=True)
    thr = int(round(float(p) * 65536.0))
    scale = np.float32(0.0) if p == 1 else np.float32(1.0) / np.float32(1.0 - p)
    return torch.from_numpy((bits >= thr).astype(np.float32) * scale).view(*shape)


def _dropout(x, p, seed, site):
    return x if p == 0 else x * dropout_mask(tuple(x.shape), p, seed, site)


def vit_forward(P, img, *, decoder, dropout, patch_size=16, heads, q_format="FP32", num_det_tokens=100,
                image_size=None, dim_head=64, grad_format=None):
    """vit_oracle.vit_forward with dropout = (p, emb_p, seed)."""
    vit_oracle._GRAD_FMT = grad_format
    fin, fout, ffn, fgelu = PLACEMENT[str(q_format)]
    dp, de, dseed = dropout
    b, c, h, w = img.shape
    p = patch_size
    gh, gw = h // p, w // p
    x = img.reshape(b, c, gh, p, gw, p).permute(0, 2, 4, 3, 5, 1).reshape(b, gh * gw, p * p * c)
    x = _linear(x, P, "patch_to_embedding", fin, fout)
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

    depth = 0
    while "transformer.layers.%d.0.fn.norm.weight" % depth in P:
        depth += 1
    x = _dropout(x, de, dseed, 3 * depth)                            # ViT.dropout (emb_dropout)
    n = x.shape[1]
    dh = dim // heads
    for l in range(depth):
        pre = "transformer.layers.%d." % l
        y = _layernorm(x, P, pre + "0.fn.norm", fin, fout)
        qkv = _linear(y, P, pre + "0.fn.fn.to_qkv", fin, fout)
        qkv = qkv.reshape(b, n, 3, heads, dh).permute(2, 0, 3, 1, 4)
        attn = ((qkv[0] @ qkv[1].transpose(-2, -1)) * dim_head ** -0.5).softmax(dim=-1)
        o = (attn @ qkv[2]).transpose(1, 2).reshape(b, n, dim)
        o = _linear(o, P, pre + "0.fn.fn.to_out.0", fin, fout)
        x = fq(_dropout(o, dp, dseed, 3 * l) + x, ffn)               # to_out.1: Dropout
        y = _layernorm(x, P, pre + "1.fn.norm", fin, fout)
        u = _linear(y, P, pre + "1.fn.fn.net.0", fin, fout)
        g = _dropout(F.gelu(fq(u, fgelu)), dp, dseed, 3 * l + 1)     # net.2: Dropout
        o = _linear(g, P, pre + "1.fn.fn.net.3", fin, fout)
        x = fq(_dropout(o, dp, dseed, 3 * l + 2) + x, ffn)           # net.4: Dropout

    if decoder == "classification":
        y = _layernorm(x[:, 0], P, "decoder.norm", fin, fout)
        return _linear(y, P, "decoder.linear", fin, fout)
    if decoder == "segmentation":
        y = _layernorm(x[:, 1:], P, "decoder.norm", fin, fout)
        y = _linear(y, P, "decoder.linear", fin, fout)
        bb, hw, cc = y.shape
        y = y.transpose(1, 2).view(bb, cc, gh, gw)
        return F.interpolate(y, size=image_size if image_size is not None else h, mode="bilinear")
    if decoder == "detection":
        t = x[:, -num_det_tokens:, :]
        return {"pred_logits": _linear(t, P, "decoder.class_embed", fin, fout),
                "pred_boxes": _linear(t, P, "decoder.bbox_embed", fin, fout).sigmoid()}
    raise ValueError(decoder)


def train_step(P, img, target, *, decoder, heads, q_format, dropout, patch_size=16, num_det_tokens=100,
               grad_format=None, loss_scale=1.0):
    """vit_oracle.train_step with dropout = (p, emb_p, seed).  Returns (output, loss, grads dict)."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    try:
        out = vit_forward(params, img, decoder=decoder, heads=heads, q_format=q_format, patch_size=patch_size,
                          num_det_tokens=num_det_tokens, grad_format=grad_format, dropout=dropout)
        if decoder == "detection":
            loss = (F.cross_entropy(out["pred_logits"].flatten(0, 1), target["labels"].flatten())
                    + (out["pred_boxes"] - target["boxes"]).abs().mean())
        else:
            loss = F.cross_entropy(out, target)
        (loss * loss_scale).backward()
    finally:
        vit_oracle._GRAD_FMT = None
    return out, loss.detach(), {k: v.grad for k, v in params.items()}
