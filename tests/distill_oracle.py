"""CPU reference of the distillation step, for the distillation tests (not collected by pytest itself).

oracle/vit_oracle.py restates the reference's forward; this module restates the student's forward with a distillation
token (models/distill.py) from that file's helpers (quantiser placement, fake-quant Linear and LayerNorm), with the
dropout masks of tests/dropout_oracle.py, and the wrapper's loss in float64 torch ops, so that autograd supplies the
backward:
  * the sequence is built as without the token (cls row, patch rows, positional add, FP16_16's FloatFunctional
    quantiser), then q_ff(token) is appended as row N - 1 of every image: no positional embedding;
  * the embedding dropout (site 3 depth) covers the whole sequence, the token row included;
  * distill_logits = Linear(LayerNorm(row N - 1)) with the classification head's quantisers.
"""
import torch
import torch.nn.functional as F

from dropout_oracle import _dropout
from oracle import vit_oracle
from oracle.vit_oracle import PLACEMENT, _layernorm, _linear, fq


def student_forward(P, img, *, heads, q_format="FP32", patch_size=16, dim_head=64, dropout=None, grad_format=None):
    """-> (student logits, distillation logits).  dropout = (p, emb_p, seed) or None."""
    vit_oracle._GRAD_FMT = grad_format
    fin, fout, ffn, fgelu = PLACEMENT[str(q_format)]
    dp, de, dseed = dropout if dropout is not None else (0.0, 0.0, 0)
    b, c, h, w = img.shape
    p = patch_size
    gh, gw = h // p, w // p
    x = img.reshape(b, c, gh, p, gw, p).permute(0, 2, 4, 3, 5, 1).reshape(b, gh * gw, p * p * c)
    x = _linear(x, P, "patch_to_embedding", fin, fout)
    dim = x.shape[-1]
    x = fq(torch.cat((P["cls_token"].repeat(b, 1, 1), x), dim=1), ffn)
    pos = P["pos_embedding"]
    pos_cls, pos_grid = pos[:, 0:1, :], pos[:, 1:, :]
    pos_grid = F.interpolate(pos_grid.transpose(1, 2).view(1, -1, 14, 14), size=(gh, gw), mode="bicubic",
                             align_corners=False).view(1, -1, gh * gw).transpose(1, 2)
    pos_full = fq(torch.cat((pos_cls, pos_grid), dim=1), ffn)
    x = fq(x + pos_full.repeat(b, 1, 1), ffn)
    x = torch.cat((x, fq(P["distillation_token"], ffn).repeat(b, 1, 1)), dim=1)

    depth = 0
    while "transformer.layers.%d.0.fn.norm.weight" % depth in P:
        depth += 1
    x = _dropout(x, de, dseed, 3 * depth)
    n = x.shape[1]
    dh = dim // heads
    for l in range(depth):
        pre = "transformer.layers.%d." % l
        y = _layernorm(x, P, pre + "0.fn.norm", fin, fout)
        qkv = _linear(y, P, pre + "0.fn.fn.to_qkv", fin, fout).reshape(b, n, 3, heads, dh).permute(2, 0, 3, 1, 4)
        attn = ((qkv[0] @ qkv[1].transpose(-2, -1)) * dim_head ** -0.5).softmax(dim=-1)
        o = _linear((attn @ qkv[2]).transpose(1, 2).reshape(b, n, dim), P, pre + "0.fn.fn.to_out.0", fin, fout)
        x = fq(_dropout(o, dp, dseed, 3 * l) + x, ffn)
        y = _layernorm(x, P, pre + "1.fn.norm", fin, fout)
        u = _linear(y, P, pre + "1.fn.fn.net.0", fin, fout)
        g = _dropout(F.gelu(fq(u, fgelu)), dp, dseed, 3 * l + 1)
        x = fq(_dropout(_linear(g, P, pre + "1.fn.fn.net.3", fin, fout), dp, dseed, 3 * l + 2) + x, ffn)

    student = _linear(_layernorm(x[:, 0], P, "decoder.norm", fin, fout), P, "decoder.linear", fin, fout)
    distill = _linear(_layernorm(x[:, -1], P, "distill_mlp.0", fin, fout), P, "distill_mlp.1", fin, fout)
    return student, distill


def loss(student, distill, teacher, labels, temperature, alpha, hard):
    """(1 - a) CE(student, labels) + a D in float64 (upstream DistillWrapper.forward)."""
    s, d, t = student.double(), distill.double(), teacher.double()
    ce = F.cross_entropy(s, labels)
    if hard:
        dl = F.cross_entropy(d, t.argmax(dim=-1))
    else:
        dl = F.kl_div(F.log_softmax(d / temperature, dim=-1), F.softmax(t / temperature, dim=-1),
                      reduction="batchmean") * temperature ** 2
    return (1 - alpha) * ce + alpha * dl


def train_step(P, img, labels, teacher, *, heads, q_format, temperature, alpha, hard, dropout=None):
    """zero_grad -> student forward with the token -> distillation loss against the given teacher logits -> backward.
    Returns (student logits, distillation logits, loss, grads dict)."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    try:
        s, d = student_forward(params, img, heads=heads, q_format=q_format, dropout=dropout)
        total = loss(s, d, teacher, labels, temperature, alpha, hard)
        total.backward()
    finally:
        vit_oracle._GRAD_FMT = None
    return s.detach(), d.detach(), total.detach(), {k: v.grad for k, v in params.items()}
