"""CPU restatement of Mixup / CutMix (include/mv_b200.h "Mixup / CutMix"): records applied to an image batch in fp32,
the soft targets and their cross-entropy in float64, and the classification step on the mixed batch."""
import torch

from oracle import vit_oracle


def records(recs):
    """int32 [B, 8] device records -> dict of CPU tensors (lam, w_self, w_other fp32; cutmix, y0, y1, x0, x1 int)."""
    r = recs.cpu()
    f = r[:, :3].view(torch.float32)
    out = {"lam": f[:, 0], "w_self": f[:, 1], "w_other": f[:, 2]}
    out.update({k: r[:, 3 + i] for i, k in enumerate(("cutmix", "y0", "y1", "x0", "x1"))})
    return out


def apply(img, rec):
    """The mixed batch: fp32 img [B, C, H, W] (CPU), rec from records().  Mixup pixels are
    fl32(fl32(w_self a) + fl32(w_other p)); CutMix boxes are copied from the partner B - 1 - b."""
    img = img.float()
    B = img.shape[0]
    out = img.clone()
    for b in range(B):
        p = img[B - 1 - b]
        if int(rec["cutmix"][b]):
            y0, y1, x0, x1 = (int(rec[k][b]) for k in ("y0", "y1", "x0", "x1"))
            out[b, :, y0:y1, x0:x1] = p[:, y0:y1, x0:x1]
        else:
            ws, wo = rec["w_self"][b], rec["w_other"][b]            # fp32 scalars: fp32 products and sum
            out[b] = (ws * img[b]) + (wo * p)
    return out


def targets(labels, lam, C, smoothing):
    """float64 [B, C]: t_b = lam_b s(y_b) + (1 - lam_b) s(y_{B-1-b}), s(y) = off + (on - off) e_y."""
    off = smoothing / C
    on = 1.0 - smoothing + off
    s = torch.full((labels.shape[0], C), off, dtype=torch.float64)
    s[torch.arange(labels.shape[0]), labels] = on
    lam = lam.double()[:, None]
    return lam * s + (1.0 - lam) * s.flip(0)


def loss(logits, labels, lam, smoothing):
    """mean_b sum_c -t_bc log_softmax(x_b)_c in the dtype of logits (float64 for the reference)."""
    t = targets(labels, lam, logits.shape[1], smoothing).to(logits.dtype)
    return (-t * torch.log_softmax(logits, dim=-1)).sum(-1).mean()


def train_step(P, img_mixed, labels, lam, smoothing, *, heads, q_format):
    """vit_oracle's classification step on the mixed batch with the soft-target loss -> (logits, loss, grads)."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    out = vit_oracle.vit_forward(params, img_mixed, decoder="classification", heads=heads, q_format=q_format)
    l = loss(out, labels, lam, smoothing)
    l.backward()
    return out, l.detach(), {k: v.grad for k, v in params.items()}
