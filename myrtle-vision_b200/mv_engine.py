"""Fused sm_100a execution of the quantised ViT encoder (patch embedding + transformer blocks).

Host-side orchestration only: every arithmetic step is a kernel of libmv_b200.so called through
the C ABI (include/mv_b200.h).  Replaces the module-by-module execution of
src/myrtle_vision/models/vit.py:267-314 (ViT.forward up to the decoder) and its autograd
backward, with the fake-quantisers of SURVEY.md Appendix A folded into the neighbouring kernels:

  forward, per block (H = the input/weight format, o = Linear/LN output format, f = FloatFunctional
  format; o and f are identity except in FP16_16):
    xn1  = H(LN(H(x)))                                   mv_layernorm_q_fwd      -> fp16
    qkv  = o(xn1 . H(Wqkv)^T + b)                        mv_gemm                 -> fp16
    att  = H(softmax(q k^T / 8) v)                       mv_attention_fwd        -> fp16
    x1   = f(o(att . H(Wo)^T + b) + x)                   mv_gemm (+residual)     -> fp32
    xn2  = H(LN(H(x1)))                                  mv_layernorm_q_fwd      -> fp16
    u,h  = o(xn2 . H(W1)^T + b),  H(gelu(u))             mv_gemm (GELU epilogue) -> fp16, fp16
    x2   = f(o(h . H(W2)^T + b) + x1)                    mv_gemm (+residual)     -> fp32
  dropout (EngineConfig.dropout / emb_dropout, training forwards only): D(y) = y * keep * s with the mask stream of
  include/mv_b200.h, fused where the tensor is produced — x0 = D_emb(embedding) (mv_dropout after mv_cls_rows),
  x1 = f(D(o(att . Wo^T + b)) + x) and x2 = f(D(o(h . W2^T + b)) + x1) in the residual epilogues, h = H(D(gelu(u)))
  with the saved gelu'(u) masked alike; the backward masks the gradient entering each dropped branch where the
  LayerNorm backward writes its fp16 operand copy and bias column sums.
  backward: straight-through quantisers (utils/quantize.py:87-89); dgrad / wgrad on the same GEMM
  kernel (wgrad reads dY and X in place as MN-major operands, split-K red.add into a flat fp32
  gradient buffer), GELU' in the dgrad epilogue, LN backward fused with the residual-gradient add,
  the fp16 operand copy and the bias-gradient column sums.

Gradients travel as fp16 tensor-core operands scaled by a power of two S chosen on the device from
the incoming gradient (the reference itself trains under GradScaler(65536), classification/
train.py:167); parameter gradients are un-scaled in fp32 before they are returned.
"""
import contextlib
import os

import torch

import mv_native as mv


class _Range:
    """`profile=True` of the reference's ViT (models/vit.py:115-124, 205-213: autograd-profiler record_function
    contexts): the same five labels, as a record_function (torch profiler) AND an NVTX range (nsys / ncu)."""

    def __init__(self, name):
        self.name = name
        self.rf = None

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)
        self.rf = torch.autograd.profiler.record_function(self.name)
        self.rf.__enter__()
        return self

    def __exit__(self, *exc):
        self.rf.__exit__(*exc)
        torch.cuda.nvtx.range_pop()
        return False


class EngineConfig:
    def __init__(self, dim, heads, mlp_dim, depth, patch, plan, dropout=0.0, emb_dropout=0.0):
        self.dim, self.heads, self.mlp_dim, self.depth, self.patch, self.plan = (
            dim, heads, mlp_dim, depth, patch, plan)
        mv.drop_params(dropout), mv.drop_params(emb_dropout)        # ValueError outside [0, 1], as nn.Dropout
        self.dropout, self.emb_dropout = float(dropout), float(emb_dropout)


PER_LAYER = 12   # ln1.w ln1.b qkv.w qkv.b out.w out.b ln2.w ln2.b fc1.w fc1.b fc2.w fc2.b

# Gradient-quantiser sites of encoder block l (include/mv_b200.h "gradient rounding stream"): 10 l + k; 10 depth is the
# patch-embedding weight, 10 depth + 1 + j the decoder's stubs (models/vit.py ViT._gfmt)
GS_LN1, GS_QKV_IN, GS_QKV_W, GS_OUT_IN, GS_OUT_W, GS_LN2, GS_FC1_IN, GS_FC1_W, GS_FC2_IN, GS_FC2_W = range(10)


def grad_round_offset(site, rank=0):
    """The stream offset of a gradient-quantiser site on data-parallel rank `rank`: site + (rank << 32)."""
    return int(site) + (int(rank) << 32)


class _Drops:
    """The dropout sites of one training forward and its backward: site ids of include/mv_b200.h ("dropout mask") and
    the seed tensor drawn for that forward.  Each method returns the `drop` argument of the mv_native calls, or None
    where the probability is 0 (the site is the identity and runs no mask code)."""

    def __init__(self, cfg, seed):
        self.p, self.pe, self.depth, self.seed = cfg.dropout, cfg.emb_dropout, cfg.depth, seed

    def _site(self, p, site):
        return (self.seed, p, site) if p > 0.0 else None

    def proj(self, l):
        return self._site(self.p, 3 * l)

    def fc1(self, l):
        return self._site(self.p, 3 * l + 1)

    def fc2(self, l):
        return self._site(self.p, 3 * l + 2)

    def emb(self):
        return self._site(self.pe, 3 * self.depth)


class EncoderEngine:
    def __init__(self, cfg, params):
        """params: [pe.w, pe.b] + PER_LAYER tensors per block, all fp32 CUDA nn.Parameters."""
        self.cfg = cfg
        self.params = list(params)
        assert len(self.params) == 2 + PER_LAYER * cfg.depth
        # debugging aids of the reference's model, off the training path: profile ranges and, per block, the module
        # the reference passes the softmax probabilities through (models/vit.py:80-82, 94 — a hook point)
        self.profile = False
        self.probes = None
        plan = cfg.plan
        if plan.inp not in ((5, 10), (8, 10), None):
            raise NotImplementedError("no tensor-core operand container for input format %r" % (plan.inp,))
        # 32-bit formats (TF32: inputs/weights on the (8,10) grid; FP32: no quantisers) run their
        # contractions as kind::tf32 on fp32 containers — what the reference's torch 1.11 does with its
        # default allow_tf32 matmuls; (8,10) values are exact tf32 operands.
        self.wide = plan.inp != (5, 10)
        # FP32 (no quantisers at all): fp32-grade arithmetic.  Linears run as 3xTF32 — operands split into
        # tf32 hi + lo parts concatenated along K (mv_split_tf32), so the kind::tf32 kernel accumulates
        # hi*hi + lo*hi + hi*lo — and attention / GELU, which have no quantiser to fuse with in this format,
        # use torch's fp32 ops.  This is the reference's "plumbing" configuration, not a performance path.
        self.exact = plan.inp is None
        # gradient quantiser of the input / weight quantisers (QPyTorch backward_number; QuantPlan.grad)
        self.gfmt = getattr(plan, "grad", None)
        if self.gfmt is not None and self.wide:
            raise NotImplementedError("a gradient format needs the 16-bit operand path (q_format=FP16_32)")
        if cfg.dim != cfg.heads * 64:
            raise ValueError("dim must equal heads * 64 (dim_head is fixed at 64, models/vit.py:178)")
        self.fmt = plan.inp
        self.dev = self.params[0].device
        self._wq = None
        self._wq_versions = None
        self._wq_capture_done = None
        self.capture_generation = 0
        sizes = [p.numel() for p in self.params]
        # gflat[0:4] is a slot that travels through the last gradient all-reduce: under data parallelism it carries
        # this rank's overflow flag to every rank (no extra collective)
        self.offsets = [4]
        for s in sizes:
            self.offsets.append(self.offsets[-1] + ((s + 3) // 4) * 4)
        self.gflat = torch.zeros(self.offsets[-1], dtype=torch.float32, device=self.dev)
        self.gviews = [self.gflat[self.offsets[i]:self.offsets[i] + sizes[i]].view_as(p)
                       for i, p in enumerate(self.params)]
        # Overflow handling in place of the reference's GradScaler (classification/train.py:167, 259-277), all on the
        # device: `overflow` is raised by the backward kernels (mv_set_overflow_flag), `scaler_state` =
        # {found_inf of the last backward, scale_target, good_steps}; an optimizer that understands found_inf
        # (utils.fused_adamw.FusedAdamW.step(found_inf=engine.found_inf)) skips the update, as GradScaler.step does
        self.overflow = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.scaler_state = torch.tensor([0.0, 1024.0, 0.0], dtype=torch.float32, device=self.dev)
        self.reducer = None      # set by parallel.DataParallel: called with flat gradient slices
        self.bucket_blocks = max(1, int(os.environ.get("MV_DP_BUCKET_BLOCKS", "3")))   # encoder blocks per all-reduce
        # True once an optimizer (utils/fused_adamw.FusedAdamW) emits q(W) / q(W)^T itself after every
        # update: a CUDA-graph capture then leaves the re-quantisation out of the graph
        self.external_requant = False
        # True for a model whose weights do not change while it is used (a distillation teacher, models/distill.py):
        # the operands are quantised once and served from the cache inside a CUDA-graph capture, so a replay does not
        # re-quantise them; outside a capture they are still rebuilt when the parameters change (e.g. load_state_dict)
        self.frozen_weights = False
        # nn.Module.training of the owning model (ViT.forward sets it): dropout acts in training forwards only
        self.training = True
        # seed of the last forward that applied dropout: int64 [1] on the device (its 64 bits are the Philox key)
        self.last_dropout_seed = None
        # None, or an int64 [1] device tensor that training forwards use instead of a fresh draw (reproduces the masks of
        # an earlier step, e.g. one replayed from a CUDA graph, given its last_dropout_seed)
        self.fixed_dropout_seed = None
        # stochastic gradient rounding (QuantPlan.grad_rounding == "stochastic" with a gradient format): the seed of the
        # last forward that drew one, an override like fixed_dropout_seed, and the seed of the running step (None when
        # this forward drew none; the decoder's stubs read it)
        self.grad_round = self.gfmt is not None and getattr(plan, "grad_rounding", "nearest") == "stochastic"
        self.last_grad_round_seed = None
        self.fixed_grad_round_seed = None
        self.step_grad_round_seed = None

    # ------------------------------------------------------------------ weights
    def _weight_indices(self):
        idx = [0]
        for l in range(self.cfg.depth):
            base = 2 + PER_LAYER * l
            idx += [base + 2, base + 4, base + 8, base + 10]
        return idx

    def quantised_weights(self):
        """weight_fake_quant of every Linear (torch.nn.qat.Linear.forward re-quantises each step):
        fp16 q(W) [out,in] for forward and q(W)^T [in,out] for dgrad; cached on parameter versions."""
        idx = self._weight_indices()
        versions = tuple(self.params[i]._version for i in idx) + tuple(
            self.params[i].data_ptr() for i in idx)
        capturing = torch.cuda.is_current_stream_capturing()
        if self._wq is not None and versions == self._wq_versions and (
                not capturing or self.external_requant):
            return self._wq
        if capturing and self._wq is not None and self._wq_capture_done == self._capture_key():
            return self._wq          # already re-quantised once inside this capture (forward)
        if capturing and self._wq is not None and self.frozen_weights:
            return self._wq
        if self.exact:
            wq = {i: (mv.split_tf32(self.params[i].detach(), 1),
                      mv.split_tf32(self.params[i].detach().t().contiguous(), 1)) for i in idx}
        else:
            wq = self._requantise_all(idx)
        self._wq, self._wq_versions = wq, versions
        # inside a CUDA-graph capture the re-quantisation must be part of the graph (weights change
        # between replays) but only once per step: backward reuses the forward's operands
        self._wq_capture_done = self._capture_key() if capturing else None
        return wq

    def _capture_key(self):
        """Identifies the running capture: the capturing stream's handle and the capture generation
        (utils.graph.GraphedTrainStep bumps it around every capture, so a flag left by an earlier capture on the
        same stream never matches a later one)."""
        return (torch.cuda.current_stream().cuda_stream, self.capture_generation)

    def _requantise_all(self, idx):
        """q(W) and q(W)^T of every Linear in ONE launch: the multi-tensor optimizer kernel (mv_adamw_step)
        in its skip mode leaves parameters and moments untouched and only emits the operand tiles, so the
        per-step weight_fake_quant of 4 * depth + 1 Linears costs one kernel instead of one each."""
        import ctypes
        from myrtle_vision.utils.fused_adamw import AdamwTensor
        dt = torch.float32 if self.wide else torch.float16
        e, m = self.fmt if self.fmt else (0, 0)
        key = tuple(self.params[i].data_ptr() for i in idx)
        tab = getattr(self, "_rq_table", None)
        if tab is None or tab[0] != key:
            wq, rows, chunk = {}, [], 0
            for i in idx:
                w = self.params[i].detach()
                r, c = w.shape
                q = torch.empty(r, c, dtype=dt, device=self.dev)
                qt = torch.empty(c, r, dtype=dt, device=self.dev)
                wq[i] = (q, qt)
                t = AdamwTensor()
                t.param, t.grad, t.exp_avg, t.exp_avg_sq = w.data_ptr(), w.data_ptr(), w.data_ptr(), w.data_ptr()
                t.wq, t.wq_t, t.n, t.rows, t.cols = q.data_ptr(), qt.data_ptr(), w.numel(), r, c
                t.wq_dtype, t.q_exp, t.q_man, t.lr, t.weight_decay, t.chunk0 = mv._DT[dt], e, m, 0.0, 0.0, chunk
                chunk += ((r + 31) // 32) * ((c + 31) // 32)
                rows.append(t)
            arr = (AdamwTensor * len(rows))(*rows)
            table = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(self.dev)
            hyper = torch.tensor([0.9, 0.999, 1e-8, 1.0, 1.0, 1.0], dtype=torch.float32, device=self.dev)  # found_inf = 1: skip
            tab = (key, wq, table, hyper, len(rows), chunk)
            self._rq_table = tab
        _, wq, table, hyper, n, chunks = tab
        mv._check(mv.lib().mv_adamw_step(ctypes.c_void_p(table.data_ptr()), n, chunks, mv._ptr(hyper),
                                         mv._stream()), "mv_adamw_step (re-quantise)")
        return wq

    def invalidate_weights(self):
        """The parameters changed behind the version counters: rebuild the operands on the next use."""
        self._wq, self._wq_versions = None, None

    def mark_weights_fresh(self):
        """The operand buffers were just rewritten from the current parameter values (fused optimizer)."""
        idx = self._weight_indices()
        self._wq_versions = tuple(self.params[i]._version for i in idx) + tuple(
            self.params[i].data_ptr() for i in idx)

    @property
    def rank(self):
        """Data-parallel rank (0 without parallel.DataParallel): the high word of the gradient rounding offsets."""
        if self.reducer is None or getattr(self.reducer, "world", 1) <= 1:
            return 0
        import torch.distributed as dist
        return dist.get_rank(self.reducer.group)

    @property
    def found_inf(self):
        """fp32 [1] on the device: 1.0 when the last backward overflowed (identical on every data-parallel rank)."""
        return self.scaler_state[0:1]

    def _gradient_scale(self, gx):
        """Power-of-two operand scale S chosen on the device: max |gx| * S lands in [target / 2, target]."""
        if self.gfmt is not None:
            # the gradient quantisers must see the gradient as autograd presents it (what QPyTorch's would see under
            # the reference's GradScaler): no rescaling here, loss scaling is the caller's
            return self._one()
        amax = torch.linalg.vector_norm(gx, float("inf")).clamp_min(1e-30)          # one reduction, no |gx| temporary
        return torch.exp2(torch.floor(torch.log2(self.scaler_state[1] / amax))).clamp(2.0 ** -60, 2.0 ** 60)

    # ------------------------------------------------------------------ forward
    def _range(self, name):
        return _Range(name) if self.profile else contextlib.nullcontext()

    def _probe_attention(self, l, qkv, B, H, N):
        """Debug only: if forward hooks are registered on block l's `attn_output` module, hand it the softmax
        probabilities [B, H, N, N] (computed unfused from the same qkv; the fused kernels never materialise them).
        The training arithmetic is not touched; Python hooks do not replay inside a captured CUDA graph."""
        m = None if self.probes is None else self.probes[l]
        if m is None or not (m._forward_hooks or m._forward_pre_hooks):
            return
        q, k = qkv.view(B, N, 3, H, 64).float().permute(2, 0, 3, 1, 4)[:2]
        m(torch.softmax(torch.matmul(q, k.transpose(-2, -1)) * 0.125, dim=-1))

    def _draw_drops(self):
        """A fresh seed per training forward with dropout, drawn on the device from torch's default CUDA generator: a
        captured CUDA graph replays the draw with a new philox offset, so every replay gets new masks, and
        torch.manual_seed makes runs repeatable.  None when dropout is off (no draw: the generator is not advanced)."""
        cfg = self.cfg
        if not self.training or (cfg.dropout == 0.0 and cfg.emb_dropout == 0.0):
            return None
        seed = self.fixed_dropout_seed
        if seed is None:
            seed = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=self.dev)
        self.last_dropout_seed = seed
        return _Drops(cfg, seed)

    def _draw_grad_round(self, save):
        """A fresh 64-bit seed per forward that may be followed by a backward, when stochastic gradient rounding is on
        (drawn after the dropout seed, on the device, like it).  None otherwise: no draw, the generator is not
        advanced."""
        if not (save and self.grad_round):
            return None
        seed = self.fixed_grad_round_seed
        if seed is None:
            seed = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=self.dev)
        self.last_grad_round_seed = seed
        return seed

    def forward(self, img, pos_full, cls_token, save, token=None, mix=None):
        """token (optional, [1, 1, D]): a distillation token appended as the last row N - 1 of every image, with no
        positional embedding (DESIGN.md section 7); pos_full then still holds the N - 1 rows of cls + grid.
        mix (optional): Mixup / CutMix records (mv_native.mix_draw): the encoder sees the mixed batch, mixed inside the
        patch gather; the saved patches are the mixed ones, so the backward needs nothing else."""
        # A training forward clears self.overflow and its backward closes the window (mv_overflow_update); inference
        # forwards report nothing.  The library keeps one process-wide flag pointer, so it is registered only while
        # this engine's own kernels run and cleared on the way out, exception or not: launches outside the step (other
        # models, standalone calls) never write into this engine's flag, nor into it after it is freed.  A captured
        # CUDA graph keeps the pointer its kernels were captured with.
        mv.set_overflow_flag(self.overflow if save else None)
        try:
            if save:
                self.overflow.zero_()
            drops = self._draw_drops()
            self.step_grad_round_seed = self._draw_grad_round(save)
            if self.wide:
                return self._forward_wide(img, pos_full, cls_token, save, drops, token, mix)
            x, saved = self._forward_16(img, pos_full, cls_token, save, drops, token, mix)
            if saved is not None:
                saved["grad_round"] = self.step_grad_round_seed
            return x, saved
        finally:
            mv.set_overflow_flag(None)

    def _embed_inputs(self, pos_full, token, N, D):
        """The patch-embedding GEMM's positional residual [N, D] and the patchify slot mode: with a token its last row
        is zero (mv_token_row overwrites that row of x afterwards) and `patches` gets a zero row at both ends."""
        pos32 = pos_full.detach().reshape(N - (token is not None), D)
        if token is None:
            return pos32.contiguous(), 1
        return torch.cat((pos32, pos32.new_zeros(1, D))), 2

    def _token_row(self, token, x, B, N, D):
        if token is not None:
            mv.token_row(token.detach().reshape(D).contiguous(), x, B, N, D, N - 1, q_ff=self.cfg.plan.ff)

    def _patchify(self, img, mix, P, out_dtype, slots):
        if mix is None:
            return mv.patchify_q(img, P, q_in=self.fmt, out_dtype=out_dtype, cls_slot=slots)
        return mv.patchify_mix_q(img, mix, P, q_in=self.fmt, out_dtype=out_dtype, cls_slot=slots)

    def _forward_16(self, img, pos_full, cls_token, save, drops, token=None, mix=None):
        cfg, plan, fmt = self.cfg, self.cfg.plan, self.fmt
        B, C, Hh, Ww = img.shape
        P = cfg.patch
        N = (Hh // P) * (Ww // P) + 1 + (token is not None)
        M, D, Mm, H = B * N, cfg.dim, cfg.mlp_dim, cfg.heads
        prm = [p.detach() for p in self.params]
        wq = self.quantised_weights()
        f16 = torch.float16
        dev = img.device

        with self._range("patch_to_embedding"):
            pos32, slots = self._embed_inputs(pos_full, token, N, D)
            patches = self._patchify(img, mix, P, f16, slots)                    # [M, P*P*C], zero token rows
            x = torch.empty(M, D, dtype=torch.float32, device=dev)
            mv.gemm(patches, wq[0][0], x, bias=prm[1], q_out=plan.out, residual=pos32, q_res=plan.ff,
                    rows_per_img=N)
            mv.cls_rows(cls_token.detach().reshape(D).contiguous(), pos32, x, B, N, D, q_ff=plan.ff)
            self._token_row(token, x, B, N, D)
            if drops and drops.emb():
                mv.dropout(x, drops.emb(), out=x)

        saved = {"B": B, "N": N, "patches": patches, "layers": [], "drops": drops,
                 "token": token is not None} if save else None
        with self._range("transformer"):
            for l in range(cfg.depth):
                b0 = 2 + PER_LAYER * l
                with self._range("transformer:attention"):
                    xn1, mean1, rstd1 = mv.layernorm_q_fwd(x, prm[b0], prm[b0 + 1], q_in=fmt, q_post=fmt)
                    qkv = torch.empty(M, 3 * D, dtype=f16, device=dev)
                    mv.gemm(xn1, wq[b0 + 2][0], qkv, bias=prm[b0 + 3], q_out=plan.out)
                    self._probe_attention(l, qkv, B, H, N)
                    att, lse = mv.attention_fwd(qkv, B, H, N, scale=0.125, q_out=fmt)
                    x1 = torch.empty(M, D, dtype=torch.float32, device=dev)
                    mv.gemm(att, wq[b0 + 4][0], x1, bias=prm[b0 + 5], q_out=plan.out, residual=x,
                            q_res=plan.ff, drop=drops and drops.proj(l))
                with self._range("transformer:feedforward"):
                    xn2, mean2, rstd2 = mv.layernorm_q_fwd(x1, prm[b0 + 6], prm[b0 + 7], q_in=fmt, q_post=fmt)
                    u = torch.empty(M, Mm, dtype=f16, device=dev)
                    h = torch.empty(M, Mm, dtype=f16, device=dev)
                    mv.gemm(xn2, wq[b0 + 8][0], h, bias=prm[b0 + 9], q_out=plan.out, aux=u,
                            epilogue=mv.EPI_GELU, q_res=fmt, drop=drops and drops.fc1(l))
                    x2 = torch.empty(M, D, dtype=torch.float32, device=dev)
                    mv.gemm(h, wq[b0 + 10][0], x2, bias=prm[b0 + 11], q_out=plan.out, residual=x1,
                            q_res=plan.ff, drop=drops and drops.fc2(l))
                if save:
                    saved["layers"].append((x, xn1, mean1, rstd1, qkv, att, lse, x1, xn2, mean2, rstd2, u, h))
                x = x2
        return x.view(B, N, D), saved

    # ----------------------------------------------------------------- backward
    def backward(self, saved, gx):
        # the overflow window of the training forward, continued for this engine's backward launches only (see forward)
        mv.set_overflow_flag(self.overflow)
        try:
            if self.wide:
                return self._backward_wide(saved, gx)
            return self._backward_16(saved, gx)
        finally:
            mv.set_overflow_flag(None)

    def _backward_16(self, saved, gx):
        cfg, fmt = self.cfg, self.fmt
        B, N = saved["B"], saved["N"]
        M, D, Mm, H = B * N, cfg.dim, cfg.mlp_dim, cfg.heads
        prm = [p.detach() for p in self.params]
        wq = self.quantised_weights()
        g = self.gviews
        dev = gx.device
        f16 = torch.float16

        # power-of-two gradient scale chosen on the device (no host sync)
        gx = gx.reshape(M, D)
        S = self._gradient_scale(gx)
        drops = saved["drops"]
        last = cfg.depth - 1
        if drops and drops.fc2(last):
            # the last block's fc2 branch receives the masked gradient (its dgrad / wgrad operand and bias column sums);
            # the residual stream keeps the unmasked fp32 one
            dx, _ = mv.scale_f32(gx, S)
            dxm = mv.dropout(dx, drops.fc2(last))
            self.gflat.zero_()
            mv.colsum(dxm, g[2 + PER_LAYER * last + 11].view(-1))
            _, dx_h = mv.scale_f32(dxm, self._one(), want_f32=False, want_f16=True)
            del dxm
        else:
            dx, dx_h = mv.scale_f32(gx, S, want_f16=True)                         # fp32 master and fp16 operand in one pass
            self.gflat.zero_()
            mv.colsum(dx, g[2 + PER_LAYER * last + 11].view(-1))           # fc2 bias of the last block

        # Gradient quantiser G (QuantPlan.grad, normally None): the backward of every QuantStub in front of a Linear is
        # the q_out of that Linear's dgrad GEMM (before the gelu' multiply for fc2's), of every stub in front of a
        # LayerNorm a rounding inside mv_layernorm_q_bwd (before the residual gradient is added), of every weight
        # quantiser a pass over the accumulated weight gradient (before the data-parallel reduction, as autograd
        # would apply it to the local gradient)
        gq = self.gfmt
        # stochastic rounding (QuantPlan.grad_rounding): every site rounds with the stream of include/mv_b200.h under
        # the seed its forward drew; gr(site) is the grad_round argument of the mv_native calls, None: nearest
        seed, rank = saved.get("grad_round"), self.rank

        def gr(site):
            return None if seed is None else (seed, grad_round_offset(site, rank))

        def wq_grad(i, site):
            if gq is not None and seed is not None:
                mv.float_quantize_dev(g[i], gq[0], gq[1], gr(site), out=g[i])
            elif gq is not None:
                mv.float_quantize(g[i], gq[0], gq[1], out=g[i])

        for l in range(last, -1, -1):
            b0 = 2 + PER_LAYER * l
            x, xn1, mean1, rstd1, qkv, att, lse, x1, xn2, mean2, rstd2, u, h = saved["layers"][l]
            s0 = 10 * l                                                     # this block's gradient-quantiser sites
            # ---- FeedForward
            du = torch.empty(M, Mm, dtype=f16, device=dev)
            # fc1's bias gradient (column sums of du) rides in the epilogue
            mv.gemm(dx_h, wq[b0 + 10][1], du, aux=u, epilogue=mv.EPI_DGELU, colsum=g[b0 + 9].view(-1), q_out=gq,
                    grad_round=gr(s0 + GS_FC2_IN))
            # fc2's [D, 4D] gradient as its transpose h^T dx: 256 x 384 tiles over 4D rows instead of 1.5 padded 256-row tiles
            mv.gemm(h, dx_h, g[b0 + 10], a_major=1, b_major=1, accumulate=True, transpose_out=True)
            wq_grad(b0 + 10, s0 + GS_FC2_W)
            dxn2 = torch.empty(M, D, dtype=f16, device=dev)
            mv.gemm(du, wq[b0 + 8][1], dxn2, tag="dgrad", q_out=gq, grad_round=gr(s0 + GS_FC1_IN))
            mv.gemm(du, xn2, g[b0 + 8], a_major=1, b_major=1, accumulate=True)
            wq_grad(b0 + 8, s0 + GS_FC1_W)
            del du
            # dx1_h and to_out's bias gradient: the masked gradient of the to_out branch (dropout site of to_out)
            dx1, dx1_h = mv.layernorm_q_bwd(dxn2, x1, prm[b0 + 6], mean2, rstd2, dres=dx, q_in=fmt,
                                            dgamma=g[b0 + 6], dbeta=g[b0 + 7], dbias_prev=g[b0 + 5],
                                            q_grad=gq, drop=drops and drops.proj(l), grad_round=gr(s0 + GS_LN2))
            # ---- Attention
            datt = torch.empty(M, D, dtype=f16, device=dev)
            mv.gemm(dx1_h, wq[b0 + 4][1], datt, tag="dgrad", q_out=gq, grad_round=gr(s0 + GS_OUT_IN))
            mv.gemm(dx1_h, att, g[b0 + 4], a_major=1, b_major=1, accumulate=True)
            wq_grad(b0 + 4, s0 + GS_OUT_W)
            dqkv = mv.attention_bwd(qkv, att, datt, lse, B, H, N, scale=0.125,
                                    dbias=g[b0 + 3].view(-1))          # to_qkv's bias gradient fused
            dxn1 = dxn2      # reuse
            mv.gemm(dqkv, wq[b0 + 2][1], dxn1, tag="dgrad", q_out=gq, grad_round=gr(s0 + GS_QKV_IN))
            mv.gemm(dqkv, xn1, g[b0 + 2], a_major=1, b_major=1, accumulate=True)
            wq_grad(b0 + 2, s0 + GS_QKV_W)
            prev_bias = g[b0 - 1] if l > 0 else None                       # fc2 bias of block l-1
            # dx_h (and prev_bias): masked with block l-1's fc2 site; below block 0 everything (dx too) with the embedding
            # site — the patch wgrad, dpos / dcls and the patch bias all lie behind that dropout
            drop = (drops.fc2(l - 1) if l > 0 else drops.emb()) if drops else None
            dx, dx_h = mv.layernorm_q_bwd(dxn1, x, prm[b0], mean1, rstd1, dres=dx1, q_in=fmt,
                                          dgamma=g[b0], dbeta=g[b0 + 1], dbias_prev=prev_bias,
                                          dx=dx, dx_f16=dx_h, q_grad=gq, drop=drop, mask_dx=l == 0,
                                          grad_round=gr(s0 + GS_LN1))
            if self.reducer is not None and l % self.bucket_blocks == 0:
                # one all-reduce per bucket of `bucket_blocks` encoder blocks (their gradient slices are contiguous),
                # issued as soon as the bucket's last wgrad is enqueued
                top = min(cfg.depth, l + self.bucket_blocks)
                lo, hi = self.offsets[b0], self.offsets[2 + PER_LAYER * top]
                self.reducer.reduce_slice(self.gflat[lo:hi], 1.0 / S)
        # ---- patch embedding: dW = dx^T patches (cls rows of `patches` are zero)
        mv.gemm(dx_h, saved["patches"], g[0], a_major=1, b_major=1, accumulate=True)
        wq_grad(0, 10 * cfg.depth)
        return self._finish_backward(dx, S, B, N, D, saved["token"])

    def _finish_backward(self, dx, S, B, N, D, token=False):
        g, dev = self.gviews, dx.device
        dpos = torch.zeros(N * D, dtype=torch.float32, device=dev)
        mv.colsum(dx.view(B, N * D), dpos)
        dpos = dpos.view(1, N, D)
        g[1].copy_(dpos[0, 1:N - token].sum(0))                            # bias: patch rows only
        inv = 1.0 / S
        slot = None
        if self.reducer is not None:
            # this rank's overflow flag rides in the slot in front of the last bucket (any positive value survives
            # the 1 / (S * world) factor: S is clamped to 2^+-60)
            self.gflat[0:1].copy_(self.overflow)
            self.reducer.reduce_slice(self.gflat[:self.offsets[2]], inv)
            self.reducer.wait()
            slot = self.gflat[0:1]
        dpos = dpos * inv
        dcls = dpos[:, 0:1, :].clone()
        dtok = None
        if token:
            # the token row has no positional embedding: its column sum is the token's gradient
            dtok = dpos[:, N - 1:N, :].clone()
            dpos = dpos[:, :N - 1, :]
        # hand autograd its own copy: self.gflat is reused (zeroed) by the next backward.  The same pass un-scales
        # (single GPU) and tests every parameter gradient for inf / NaN (the overflow sink)
        if self.reducer is not None:
            out, _ = mv.scale_f32(self.gflat, self._one(), invert=False)
        else:
            out, _ = mv.scale_f32(self.gflat, S, invert=True)
        mv.overflow_update(self.overflow, self.scaler_state, shared_slot=slot)
        grads = [out[self.offsets[i]:self.offsets[i] + p.numel()].view_as(p)
                 for i, p in enumerate(self.params)]
        return dpos, dcls, dtok, grads

    def _one(self):
        if getattr(self, "_one_t", None) is None:
            self._one_t = torch.ones(1, dtype=torch.float32, device=self.dev)
        return self._one_t


    # ------------------------------------------------- 32-bit formats (TF32 / FP32)
    # Same step as above on fp32 containers.  Every Linear is a kind::tf32 GEMM on K-major operands;
    # wgrad therefore takes explicit transposes (mv_widen_transpose) instead of the in-place MN-major
    # reads of the 16-bit path.  Attention keeps the fp16 tcgen05 kernels: qkv / attention output /
    # their gradients carry 11 significant bits, the same as a tf32 operand.
    def _forward_wide(self, img, pos_full, cls_token, save, drops, token=None, mix=None):
        cfg, plan, fmt = self.cfg, self.cfg.plan, self.fmt
        B, C, Hh, Ww = img.shape
        P = cfg.patch
        N = (Hh // P) * (Ww // P) + 1 + (token is not None)
        M, D, Mm, H = B * N, cfg.dim, cfg.mlp_dim, cfg.heads
        prm = [p.detach() for p in self.params]
        wq = self.quantised_weights()
        f16, f32 = torch.float16, torch.float32
        dev = img.device
        ex = self.exact
        A_ = (lambda t: mv.split_tf32(t, 0)) if ex else (lambda t: t)        # A operand of a Linear

        pos32, slots = self._embed_inputs(pos_full, token, N, D)
        patches = self._patchify(img, mix, P, f32, slots)
        x = torch.empty(M, D, dtype=f32, device=dev)
        mv.gemm(A_(patches), wq[0][0], x, bias=prm[1], q_out=plan.out, residual=pos32, q_res=plan.ff,
                rows_per_img=N)
        mv.cls_rows(cls_token.detach().reshape(D).contiguous(), pos32, x, B, N, D, q_ff=plan.ff)
        self._token_row(token, x, B, N, D)
        if drops and drops.emb():
            mv.dropout(x, drops.emb(), out=x)

        def linear_res(a, w, bias, res, drop):
            # x + D(Linear(a)): the single-CTA kind::tf32 kernel has no dropout epilogue, so the mask is a pass of its own
            y = torch.empty(M, D, dtype=f32, device=dev)
            if drop is None:
                return mv.gemm(a, w, y, bias=bias, q_out=plan.out, residual=res, q_res=plan.ff)
            mv.gemm(a, w, y, bias=bias, q_out=plan.out)
            mv.dropout(y, drop, out=y)
            y.add_(res)
            if plan.ff:
                mv.float_quantize(y, plan.ff[0], plan.ff[1], out=y)
            return y

        saved = {"B": B, "N": N, "patches": patches, "layers": [], "drops": drops,
                 "token": token is not None} if save else None
        for l in range(cfg.depth):
            b0 = 2 + PER_LAYER * l
            xn1, mean1, rstd1 = mv.layernorm_q_fwd(x, prm[b0], prm[b0 + 1], q_in=fmt, q_post=fmt,
                                                   out_dtype=f32)
            qkv = torch.empty(M, 3 * D, dtype=f32 if ex else f16, device=dev)
            mv.gemm(A_(xn1), wq[b0 + 2][0], qkv, bias=prm[b0 + 3], q_out=plan.out)
            self._probe_attention(l, qkv, B, H, N)
            if ex:
                att, lse = self._attention_exact_fwd(qkv, B, H, N)           # lse slot holds the probabilities
                att16 = att
            else:
                att16, lse = mv.attention_fwd(qkv, B, H, N, scale=0.125, q_out=fmt)
                att, _ = mv.widen_transpose(att16, want_copy=True, want_t=False)
            x1 = linear_res(A_(att), wq[b0 + 4][0], prm[b0 + 5], x, drops and drops.proj(l))
            xn2, mean2, rstd2 = mv.layernorm_q_fwd(x1, prm[b0 + 6], prm[b0 + 7], q_in=fmt, q_post=fmt,
                                                   out_dtype=f32)
            h = torch.empty(M, Mm, dtype=f32, device=dev)
            d1 = drops and drops.fc1(l)
            if ex:
                gd = torch.empty(M, Mm, dtype=f32, device=dev)               # u (pre-GELU), fp32
                mv.gemm(A_(xn2), wq[b0 + 8][0], gd, bias=prm[b0 + 9])
                h = torch.nn.functional.gelu(gd)
                if d1:
                    mv.dropout(h, d1, out=h)
            else:
                # gelu'(u); with dropout the backward applies the mask after the gelu' multiply (mv_dropout on du)
                gd = torch.empty(M, Mm, dtype=f16, device=dev)
                mv.gemm(xn2, wq[b0 + 8][0], h, bias=prm[b0 + 9], q_out=plan.out, aux=gd,
                        epilogue=mv.EPI_GELU, q_res=None if d1 else fmt)
                if d1:
                    mv.dropout(h, d1, out=h)
                    if fmt:
                        mv.float_quantize(h, fmt[0], fmt[1], out=h)
            x2 = linear_res(A_(h), wq[b0 + 10][0], prm[b0 + 11], x1, drops and drops.fc2(l))
            if save:
                saved["layers"].append((x, xn1, mean1, rstd1, qkv, att16, lse, x1, xn2, mean2, rstd2, gd, h))
            x = x2
        return x.view(B, N, D), saved

    @staticmethod
    def _attention_exact_fwd(qkv, B, H, N):
        q, k, v = qkv.view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
        prob = torch.softmax(torch.matmul(q, k.transpose(-2, -1)) * 0.125, dim=-1)
        return torch.matmul(prob, v).transpose(1, 2).reshape(B * N, H * 64), prob

    @staticmethod
    def _attention_exact_bwd(qkv, prob, d_att, B, H, N):
        q, k, v = qkv.view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
        do = d_att.view(B, N, H, 64).transpose(1, 2)
        dv = torch.matmul(prob.transpose(-2, -1), do)
        dp = torch.matmul(do, v.transpose(-2, -1))
        ds = prob * (dp - (dp * prob).sum(-1, keepdim=True)) * 0.125
        dq, dk = torch.matmul(ds, k), torch.matmul(ds.transpose(-2, -1), q)
        return torch.stack((dq, dk, dv), dim=0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * H * 64)

    def _backward_wide(self, saved, gx):
        cfg, fmt = self.cfg, self.fmt
        B, N = saved["B"], saved["N"]
        M, D, Mm, H = B * N, cfg.dim, cfg.mlp_dim, cfg.heads
        prm = [p.detach() for p in self.params]
        wq = self.quantised_weights()
        g = self.gviews
        dev = gx.device
        f16, f32 = torch.float16, torch.float32

        ex = self.exact
        A_ = (lambda t: mv.split_tf32(t, 0)) if ex else (lambda t: t)

        def wgrad(dy, act, out):                       # out[o, i] += sum_m dy[m, o] act[m, i]
            _, dy_t = mv.widen_transpose(dy, padded=ex)
            _, act_t = mv.widen_transpose(act, padded=ex)
            if ex:
                dy_t, act_t = mv.split_tf32(dy_t, 0), mv.split_tf32(act_t, 1)
            mv.gemm(dy_t, act_t, out, accumulate=True)

        # the fp16 attention backward wants its gradient operand inside fp16's range: same
        # power-of-two scale as the 16-bit path, removed from the parameter gradients at the end
        gx = gx.reshape(M, D)
        S = self._gradient_scale(gx)
        dx, _ = mv.scale_f32(gx, S)
        self.gflat.zero_()
        last = cfg.depth - 1
        drops = saved["drops"]
        # with dropout each masked branch gradient is a pass of its own (mv_dropout) and its bias gradient a colsum of it
        dropping = bool(drops and drops.p > 0.0)
        if not dropping:
            mv.colsum(dx, g[2 + PER_LAYER * last + 11].view(-1))

        for l in range(last, -1, -1):
            b0 = 2 + PER_LAYER * l
            x, xn1, mean1, rstd1, qkv, att16, lse, x1, xn2, mean2, rstd2, gd, h = saved["layers"][l]
            # ---- FeedForward
            dxm = dx
            if dropping:
                dxm = mv.dropout(dx, drops.fc2(l))
                mv.colsum(dxm, g[b0 + 11].view(-1))
            du = torch.empty(M, Mm, dtype=f32, device=dev)
            if ex:
                mv.gemm(A_(dxm), wq[b0 + 10][1], du)
                u = gd                                                       # gelu'(u) = Phi(u) + u phi(u)
                du.mul_(0.5 * (1.0 + torch.erf(u * 0.7071067811865476))
                        + u * torch.exp(-0.5 * u * u) * 0.3989422804014327)
            else:
                mv.gemm(dxm, wq[b0 + 10][1], du, aux=gd, epilogue=mv.EPI_DGELU)
            if dropping:
                mv.dropout(du, drops.fc1(l), out=du)
            wgrad(dxm, h, g[b0 + 10])
            del dxm
            dxn2 = torch.empty(M, D, dtype=f32, device=dev)
            mv.gemm(A_(du), wq[b0 + 8][1], dxn2, tag="dgrad")
            wgrad(du, xn2, g[b0 + 8])
            mv.colsum(du, g[b0 + 9].view(-1))
            del du
            dx1, _ = mv.layernorm_q_bwd(dxn2, x1, prm[b0 + 6], mean2, rstd2, dres=dx, q_in=fmt,
                                        dgamma=g[b0 + 6], dbeta=g[b0 + 7],
                                        dbias_prev=None if dropping else g[b0 + 5], want_f16=False)
            # ---- Attention
            dx1m = dx1
            if dropping:
                dx1m = mv.dropout(dx1, drops.proj(l))
                mv.colsum(dx1m, g[b0 + 5].view(-1))
            datt = torch.empty(M, D, dtype=f32 if ex else f16, device=dev)
            mv.gemm(A_(dx1m), wq[b0 + 4][1], datt, tag="dgrad")
            wgrad(dx1m, att16, g[b0 + 4])
            del dx1m
            if ex:
                dqkv16 = dqkv = self._attention_exact_bwd(qkv, lse, datt, B, H, N)
                _, dqkv_t = mv.widen_transpose(dqkv, padded=True)
            else:
                dqkv16 = mv.attention_bwd(qkv, att16, datt, lse, B, H, N, scale=0.125, dbias=g[b0 + 3].view(-1))
                dqkv, dqkv_t = mv.widen_transpose(dqkv16, want_copy=True)
            dxn1 = dxn2
            mv.gemm(A_(dqkv), wq[b0 + 2][1], dxn1, tag="dgrad")
            _, xn1_t = mv.widen_transpose(xn1, padded=ex)
            if ex:
                dqkv_t, xn1_t = mv.split_tf32(dqkv_t, 0), mv.split_tf32(xn1_t, 1)
            mv.gemm(dqkv_t, xn1_t, g[b0 + 2], accumulate=True)
            if ex:
                mv.colsum(dqkv16, g[b0 + 3].view(-1))
            prev_bias = g[b0 - 1] if l > 0 and not dropping else None
            dx, _ = mv.layernorm_q_bwd(dxn1, x, prm[b0], mean1, rstd1, dres=dx1, q_in=fmt,
                                       dgamma=g[b0], dbeta=g[b0 + 1], dbias_prev=prev_bias,
                                       want_f16=False, dx=dx)
            if self.reducer is not None and l % self.bucket_blocks == 0:
                # one all-reduce per bucket of `bucket_blocks` encoder blocks (their gradient slices are contiguous),
                # issued as soon as the bucket's last wgrad is enqueued
                top = min(cfg.depth, l + self.bucket_blocks)
                lo, hi = self.offsets[b0], self.offsets[2 + PER_LAYER * top]
                self.reducer.reduce_slice(self.gflat[lo:hi], 1.0 / S)
        if drops and drops.emb():
            mv.dropout(dx, drops.emb(), out=dx)
        wgrad(dx, saved["patches"], g[0])
        return self._finish_backward(dx, S, B, N, D, saved["token"])


class EncoderFunction(torch.autograd.Function):
    @classmethod
    def apply(cls, engine, img, pos_full, cls_token, *params, token=None, mix=None):
        """token: optional distillation token [1, 1, D]; mix: optional Mixup / CutMix records (EncoderEngine.forward)."""
        # ctx.needs_input_grad follows requires_grad even under torch.no_grad(), and forward() itself always runs with
        # grad mode off, so grad mode is read here: without it the forward saves nothing and reports into no flag
        if not torch.is_grad_enabled():
            return engine.forward(img, pos_full, cls_token, save=False, token=token, mix=mix)[0]
        return super().apply(engine, img, pos_full, cls_token, token, mix, *params)

    @staticmethod
    def forward(ctx, engine, img, pos_full, cls_token, token, mix, *params):
        need = any(ctx.needs_input_grad)      # False when no input requires a gradient
        with torch.no_grad():
            x, saved = engine.forward(img, pos_full, cls_token, save=need, token=token, mix=mix)
        ctx.engine, ctx.saved = engine, saved
        return x

    @staticmethod
    def backward(ctx, gx):
        engine, saved = ctx.engine, ctx.saved
        if saved is None:
            raise RuntimeError("backward through an encoder forward that ran without grad")
        if engine.reducer is not None:
            engine.reducer.queue_finalize()
        with torch.no_grad():
            dpos, dcls, dtok, g = engine.backward(saved, gx.contiguous())
        ctx.saved = None
        return (None, None, dpos, dcls, dtok, None) + tuple(g)
