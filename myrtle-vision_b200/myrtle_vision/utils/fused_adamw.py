"""AdamW for the B200 path: one multi-tensor kernel launch per step, fused with the next step's
weight fake-quantisation (SURVEY.md §8f.1; reference optimizer: timm AdamW built in
classification/train.py:161-166 and stepped at :274-277).

`FusedAdamW(params, lr, betas, eps, weight_decay, model=vit)` behaves like `torch.optim.AdamW`
(same update rule, `param_groups` for the lr scheduler, `state_dict()` with `exp_avg` /
`exp_avg_sq` / `step`).  When `model` is given, the Linear weights of its fused encoder are
updated by 32x32 tiles and the kernel writes q(W) and q(W)^T straight into the engine's
tensor-core operand buffers, so the forward that follows does not re-quantise them.

`step(inv_scale=None, found_inf=None)` takes optional DEVICE scalars with GradScaler semantics
(gradients are multiplied by inv_scale; a non-zero found_inf skips the update) so that a scaled
training loop needs no host synchronisation.  There is no CPU fallback.
"""
import ctypes

import torch

import mv_native as mv


class AdamwTensor(ctypes.Structure):
    _fields_ = [("param", ctypes.c_void_p), ("grad", ctypes.c_void_p), ("exp_avg", ctypes.c_void_p),
                ("exp_avg_sq", ctypes.c_void_p), ("wq", ctypes.c_void_p), ("wq_t", ctypes.c_void_p),
                ("n", ctypes.c_int64), ("rows", ctypes.c_int), ("cols", ctypes.c_int),
                ("wq_dtype", ctypes.c_int), ("q_exp", ctypes.c_int), ("q_man", ctypes.c_int),
                ("lr", ctypes.c_float), ("weight_decay", ctypes.c_float), ("chunk0", ctypes.c_int)]


class AdamwLpTensor(ctypes.Structure):
    """mv_adamw_lp_tensor: the per-tensor side table of mv_adamw_lp_step (qtorch.optim.OptimLP's fused path)."""
    _fields_ = [("acc", ctypes.c_void_p), ("grad_out", ctypes.c_void_p), ("index", ctypes.c_uint32)]


class LpQuant(ctypes.Structure):
    """mv_lp_quant: one quantiser site of mv_adamw_lp_step."""
    _fields_ = [("kind", ctypes.c_int), ("rounding", ctypes.c_int), ("exp_bits", ctypes.c_int),
                ("man_bits", ctypes.c_int), ("wl", ctypes.c_int), ("fl", ctypes.c_int), ("clamp", ctypes.c_int),
                ("symmetric", ctypes.c_int)]


class OptimLpSpec(ctypes.Structure):
    """mv_optim_lp: the five quantisers, gradient scaling and rounding seed of mv_adamw_lp_step."""
    _fields_ = [("grad", LpQuant), ("exp_avg", LpQuant), ("exp_avg_sq", LpQuant), ("acc", LpQuant),
                ("weight", LpQuant), ("grad_scaling", ctypes.c_float), ("seed", ctypes.c_uint64)]


class FusedAdamW(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, model=None):
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay))
        self.model = model
        self._engine = None
        self._table = None          # (host bytes, device uint8 tensor, key)
        self._hyper = None
        self._step0 = None          # steps already taken, when restored by a wrapper (qtorch.optim.OptimLP)
        for group in self.param_groups:
            for p in group["params"]:
                if not p.is_cuda:
                    raise mv.MvError("FusedAdamW needs CUDA parameters (there is no CPU fallback)")
        b0 = self.param_groups[0]["betas"]
        if any(g["betas"] != b0 or g["eps"] != self.param_groups[0]["eps"] for g in self.param_groups):
            raise ValueError("FusedAdamW: betas / eps must be the same for all groups")

    # ------------------------------------------------------------------ engine operands
    def _operands(self):
        """{id(weight): (q, q_t, fmt)} of the fused encoder's Linear weights (empty without a model)."""
        if self.model is None:
            return {}
        engine = self.model.engine()
        if engine is not self._engine:
            self._engine, self._table = engine, None
        if engine.exact:
            # FP32: the engine's operands are 3xTF32 split buffers ([r, 3c] / [c, 3r]), not plain q(W) / q(W)^T
            # tiles — the kernel must not write into them; the engine re-splits after every update instead
            return {}
        engine.external_requant = True
        wq = engine.quantised_weights()
        return {id(engine.params[i]): (q, qt, engine.fmt) for i, (q, qt) in wq.items()}

    def _state_of(self, p):
        st = self.state[p]
        if not st:
            st["step"] = 0
            st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return st

    def _build_table(self, lp=None):
        ops = self._operands()
        rows, key, chunk = [], [], 0
        self._updated = []
        k = -1
        for group in self.param_groups:
            for p in group["params"]:
                k += 1
                if p.grad is None:
                    continue
                if p.grad.dtype != torch.float32 or p.dtype != torch.float32 or not p.is_contiguous():
                    raise mv.MvError("FusedAdamW: parameters and gradients must be contiguous fp32")
                g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
                st = self._state_of(p)
                t = AdamwTensor()
                t.param, t.grad = p.data_ptr(), g.data_ptr()
                t.exp_avg, t.exp_avg_sq = st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()
                t.n, t.lr, t.weight_decay, t.chunk0 = p.numel(), group["lr"], group["weight_decay"], chunk
                op = ops.get(id(p))
                if op is not None:
                    q, qt, fmt = op
                    t.wq, t.wq_t = q.data_ptr(), qt.data_ptr()
                    t.rows, t.cols = p.shape
                    t.wq_dtype = mv._DT[q.dtype]
                    t.q_exp, t.q_man = fmt if fmt else (0, 0)
                    chunk += ((t.rows + 31) // 32) * ((t.cols + 31) // 32)
                else:
                    chunk += (p.numel() + 1023) // 1024
                x = None
                if lp is not None:
                    x = AdamwLpTensor()
                    x.acc, x.grad_out = lp.side(p, k, g)
                    x.index = k
                rows.append((t, g, x))
                self._updated.append((t, p))
                key.append((t.param, t.grad, t.wq, float(t.lr), float(t.weight_decay)) +
                           ((x.acc, x.grad_out, x.index) if x is not None else ()))
        return rows, tuple(key), chunk

    @torch.no_grad()
    def step(self, closure=None, inv_scale=None, found_inf=None):
        return self._fused_step(closure, inv_scale, found_inf)

    @torch.no_grad()
    def _fused_step(self, closure, inv_scale, found_inf, lp=None):
        """lp (qtorch.optim.OptimLP's fused path): `spec` (an OptimLpSpec) and `side(p, k, g)` -> (acc, grad_out)
        pointers of parameter p, index k, contiguous gradient g; the launch is mv_adamw_lp_step."""
        loss = closure() if closure is not None else None
        rows, key, chunks = self._build_table(lp)
        if not rows:
            return loss
        dev = self.param_groups[0]["params"][0].device
        if self._table is None or self._table[2] != key:
            arr = (AdamwTensor * len(rows))(*[t for t, _, _ in rows])
            data = bytes(arr)
            if lp is not None:
                data += bytes((AdamwLpTensor * len(rows))(*[x for _, _, x in rows]))
            host = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
            table = torch.empty(host.numel(), dtype=torch.uint8, device=dev)
            table.copy_(host, non_blocking=True)
            self._table = (host, table, key, len(bytes(arr)))
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is not None:
                    self.state[p]["step"] += 1
        g0 = self.param_groups[0]
        if self._hyper is None:
            # step count lives on the device from here on: no per-step host -> device traffic
            done = max((st["step"] for st in self.state.values() if st), default=1) - 1
            if self._step0 is not None:
                done = self._step0
            self._hyper = torch.tensor([g0["betas"][0], g0["betas"][1], g0["eps"], float(done), 1.0, 0.0],
                                       dtype=torch.float32, device=dev)
            self._one = torch.ones(1, dtype=torch.float32, device=dev)
        hy = self._hyper
        hy[4:5].copy_(inv_scale.reshape(1) if inv_scale is not None else self._one)
        if found_inf is not None:
            hy[5:6].copy_(found_inf.reshape(1))
            hy[3:4].add_(1.0 - hy[5:6].ne(0).float())     # a skipped step does not advance the count
        else:
            hy[5:6].zero_()
            hy[3:4].add_(1.0)
        keep = [g for _, g, _ in rows]                # contiguous gradient copies stay alive for the launch
        if lp is None:
            mv._check(mv.lib().mv_adamw_step(ctypes.c_void_p(self._table[1].data_ptr()), len(rows), chunks,
                                             mv._ptr(hy), mv._stream()), "mv_adamw_step")
        else:
            base = self._table[1].data_ptr()
            mv._check(mv.lib().mv_adamw_lp_step(ctypes.c_void_p(base), ctypes.c_void_p(base + self._table[3]),
                                                len(rows), chunks, mv._ptr(hy), ctypes.byref(lp.spec), mv._stream()),
                      "mv_adamw_lp_step")
            for (_, g, x), (_, p) in zip(rows, self._updated):
                if x.grad_out and g is not p.grad:
                    p.grad.copy_(g)                   # a strided gradient was quantised in its contiguous copy
        del keep
        # the kernel wrote the parameters through raw pointers: let every version-keyed cache see the update
        torch.autograd.graph.increment_version([p for _, p in self._updated])
        if self._engine is not None:
            if self._engine.exact:
                self._engine.invalidate_weights()
            else:
                self._engine.mark_weights_fresh()
        return loss

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._hyper = None          # re-derive the device step count from the restored state
        self._table = None
        self._step0 = None
