#!/usr/bin/env python
"""bench.py — train images/s of the quantised ViT fwd+bwd step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a path
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                          # the reference's CPU path
    python bench.py --dump-outputs DIR ...                        # + what the last timed step computed, DIR/*.npy

Workload (BASELINE.json configs[1]; SURVEY.md §8d config 2): ViT-Small (D=384, L=12, h=6,
M=1536, patch 16), classification, 45 classes, 256x256x3 synthetic RESISC45-shaped images,
q_format FP16_32, batch 256 per GPU, random-init weights.  One step = zero_grad -> forward ->
CrossEntropy -> backward (+ NCCL gradient all-reduce for N > 1), the span the reference times
in classification/train.py:239-264.  Weak scaling: 256 images per GPU.

Prints ONE JSON line (rank 0).  `value` has inputs resident in HBM; `e2e` copies every step's
batch from pinned host memory and reads the loss back.  `roofline` describes the dominant kernel
class of the step, timed with CUDA events inside the timed region; `cpu_baseline` times the
oracle port of the reference (stock PyTorch CPU ops + the C restatement of QPyTorch quant_cpu)
on a bounded sample on this box's host cores.  `quant_kernels` (N=1) is the second half of the
metric: HBM GB/s of the standalone fake-quant kernel on 2^28 fp32 values, nearest and stochastic.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "myrtle-vision_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

ARCH = dict(dim=384, depth=12, heads=6, mlp_dim=1536)
IMAGE, PATCH, CLASSES = 256, 16, 45
METRIC = "train images/sec, quantised ViT fwd+bwd"
DTYPES = {"FP16_32": "f16 tensor-core operands, f32 accumulate: fake-quantised tensors are exact in their f16 containers; the "
                     "tensors the reference leaves in f32 (qkv, attention probabilities, activation gradients) are also "
                     "rounded to f16 (11 significant bits, f16 range; saturation raises the device overflow flag)",
          "FP16_16": "f16 tensor-core operands (exact fake-quant containers; attention probabilities and activation "
                     "gradients rounded to f16, overflow flagged), f32 accumulate",
          "TF32": "tf32 operands (exact (8,10) fake-quant values in f32 containers), f32 accumulate",
          "FP32": "tf32 tensor-core products of f32 operands, f32 accumulate"}


def flops_per_image(n_tokens, dim, depth, mlp, classes, patch_dim=768):
    fwd = 2 * (n_tokens - 1) * patch_dim * dim + depth * (
        2 * n_tokens * (3 * dim * dim + dim * dim + 2 * dim * mlp) + 4 * n_tokens * n_tokens * dim
    ) + 2 * dim * classes
    return 3 * fwd


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._read, daemon=True).start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Median SM clock and throttle reasons of the samples taken inside [t0, t1] (host times around the
        timed region).  nvidia-smi needs a few hundred ms to deliver its first row, so the sampler is
        started before the warm-up; if the timed region itself is shorter than the sampling period the
        window is widened to the warm-up steps right before it (same load)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = self.rows
        if t0 is not None:
            inside = [r for ts, r in rows if t0 <= ts <= t1 + 0.15]
            if len(inside) < 2:
                inside = [r for ts, r in rows if t0 - 1.0 <= ts <= t1 + 0.25]
            rows = inside
        else:
            rows = [r for _, r in rows]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
def cpu_port_throughput(batch, steps, warmup, q_format):
    """The reference's CPU path restated (oracle/vit_oracle.py): img/s of zero_grad -> fwd -> CE ->
    bwd on `batch` images per step, all host threads torch wants to use."""
    import torch
    from oracle import vit_oracle
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host core it can
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, RuntimeError):
        pass
    torch.manual_seed(1234)
    P = vit_oracle.init_params(decoder="classification", num_classes=CLASSES, seed=1234, **ARCH)
    g = torch.Generator().manual_seed(1234)
    img = torch.randn(batch, 3, IMAGE, IMAGE, generator=g).clamp(-1, 1)
    tgt = torch.randint(0, CLASSES, (batch,), generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        vit_oracle.train_step(P, img, tgt, decoder="classification", heads=ARCH["heads"], q_format=q_format)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    return batch / mean, mean * 1e3, torch.get_num_threads()


def cpu_reference_throughput(batch, steps, warmup, q_format):
    """The UNMODIFIED reference (`oracle/_ref/myrtle_vision`, staged by oracle/make_ref.py) through the qtorch
    shim: img/s of the span classification/train.py:239-264 times (zero_grad -> forward -> CE -> backward) on
    `batch` images per step, all host threads.  Raises ImportError when oracle/_ref is not staged."""
    import torch
    import torch.nn.functional as F
    from oracle import make_ref
    ref_vit = make_ref.import_reference()
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, RuntimeError):
        pass
    torch.manual_seed(1234)
    model = ref_vit.ViT(decoder="classification", image_size=IMAGE, patch_size=PATCH, num_classes=CLASSES,
                        dim=ARCH["dim"], depth=ARCH["depth"], heads=ARCH["heads"], mlp_dim=ARCH["mlp_dim"],
                        q_format=q_format).train()
    g = torch.Generator().manual_seed(1234)
    img = torch.randn(batch, 3, IMAGE, IMAGE, generator=g).clamp(-1, 1)
    tgt = torch.randint(0, CLASSES, (batch,), generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        model.zero_grad()
        F.cross_entropy(model(img), tgt).backward()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    return batch / mean, mean * 1e3, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = args.ref_batch
    steps, warmup = args.steps, max(1, min(args.warmup, 1))
    try:
        ips, ms, threads = cpu_reference_throughput(batch, steps, warmup, args.q_format)
        kind, what = "reference", "unmodified reference package (oracle/_ref) + qtorch shim over oracle/quant_oracle.c"
    except ImportError as e:
        sys.stderr.write("reference arm: %s — timing the oracle port instead\n" % e)
        ips, ms, threads = cpu_port_throughput(batch, steps, warmup, args.q_format)
        kind, what = "port", "oracle/vit_oracle.py (restatement of the reference) + oracle/quant_oracle.c"
    extra = {}
    if args.ref_batch2 and kind == "reference":
        # second, larger sample (SURVEY.md section 8d: "batch 8 and, if time allows, 32")
        ips2, ms2, _ = cpu_reference_throughput(args.ref_batch2, max(1, min(steps, 2)), 1, args.q_format)
        extra = {"batch_%d" % args.ref_batch2: {"value": ips2, "ms_per_step": ms2}}
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (fake-quantised to fp16 values)", "data": "synthetic",
        "config": {"workload": "ViT-Small cls 256x256x3, 45 classes, q_format=%s, batch %d/GPU, fwd+CE+bwd"
                               % (args.q_format, args.batch),
                   "sample": "each step is batch %d of that workload on the host cores (bounded CPU sample)" % batch,
                   "parallelism": "cpu, %d threads" % threads},
        "cpu_baseline": dict({"value": ips, "unit": "images/s", "cores": threads, "kind": kind, "what": what,
                              "sample": "%d steps of batch %d (same model/input shape), host cores=%d"
                                        % (steps, batch, os.cpu_count())}, **extra),
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(q_format):
    """`cpu_baseline` of the B200 arm: the reference arm in a child process (this process has this repo's own
    `myrtle_vision` package imported, the reference's has the same name)."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2",
                              "--warmup", "1", "--q-format", q_format, "--ref-batch2", "0"],
                             capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        sys.stderr.write("cpu_baseline child printed no JSON: %s\n" % out.stderr[-500:])
    except (subprocess.SubprocessError, OSError, ValueError, KeyError) as e:
        sys.stderr.write("cpu_baseline child failed: %r\n" % (e,))
    return None


# ------------------------------------------------------------------------------------------
def roofline_entries(kern, work, steps, peaks):
    """Per kernel class: launches, ms per step and — from the ALGORITHMIC flop / bytes of one launch (recorded by
    mv_native at call time; DESIGN.md section 4) — the roofline that bounds it: whichever of flop / tensor peak and
    bytes / HBM peak is the longer time.  Returns (breakdown dict, entry of the class with the most time)."""
    t_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    h_peak = peaks.get("hbm_gbs", 6650.0)
    breakdown, top = {}, None
    for name, (cnt, tot) in sorted(kern.items(), key=lambda kv: -kv[1][1]):
        entry = {"launches_per_step": cnt / steps, "ms_per_step": tot / steps}
        flop, nbytes = work.get(name, (0.0, 0.0))
        if cnt and (flop or nbytes):
            avg_ms = tot / cnt
            t_tensor = flop / (t_peak * 1e9)          # ms at the sustained tensor peak
            t_hbm = nbytes / (h_peak * 1e6)           # ms at the measured copy bandwidth
            if t_tensor >= t_hbm:
                entry.update({"bound": "tensor", "achieved": flop / avg_ms / 1e9, "unit": "TFLOP/s", "peak": t_peak,
                              "frac": t_tensor / avg_ms})
            else:
                entry.update({"bound": "hbm", "achieved": nbytes / avg_ms / 1e6, "unit": "GB/s", "peak": h_peak,
                              "frac": t_hbm / avg_ms})
            entry.update({"avg_launch_ms": avg_ms, "floor_ms": max(t_tensor, t_hbm),
                          "algorithmic_flop": flop, "algorithmic_bytes": nbytes})
            if top is None:
                top = dict(entry, kernel=name)
        breakdown[name] = entry
    return breakdown, top


def build_task(task, q_format, batch, dev, arch=None):
    """(model, criterion, [two device batches]) of a BASELINE.json config: classification 256^2 / 45 classes,
    segmentation 256^2 / 17 classes (fused upsample + CE), detection 800^2 / 20 classes (N = 2501, padded targets,
    device matching).  Synthetic RESISC45 / DLRSD / DIOR-shaped data, random-init weights."""
    import torch
    from myrtle_vision.datasets.synthetic import SyntheticVision, detection_collate
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.trainer import build_criterion, to_device
    size, classes = {"classification": (IMAGE, CLASSES), "segmentation": (256, 17), "detection": (800, 20)}[task]
    torch.manual_seed(1234)
    model = ViT(decoder=task, image_size=size, patch_size=PATCH, num_classes=classes, q_format=q_format,
                **(arch or ARCH)).to(dev).train()
    if task == "classification":
        g = torch.Generator().manual_seed(1234)
        batches = [(torch.randn(batch, 3, size, size, generator=g).clamp(-1, 1),
                    torch.randint(0, classes, (batch,), generator=g)) for _ in range(2)]
    else:
        ds = SyntheticVision(task, 2 * batch, size, classes, seed=1234)
        items = [ds[i] for i in range(2 * batch)]
        if task == "detection":
            from myrtle_vision.models.matcher import pad_targets
            batches = [detection_collate(items[:batch]), detection_collate(items[batch:])]
            cap = -(-max(int(t["boxes"].shape[0]) for _, ts in batches for t in ts) // 16) * 16
            batches = [(img, pad_targets(ts, capacity=cap)) for img, ts in batches]
        else:
            batches = [(torch.stack([a for a, _ in part]), torch.stack([b for _, b in part]))
                       for part in (items[:batch], items[batch:])]
    batches = [(img.to(dev), to_device(t, dev)) for img, t in batches]
    cfg = {"loss_ce": 1.0, "class_error": 0.0, "loss_bbox": 5.0, "loss_giou": 2.0, "cardinality_error": 0.0,
           "eos_coef": 0.1, "fused_seg_loss": True}
    criterion = build_criterion(task, cfg, classes, dev)
    if task == "segmentation":
        model.decoder.fused_loss = True
    return model, criterion, batches, (size // PATCH) ** 2 + 1


def time_config(name, task, q_format, batch, dev, steps, peaks):
    """One secondary BASELINE.json config on this GPU: a short eager leg for the per-kernel roofline, then the step
    as one CUDA graph, `steps` timed replays after 10 warm-up replays (inputs resident, alternating batches)."""
    import torch
    import mv_native
    from myrtle_vision.utils.graph import GraphedTrainStep
    model, criterion, batches, n_tok = build_task(task, q_format, batch, dev)

    def eager(img, tgt):
        model.zero_grad(set_to_none=True)
        loss = criterion(model(img), tgt)
        loss.backward()
        return loss

    for i in range(3):
        eager(*batches[i % 2])
    torch.cuda.synchronize()
    mv_native.enable_timing(True)
    for i in range(2):
        eager(*batches[i % 2])
    torch.cuda.synchronize()
    breakdown, top = roofline_entries(mv_native.timing_summary(), mv_native.work_summary(), 2, peaks)
    mv_native.enable_timing(False)
    gs = GraphedTrainStep(model, criterion, *batches[0])
    for i in range(10):
        gs(*batches[i % 2])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        gs(*batches[i % 2])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    fl = flops_per_image(n_tok, ARCH["dim"], ARCH["depth"], ARCH["mlp_dim"], 0)
    out = {"workload": name, "images_per_s": batch / ms * 1e3, "ms_per_step": ms, "batch": batch, "tokens": n_tok,
           "q_format": q_format, "steps": steps, "model_tflops": batch / ms * 1e3 * fl / 1e12,
           "dominant_kernel": ({k: top[k] for k in ("kernel", "bound", "achieved", "unit", "frac", "avg_launch_ms")}
                               if top else None),
           "top_kernels_ms_per_step": {k: round(v["ms_per_step"], 3) for k, v in list(breakdown.items())[:6]}}
    del gs, model, criterion, batches
    torch.cuda.empty_cache()
    return out


def quant_microbench(dev, peaks):
    """Second half of BASELINE.json's metric: HBM GB/s of the standalone fake-quant kernels, SURVEY.md section 8d set.
    Input (i): 2^28 fp32 = 1 GiB, randn * exp(U(-12, 8)) (normal, subnormal and saturating branches all run);
    algorithmic bytes per element: 8 (fp32 -> fp32), 6 (fp16 container), 12 (block: max pass + quant pass).  Every
    launch moves >= 1.5 GiB, far beyond the 126 MB L2.  Input (ii): model-shaped tensors, rotated over enough
    buffers that consecutive launches never find their data in L2."""
    import torch
    import mv_native
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    gq = torch.Generator(device=dev).manual_seed(1234)
    nq = 1 << 28
    xq = torch.randn(nq, device=dev, generator=gq)
    xq.mul_(torch.exp(torch.empty(nq, device=dev).uniform_(-12, 8, generator=gq)))
    oq = torch.empty_like(xq)
    oh = torch.empty(nq, dtype=torch.float16, device=dev)
    x2 = xq.view(16384, 16384)
    quant = {"unit": "GB/s", "elements": nq, "peak": hbm_peak,
             "peak_source": "MEASURED_PEAKS.json (hbm_gbs)" if peaks else "fallback",
             "input": "randn * exp(U(-12, 8)), 2^28 fp32, seed 1234"}

    def timed(fn, bytes_per_launch, reps=10):
        for _ in range(3):
            fn()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for _ in range(reps):
            fn()
        q1.record()
        torch.cuda.synchronize()
        gbs = bytes_per_launch * reps / q0.elapsed_time(q1) / 1e6
        return {"value": gbs, "frac": gbs / hbm_peak, "bytes_per_element": bytes_per_launch / nq}

    st = dict(rounding="stochastic", seed=1234, offset=0)
    cases = [
        ("float(5,10) nearest", lambda: mv_native.float_quantize(xq, 5, 10, out=oq), 8),
        ("float(5,10) stochastic", lambda: mv_native.float_quantize(xq, 5, 10, out=oq, **st), 8),
        ("float(8,10) nearest", lambda: mv_native.float_quantize(xq, 8, 10, out=oq), 8),
        ("float(8,10) stochastic", lambda: mv_native.float_quantize(xq, 8, 10, out=oq, **st), 8),
        ("float(5,10) nearest -> fp16 container", lambda: mv_native.float_quantize(xq, 5, 10, out=oh), 6),
        ("float(5,10) stochastic -> fp16 container", lambda: mv_native.float_quantize(xq, 5, 10, out=oh, **st), 6),
    ]
    for fl in (9, 8, 7):                      # the reference's three 11-bit fixed-point formats (utils/quantize.py:58-72)
        cases.append(("fixed(11,%d) nearest" % fl, lambda fl=fl: mv_native.fixed_point_quantize(xq, 11, fl, out=oq), 8))
        cases.append(("fixed(11,%d) stochastic" % fl,
                      lambda fl=fl: mv_native.fixed_point_quantize(xq, 11, fl, out=oq, **st), 8))
    cases += [
        ("block(wl=8, dim=-1) nearest", lambda: mv_native.block_quantize(xq, 8, dim=-1, out=oq), 12),
        ("block(wl=8, dim=0) nearest", lambda: mv_native.block_quantize(x2, 8, dim=0, out=oq.view(16384, 16384)), 12),
        ("block(wl=8, dim=0) stochastic",
         lambda: mv_native.block_quantize(x2, 8, dim=0, out=oq.view(16384, 16384), **st), 12),
    ]
    for label, fn, bpe in cases:
        quant[label] = timed(fn, float(bpe) * nq)
    # (ii) model-shaped activations / weights of ViT-Small at batch 256, float(5,10) nearest, rotating buffers
    shaped = {}
    for shape in ((256, 257, 384), (256, 257, 1536), (256, 256, 768), (1536, 384)):
        n = 1
        for d in shape:
            n *= d
        copies = max(2, min(64, (1 << 28) // n))
        ins = [xq[i * n:(i + 1) * n].view(shape) for i in range(copies)]
        outs = [oq[i * n:(i + 1) * n].view(shape) for i in range(copies)]
        it = {"i": 0}

        def fn():
            k = it["i"] % copies
            it["i"] += 1
            mv_native.float_quantize(ins[k], 5, 10, out=outs[k])
        for _ in range(copies):
            fn()
        reps = 4 * copies
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for _ in range(reps):
            fn()
        q1.record()
        torch.cuda.synchronize()
        us = q0.elapsed_time(q1) / reps * 1e3
        shaped["x".join(str(d) for d in shape)] = {"us_per_launch": us, "value": 8.0 * n / us / 1e3,
                                                   "frac": 8.0 * n / us / 1e3 / hbm_peak, "buffers": copies}
    quant["model_shaped float(5,10) nearest"] = shaped
    del xq, oq, oh
    torch.cuda.empty_cache()
    return quant


DUMP_MAX_ELEMENTS = 1 << 18       # per array; with it the ViT-Small gradients come to 47 MB


def dump_outputs(out_dir, arrays):
    """Write each (name, tensor) as out_dir/<name>.npy in float32.  An array of more than DUMP_MAX_ELEMENTS values
    is written as a fixed, seeded sample of its flattened values (sorted positions, the same in every run), so the
    dumps of two builds can be compared value for value."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays:
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(1234).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))
            a = a.reshape(-1)[idx]
        total += a.nbytes
        assert total <= 64e6, "output dump exceeds 64 MB at %s" % name
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    import mv_native
    from myrtle_vision.models.vit import ViT
    from myrtle_vision.utils.parallel import DataParallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    torch.manual_seed(1234)
    model = ViT(decoder="classification", image_size=IMAGE, patch_size=PATCH, num_classes=CLASSES,
                q_format=args.q_format, **ARCH).to(dev).train()
    net = DataParallel(model) if world > 1 else model
    g = torch.Generator().manual_seed(1234 + rank)
    host = [(torch.randn(B, 3, IMAGE, IMAGE, generator=g).clamp(-1, 1).pin_memory(),
             torch.randint(0, CLASSES, (B,), generator=g).pin_memory()) for _ in range(2)]
    resident = [(a.to(dev), b.to(dev)) for a, b in host]

    def step(img, y):
        model.zero_grad(set_to_none=True)
        out = net(img)
        loss = F.cross_entropy(out, y)
        loss.backward()
        step.logits = out.detach()        # detached: a live autograd graph breaks the CUDA-graph capture below
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(args.warmup):
        step(*resident[i % 2])
    # ---- eager region: per-kernel-class CUDA-event timing (roofline / breakdown) + host enqueue cost
    mv_native.enable_timing(rank == 0 and not args.no_kernel_timing)
    barrier()
    n0 = mv_native.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        step(*resident[i % 2])
    host_enqueue_ms = (time.perf_counter() - t_host0) / args.steps * 1e3
    e1.record()
    barrier()
    ms_eager = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    launches_per_step = (mv_native.launch_count() - n0) // args.steps
    kern, work = mv_native.timing_summary(), mv_native.work_summary()
    mv_native.enable_timing(False)

    # ---- timed region 1 (`value`): the same step captured in a CUDA graph, inputs resident in HBM
    use_graph = not args.no_graph
    if use_graph:
        from myrtle_vision.utils.graph import GraphedTrainStep
        gstep = GraphedTrainStep(net, F.cross_entropy, resident[0][0], resident[0][1])
        run_step = lambda img, y: gstep(img, y)
    else:
        run_step = step
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                     # before the warm-up: the first nvidia-smi row takes a while
    for i in range(max(args.warmup, 25)):   # >= 0.5 s of the same load ahead of the timed region
        run_step(*resident[i % 2])
    barrier()
    t_wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        run_step(*resident[i % 2])
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    launches = launches_per_step * args.steps
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None

    # data parallel: the same graph without the gradient all-reduces -> the communication time that backward does
    # not hide (exposed_comm_ms), measured in this run instead of inferred from a separate N = 1 run
    exposed_comm_ms = None
    if world > 1 and use_graph:
        eng = model.engine()
        saved_reducer, eng.reducer = eng.reducer, None
        g2 = GraphedTrainStep(model, F.cross_entropy, resident[0][0], resident[0][1])
        for i in range(10):
            g2(*resident[i % 2])
        barrier()
        e0.record()
        for i in range(args.steps):
            g2(*resident[i % 2])
        e1.record()
        barrier()
        ms_nocomm = max_over_ranks(e0.elapsed_time(e1) / args.steps)
        exposed_comm_ms = ms_step - ms_nocomm
        eng.reducer = saved_reducer
        del g2

    # ---- timed region 2 (e2e): every step copies its batch from pinned host memory (prefetched one
    # step ahead on a copy stream) and reads the loss back to the host
    copy_stream = torch.cuda.Stream()
    bufs = [(torch.empty_like(resident[0][0]), torch.empty_like(resident[0][1])) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            bufs[s][0].copy_(host[s][0], non_blocking=True)
            bufs[s][1].copy_(host[s][1], non_blocking=True)
            ready[s].record(copy_stream)

    for s in range(2):
        consumed[s].record()
    barrier()
    t_e2e0 = torch.cuda.Event(enable_timing=True); t_e2e1 = torch.cuda.Event(enable_timing=True)
    t_e2e0.record()
    prefetch(0)
    loss_host = 0.0
    for i in range(args.steps):
        s = i % 2
        if i + 1 < args.steps:
            prefetch(i + 1)
        torch.cuda.current_stream().wait_event(ready[s])
        loss = run_step(*bufs[s])
        consumed[s].record()
        loss_host = loss.item()                       # device -> host read of the step result
    t_e2e1.record()
    barrier()
    ms_e2e = max_over_ranks(t_e2e0.elapsed_time(t_e2e1) / args.steps)
    h2d = B * 3 * IMAGE * IMAGE * 4 + B * 8
    d2h = 4

    if world > 1:
        # Tear-down: the captured graph holds NCCL work, and destroy_process_group() has been seen to
        # hang behind it.  All ranks meet here; non-zero ranks then leave without running destructors.
        dist.barrier()
        torch.cuda.synchronize()
    if rank != 0:
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)

    if args.dump_outputs:                 # the e2e loop ran the last timed step
        dump_outputs(args.dump_outputs, [("loss", loss), ("logits", gstep.output if use_graph else step.logits)] +
                     [("grad." + n, p.grad) for n, p in model.named_parameters() if p.grad is not None])

    # ---- roofline of the dominant kernel class
    # measured peaks of this GPU, if a measurement left them next to bench.py; the fallbacks are used otherwise
    peaks = {}
    if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    n_tok = (IMAGE // PATCH) ** 2 + 1
    D, Mm, L = ARCH["dim"], ARCH["mlp_dim"], ARCH["depth"]
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_launch", {})
    breakdown, roofline = {}, None
    if kern:
        breakdown, top = roofline_entries(kern, work, args.steps, peaks)
        if top is not None:              # the dominant kernel (most time per step)
            roofline = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"],
                        "peak": top["peak"], "unit": top["unit"], "frac": top["frac"],
                        "traffic": traffic.get(top["kernel"]),
                        "peak_source": "MEASURED_PEAKS.json (%s)" % ("bf16_tflops_sustained" if top["bound"] == "tensor"
                                                                     else "hbm_gbs") if peaks else "fallback",
                        "avg_launch_ms": top["avg_launch_ms"],
                        "algorithmic_per_launch": top["algorithmic_flop"] if top["bound"] == "tensor"
                        else top["algorithmic_bytes"]}

    # the main model is done: release it before the secondary workloads
    if world == 1:
        del model, net, resident, bufs
        if use_graph:
            del gstep, run_step
        torch.cuda.empty_cache()

    # BASELINE.json's other configs and the secondary formats of config 2, on this GPU, same harness
    # (segmentation/train.py:254-290, detection/train.py:247-287; SURVEY.md section 8d)
    configs = None
    if world == 1 and not args.no_configs:
        configs = {}
        for name, task, fmt, bsz in (("cls256 FP16_16", "classification", "FP16_16", args.batch),
                                     ("cls256 TF32", "classification", "TF32", args.batch),
                                     ("seg256 (config 4)", "segmentation", args.q_format, args.batch),
                                     ("det800 (config 5)", "detection", args.q_format, 8)):
            try:
                configs[name] = time_config(name, task, fmt, bsz, dev, args.steps, peaks)
            except Exception as e:       # a secondary workload must not cost the headline line
                configs[name] = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()

    quant = quant_microbench(dev, peaks) if world == 1 and not args.no_quant_bench else None

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess(args.q_format)
        if cpu is None:
            ips, ms_cpu, threads = cpu_port_throughput(8, 2, 1, args.q_format)
            cpu = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                   "sample": "2 timed steps of batch 8, same model and image shape (%.0f ms/step), host cpu_count=%d"
                             % (ms_cpu, os.cpu_count())}

    value = world * B / ms_step * 1e3
    fl = flops_per_image(n_tok, D, L, Mm, CLASSES)
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPES[args.q_format],
        "data": "synthetic",
        "config": {"workload": "ViT-Small cls 256x256x3, 45 classes, q_format=%s, batch %d/GPU, fwd+CE+bwd%s"
                               % (args.q_format, B, " + NCCL grad all-reduce" if world > 1 else ""),
                   "global_batch": world * B, "parallelism": "dp%d" % world,
                   "launch": "whole step captured in one CUDA graph (myrtle_vision.utils.graph.GraphedTrainStep)" if use_graph else "eager launches",
                   "l2": "per-step working set (~11 GB of activations) >> 126 MB L2; two alternating input batches"},
        "clocks": clocks,
        "e2e": {"value": world * B / ms_e2e * 1e3, "unit": "images/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "last_loss": loss_host},
        "gpu_launches": launches,
        "cuda_graph": use_graph,
        "exposed_comm_ms": exposed_comm_ms,
        "eager_ms_per_step": ms_eager,
        "host_enqueue_ms_per_step_eager": host_enqueue_ms,
        "model_tflops": value * fl / 1e12,
        "roofline": roofline,
        "kernels": breakdown,
        "configs": configs,
        "quant_kernels": quant,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--q-format", default="FP16_32", choices=["FP16_32", "FP16_16", "TF32", "FP32"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--ref-batch", type=int, default=8, help="reference arm: images per CPU step")
    ap.add_argument("--ref-batch2", type=int, default=32, help="reference arm: second, larger sample (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--no-quant-bench", action="store_true", help="skip the fake-quant kernel GB/s microbench")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary workloads (FP16_16, TF32, seg256, det800)")
    ap.add_argument("--no-graph", action="store_true", help="time the eagerly launched step instead of the CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, logits and parameter gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_b200(args)


if __name__ == "__main__":
    main()
