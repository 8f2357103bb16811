#!/usr/bin/env python
"""Headline benchmark: images/sec of the ResNet-50 training step (bf16, synthetic 3x224x224, bs=256 per GPU).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W     (the reference's own CPU train_one_epoch on the host cores)
  python bench.py --steps K --warmup W --dump-outputs DIR   (also writes what the last timed step computed, as .npy files)

One step = forward + soft-max cross-entropy + backward + gradient all-reduce + SGD(momentum) update, i.e. the body of the
reference's train_one_epoch (classification/resnet/utils.py:35-55) in the DDP pattern of others/train_with_DDP.
Prints ONE JSON line (rank 0).  `value` times the step with the batch already resident in HBM; `e2e` times the same public
API call with the batch copied from pinned host memory every step and the loss read back to the host.
BASELINE.json's metric names ResNet-50 AND ViT-B/16: the line's `value` is ResNet-50 (configs[1]) and its `secondary` block
holds the same measurements (value / ms_per_step / e2e / step_roofline / roofline / kernels) of ViT-B/16 bs 256 (configs[2]),
taken in the same invocation.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# per-image algorithmic work, fwd+bwd = 3 x forward (BASELINE.md section 2): GFLOP (GEMM-like ops) and MB of HBM traffic
MODELS = {
    "resnet50": {"gflop": 24.53, "mb": 3 * 43.8, "batch": 256, "label": "ResNet-50",
                 "workload": "classification/resnet ResNet-50 bf16, synthetic 3x224x224, bs=256/GPU (BASELINE.json configs[1])"},
    "vit_b16": {"gflop": 105.38, "mb": 3 * 73.9, "batch": 256, "label": "ViT-B/16",
                "workload": "classification/vision_transformer ViT-B/16 bf16, synthetic 3x224x224, bs=256/GPU (BASELINE.json configs[2])"},
    "convnext_tiny": {"gflop": 26.73, "mb": 3 * 54.2, "batch": 256, "label": "ConvNeXt-T",
                      "workload": "classification/convNext ConvNeXt-T bf16, synthetic 3x224x224, bs=256/GPU, drop_path 0 (BASELINE.json configs[4])"},
    "swin_tiny": {"gflop": 26.94, "mb": 3 * 60.1, "batch": 128, "label": "Swin-T",
                  "workload": "classification/swin_transformer Swin-T bf16, synthetic 3x224x224, bs=128/GPU, drop_path 0 (BASELINE.json configs[3])"},
}


def metric_label(model):
    """ONE metric string per model, shared by the B200 arm and the reference arm (the driver matches the two lines on it)."""
    return f"images/sec ({MODELS[model]['label']} training step)"


ADAMW_MODELS = ("convnext_tiny", "swin_tiny")   # AdamW(lr 5e-4, wd 5e-2): convNext/train.py:96,102; swin config.py:133-162
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons of this rank's GPU during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------------- reference arm
REF_BATCH = 16   # fixed per-step sample of the bs-256 workload (SURVEY 8(d): bs 16, fp32, all host cores)


def host_cores():
    """Logical CPUs this process may use: scheduler affinity, capped by the cgroup CPU quota when one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def best_thread_count(model, limit):
    """Pick the intra-op thread count the reference actually runs fastest with on this box: "all host cores" is the intent,
    but on the shared GPU hosts 128 OpenMP threads ran a 16-image step 70x SLOWER than 8 did (oversubscribed hyper-threads /
    noisy neighbours).  Probe a small forward pass with 8, 16, 32, ... <= limit threads and stop once it gets slower."""
    import torch

    x = torch.randn(4, 3, 224, 224)
    cands = [c for c in (8, 16, 32, 64, 128, 256) if c < limit] + [limit]
    best, best_t = cands[0], None
    was_training = model.training
    model.eval()
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            model(x)
            t0 = time.time()
            model(x)
            dt = time.time() - t0
            if best_t is None or dt < best_t:
                best, best_t = c, dt
            elif dt > 1.25 * best_t:
                break
    model.train(was_training)
    torch.set_num_threads(best)
    return best


def cpu_reference_run(steps, warmup, batch=REF_BATCH):
    """The reference's CPU training path on `batch` synthetic images per step, fp32, ALL host cores (whatever
    OMP_NUM_THREADS torchrun exported).  kind "reference": the unmodified reference module + its own train_one_epoch
    (classification/resnet/{models/networks.py,utils.py}, staged under oracle/_ref by oracle/build_ref.py); kind "port": the
    oracle restatement (bit-identical to the reference, tests/golden/make_golden.py) when oracle/_ref is absent."""
    import torch

    avail = host_cores()
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, 224, 224, generator=g)
    y = torch.randint(0, 1000, (batch,), generator=g)
    from oracle import build_ref

    if build_ref.available():
        kind = "reference"
        net = build_ref.load("resnet", "models/networks")
        utils = build_ref.load("resnet", "utils")
        torch.manual_seed(0)
        model = net.resnet50()
        cores = best_thread_count(model, avail)
        opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-5)   # resnet/train.py:96
        loss_fn = torch.nn.CrossEntropyLoss()
        dev = torch.device("cpu")

        def run(n):   # one "epoch" of n steps through the reference's own loop (it prints per step: stdout -> stderr here)
            utils.train_one_epoch(model, [(x, y)] * n, dev, opt, loss_fn, 0)
        what = "the reference's train_one_epoch on its own resnet50()"
    else:
        kind = "port"
        from deeplearning_b200.classification.resnet.models.networks import resnet50
        from oracle.resnet import resnet_forward
        from oracle.train_loop import CpuSgdTrainer

        torch.manual_seed(0)
        probe = resnet50()
        state = {k: v.clone() for k, v in probe.state_dict().items()}
        from oracle import build_ref as _b  # noqa: F401  (the port arm probes thread counts on the oracle forward)

        class _Fwd(torch.nn.Module):
            def forward(self, xx):
                return resnet_forward(state, xx, train=False)

        cores = best_thread_count(_Fwd(), avail)
        tr = CpuSgdTrainer(resnet_forward, state, lr=0.01, momentum=0.9, weight_decay=5e-5)

        def run(n):
            for _ in range(n):
                tr.step(x, y)
        what = "the oracle port of the reference ResNet-50 loop"
    if warmup:
        run(warmup)
    t0 = time.time()
    run(steps)
    dt = time.time() - t0
    return {"value": batch * steps / dt, "unit": "images/sec", "cores": cores, "kind": kind,
            "sample": f"{steps} SGD steps of {what} (fp32, CPU, {cores} threads = fastest of the {avail} logical CPUs available) "
                      f"on {batch} synthetic 3x224x224 images each",
            "ms_per_step": dt / steps * 1e3, "batch": batch}


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else a library prints while the bench runs
    (e.g. NCCL's version banner, the reference loop's per-step prints) was redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_run(args.steps, args.warmup)
    line = {"impl": "reference", "metric": metric_label("resnet50"), "value": cb["value"], "unit": "images/sec",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": MODELS["resnet50"]["workload"],
                       "device": "CPU fp32 (the reference's own device default, resnet/train.py:151)",
                       "per_step_batch": cb["batch"], "optimizer": "SGD(momentum=0.9, weight_decay=5e-5)"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------------- B200 arm
def build_model(name, dev):
    if name == "resnet50":
        from deeplearning_b200.classification.resnet.models.networks import resnet50

        return resnet50().to(dev).train()
    if name == "vit_b16":
        from deeplearning_b200.classification.vision_transformer.vit_model import vit_base_patch16_224_in21k

        return vit_base_patch16_224_in21k(num_classes=1000, has_logits=False).to(dev).train()
    if name == "swin_tiny":
        from deeplearning_b200.classification.swin_transformer.models.swin_transformer import SwinTransformer

        return SwinTransformer(drop_path_rate=0.0).to(dev).train()   # Swin-T defaults, stochastic depth off (SURVEY 8(d))
    from deeplearning_b200.classification.convNext.models.networks import ConvNeXt

    # convnext_tiny(1000) with stochastic depth off (SURVEY 8(d) config 5)
    return ConvNeXt(depths=[3, 3, 9, 3], dims=[96, 192, 384, 768], num_classes=1000, drop_path_rate=0.0).to(dev).train()


def optimizer_desc(name):
    return ("AdamW(lr=5e-4, wd=5e-2, decay groups, clip_grad_norm 5.0)" if name == "swin_tiny" else
            "AdamW(lr=5e-4, wd=5e-2, decay groups)" if name in ADAMW_MODELS else "SGD(momentum=0.9, weight_decay=5e-5)")


DUMP_PARAM_SAMPLE = 1 << 20   # parameters per model written by --dump-outputs (4 MB in fp32)


def dump_outputs(out_dir, name, loss, correct, flat_p):
    """What the last timed step returned (loss, per-sample correct flags) and a fixed, seeded sample of the parameters it
    updated, as float32 DIR/<model>_<array>.npy: two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n = flat_p.numel()
    idx = torch.randint(0, n, (min(n, DUMP_PARAM_SAMPLE),), generator=torch.Generator().manual_seed(0)).unique()
    arrays = {"loss": loss, "correct": correct, "params_sample": flat_p[idx.to(flat_p.device)]}
    for key, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}_{key}.npy"), t.detach().float().cpu().numpy())


def measure(name, args, dev, world, rank, local_rank, batch=None):
    """All measurements of one model: device-resident throughput, e2e, per-kernel spans.  Returns the JSON dict (every rank
    runs everything; only rank 0's dict carries the roofline / kernel table)."""
    import torch
    import torch.distributed as dist

    from deeplearning_b200 import ops
    from deeplearning_b200.engine.trainer import TrainStep

    spec = MODELS[name]
    B = batch or spec["batch"]
    warmup = max(args.warmup, 3)   # the timing rules ask for >= 3 warm-up steps; the line reports the number actually run
    torch.manual_seed(0)  # identical init on every rank (and broadcast from rank 0 inside TrainStep)
    model = build_model(name, dev)
    if name == "swin_tiny":       # Swin recipe: AdamW + clip_grad_norm_(5.0) (main.py:197, config.py TRAIN.CLIP_GRAD)
        trainer = TrainStep(model, lr=5e-4, weight_decay=5e-2, optimizer="adamw", clip_grad=5.0)
    elif name in ADAMW_MODELS:    # AdamW(lr 5e-4, wd 5e-2) with the reference's decay groups
        trainer = TrainStep(model, lr=5e-4, weight_decay=5e-2, optimizer="adamw")
    else:                         # SGD(momentum 0.9, wd 5e-5) (resnet/train.py:96, vision_transformer/train.py:94)
        trainer = TrainStep(model, lr=0.01, momentum=0.9, weight_decay=5e-5)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    images = torch.randn(B, 3, 224, 224, device=dev, generator=g)
    labels = torch.randint(0, 1000, (B,), device=dev, generator=torch.Generator(device=dev).manual_seed(4321 + rank))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- device-resident timing ---------------------------------------------------------------------------------
    launches0 = ops.launch_count()
    trainer.step_eager(images, labels)          # one eager step: counts this library's kernel launches per step
    launches_per_step = ops.launch_count() - launches0
    if not args.eager:
        trainer.capture(images, labels)         # whole step (fwd+CE+bwd+all-reduce+update)
    for _ in range(warmup):
        loss, _ = trainer.step(images, labels)
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, correct = trainer.step(images, labels)
    e1.record()
    sync_all()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = launches_per_step * args.steps   # graph replays launch the same kernels the eager step does
    clocks = sampler.stop()
    final_loss = float(loss)
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, name, loss, correct, trainer.arena.flat_p)

    # ---- end-to-end: pinned host batch -> H2D every step (double-buffered on a copy stream), loss read back ---------
    host_imgs = [torch.randn(B, 3, 224, 224).pin_memory() for _ in range(2)]
    host_lbls = [torch.randint(0, 1000, (B,)).pin_memory() for _ in range(2)]
    dev_imgs = [torch.empty_like(images) for _ in range(2)]
    dev_lbls = [torch.empty_like(labels) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i])
            dev_imgs[i].copy_(host_imgs[i], non_blocking=True)
            dev_lbls[i].copy_(host_lbls[i], non_blocking=True)
            ready[i].record(copy_stream)

    def e2e_loop(n):
        for i in range(2):
            consumed[i].record()
        prefetch(0)
        out = 0.0
        for s in range(n):
            cur = s & 1
            if s + 1 < n:
                prefetch(cur ^ 1)
            torch.cuda.current_stream().wait_event(ready[cur])
            l, _ = trainer.step(dev_imgs[cur], dev_lbls[cur])
            consumed[cur].record()
            out = l.item()  # D2H read of the step's result, every step
        return out

    e2e_loop(2)
    sync_all()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    sync_all()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)
    h2d = B * 3 * 224 * 224 * 4 + B * 8

    # ---- optional: the same end-to-end loop fed DECODED uint8 NHWC images (GPU input pipeline, SURVEY 8(f)-1): ToTensor +
    # Normalize run on the device inside the step, the host->device copy is 4x smaller.  Reported beside `e2e`, not instead of it
    # (the reference's loader hands the model float tensors, which is what `e2e` copies).
    e2e_u8 = None
    if name == "resnet50" and not args.eager:
        u8_host = [torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8).pin_memory() for _ in range(2)]
        u8_dev = [torch.empty(B, 224, 224, 3, dtype=torch.uint8, device=dev) for _ in range(2)]
        trainer.capture(u8_dev[0], dev_lbls[0])

        def prefetch8(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i])
                u8_dev[i].copy_(u8_host[i], non_blocking=True)
                dev_lbls[i].copy_(host_lbls[i], non_blocking=True)
                ready[i].record(copy_stream)

        def loop8(n):
            for i in range(2):
                consumed[i].record()
            prefetch8(0)
            out = 0.0
            for s in range(n):
                cur = s & 1
                if s + 1 < n:
                    prefetch8(cur ^ 1)
                torch.cuda.current_stream().wait_event(ready[cur])
                l, _ = trainer.step(u8_dev[cur], dev_lbls[cur])
                consumed[cur].record()
                out = l.item()
            return out

        loop8(2)
        sync_all()
        t0 = time.perf_counter()
        loop8(args.steps)
        sync_all()
        u8_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        e2e_u8 = {"value": world * B * args.steps / (u8_ms / 1e3), "unit": "images/sec",
                  "h2d_bytes_per_step": B * 224 * 224 * 3 + B * 8, "d2h_bytes_per_step": 4, "ms_per_step": u8_ms / args.steps,
                  "input": "decoded uint8 NHWC; ToTensor + Normalize fused into the stem operand on the device"}

    line = {"metric": metric_label(name), "value": value, "unit": "images/sec", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": spec["workload"],
                       "per_gpu_batch": B, "global_batch": world * B, "parallelism": f"dp{world}",
                       "optimizer": optimizer_desc(name),
                       "step": "fwd+CE+bwd+allreduce+optimizer",
                       "launch": "eager" if args.eager else "CUDA graph replay",
                       "l2": "working set (>10 GB of activations per step) is far larger than the 126 MB L2; no flush needed"},
            "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches), "clocks": clocks, "final_loss": final_loss}
    if e2e_u8 is not None:
        line["e2e_uint8"] = e2e_u8

    # per-kernel roofline: one extra step with CUDA-event spans around every C-ABI op on the launching stream.  Every rank
    # runs the step (it contains the gradient all-reduce); only rank 0 records spans.
    trainer.step_eager(images, labels)   # torch.cuda.graph() emptied the allocator cache: re-warm it outside the spans
    sync_all()
    if rank == 0:
        with ops.Profiler(run_ahead_ms=120.0) as prof:
            trainer.step_eager(images, labels)
    else:
        trainer.step_eager(images, labels)
    sync_all()
    if rank == 0:
        peaks = load_peaks()
        per_gpu = value / world
        line["step_roofline"] = {
            "hbm_frac": per_gpu * spec["mb"] * 1e6 / (peaks["hbm_gbs"] * 1e9),
            "tensor_frac": per_gpu * spec["gflop"] * 1e9 / (peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]) * 1e12),
            "peaks": peaks["_source"]}
        agg = prof.summary()
        tot = sum(a["ms"] for a in agg.values())
        kernels = []
        for kname, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
            kernels.append({"kernel": kname, "calls": a["calls"], "ms": round(a["ms"], 3), "share": round(a["ms"] / tot, 4),
                            "GBps": round(a["bytes"] / a["ms"] / 1e6, 1), "TFLOPs": round(a["flops"] / a["ms"] / 1e9, 1)})
        top = kernels[0]
        a = agg[top["kernel"]]
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(name, {}).get(top["kernel"])
        flops_bound = a["flops"] > 0 and (a["flops"] / (peaks["bf16_tflops_sustained"] * 1e12)) > (a["bytes"] / (peaks["hbm_gbs"] * 1e9))
        if flops_bound:
            ach, peak, unit = a["flops"] / a["ms"] / 1e9, peaks["bf16_tflops_sustained"], "TFLOP/s"
        else:
            ach, peak, unit = a["bytes"] / a["ms"] / 1e6, peaks["hbm_gbs"], "GB/s"
        line["roofline"] = {"bound": "tensor" if flops_bound else "hbm", "kernel": top["kernel"], "achieved": ach, "peak": peak,
                            "unit": unit, "frac": ach / peak, "traffic": traffic, "launches_per_step": a["calls"],
                            "avg_launch_ms": a["ms"] / a["calls"], "peaks": peaks["_source"],
                            "how": "CUDA-event spans on the launching stream over one extra eager step after the timed region (host enqueues ahead of the device behind a spin kernel, so spans hold no launch gaps); "
                                   "algorithmic bytes = tensors read+written once per launch"}
        line["kernels"] = kernels
    # release this model's activations / graphs before the next one is measured
    del trainer, model, images, labels, host_imgs, host_lbls, dev_imgs, dev_lbls
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    return line


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: no CUDA device visible (there is no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    line = measure(args.model, args, dev, world, rank, local_rank, args.batch or None)
    if args.model == "resnet50" and not args.no_secondary:
        # BASELINE.json's metric is quoted on ResNet-50 AND ViT-B/16: same measurements, same invocation, as a sub-block
        sec = measure("vit_b16", args, dev, world, rank, local_rank)
        line["secondary"] = {k: sec[k] for k in ("metric", "value", "unit", "ms_per_step", "config", "e2e", "gpu_launches",
                                                  "clocks", "final_loss", "step_roofline", "roofline", "kernels") if k in sec}
        line["gpu_launches"] += sec["gpu_launches"]
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and args.model == "resnet50":
            cb = cpu_reference_run(3, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the BASELINE config's, 256)")
    ap.add_argument("--model", default="resnet50", choices=sorted(MODELS), help="resnet50 = BASELINE configs[1] (headline)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the ViT-B/16 block of the default (resnet50) line")
    ap.add_argument("--eager", action="store_true", help="do not capture the step into CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's loss, correct flags and a seeded sample of the updated "
                         "parameters of each measured model to DIR/<model>_<array>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 training step (--impl b200)")
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)  # stdout of this process (and of native libraries) -> stderr; emit() writes the JSON line to the saved fd
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
