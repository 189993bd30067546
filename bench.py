#!/usr/bin/env python
"""Headline benchmark: ViT-B/16 224px bf16 training images/sec (BASELINE.json `metric`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1..5 | --model NAME --batch B] [--impl ours|reference]
                  [--dump-outputs DIR]

--config selects one of BASELINE.json's configs as written (default 3 = the headline: vit_base_patch16_224, batch 256/GPU):
  1 vit_tiny_patch16_224 batch 8            2 vit_small_patch16_224 batch 256        3 vit_base_patch16_224 batch 256
  4 deit_base_distilled_patch16_224 batch 256, StudentWithDistillation(student, frozen RegNetY-16GF teacher, channels-last
    bf16, no_grad) + DistillationLoss(hard) with distilled_training on   5 vit_large_patch16_384 batch 64

One process per GPU (torchrun for N>1).  A step = forward + loss + backward + AdamW on one synthetic batch.
Prints ONE JSON line (rank 0).  `value` is timed with inputs resident in HBM; `e2e` goes through the public
API (`engine.train_one_epoch`) with pinned host batches (H2D copy + loss read-back inside the timed region).
`roofline` times every tcgen05 GEMM launch of the timed region with CUDA events; `cpu_baseline` times the
CPU oracle (restated reference eager path) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# stdout carries exactly ONE JSON line.  Libraries print there too (NCCL's "NCCL version ..." banner at NCCL_DEBUG=WARN
# ignores NCCL_DEBUG_FILE on this image), so file descriptor 1 points at stderr while the benchmark runs and is only
# restored for the final print.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: str) -> None:
    sys.stdout.flush()
    os.dup2(_REAL_STDOUT, 1)
    print(line, flush=True)

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

#: algorithmic train GFLOP per image (SURVEY §8 header formula), used for the tensor-roofline fraction
TRAIN_GFLOP_PER_IMG = {
    "vit_tiny_patch16_224": 7.464, "vit_small_patch16_224": 27.478, "vit_base_patch16_224": 105.152,
    "deit_base_distilled_patch16_224": 105.710, "vit_large_patch16_384": 1145.492, "my_vit_b": 105.152,
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tf=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"], hbm=d["hbm_gbs"], src="measured")
    return dict(tf=1400.0, tf_burst=1590.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


#: BASELINE.json `configs`, in order: (model, per-GPU batch, distillation teacher)
CONFIGS = {
    1: ("vit_tiny_patch16_224", 8, None),
    2: ("vit_small_patch16_224", 256, None),
    3: ("vit_base_patch16_224", 256, None),
    4: ("deit_base_distilled_patch16_224", 256, "regnet_y_16gf"),
    5: ("vit_large_patch16_384", 64, None),
}


class Teacher(torch.nn.Module):
    """Frozen forward-only distillation teacher (/root/reference/main.py:691-742): torchvision RegNetY-16GF (83.6 M
    parameters, random init: there is no network for checkpoints), channels-last bf16, eval mode.  Library (cuDNN)
    convolutions: the teacher is not a custom-kernel target (SURVEY §8 a12); its time is reported separately."""

    def __init__(self, name, device):
        super().__init__()
        import torchvision

        torch.backends.cudnn.benchmark = True   # grouped 3x3 convolutions: let cuDNN time its algorithms once
        self.net = getattr(torchvision.models, name)(weights=None, num_classes=1000).to(device).eval()
        self.net = self.net.to(memory_format=torch.channels_last).bfloat16()
        for p in self.net.parameters():
            p.requires_grad = False

    def train(self, mode=True):   # stays in eval mode inside the training wrapper (main.py:737-740)
        return super().train(False)

    @torch.no_grad()
    def forward(self, x):
        return self.net(x.to(dtype=torch.bfloat16, memory_format=torch.channels_last)).float()


def build(model_name, batch, device, drop_path, teacher=None):
    from vision_transformers_torch_xla_b200 import optim_factory
    from vision_transformers_torch_xla_b200.losses import DistillationLoss, SoftTargetCrossEntropy, StudentWithDistillation
    from vision_transformers_torch_xla_b200.models import create_model

    torch.manual_seed(0)
    kw = dict(num_classes=1000, drop_path_rate=drop_path)
    if not model_name.startswith("deit_"):
        kw["global_pool"] = "avg"  # what reference main.py:643-649 passes
    model = create_model(model_name, pretrained=False, **kw).to(device)
    model.train()

    class Args:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 1e-3, 0.05, 1e-8, None

    opt = optim_factory.create_optimizer(Args, model)   # (main.py:868-878: the optimizer sees the student only)
    crit = SoftTargetCrossEntropy()
    if teacher is None:
        return model, model, opt, crit
    if hasattr(model, "set_distilled_training"):
        model.set_distilled_training(True)              # (cls, dist) heads -> DeiT hard distillation
    wrapped = StudentWithDistillation(model, Teacher(teacher, device))
    wrapped.train()
    return model, wrapped, opt, DistillationLoss(crit, alpha=0.5, temperature=1.0, hard=True)


def soft_targets(labels, num_classes=1000, lam=0.7, smoothing=0.1):
    """Mixup-style soft targets made on the host for the synthetic batches: lam * onehot_s(y) + (1 - lam) * onehot_s(y.flip(0))
    with timm's smoothed one-hot (on 1 - eps + eps / C, off eps / C)."""
    off = smoothing / num_classes
    on = 1.0 - smoothing + off

    def one_hot(y):
        return torch.full((y.shape[0], num_classes), off).scatter_(1, y.view(-1, 1), on)

    return lam * one_hot(labels) + (1.0 - lam) * one_hot(labels.flip(0))


def synth_batch(batch, img, gen):
    """ImageNet-shaped synthetic batch: N(0,1) images, mixup-style soft targets (smoothing 0.1), hard labels."""
    x = torch.randn(batch, 3, img, img, generator=gen)
    labels = torch.randint(0, 1000, (batch,), generator=gen)
    return x, soft_targets(labels), labels


#: --dump-outputs writes an array of more elements than this as a seeded sample of that many: at most five arrays (loss,
#: up to three outputs, parameters) of 8 MB of float32 each keep a dump well under 64 MB
DUMP_MAX_ELEMS = 1 << 21


def _dump_array(t):
    """``t`` as float32, or, if it has more than DUMP_MAX_ELEMS elements, the flat sample at fixed seeded positions."""
    t = t.detach().float()
    if t.numel() <= DUMP_MAX_ELEMS:
        return t
    idx = torch.randint(0, t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
    return t.reshape(-1)[idx.to(t.device)]


def dump_outputs(out_dir, loss, output, model):
    """Write what one training step computed as float32 ``out_dir/<name>.npy``: ``loss``; the model output (``output``, or
    ``output_0``, ``output_1``, ... for nested tuples, in order: (student (cls, dist), teacher) logits with a distillation
    teacher); ``params``, every parameter of ``model`` after the optimizer step, flattened in ``model.parameters()`` order."""
    import numpy as np

    outs = []

    def flatten(o):
        if isinstance(o, (tuple, list)):
            for v in o:
                flatten(v)
        else:
            outs.append(o)

    flatten(output)
    arrays = {"loss": loss}
    arrays.update({"output": outs[0]} if len(outs) == 1 else {f"output_{i}": t for i, t in enumerate(outs)})
    arrays["params"] = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), _dump_array(t).cpu().numpy())


def run_reference(args):
    """CPU arm: the restated reference eager path (oracle) on the host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import vit_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    sample_b = 8
    torch.manual_seed(0)
    kw = dict(num_classes=1000)
    if not args.model.startswith("deit_"):
        kw["global_pool"] = "avg"
    model = O.create_model(args.model, **kw)
    model.train()
    opt = O.create_optimizer(model, lr=1e-3, weight_decay=0.05)
    crit = O.SoftTargetCrossEntropy()
    img = model.patch_embed.img_size[0]
    gen = torch.Generator().manual_seed(0)
    x, y, _ = synth_batch(sample_b, img, gen)
    for _ in range(args.warmup):
        O.train_step(model, crit, opt, x, y)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss, out = O.train_step(model, crit, opt, x, y)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, out, model)
    v = sample_b / dt
    cores = torch.get_num_threads()
    sample = f"{args.model} fwd+bwd+AdamW fp32 eager CPU, batch {sample_b} per step (bounded sample of batch {args.batch})"
    emit(json.dumps({
        "impl": "reference", "metric": "train images/sec", "value": v, "unit": "img/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} train step, {img}x{img}, batch {args.batch}/GPU", "sample_batch": sample_b},
        "cpu_baseline": {"value": v, "unit": "img/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def cpu_baseline(model_name, batch):
    from oracle import vit_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    sample_b = 8
    kw = dict(num_classes=1000)
    if not model_name.startswith("deit_"):
        kw["global_pool"] = "avg"
    torch.manual_seed(0)
    model = O.create_model(model_name, **kw)
    model.train()
    opt = O.create_optimizer(model, lr=1e-3, weight_decay=0.05)
    crit = O.SoftTargetCrossEntropy()
    img = model.patch_embed.img_size[0]
    x, y, _ = synth_batch(sample_b, img, torch.Generator().manual_seed(0))
    O.train_step(model, crit, opt, x, y)
    n, t0 = 0, time.perf_counter()
    while n < 3 or (time.perf_counter() - t0 < 8 and n < 20):
        O.train_step(model, crit, opt, x, y)
        n += 1
    dt = (time.perf_counter() - t0) / n
    return {"value": sample_b / dt, "unit": "img/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{model_name} fwd+bwd+AdamW fp32 eager on CPU, batch {sample_b}, {n} timed steps "
                      f"({dt * 1e3:.0f} ms/step)"}


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant GEMM from a committed `ncu --set full` capture of
# the same kernel at the same shape, keyed by GEMM family: (bytes, capture file, build id of the library that was profiled).
# Read from profiles/ncu_traffic.json so that a new capture updates the number without touching this file; a capture taken
# from a different build of the library is still reported but flagged (`traffic_build` != `build`).
def ncu_traffic():
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


def roofline(by_shape, family_tf, n_launches, gemm_ms_per_step, pk, build_id):
    """The dominant kernel = the GEMM role/shape with the largest summed device time inside the timed region; every
    launch was bracketed by CUDA events on the launching stream.  `family_*` is the same over all gemm_kernel launches."""
    if not by_shape:
        return None
    from vision_transformers_torch_xla_b200 import _lib as L

    fam, (fl, ms, n) = max(by_shape.items(), key=lambda kv: kv[1][1])
    tf = fl / (ms * 1e-3) / 1e12
    t = ncu_traffic().get(fam, {})
    return {"bound": "tensor", "kernel": f"vitk gemm_kernel (tcgen05 cta_group::2) {fam}", "achieved": tf, "peak": pk["tf"],
            "unit": "TFLOP/s", "frac": tf / pk["tf"], "traffic": t.get("bytes"), "traffic_source": t.get("source"),
            "traffic_build": t.get("build_id"), "build": build_id,
            # the capture is of THIS kernel as long as the GEMM sources are the ones it was taken from
            "traffic_kernel_source_id": t.get("kernel_source_id"),
            "kernel_source_id": L.source_id(("csrc/vitk_gemm.cu", "csrc/vitk_common.cuh")),
            "launches_timed": n, "us_per_launch": ms * 1e3 / n, "flop_per_launch": fl / n,
            "peak_source": f"bf16_tflops_sustained, {pk['src']}",
            "family_achieved": family_tf, "family_frac": (family_tf / pk["tf"]) if family_tf else None,
            "family_launches_timed": n_launches, "family_ms_per_step": gemm_ms_per_step,
            "by_shape_us": {k: round(v[1] * 1e3 / v[2], 1) for k, v in sorted(by_shape.items(), key=lambda kv: -kv[1][1])[:8]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", type=int, default=None, choices=sorted(CONFIGS), help="BASELINE.json config number")
    ap.add_argument("--model", default=None)
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch")
    ap.add_argument("--teacher", default=None, help="torchvision model name of a frozen distillation teacher")
    ap.add_argument("--drop-path", type=float, default=0.1, help="reference launch value (run_train.sh:58)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="print a per-kernel-family time table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last one's loss, model outputs and updated parameters as float32 "
                         "DIR/<name>.npy (a seeded sample of an array above 2M elements); the inputs are seeded, so two "
                         "builds run with the same arguments can be compared array for array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg_model, cfg_batch, cfg_teacher = CONFIGS[args.config if args.config is not None else 3]
    if args.config is None and args.model is not None:
        cfg_teacher = None
    args.model = args.model or cfg_model
    args.batch = args.batch or cfg_batch
    args.teacher = args.teacher or cfg_teacher

    if args.impl == "reference":
        run_reference(args)
        return

    from vision_transformers_torch_xla_b200 import _lib as L
    from vision_transformers_torch_xla_b200 import engine, utils
    from vision_transformers_torch_xla_b200.mixup import Mixup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    distributed = utils.init_distributed_mode(None, backend="nccl") if world > 1 else False
    lib = L.load()
    build_id = lib.vitk_build_id().decode()

    model, step_model, opt, crit = build(args.model, args.batch, dev, args.drop_path, args.teacher)
    train_model = step_model
    if distributed:
        from vision_transformers_torch_xla_b200.parallel import DataParallel

        train_model = DataParallel(step_model, optimizer=opt)
    img = model.patch_embed.img_size[0]
    gen = torch.Generator().manual_seed(1234 + rank)
    host = [tuple(t.pin_memory() for t in synth_batch(args.batch, img, gen)) for _ in range(2)]
    dev_batches = [(x.to(dev), y.to(dev)) for x, y, _ in host]

    def step(i):
        x, y = dev_batches[i % 2]
        out = train_model(x)
        loss = crit(out, y)
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss, out

    def barrier():
        if distributed:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()

    # ---------------- timed region 1: inputs resident in HBM ----------------
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("VITK_BENCH_NO_SAMPLER") != "1":
        sampler.start()
    if os.environ.get("VITK_BENCH_NO_GEMM_TIMING") != "1":
        L.gemm_timing_begin()
    launches0 = L.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        loss, out = step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = L.launch_count - launches0
    (gemm_flops, gemm_ms, gemm_n), gemm_by_shape = L.gemm_timing_end_by_shape()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if distributed:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * args.batch * args.steps / (ms / 1e3)
    final_loss = float(loss.item())
    # before the teacher timing and the end-to-end region run the model again
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, out, model)

    # the frozen teacher's forward alone (library convolutions), so that the student's share of the step is visible
    teacher_ms = None
    if args.teacher is not None:
        x = dev_batches[0][0]
        for _ in range(2):
            step_model.teacher(x)
        barrier()
        e0.record()
        for _ in range(5):
            step_model.teacher(x)
        e1.record()
        barrier()
        teacher_ms = e0.elapsed_time(e1) / 5

    # ---------------- timed region 2: end to end through engine.train_one_epoch ----------------
    # what a user of the reference runs per step (engine.py:259-274): pinned host batch of fp32 images + int64 labels ->
    # H2D -> Mixup / CutMix + label smoothing on the device (timm.data.Mixup as main.py:622-629 builds it) -> model ->
    # criterion -> backward -> step, with the loss read back every step
    e2e = None
    if not args.no_e2e:
        fetch_times = []
        mixup_fn = Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, prob=1.0, switch_prob=0.5, mode="batch", label_smoothing=0.1,
                         num_classes=1000)
        if os.environ.get("VITK_BENCH_E2E_NO_MIXUP") == "1":
            mixup_fn = None

        class _Loader:   # pinned host batches; notes when the engine asks for each one (diagnostics on stderr only)
            def __init__(self, n):
                self.n = n

            def __len__(self):
                return self.n

            def __iter__(self):
                for i in range(self.n):
                    fetch_times.append(time.perf_counter())
                    x, soft, labels = host[i % 2]
                    yield (x, labels) if mixup_fn is not None else (x, soft)

        # untimed warm-up of the end-to-end path itself (the engine's own small torch ops, the prefetcher's buffers and
        # stream, pinned read-back buffers: first use costs 0.2-0.5 s of lazy CUDA module loading and allocation)
        engine.train_one_epoch(train_model, crit, _Loader(args.warmup), opt, dev, 0, None, mixup_fn=mixup_fn, log_freq=1,
                               update_freq=1, quiet=True)
        fetch_times.clear()
        barrier()
        e0.record()
        engine.train_one_epoch(train_model, crit, _Loader(args.steps), opt, dev, 0, None, mixup_fn=mixup_fn, log_freq=1,
                               update_freq=1, quiet=True)
        e1.record()
        barrier()
        if rank == 0 and len(fetch_times) > 2:
            gaps = sorted((b - a) * 1e3 for a, b in zip(fetch_times, fetch_times[1:]))
            print(f"[e2e] host interval between batch fetches: median {gaps[len(gaps) // 2]:.1f} ms, max {gaps[-1]:.1f} ms, "
                  f"first fetch -> last fetch {1e3 * (fetch_times[-1] - fetch_times[0]):.1f} ms", file=sys.stderr)
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if distributed:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        h2d = host[0][0].numel() * host[0][0].element_size() + host[0][2].numel() * host[0][2].element_size()
        e2e = {"value": world * args.batch * args.steps / (float(t.item()) / 1e3), "unit": "img/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
               "api": "engine.train_one_epoch(model, criterion, pinned-host loader of (fp32 images, int64 labels) -> side-stream "
                      "H2D prefetch -> device Mixup/CutMix + label smoothing -> fwd/bwd -> FusedAdamW, log_freq=1: loss read "
                      "back every step, one step deferred)"}

    if args.breakdown and rank == 0:
        L.breakdown_begin()
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        for fam, (n, tms) in sorted(L.breakdown_end().items(), key=lambda kv: -kv[1][1]):
            print(f"  {fam:24s} {n / 3:7.1f} launches/step {tms / 3:9.3f} ms/step", file=sys.stderr)

    if distributed:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    pk = peaks()
    gflop_img = TRAIN_GFLOP_PER_IMG.get(args.model)
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
    loss_name = "SoftTargetCE" if args.teacher is None else \
        f"DistillationLoss(hard, SoftTargetCE base) with a frozen {args.teacher} teacher forward (channels-last bf16)"
    out = {
        "metric": "train images/sec", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.model} train step (fwd + {loss_name} + bwd + AdamW), {img}x{img}, batch "
                               f"{args.batch}/GPU, drop_path {args.drop_path}",
                   "baseline_config": args.config if args.config is not None else (3 if args.model == CONFIGS[3][0] and args.batch == CONFIGS[3][1] else None),
                   "global_batch": world * args.batch,
                   "parallelism": f"dp{world}", "grad_allreduce": os.environ.get("VITK_DP_GRAD", "bf16") + "/" + os.environ.get("VITK_DP_SYNC", "step") if world > 1 else None,
                   "l2": "per-step working set (>10 GB of activations) >> 126 MB L2",
                   "final_loss": final_loss, "teacher_fwd_ms_per_step": teacher_ms},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "roofline": roofline(gemm_by_shape, achieved_tf, gemm_n, gemm_ms / args.steps, pk, build_id),
    }
    if gflop_img:
        step_tf = value / world * gflop_img * 1e9 / 1e12
        out["model_flops"] = {"train_gflop_per_img": gflop_img, "achieved_tflops_per_gpu": step_tf,
                              "frac_of_measured_sustained": step_tf / pk["tf"], "frac_of_nominal_2250": step_tf / 2250.0,
                              "counts": "student GEMMs + attention only (SURVEY section 8 formula)" + ("; the teacher forward is extra, uncounted work inside the step" if args.teacher else "")}
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args.model, args.batch)
    emit(json.dumps(out))


if __name__ == "__main__":
    main()
