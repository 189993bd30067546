"""Training / evaluation loops with the call contract of /root/reference/engine.py.

``train_one_epoch`` keeps the reference signature (engine.py:19-24) and the semantics of its eager branch
(257-274): per-iteration LR/WD schedule write (98-103, including the ``is not None`` quirk that also
rewrites the no-decay group — SURVEY Appendix D #1), ``loss / update_freq``, backward, step every
``update_freq`` micro-batches, ``zero_grad``, optional EMA, meters, returned ``{meter: global_avg}``.
What changes underneath: model, criterion and optimizer run on the vitk sm_100a kernels, gradient
averaging across ranks is the NCCL all-reduce of ``parallel.DataParallel`` (one bf16 all-reduce of the flat
gradient after backward; micro-batches that do not end in ``optimizer.step()`` run under ``no_sync()``), gradient
clipping acts on the reduced gradient, and the device is only synchronised when a metric is actually read (every
``log_freq`` steps) instead of after every step (engine.py:278-279, 290-299).
"""
from __future__ import annotations

import contextlib
from typing import Iterable

import torch

from . import utils
from .losses import CrossEntropyLoss


def train_one_epoch(model: torch.nn.Module, criterion: torch.nn.Module, data_loader: Iterable,
                    optimizer: torch.optim.Optimizer, device: torch.device, epoch: int, loss_scaler=None,
                    max_norm: float = 0, model_ema=None, mixup_fn=None, log_writer=None, wandb_logger=None,
                    start_steps=None, lr_schedule_values=None, wd_schedule_values=None,
                    num_training_steps_per_epoch=None, update_freq=None, use_amp=False, tpu: bool = False,
                    log_freq: int = 10, wd_quirk: bool = True, quiet: bool = True):
    if tpu:
        raise NotImplementedError("tpu=True selects the reference's torch_xla branch; this build targets B200 (CUDA)")
    if loss_scaler is not None and use_amp:
        raise NotImplementedError("GradScaler/AMP is not used: the kernels compute in bf16 with fp32 accumulation "
                                  "and fp32 master weights, no loss scaling is needed")
    update_freq = update_freq or 1
    start_steps = start_steps or 0
    model.train(True)
    metric_logger = utils.MetricLogger(delimiter="  ")
    header = f"Epoch: [{epoch}]"
    if log_writer is not None and num_training_steps_per_epoch is not None:
        log_writer.set_step(epoch * num_training_steps_per_epoch * update_freq)
    optimizer.zero_grad()
    last_loss = None
    on_gpu = torch.device(device).type == "cuda"
    pinned = [torch.empty(2, dtype=torch.float32, pin_memory=on_gpu) for _ in range(2)]
    pending = None

    def _enqueue_read(loss_t, acc_t, nsamp, lr_now, buf):
        vals = torch.stack([loss_t.detach().float().reshape(()), (acc_t if acc_t is not None else loss_t.detach()).float().reshape(())])
        buf.copy_(vals, non_blocking=True)
        ev = None
        if on_gpu:
            ev = torch.cuda.Event()
            ev.record()
        return ev, buf, acc_t is not None, nsamp, lr_now

    def _consume(p):
        ev, buf, has_acc, nsamp, lr_now = p
        if ev is not None:
            ev.synchronize()
        metric_logger.update(loss=float(buf[0]))
        if has_acc:
            metric_logger.meters["class_acc"].update(float(buf[1]), n=nsamp)
        metric_logger.update(lr=lr_now)
        if log_writer is not None:
            log_writer.update(loss=metric_logger.meters["loss"].value, lr=lr_now)
        if wandb_logger is not None:
            wandb_logger._wandb.log({"train/loss": metric_logger.meters["loss"].value, "train/learning_rate": lr_now,
                                     "train/epoch": epoch})

    if on_gpu:
        data_loader = utils.DevicePrefetcher(data_loader, torch.device(device))   # H2D of batch i+1 overlaps step i
    for data_iter_step, (samples, targets) in enumerate(metric_logger.log_every(data_loader, 10, header, quiet=quiet)):
        step = data_iter_step // update_freq
        if num_training_steps_per_epoch is not None and step >= num_training_steps_per_epoch:
            continue
        it = start_steps + step
        if (lr_schedule_values is not None or wd_schedule_values is not None) and data_iter_step % update_freq == 0:
            for param_group in optimizer.param_groups:
                if lr_schedule_values is not None:
                    param_group["lr"] = lr_schedule_values[it] * param_group.get("lr_scale", 1.0)
                if wd_schedule_values is not None:
                    wd = param_group.get("weight_decay", None)
                    if (wd is not None) if wd_quirk else (wd is not None and wd > 0):
                        param_group["weight_decay"] = wd_schedule_values[it]
        # the device-side Mixup / CutMix (mixup.Mixup) works on the batch where it will be consumed
        samples = samples.to(device, non_blocking=True)
        targets = targets.to(device, non_blocking=True)
        if mixup_fn is not None:
            samples, targets = mixup_fn(samples, targets)

        output = model(samples)
        loss = criterion(output, targets)
        if update_freq != 1:
            loss = loss / update_freq
        stepping = (data_iter_step + 1) % update_freq == 0
        # gradients of micro-batches that do not end in a step are only accumulated locally (DDP's no_sync)
        with (model.no_sync() if not stepping and hasattr(model, "no_sync") else contextlib.nullcontext()):
            loss.backward()
        if stepping:
            if max_norm and max_norm > 0:
                clip_grad_norm_(optimizer, max_norm)
            optimizer.step()
            optimizer.zero_grad()
            if model_ema is not None and hasattr(model_ema, "update"):   # (an EMA fused into FusedAdamW needs no call)
                model_ema.update(model)
        last_loss = loss

        if mixup_fn is None and not isinstance(output, tuple) and targets.dtype == torch.int64:
            class_acc = (output.max(-1)[-1] == targets).float().mean()
        else:
            class_acc = None
        lr = optimizer.param_groups[0]["lr"]
        if data_iter_step % log_freq == 0 or data_iter_step < 5:
            # The device -> host read of this step's loss is asynchronous (pinned buffer + event) and consumed one step
            # later, so the host keeps enqueuing the next step while the GPU finishes this one; the reference blocks on
            # loss.item() after every step (/root/reference/engine.py:278-299).
            if pending is not None:
                _consume(pending)
            pending = _enqueue_read(loss, class_acc, samples.size(0), lr, pinned[data_iter_step & 1])
    if pending is not None:
        _consume(pending)
    if last_loss is not None and "loss" not in metric_logger.meters:
        metric_logger.update(loss=last_loss.item())
    metric_logger.synchronize_between_processes()
    return {k: meter.global_avg for k, meter in metric_logger.meters.items()}


def clip_grad_norm_(optimizer, max_norm: float) -> torch.Tensor:
    """``torch.nn.utils.clip_grad_norm_`` semantics on the flat gradient buffer(s), for the gradient the optimizer will
    actually apply: the data-parallel all-reduce is completed first (``optimizer.sync_gradients()``; idempotent, so
    ``step()`` does not reduce again), the global L2 norm is that of the gradient MEAN over the replicas, and every
    rank derives the same coefficient.  Nothing is read back and the gradients are not rewritten: the coefficient
    ``min(1, max_norm / (norm + 1e-6))`` stays on the device and the AdamW kernel multiplies it in.  Returns the norm
    (device scalar).  (The reference's TPU branch clips the local gradient BEFORE the cross-replica mean,
    /root/reference/engine.py:175-185 — SURVEY Appendix D #4; its eager branch never clips.)"""
    from . import _lib as L
    from .optim_factory import FusedAdamW

    if not isinstance(optimizer, FusedAdamW):
        raise NotImplementedError("clip_grad_norm_ is built for FusedAdamW")
    if optimizer._plan is None or any(not e["store"].valid() for e in optimizer._plan):
        optimizer._build_plan()
    optimizer.sync_gradients()
    dev = optimizer._plan[0]["store"].device
    buf = torch.zeros(3, device=dev)   # [sum of squares, coefficient, norm]
    if optimizer.grad_lowp is not None:
        L.sumsq(optimizer.grad_lowp, buf[0:1])
    else:
        for e in optimizer._plan:
            L.sumsq(e["store"].grad, buf[0:1])
    L.clip_coef(buf[0:1], optimizer.grad_scale, float(max_norm), buf[1:2], buf[2:3])
    optimizer.grad_scale_dev = buf[1:2]
    return buf[2]


@torch.no_grad()
def evaluate(data_loader, model, device, use_amp=False, tpu: bool = False):
    """/root/reference/engine.py:339-430: CE loss + top-1/top-5 accuracy meters over the loader."""
    if tpu:
        raise NotImplementedError("tpu=True selects the reference's torch_xla branch; this build targets B200 (CUDA)")
    criterion = CrossEntropyLoss()
    metric_logger = utils.MetricLogger(delimiter="  ")
    model.eval()
    for images, target in data_loader:
        images = images.to(device, non_blocking=True)
        target = target.to(device, non_blocking=True)
        output = model(images)
        if isinstance(output, tuple):
            output = output[0]
        loss = criterion(output, target)
        acc1, acc5 = utils.accuracy(output, target, topk=(1, 5))
        batch_size = images.shape[0]
        metric_logger.update(loss=loss.item())
        metric_logger.meters["acc1"].update(acc1.item(), n=batch_size)
        metric_logger.meters["acc5"].update(acc5.item(), n=batch_size)
    metric_logger.synchronize_between_processes()
    return {k: meter.global_avg for k, meter in metric_logger.meters.items()}
