"""2-GPU NCCL data parallelism on real devices (skipped with fewer than 2 GPUs).

  * both wire formats, as ``DataParallel`` selects them, give every rank the SUM of the per-rank gradients: bf16 when
    FusedAdamW is attached (it reads the summed gradient from ``grad_lowp``), fp32 in place without an optimizer;
    FusedAdamW applies 1/world, replicas stay identical, and the result equals a single process that sees both batches;
  * ``engine.train_one_epoch`` with ``update_freq = 2`` (micro-batches that do not step run under ``no_sync()``) and
    gradient clipping, on the bf16 wire, matches a single process that sees every micro-batch;
  * gradient clipping acts on the reduced gradient: both ranks derive the same norm, equal to the norm of the
    single-process gradient mean."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _setup(rank, world, port, with_opt=True):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from vision_transformers_torch_xla_b200 import optim_factory, utils
    from vision_transformers_torch_xla_b200.models import create_model
    from vision_transformers_torch_xla_b200.parallel import DataParallel

    assert utils.init_distributed_mode(None, backend="nccl")
    dev = torch.device("cuda", rank)
    torch.manual_seed(100 + rank)  # replicas start different; DataParallel broadcasts rank 0
    model = create_model("vit_tiny_patch16_224", num_classes=1000, global_pool="avg").to(dev)

    class Args:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 1e-3, 0.05, 1e-8, None

    opt = optim_factory.create_optimizer(Args, model)
    dp = DataParallel(model, optimizer=opt if with_opt else None)
    return dev, model, opt, dp, Args


def _single(dev, model, Args):
    """A single-process replica with the same weights (for the 'sees every batch' reference)."""
    from vision_transformers_torch_xla_b200 import optim_factory
    from vision_transformers_torch_xla_b200.models import create_model

    ref = create_model("vit_tiny_patch16_224", num_classes=1000, global_pool="avg").to(dev)
    ref.load_state_dict(model.state_dict())
    ref.train()
    return ref, optim_factory.create_optimizer(Args, ref)


def _worker_sum(rank, world, port, q, wire):
    try:
        from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
        from vision_transformers_torch_xla_b200.store import get_store

        # bf16 wire: FusedAdamW attached at construction; fp32 wire: no optimizer until after the reduction
        dev, model, opt, dp, Args = _setup(rank, world, port, with_opt=wire == "bf16")
        g = torch.Generator().manual_seed(7)
        xs = [torch.randn(4, 3, 224, 224, generator=g) for _ in range(world)]
        ys = [torch.softmax(torch.randn(4, 1000, generator=g) * 3, -1) for _ in range(world)]
        crit = SoftTargetCrossEntropy()
        dp.train()
        crit(dp(xs[rank].to(dev)), ys[rank].to(dev)).backward()
        dp.finish_gradient_sync()
        torch.cuda.synchronize()
        lowp = opt.grad_lowp is not None
        assert lowp == (wire == "bf16")
        grad_sum = (opt.grad_lowp.float() if lowp else dp.store.grad).clone()
        other = [torch.zeros_like(grad_sum) for _ in range(world)]
        dist.all_gather(other, grad_sum)
        assert all(torch.equal(other[0], o) for o in other), "ranks hold different reduced gradients"
        if rank == 0:
            ref, _ = _single(dev, model, Args)
            for x, y in zip(xs, ys):
                crit(ref(x.to(dev)), y.to(dev)).backward()
            rg = get_store(ref).grad
            err = float((grad_sum - rg).abs().max() / rg.abs().max())
            # identical kernels; only the atomic accumulation order (and, for bf16, one rounding per rank) differs
            assert err < (6e-3 if lowp else 1e-3), err
        if not lowp:
            dp.attach_optimizer(opt)
        opt.step()
        opt.zero_grad()
        torch.cuda.synchronize()
        flat = [torch.zeros_like(dp.store.flat) for _ in range(world)]
        dist.all_gather(flat, dp.store.flat)
        assert all(torch.equal(flat[0], f) for f in flat), "replicas diverged after the optimizer step"
        assert opt.grad_scale == 1.0 / world and opt.grad_lowp is None
        assert float(dp.store.grad.abs().max()) == 0.0, "the fp32 gradient buffer is zeroed by the AdamW launch"
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, traceback.format_exc()[-1500:]))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _worker_engine(rank, world, port, q):
    """update_freq = 2 through engine.train_one_epoch + clipping, against one process that sees all four micro-batches."""
    try:
        from vision_transformers_torch_xla_b200 import engine
        from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy

        dev, model, opt, dp, Args = _setup(rank, world, port)
        g = torch.Generator().manual_seed(11)
        # 2 optimizer steps x 2 micro-batches per rank; rank r sees micro-batches [4r, 4r + 4)
        xs = [torch.randn(4, 3, 224, 224, generator=g) for _ in range(4 * world)]
        ys = [torch.softmax(torch.randn(4, 1000, generator=g) * 3, -1) for _ in range(4 * world)]
        mine = [(xs[4 * rank + i], ys[4 * rank + i]) for i in range(4)]
        crit = SoftTargetCrossEntropy()
        if rank == 0:
            ref, opt_ref = _single(dev, model, Args)
        engine.train_one_epoch(dp, crit, mine, opt, dev, 0, None, max_norm=0.05, update_freq=2, log_freq=1)
        torch.cuda.synchronize()
        flat = [torch.zeros_like(dp.store.flat) for _ in range(world)]
        dist.all_gather(flat, dp.store.flat)
        assert all(torch.equal(flat[0], f) for f in flat), "replicas diverged"
        if rank == 0:
            # the same two steps in one process: step s averages micro-batches {2s, 2s+1} of every rank, i.e. the
            # mean over world * 2 micro-batches = update_freq 2 * world with the loss divided accordingly
            # (a plain loop, not the engine: its end-of-epoch meter reduction is a collective rank 1 no longer joins)
            for s in range(2):
                for r in range(world):
                    for i in range(2):
                        x, y = xs[4 * r + 2 * s + i], ys[4 * r + 2 * s + i]
                        (crit(ref(x.to(dev)), y.to(dev)) / (2 * world)).backward()
                engine.clip_grad_norm_(opt_ref, 0.05)
                opt_ref.step()
                opt_ref.zero_grad()

            def rms_err(a, b):
                return float((a.double() - b.double()).pow(2).mean().sqrt() / b.double().pow(2).mean().sqrt())

            refp = dict(ref.named_parameters())
            worst = max((rms_err(p.data, refp[n].data), n) for n, p in model.named_parameters() if p.ndim == 2)
            # two clipped AdamW steps from the same start.  Adam's first steps are ~ lr * sign(g): an element whose
            # gradient is within the bf16 wire's rounding of zero (2^-9 per element) may flip (2 lr = 10 % of a weight's
            # RMS), so the weight matrices are held to 2e-2 rms (the [1, 1, D] tokens start at ~1e-6 and ARE their first
            # two Adam steps)
            assert worst[0] < 2e-2, worst
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, traceback.format_exc()[-1500:]))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _run(worker, *args):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, 2, port, q) + args) for r in range(2)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert results == {0: "ok", 1: "ok"}, results


@pytest.mark.parametrize("wire", ["bf16", "fp32"])
def test_data_parallel_two_gpus(wire):
    _run(_worker_sum, wire)


def test_engine_update_freq_and_clipping_two_gpus():
    _run(_worker_engine)
