"""world_size-2 data-parallel plumbing on CPU (gloo): replica broadcast, the gradient marked pending by the backward's
hook and reduced by the optimizer's pre-step hook (fp32 in place, since the gradient is not on CUDA), 1/world folded
into the optimizer, no_sync() and exactly-once reduction under gradient accumulation, meter reduction."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn


class Tiny(nn.Module):
    def __init__(self):
        super().__init__()
        self.cls_token = nn.Parameter(torch.randn(1, 1, 8))
        self.blocks = nn.Sequential(nn.Linear(8, 8), nn.Linear(8, 8))
        self.head = nn.Linear(8, 4)


class FakeOpt:
    def __init__(self):
        self.grad_scale = 1.0
        self.pre_step_hooks = []

    def step(self):
        for h in self.pre_step_hooks:
            h(self)


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from vision_transformers_torch_xla_b200 import store as S
        from vision_transformers_torch_xla_b200 import utils
        from vision_transformers_torch_xla_b200.parallel import DataParallel

        torch.manual_seed(100 + rank)  # different replicas before the broadcast
        m = Tiny()
        st = S.ParamStore(m, allow_cpu=True)
        m.__dict__["_vitk_store"] = st
        opt = FakeOpt()
        dp = DataParallel(m, optimizer=opt)
        assert dp.store is st and opt.grad_scale == 1.0 / world
        # 1) identical replicas after construction
        flat = [torch.zeros_like(st.flat) for _ in range(world)]
        dist.all_gather(flat, st.flat)
        assert all(torch.equal(flat[0], f) for f in flat)
        # 2) the backward's hook marks the gradient pending; the optimizer's pre-step hook reduces it in one all-reduce of
        #    the flat buffer (fp32 in place: the gradient is not on CUDA).  Grads are SUMMED (the mean is in grad_scale).
        st.grad.fill_(float(rank + 1))
        st.fire_grad_ready()
        assert dp._pending
        opt.step()
        assert not dp._pending and not hasattr(opt, "grad_lowp")
        assert torch.equal(st.grad, torch.full_like(st.grad, float(sum(range(1, world + 1)))))
        assert torch.equal(m.head.weight.grad, torch.full_like(m.head.weight, 3.0))  # p.grad views the flat buffer
        # 3) no_sync(): gradient accumulation micro-steps do not communicate
        st.grad.fill_(float(rank + 1))
        with dp.no_sync():
            st.fire_grad_ready()
        assert not dp._pending
        opt.step()
        assert float(st.grad[0]) == float(rank + 1)
        # 4) update_freq = 2 the way engine.train_one_epoch drives it: micro-batch 1 under no_sync(), micro-batch 2
        #    synchronised -> the ACCUMULATED gradient is reduced exactly once (a reduction per micro-batch would count
        #    the first micro-batch world_size times)
        st.grad.zero_()
        with dp.no_sync():
            st.grad.add_(float(rank + 1))
            st.fire_grad_ready()
        assert not dp._pending
        st.grad.add_(10.0 * (rank + 1))
        st.fire_grad_ready()
        dp.finish_gradient_sync()
        dp.finish_gradient_sync()   # idempotent: clipping syncs first, step() must not reduce again
        opt.step()
        assert torch.equal(st.grad, torch.full_like(st.grad, 11.0 * sum(range(1, world + 1))))
        # 5) metric meters reduce across ranks like the reference's SmoothedValue.synchronize_between_processes
        sv = utils.SmoothedValue()
        sv.update(float(rank + 1), n=1)
        sv.synchronize_between_processes()
        assert sv.count == world and sv.total == 3.0 and utils.get_world_size() == world and utils.get_rank() == rank
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_data_parallel_world2_gloo_one_allreduce():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert results == {0: "ok", 1: "ok"}, results
