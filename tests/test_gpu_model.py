"""Whole-model parity on the GPU: the vitk model (bf16 tensor-core kernels, fp32 accumulate, fp32 residual
stream and master weights) against the eager fp32 oracle with identical weights and inputs.

Metrics and stated tolerances for bf16 tensor-core compute against the fp32 oracle:
  * rel_err  = max|a-b| / rms(b)          (north-star metric)  activations <= 2e-2
  * elem_err = max|a-b| / (|b| + rms(b))  used where the tensor is heavy-tailed (logits of a single token,
               gradients whose RMS is dominated by a handful of label rows): <= 3e-2 ... 5e-2
  * rms_err  = rms(a-b) / rms(b)          typical error: <= 1e-2, and cosine similarity >= 0.999 for gradients
  * loss trajectories over 200 AdamW steps: <= 5e-3 relative over the first 20 steps, <= 5e-2 throughout.
"""
import math

import pytest
import torch

from conftest import cos_sim, elem_err, rel_err, rms_err

pytestmark = pytest.mark.gpu


def _pair(name, dev, **kw):
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200.models import create_model

    torch.manual_seed(0)
    ref = O.create_model(name, **kw).to(dev)
    mine = create_model(name, **kw).to(dev)
    missing = mine.load_state_dict(ref.state_dict(), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return ref, mine


@pytest.mark.parametrize("name,kw", [
    ("vit_tiny_patch16_224", dict(num_classes=1000, global_pool="avg")),
    ("vit_tiny_patch16_224", dict(num_classes=1000, global_pool="token")),
    ("vit_small_patch16_224", dict(num_classes=100, global_pool="avg")),  # ragged class count (100 % 8 != 0)
    ("deit_tiny_distilled_patch16_224", dict(num_classes=1000)),
])
def test_forward_logits(cuda_device, name, kw):
    ref, mine = _pair(name, cuda_device, **kw)
    ref.eval()
    mine.eval()
    x = torch.randn(6, 3, 224, 224, device=cuda_device)
    with torch.no_grad():
        want = ref(x)
        got = mine(x)
    assert got.shape == want.shape and got.dtype == torch.float32
    assert elem_err(got, want) < 3e-2 and rms_err(got, want) < 1e-2


@pytest.mark.parametrize("name,kw", [
    ("vit_tiny_patch16_224", dict(num_classes=1000)),                 # the image is the patch GEMM's operand
    ("vit_small_patch16_224", dict(num_classes=100, patch_size=8)),   # im2col PatchEmbed, N = 785
])
def test_bf16_image_matches_its_fp32_copy(cuda_device, name, kw):
    """A bf16 image batch gives the same logits, bit for bit, as the fp32 batch that holds the same values."""
    from vision_transformers_torch_xla_b200.models import create_model

    torch.manual_seed(0)
    model = create_model(name, **kw).to(cuda_device).eval()
    x = torch.randn(4, 3, 224, 224, device=cuda_device).bfloat16()
    with torch.no_grad():
        got = model(x)
        want = model(x.float())
    assert torch.equal(got, want)


def test_per_layer_activations_and_grads(cuda_device):
    ref, mine = _pair("vit_tiny_patch16_224", cuda_device, num_classes=1000, global_pool="avg")
    ref.train()
    mine.train()
    B = 8
    x = torch.randn(B, 3, 224, 224, device=cuda_device)
    tgt = torch.softmax(torch.randn(B, 1000, device=cuda_device) * 3, -1)
    acts = {"ref": [], "mine": []}
    grads = {"ref": [], "mine": []}

    def hook(store_a, store_g):
        def fn(mod, inp, out):
            store_a.append(out.detach())
            out.register_hook(lambda g: store_g.append(g.detach()))
        return fn

    for blk in ref.blocks:
        blk.register_forward_hook(hook(acts["ref"], grads["ref"]))
    for blk in mine.blocks:
        blk.register_forward_hook(hook(acts["mine"], grads["mine"]))

    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy

    loss_ref = O.SoftTargetCrossEntropy()(ref(x), tgt)
    loss_ref.backward()
    loss = SoftTargetCrossEntropy()(mine(x), tgt)
    loss.backward()
    assert abs(loss.item() - loss_ref.item()) < 2e-3 * abs(loss_ref.item())
    assert len(acts["mine"]) == 12 and len(grads["mine"]) == 12
    for i, (a, b) in enumerate(zip(acts["mine"], acts["ref"])):
        assert rel_err(a, b) < 2e-2, f"activation of block {i}"
    worst_g = max((elem_err(a, b), rms_err(a, b), i) for i, (a, b) in enumerate(zip(grads["mine"], grads["ref"])))
    print("worst residual-stream gradient (elem_err, rms_err, #):", worst_g)
    for i, (a, b) in enumerate(zip(grads["mine"], grads["ref"])):  # appended in reverse block order on both sides
        assert elem_err(a, b) < 5e-2 and rms_err(a, b) < 1e-2, f"residual-stream gradient #{i}"
    refp = dict(ref.named_parameters())
    worst = ("", 0.0)
    for n, p in mine.named_parameters():
        assert p.grad is not None, n
        e = elem_err(p.grad, refp[n].grad)
        if e > worst[1]:
            worst = (n, e)
        # typical error and direction are the criteria; the worst single element (heavy-tailed sums over the batch,
        # e.g. pos_embed.grad) is only sanity-bounded
        assert rms_err(p.grad, refp[n].grad) < 1.5e-2 and cos_sim(p.grad, refp[n].grad) > 0.999, n
        assert e < 0.25, f"grad of {n}: {e}"
    print("worst param-grad rel err:", worst)


def test_gradient_accumulation_and_zero_grad(cuda_device):
    _, mine = _pair("vit_tiny_patch16_224", cuda_device, num_classes=1000, global_pool="avg")
    from vision_transformers_torch_xla_b200.losses import LabelSmoothingCrossEntropy

    mine.train()
    x = torch.randn(4, 3, 224, 224, device=cuda_device)
    y = torch.randint(0, 1000, (4,), device=cuda_device)
    crit = LabelSmoothingCrossEntropy(0.1)
    crit(mine(x), y).backward()
    g1 = mine.head.weight.grad.clone()
    crit(mine(x), y).backward()
    assert rel_err(mine.head.weight.grad, 2 * g1) < 1e-3  # accumulates like autograd
    for p in mine.parameters():
        p.grad = None  # what torch's zero_grad(set_to_none=True) does
    crit(mine(x), y).backward()
    assert rel_err(mine.head.weight.grad, g1) < 1e-3


def test_loss_trajectory_200_steps(cuda_device):
    """200 AdamW steps on fixed synthetic batches: vitk model + FusedAdamW vs oracle + torch.optim.AdamW."""
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200 import optim_factory
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy

    ref, mine = _pair("vit_tiny_patch16_224", cuda_device, num_classes=1000, global_pool="avg", drop_path_rate=0.0)
    ref.train()
    mine.train()
    B, steps = 8, 200
    g = torch.Generator(device="cpu").manual_seed(1)
    xs = [torch.randn(B, 3, 224, 224, generator=g).to(cuda_device) for _ in range(4)]
    ys = [O.mixup_soft_targets(torch.randint(0, 1000, (B,), generator=g)).to(cuda_device) for _ in range(4)]
    opt_ref = O.create_optimizer(ref, lr=5e-4, weight_decay=0.05)

    class Args:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 5e-4, 0.05, 1e-8, None

    opt = optim_factory.create_optimizer(Args, mine)
    assert [len(gp["params"]) for gp in opt.param_groups] == [len(gp["params"]) for gp in opt_ref.param_groups]
    lr_sched = O.cosine_scheduler(5e-4, 1e-6, 1, steps, warmup_epochs=1, warmup_steps=20)
    wd_sched = O.cosine_scheduler(0.05, 0.05, 1, steps)
    crit_ref, crit = O.SoftTargetCrossEntropy(), SoftTargetCrossEntropy()
    l_ref, l_mine = [], []
    for it in range(steps):
        O.apply_schedules(opt_ref, it, lr_sched, wd_sched)
        O.apply_schedules(opt, it, lr_sched, wd_sched)
        loss_r, _ = O.train_step(ref, crit_ref, opt_ref, xs[it % 4], ys[it % 4])
        loss_m, _ = O.train_step(mine, crit, opt, xs[it % 4], ys[it % 4])
        l_ref.append(float(loss_r))
        l_mine.append(float(loss_m))
    l_ref, l_mine = torch.tensor(l_ref), torch.tensor(l_mine)
    assert l_ref[-1] < 0.8 * l_ref[0], "oracle did not learn; test is vacuous"
    rel = ((l_mine - l_ref).abs() / l_ref.abs().clamp_min(1e-3))
    print("trajectory: first", l_ref[0].item(), l_mine[0].item(), "last", l_ref[-1].item(), l_mine[-1].item(),
          "max rel dev", rel.max().item())
    assert rel[:20].max() < 5e-3
    assert rel.max() < 5e-2
    # weights stay close too.  Only matrices are compared: Adam turns a mathematically-zero gradient (e.g. the key
    # bias, which softmax is invariant to) into a +-lr random walk of rounding noise, so 1-D parameters whose true
    # gradient vanishes legitimately differ between any two floating-point implementations.
    refp = dict(ref.named_parameters())
    worst = max(((rms_err(p.data, refp[n].data), n) for n, p in mine.named_parameters() if p.ndim >= 2))
    print("worst weight rms err after 200 steps:", worst)
    assert worst[0] < 5e-2, worst


def test_kd_flow_like_reference_test_kd(cuda_device):
    """/root/reference/test_kd.py:18-126: student + teacher + wrapper + DistillationLoss on random input."""
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200.losses import (DistillationLoss, LabelSmoothingCrossEntropy,
                                                         StudentWithDistillation)
    from vision_transformers_torch_xla_b200.models import create_model

    torch.manual_seed(0)
    student = create_model("vit_tiny_patch16_224", pretrained=False, num_classes=1000, global_pool="avg").to(cuda_device)
    teacher = create_model("vit_small_patch16_224", pretrained=False, num_classes=1000, global_pool="avg").to(cuda_device)
    for p in teacher.parameters():
        p.requires_grad = False
    teacher.eval()
    model = StudentWithDistillation(student, teacher)
    crit = DistillationLoss(LabelSmoothingCrossEntropy(0.1), alpha=0.7, temperature=4.0)
    x = torch.randn(4, 3, 224, 224, device=cuda_device)
    y = torch.randint(0, 1000, (4,), device=cuda_device)
    model.train()
    teacher.eval()
    out = model(x)
    assert isinstance(out, tuple) and out[0].shape == (4, 1000) and out[1].shape == (4, 1000)
    loss = crit(out, y)
    loss.backward()
    assert student.head.weight.grad is not None and float(student.head.weight.grad.abs().sum()) > 0
    assert teacher.head.weight.grad is None or float(teacher.head.weight.grad.abs().sum()) == 0
    # same numbers as the oracle's DistillationLoss on the same logits
    want = O.DistillationLoss(O.LabelSmoothingCrossEntropy(0.1), 0.7, 4.0)((out[0].detach(), out[1].detach()), y)
    assert abs(loss.item() - want.item()) < 1e-4 * max(1.0, abs(want.item()))
    model.eval()
    assert isinstance(model(x), torch.Tensor)


def test_deit_distilled_hard_kd(cuda_device):
    from vision_transformers_torch_xla_b200.losses import DistillationLoss, LabelSmoothingCrossEntropy
    from oracle import vit_oracle as O

    ref, mine = _pair("deit_tiny_distilled_patch16_224", cuda_device, num_classes=1000)
    for m in (ref, mine):
        m.train()
        m.set_distilled_training(True)
    x = torch.randn(4, 3, 224, 224, device=cuda_device)
    y = torch.randint(0, 1000, (4,), device=cuda_device)
    teacher_logits = torch.randn(4, 1000, device=cuda_device)
    out_r, out_m = ref(x), mine(x)
    assert isinstance(out_m, tuple) and len(out_m) == 2
    l_r = O.DistillationLoss(O.LabelSmoothingCrossEntropy(0.1), 0.5, 1.0, hard=True)((out_r, teacher_logits), y)
    l_m = DistillationLoss(LabelSmoothingCrossEntropy(0.1), 0.5, 1.0, hard=True)((out_m, teacher_logits), y)
    l_r.backward()
    l_m.backward()
    assert abs(l_r.item() - l_m.item()) < 5e-3 * abs(l_r.item())
    refp = dict(ref.named_parameters())
    # only the cls/dist token rows carry loss here and B = 4, so these gradients are extremely heavy-tailed:
    # judge them by direction (cosine) and typical error (rms) instead of the worst element
    errs = {n: (rms_err(p.grad, refp[n].grad), cos_sim(p.grad, refp[n].grad)) for n, p in mine.named_parameters()}
    bad = {n: e for n, e in errs.items() if not (e[0] < 2e-2 and e[1] > 0.9995)}
    print("deit hard-KD grads: worst", max(errs.items(), key=lambda kv: kv[1][0]), "bad:", bad)
    assert not bad, bad
    mine.eval()
    ref.eval()
    with torch.no_grad():
        assert elem_err(mine(x), ref(x)) < 3e-2


def test_engine_train_one_epoch_and_evaluate(cuda_device):
    from vision_transformers_torch_xla_b200 import engine, optim_factory, utils
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model
    from oracle import vit_oracle as O

    torch.manual_seed(0)
    model = create_model("vit_tiny_patch16_224", num_classes=1000, global_pool="avg", drop_path_rate=0.1).to(cuda_device)

    class Args:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 1e-3, 0.05, 1e-8, None

    opt = optim_factory.create_optimizer(Args, model)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(8, 3, 224, 224, generator=g)
    y = O.mixup_soft_targets(torch.randint(0, 1000, (8,), generator=g))
    loader = [(x, y)] * 12
    lr = utils.cosine_scheduler(1e-3, 1e-5, 1, 6, warmup_steps=2, warmup_epochs=1)
    wd = utils.cosine_scheduler(0.05, 0.05, 1, 6)
    stats = engine.train_one_epoch(model, SoftTargetCrossEntropy(), loader, opt, cuda_device, 0, None, start_steps=0,
                                   lr_schedule_values=lr, wd_schedule_values=wd, num_training_steps_per_epoch=6,
                                   update_freq=2, log_freq=1)
    assert set(stats) >= {"loss", "lr"} and math.isfinite(stats["loss"])
    assert all(gp["weight_decay"] == 0.05 for gp in opt.param_groups)  # reference quirk: no_decay group overwritten too
    ev = engine.evaluate([(x, torch.randint(0, 1000, (8,)))], model, cuda_device)
    assert set(ev) == {"loss", "acc1", "acc5"} and math.isfinite(ev["loss"])


def test_layerscale_matches_oracle(cuda_device):
    """init_values -> LayerScale (/root/reference/models/vision_transformer.py:80-106): forward through the residual
    epilogue's column scale, gamma gradients from the branch's weight gradients (vitk_layerscale_grad)."""
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model
    from oracle import vit_oracle as O

    torch.manual_seed(0)
    kw = dict(num_classes=1000, global_pool="avg", init_values=0.1)
    ref = O.create_model("vit_tiny_patch16_224", **kw).to(cuda_device)
    mine = create_model("vit_tiny_patch16_224", **kw).to(cuda_device)
    assert set(mine.state_dict()) == set(ref.state_dict()) and "blocks.0.ls1.gamma" in mine.state_dict()
    with torch.no_grad():   # make the scales non-uniform so that a wrong channel mapping cannot hide
        for blk in ref.blocks:
            blk.ls1.gamma.mul_(torch.rand_like(blk.ls1.gamma) + 0.5)
            blk.ls2.gamma.mul_(torch.rand_like(blk.ls2.gamma) + 0.5)
    mine.load_state_dict(ref.state_dict())
    ref.train()
    mine.train()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(4, 3, 224, 224, generator=g).to(cuda_device)
    y = O.mixup_soft_targets(torch.randint(0, 1000, (4,), generator=g)).to(cuda_device)
    out_ref = ref(x)
    O.SoftTargetCrossEntropy()(out_ref, y).backward()
    out = mine(x)
    SoftTargetCrossEntropy()(out, y).backward()
    assert rel_err(out, out_ref) < 2e-2
    for name in ("blocks.0.ls1.gamma", "blocks.5.ls2.gamma", "blocks.11.ls1.gamma", "blocks.11.ls2.gamma", "blocks.3.mlp.fc2.weight",
                 "blocks.3.attn.proj.weight", "blocks.0.attn.qkv.weight"):
        a = dict(mine.named_parameters())[name].grad
        b = dict(ref.named_parameters())[name].grad
        assert rms_err(a, b) < 2e-2 and cos_sim(a, b) > 0.999, name
    # gradient accumulation: a second backward doubles dgamma (it is recomputed from the accumulated weight gradient)
    g1 = mine.blocks[5].ls2.gamma.grad.clone()
    SoftTargetCrossEntropy()(mine(x), y).backward()
    assert rms_err(mine.blocks[5].ls2.gamma.grad, 2 * g1) < 1e-2


def test_checkpoint_save_resume(cuda_device, tmp_path):
    """Reference format (/root/reference/utils/__init__.py:686-770): {'model','optimizer','epoch','scaler','args',
    'model_ema'}; resuming restores weights, Adam moments, step count and the fused EMA (the split-K wgrad
    reductions are fp32 atomics, so two runs agree to rounding, not bitwise; a lost moment or step count shows up at 1e-3)."""
    import argparse

    from vision_transformers_torch_xla_b200 import optim_factory, utils
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model
    from oracle import vit_oracle as O

    class OptArgs:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 1e-3, 0.05, 1e-8, None

    g = torch.Generator().manual_seed(0)
    x = torch.randn(4, 3, 224, 224, generator=g).to(cuda_device)
    y = O.mixup_soft_targets(torch.randint(0, 1000, (4,), generator=g)).to(cuda_device)
    crit = SoftTargetCrossEntropy()

    def make():
        torch.manual_seed(0)
        m = create_model("vit_tiny_patch16_224", num_classes=1000, global_pool="avg").to(cuda_device)
        o = optim_factory.create_optimizer(OptArgs, m)
        return m, o

    def steps(m, o, n):
        for _ in range(n):
            crit(m(x), y).backward()
            o.step()
            o.zero_grad()

    a, oa = make()
    crit(a(x), y).backward()   # the flat store (and with it the optimizer plan) exists after the first forward
    oa.zero_grad()
    oa.enable_ema(0.9)
    steps(a, oa, 2)
    args = argparse.Namespace(output_dir=str(tmp_path), save_ckpt_num=3, save_ckpt_freq=1, auto_resume=True, resume="",
                              start_epoch=0)
    path = utils.save_model(args, 0, a, a, oa, None, model_ema=True)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert set(ck) == {"model", "optimizer", "epoch", "scaler", "args", "model_ema"} and ck["epoch"] == 0
    assert set(ck["model"]) == set(a.state_dict()) == set(ck["model_ema"])
    assert set(ck["optimizer"]) == {"state", "param_groups"}
    steps(a, oa, 2)

    b, ob = make()
    crit(b(x), y).backward()
    ob.zero_grad()
    ob.enable_ema(0.9)
    utils.auto_load_model(args, b, b, ob, None, model_ema=True)
    assert args.start_epoch == 1
    # the restored state is exactly the saved one: weights, both Adam moments, step count, EMA
    for n2, p2 in b.named_parameters():
        assert torch.equal(p2.detach().cpu(), ck["model"][n2]), n2
    saved = ck["optimizer"]["state"]
    for i, p2 in enumerate(pp for gp in ob.param_groups for pp in gp["params"]):
        assert torch.equal(ob.state[p2]["exp_avg"].cpu(), saved[i]["exp_avg"]) and \
            torch.equal(ob.state[p2]["exp_avg_sq"].cpu(), saved[i]["exp_avg_sq"]), i
    assert ob._step == 2
    assert torch.equal(utils.ema_state_dict(b, ob)["blocks.3.mlp.fc1.weight"], ck["model_ema"]["blocks.3.mlp.fc1.weight"])
    # and training continues from there (elements with ~zero gradient move by up to lr under the atomics' rounding noise)
    steps(b, ob, 2)
    for (n1, p1), (n2, p2) in zip(a.named_parameters(), b.named_parameters()):
        # (the key bias has an exactly-zero true gradient: Adam turns its rounding noise into +-lr steps)
        assert (p1 - p2).abs().max().item() < 2.5e-3 and (p1 - p2).abs().mean().item() < 2e-4, n1
    assert int(float(next(iter(ob.state.values()))["step"])) == 4


def test_standalone_modules(cuda_device):
    """Attention / Mlp / LayerNorm / PatchEmbed / Block are usable on their own (reference plug points)."""
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200.models import Attention, Block, LayerNorm, Mlp, PatchEmbed

    torch.manual_seed(0)
    B, N, D = 2, 197, 192
    x = torch.randn(B, N, D, device=cuda_device)
    pairs = [
        (O.Attention(D, num_heads=3, qkv_bias=True), Attention(D, num_heads=3, qkv_bias=True)),
        (O.Mlp(D, 4 * D), Mlp(D, 4 * D)),
        (O.LayerNorm(D), LayerNorm(D)),
        (O.Block(D, 3, qkv_bias=True), Block(D, 3, qkv_bias=True)),
    ]
    for ref, mine in pairs:
        ref, mine = ref.to(cuda_device), mine.to(cuda_device)
        mine.load_state_dict(ref.state_dict())
        xr = x.clone().requires_grad_(True)
        xm = x.clone().requires_grad_(True)
        yr, ym = ref(xr), mine(xm)
        assert rel_err(ym, yr) < 2e-2, type(ref).__name__
        go = torch.randn_like(yr)
        yr.backward(go)
        ym.backward(go)
        assert rel_err(xm.grad, xr.grad) < 3e-2, type(ref).__name__
        for (n, pr), (_, pm) in zip(ref.named_parameters(), mine.named_parameters()):
            assert elem_err(pm.grad, pr.grad) < 4e-2, f"{type(ref).__name__}.{n}"
    pe_r, pe_m = O.PatchEmbed(224, 16, 3, D).to(cuda_device), PatchEmbed(224, 16, 3, D).to(cuda_device)
    pe_m.load_state_dict(pe_r.state_dict())
    img = torch.randn(2, 3, 224, 224, device=cuda_device)
    assert rel_err(pe_m(img), pe_r(img)) < 2e-2


def test_unsupported_options_raise():
    from vision_transformers_torch_xla_b200.models import VisionTransformer, create_model

    with pytest.raises(NotImplementedError):
        VisionTransformer(qk_norm=True)
    with pytest.raises(NotImplementedError):
        VisionTransformer(global_pool="map")
    with pytest.raises(NotImplementedError):
        create_model("vit_tiny_patch16_224", pretrained=True)
    with pytest.raises(RuntimeError):
        create_model("resnet50")
