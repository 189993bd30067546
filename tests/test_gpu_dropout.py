"""GPU: nn.Dropout sites of the reference model (timm Attention.proj_drop, Mlp.drop1 / drop2, pos_drop, head_drop;
/root/reference/models/vision_transformer.py:149-171, 571, 617, 780, 987-990) on the sm_100a path.

The keep masks come from one Philox kernel (vitk_dropout_mask); inside a Block they are applied in the proj / fc1 / fc2 GEMM
epilogues (vitk_gemm_args.mask) and, in the backward, by one in-place multiply of the branch gradient.  RNG streams differ
from torch's, so parity is checked the way DropPath is: the masks are fixed by the test and fed to both sides — the oracle's
nn.Dropout modules are overridden by forward hooks, the CUDA path reads them through ops.dropout_source.
"""
import math

import pytest
import torch

from conftest import cos_sim, elem_err, rel_err, report, rms_err

pytestmark = pytest.mark.gpu


def test_dropout_mask_kernel(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    n = 1_000_003   # not a multiple of 8: the tail bytes are written one by one
    for p in (0.1, 0.5, 0.9):
        m = torch.full((n + 5,), 7, dtype=torch.uint8, device=cuda_device)
        L.dropout_mask(m[:n], p, 1234, 1)
        assert set(m[:n].unique().tolist()) <= {0, 1} and m[n:].eq(7).all()   # nothing past the end
        keep = m[:n].float().mean().item()
        assert abs(keep - (1 - p)) < 5 * math.sqrt(p * (1 - p) / n), (p, keep)
        m2 = torch.empty(n, dtype=torch.uint8, device=cuda_device)
        L.dropout_mask(m2, p, 1234, 1)
        assert torch.equal(m[:n], m2)                       # same seed and offset: same mask
        L.dropout_mask(m2, p, 1234, 2)
        agree = (m[:n] == m2).float().mean().item()         # another offset: an independent draw
        assert abs(agree - (p * p + (1 - p) * (1 - p))) < 5e-3, (p, agree)
    with pytest.raises(L.VitkError):
        L.dropout_mask(m2, 1.0, 0, 0)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_mask_mul(cuda_device, dtype):
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(0)
    rows, cols = 333, 776
    x = torch.randn(rows, cols, device=cuda_device).to(dtype)
    m = (torch.rand(rows, cols, device=cuda_device) > 0.3).to(torch.uint8)
    want = (x.float() * m.float() * 1.25).to(dtype)
    L.mask_mul_(x, m, 1.25, rows, cols)
    assert torch.equal(x, want)


@pytest.mark.parametrize("M,N,K", [(394, 3072, 768), (1000, 768, 192), (130, 256, 64), (2049, 1536, 384)])
def test_gemm_gelu_epilogue_with_dropout(cuda_device, M, N, K):
    """Mlp.drop1 inside the fc1 epilogue: out = gelu(h) * m / keep, aux = gelu'(h) * m / keep."""
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(1)
    x = torch.randn(M, K, device=cuda_device).bfloat16()
    w = (torch.randn(N, K, device=cuda_device) * K ** -0.5).bfloat16()
    b = torch.randn(N, device=cuda_device)
    m = (torch.rand(M, N, device=cuda_device) > 0.25).to(torch.uint8)
    s = 1.0 / 0.75
    out = torch.full((M, N), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    aux = torch.full((M, N), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    L.gemm(x, w, out, M=M, N=N, K=K, epilogue=L.EPI_GELU, bias=b, aux=aux, mask=m, mask_scale=s)
    h = (x.float() @ w.float().t() + b).requires_grad_(True)
    act = torch.nn.functional.gelu(h)
    (dact,) = torch.autograd.grad(act.sum(), h)
    report("gelu*mask", out.float(), act.detach() * m * s)
    assert elem_err(out.float(), act.detach() * m * s) < 1e-2
    assert elem_err(aux.float(), dact * m * s) < 1.2e-2
    dropped = m == 0
    assert out[dropped].eq(0).all() and aux[dropped].eq(0).all()   # exactly zero, not merely small


@pytest.mark.parametrize("M,N,K", [(394, 768, 3072), (394, 768, 768), (1000, 384, 384), (300, 200, 256)])
@pytest.mark.parametrize("scales", [False, True])
def test_gemm_resid_epilogue_with_dropout(cuda_device, M, N, K, scales):
    """proj_drop / Mlp.drop2 inside the residual epilogue: out = resid + rowscale * colscale * m / keep * (acc + bias), for
    the short-K launches that would otherwise take the TMA-ring variant as well as the long-K ones."""
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(2)
    rpg = 50 if M % 50 == 0 else M // 2
    x = torch.randn(M, K, device=cuda_device).bfloat16()
    w = (torch.randn(N, K, device=cuda_device) * K ** -0.5).bfloat16()
    b = torch.randn(N, device=cuda_device)
    r = torch.randn(M, N, device=cuda_device)
    rs = (torch.rand((M + rpg - 1) // rpg, device=cuda_device) > 0.3).float() / 0.7 if scales else None
    cs = torch.rand(N, device=cuda_device) if scales else None
    m = (torch.rand(M, N, device=cuda_device) > 0.1).to(torch.uint8)
    s = 1.0 / 0.9
    out = torch.full((M, N), float("nan"), device=cuda_device)
    L.gemm(x, w, out, M=M, N=N, K=K, epilogue=L.EPI_RESID, bias=b, resid=r, rowscale=rs, rows_per_group=rpg, colscale=cs,
           mask=m, mask_scale=s)
    branch = (x.float() @ w.float().t() + b) * m * s
    if scales:
        branch = branch * rs.repeat_interleave(rpg)[:M, None] * cs
    report("resid+drop", out, r + branch)
    assert rel_err(out - r, branch) < 1e-2
    assert torch.equal(out[m == 0], r[m == 0])   # a dropped element passes the residual through untouched


def test_gemm_mask_is_rejected_where_it_has_no_epilogue(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    x = torch.zeros(128, 64, device=cuda_device, dtype=torch.bfloat16)
    w = torch.zeros(64, 64, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(128, 64, device=cuda_device, dtype=torch.bfloat16)
    m = torch.ones(128, 64, device=cuda_device, dtype=torch.uint8)
    with pytest.raises(L.VitkError):
        L.gemm(x, w, out, M=128, N=64, K=64, epilogue=L.EPI_BF16, mask=m, mask_scale=2.0)


@pytest.mark.parametrize("B,N,H,hd", [(2, 197, 3, 64), (1, 100, 2, 64), (1, 300, 2, 64), (2, 197, 2, 72), (2, 198, 2, 48),
                                      (3, 577, 4, 64), (3, 640, 4, 64),
                                      (2, 100, 2, 72)])
def test_attention_dropout_kernels(cuda_device, B, N, H, hd):
    """attn_drop: out = (softmax(S) * m / keep) V with lse of the undropped scores; backward through the same mask.
    Against torch on the same bf16-rounded qkv and the same mask (N <= 128, 128 < N <= 256, N > 256, wide and narrow heads)."""
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(0)
    p_drop = 0.2
    s = 1.0 / (1.0 - p_drop)
    qkv = torch.randn(B, N, 3 * H * hd, device=cuda_device).bfloat16()
    dout = torch.randn(B, N, H * hd, device=cuda_device).bfloat16()
    mask = (torch.rand(B, H, N, N, device=cuda_device) >= p_drop).to(torch.uint8)
    out = torch.full((B, N, H * hd), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    lse = torch.full((B, H, N), float("nan"), device=cuda_device)
    dqkv = torch.full((B, N, 3 * H * hd), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5, keep_mask=mask, keep_scale=s)
    L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, hd, hd ** -0.5, keep_mask=mask, keep_scale=s)
    q, k, v = (t.detach().requires_grad_(True) for t in qkv.float().view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0))
    sc = (q @ k.transpose(-1, -2)) * hd ** -0.5
    ref = ((torch.softmax(sc, -1) * mask.float() * s) @ v).transpose(1, 2).reshape(B, N, H * hd)
    ref.backward(dout.float())
    g = torch.stack([q.grad, k.grad, v.grad], 0).permute(1, 3, 0, 2, 4).reshape(B, N, 3 * H * hd)
    report("attn_drop out", out.float(), ref.detach())
    assert elem_err(out.float(), ref.detach()) < 1.5e-2 and rms_err(out.float(), ref.detach()) < 5e-3
    assert rel_err(lse, torch.logsumexp(sc.detach(), -1)) < 5e-3
    d, r = dqkv.float().view(B, N, 3, H * hd), g.view(B, N, 3, H * hd)
    for i, name in enumerate("qkv"):
        report(f"attn_drop d{name}", d[:, :, i], r[:, :, i])
        assert rms_err(d[:, :, i], r[:, :, i]) < 8e-3 and elem_err(d[:, :, i], r[:, :, i]) < 3e-2, name


class fixed_dropout:
    """Fixes the keep mask of every nn.Dropout site: forward hooks on the oracle's modules, ops.dropout_source for the CUDA
    path.  Masks are drawn once per site name from a seeded CPU generator."""

    def __init__(self, ref, device, seed=11):
        self.device, self.gen, self.masks, self.hooks = device, torch.Generator().manual_seed(seed), {}, []
        for name, mod in ref.named_modules():
            if isinstance(mod, torch.nn.Dropout) and mod.p > 0:
                self.hooks.append(mod.register_forward_hook(self._hook(name, mod.p)))

    def mask(self, site, rows, cols, p):
        if site not in self.masks:
            self.masks[site] = (torch.rand(rows, cols, generator=self.gen) >= p).to(torch.uint8).to(self.device)
        assert self.masks[site].shape == (rows, cols), (site, self.masks[site].shape, rows, cols)
        return self.masks[site]

    def _hook(self, name, p):
        def fn(mod, inp, out):
            if not mod.training:
                return out
            x = inp[0]
            cols = x.shape[-1]
            m = self.mask(name, x.numel() // cols, cols, p)
            return x * m.view(x.shape).to(x.dtype) / (1.0 - p)
        return fn

    def source(self, site, rows, cols, p, device):
        return self.mask(site, rows, cols, p)

    def close(self):
        for h in self.hooks:
            h.remove()


@pytest.mark.parametrize("kw", [dict(proj_drop_rate=0.1), dict(pos_drop_rate=0.1, drop_rate=0.2),
                                dict(proj_drop_rate=0.2, pos_drop_rate=0.1, drop_rate=0.1, drop_path_rate=0.1, init_values=0.1),
                                dict(proj_drop_rate=0.1, global_pool="token"), dict(attn_drop_rate=0.1),
                                dict(attn_drop_rate=0.2, proj_drop_rate=0.1, drop_path_rate=0.1)],
                         ids=["proj", "pos+head", "all+droppath+layerscale", "proj-token", "attn", "attn+proj+droppath"])
def test_model_with_dropout_matches_oracle(cuda_device, kw):
    """ViT-Ti/16 with dropout at every built site against the fp32 oracle with the SAME masks: logits, loss, every block's
    output, every parameter gradient.  Tolerances are those of tests/test_gpu_configs.py."""
    from oracle import vit_oracle as O
    from test_gpu_configs import record_masks, replay
    from vision_transformers_torch_xla_b200 import ops
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model

    dev, B = cuda_device, 6
    kw = dict(dict(num_classes=1000, global_pool="avg"), **kw)
    torch.manual_seed(0)
    # attn_drop: the oracle's unfused attention path applies it as an nn.Dropout module on the softmax (hookable); the fused
    # SDPA call would draw its own mask inside the kernel
    ref = O.create_model("vit_tiny_patch16_224", fused_attn=not kw.get("attn_drop_rate"), **kw).to(dev)
    mine = create_model("vit_tiny_patch16_224", **kw).to(dev)
    mine.load_state_dict(ref.state_dict())
    ref.train()
    mine.train()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, 3, 224, 224, generator=g).to(dev)
    tgt = O.mixup_soft_targets(torch.randint(0, 1000, (B,), generator=g)).to(dev)

    acts = {"ref": [], "mine": []}
    handles = [blk.register_forward_hook(lambda mod, inp, out: acts["ref"].append(out.detach())) for blk in ref.blocks]
    for blk in mine.blocks:
        blk.register_forward_hook(lambda mod, inp, out: acts["mine"].append(out.detach()))
    fix = fixed_dropout(ref, dev)
    rec = record_masks(ref)
    out_ref = ref(x)
    rec.close()
    loss_ref = O.SoftTargetCrossEntropy()(out_ref, tgt)
    loss_ref.backward()
    fix.close()
    for h in handles:
        h.remove()
    n_sites = sum(1 for _, m in ref.named_modules() if isinstance(m, torch.nn.Dropout) and m.p > 0)
    assert len(fix.masks) == n_sites and all(0 < float(m.float().mean()) < 1 for m in fix.masks.values())

    ops.dropout_source = fix.source
    ops.mask_source = replay(rec.masks) if rec.masks else None
    try:
        out = mine(x)
    finally:
        ops.dropout_source = None
        ops.mask_source = None
    loss = SoftTargetCrossEntropy()(out, tgt)
    loss.backward()

    report("logits", out, out_ref)
    assert elem_err(out, out_ref) < 3e-2 and rms_err(out, out_ref) < 1e-2
    assert abs(loss.item() - loss_ref.item()) < 2e-3 * abs(loss_ref.item()), (loss.item(), loss_ref.item())
    for i, (a, b) in enumerate(zip(acts["mine"], acts["ref"])):
        assert elem_err(a, b) < 3e-2 and rms_err(a, b) < 7e-3, i
    ref_grads = dict(ref.named_parameters())
    worst = (0.0, "")
    for n, p in mine.named_parameters():
        a, b = p.grad, ref_grads[n].grad
        assert a is not None and b is not None, n
        worst = max(worst, (rms_err(a, b), n))
        assert rms_err(a, b) < 1.5e-2 and cos_sim(a, b) > 0.999, (n, rms_err(a, b), cos_sim(a, b))
    print(f"[parity] dropout {kw}: loss {loss.item():.6f} vs {loss_ref.item():.6f}, worst gradient rms err {worst[0]:.2e} ({worst[1]})")


def test_dropout_is_off_in_eval_and_random_in_train(cuda_device):
    from vision_transformers_torch_xla_b200.models import create_model
    torch.manual_seed(0)
    model = create_model("vit_tiny_patch16_224", num_classes=10, proj_drop_rate=0.3, pos_drop_rate=0.1, drop_rate=0.1).to(cuda_device)
    x = torch.randn(2, 3, 224, 224, device=cuda_device)
    model.eval()
    with torch.no_grad():
        a, b = model(x), model(x)
    assert torch.equal(a, b)
    model.train()
    with torch.no_grad():
        c, d = model(x), model(x)
    assert not torch.equal(c, d) and torch.isfinite(c).all()


def test_stand_alone_modules_with_dropout(cuda_device):
    """Mlp(drop=p) and Attention(proj_drop=p) used on their own (the reference's leaf plug points, models/_compat.py)."""
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200 import ops
    from vision_transformers_torch_xla_b200.models.vision_transformer import Attention, Mlp
    dev = cuda_device
    torch.manual_seed(0)
    x = torch.randn(4, 50, 192, device=dev)
    for mine, ref in ((Mlp(192, 768, drop=0.2).to(dev), O.Mlp(192, 768, drop=0.2).to(dev)),
                      (Attention(192, num_heads=3, qkv_bias=True, proj_drop=0.2).to(dev),
                       O.Attention(192, num_heads=3, qkv_bias=True, proj_drop=0.2).to(dev))):
        mine.load_state_dict(ref.state_dict())
        mine.train()
        ref.train()
        fix = fixed_dropout(ref, dev)
        xr = x.clone().requires_grad_(True)
        yr = ref(xr)
        yr.square().sum().backward()
        fix.close()
        # stand-alone sites are named without the block prefix: map them onto the oracle's module names
        alias = {"mlp.drop1": "drop1", "mlp.drop2": "drop2", "attn.proj_drop": "proj_drop"}
        ops.dropout_source = lambda site, rows, cols, p, device: fix.mask(alias[site], rows, cols, p)
        try:
            xm = x.clone().requires_grad_(True)
            ym = mine(xm)
        finally:
            ops.dropout_source = None
        ym.square().sum().backward()
        assert rms_err(ym, yr) < 7e-3 and rms_err(xm.grad, xr.grad) < 1.5e-2, (type(mine).__name__, rms_err(ym, yr))
        for (n, p), (_, q) in zip(mine.named_parameters(), ref.named_parameters()):
            assert rms_err(p.grad, q.grad) < 1.5e-2, n
