"""Attention above 640 tokens (448 / 512 px at patch 16, 224 px at patch 8): the unmasked forward runs attn_fwd6, the
forward with an attention-dropout keep mask runs the kv-streaming attn_fwd_stream_kernel, the backward runs the streaming
kernel for both.  The kernel checks are those of test_gpu_attn.py / test_gpu_dropout.py at their own tolerances, the
model checks those of test_gpu_configs.py."""
import pytest
import torch

import test_gpu_attn
import test_gpu_configs
import test_gpu_dropout
from conftest import cos_sim, elem_err, rms_err

pytestmark = pytest.mark.gpu

N_MAX = 4224   # the longest sequence the attention kernels accept (1024 px at patch 16 is N = 4097)


@pytest.mark.parametrize("hd", [64, 48, 32])
@pytest.mark.parametrize("B,N,H", [(2, 641, 3), (1, 700, 2), (4, 785, 12), (2, 1025, 4), (1, 2305, 2), (1, N_MAX, 2)])
def test_long_attn_fwd_bwd(cuda_device, B, N, H, hd):
    test_gpu_attn.test_attn_fwd(cuda_device, B, N, H, hd)
    test_gpu_attn.test_attn_bwd(cuda_device, B, N, H, hd)


@pytest.mark.parametrize("B,N,H,hd", [(2, 785, 3, 64), (1, 1025, 2, 48), (1, 2305, 1, 64)])
def test_long_attention_dropout_kernels(cuda_device, B, N, H, hd):
    test_gpu_dropout.test_attention_dropout_kernels(cuda_device, B, N, H, hd)


def test_long_attn_limit_raises(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    B, N, H, hd = 1, N_MAX + 1, 1, 64
    qkv = torch.zeros(B, N, 3 * H * hd, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(B, N, H * hd, device=cuda_device, dtype=torch.bfloat16)
    lse = torch.zeros(B, H, N, device=cuda_device)
    mask = torch.ones(B, H, N, N, device=cuda_device, dtype=torch.uint8)
    with pytest.raises(L.VitkError):
        L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5)
    with pytest.raises(L.VitkError):
        L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5, keep_mask=mask, keep_scale=1.25)
    with pytest.raises(L.VitkError):
        L.attn_bwd(qkv, out, out, lse, torch.zeros_like(qkv), B, N, H, hd, hd ** -0.5)


_KW = dict(num_classes=1000, global_pool="avg", drop_path_rate=0.1)


@pytest.mark.parametrize("name,kw,B,gtol", [
    ("vit_base_patch16_224", dict(_KW, img_size=448), 2, 1.5e-2),     # N = 785
    ("vit_small_patch16_224", dict(_KW, img_size=512), 2, 1.5e-2),    # N = 1025
    ("vit_small_patch16_224", dict(_KW, patch_size=8), 2, 1.5e-2),    # N = 785 through the im2col PatchEmbed
], ids=["vit_base_448", "vit_small_512", "vit_small_patch8"])
def test_long_seq_config_matches_oracle(cuda_device, name, kw, B, gtol):
    test_gpu_configs.test_config_activations_logits_and_all_gradients(cuda_device, name, kw, B, gtol)


def test_long_seq_model_with_attention_dropout_matches_oracle(cuda_device):
    """ViT-Ti/16 at 448 px (N = 785) with attn_drop 0.1: the keep masks are fixed through ops.dropout_source (and forward
    hooks on the oracle's unfused attention), the DropPath masks replayed; logits, loss, every block's output and every
    parameter gradient at the tolerances of test_gpu_dropout.test_model_with_dropout_matches_oracle."""
    from oracle import vit_oracle as O
    from vision_transformers_torch_xla_b200 import ops
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model

    dev, B = cuda_device, 2
    kw = dict(_KW, img_size=448, attn_drop_rate=0.1)
    torch.manual_seed(0)
    ref = O.create_model("vit_tiny_patch16_224", fused_attn=False, **kw).to(dev)
    mine = create_model("vit_tiny_patch16_224", **kw).to(dev)
    mine.load_state_dict(ref.state_dict())
    ref.train()
    mine.train()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, 3, 448, 448, generator=g).to(dev)
    tgt = O.mixup_soft_targets(torch.randint(0, 1000, (B,), generator=g)).to(dev)

    acts = {"ref": [], "mine": []}
    handles = [blk.register_forward_hook(lambda mod, inp, out: acts["ref"].append(out.detach())) for blk in ref.blocks]
    for blk in mine.blocks:
        blk.register_forward_hook(lambda mod, inp, out: acts["mine"].append(out.detach()))
    fix = test_gpu_dropout.fixed_dropout(ref, dev)
    rec = test_gpu_configs.record_masks(ref)
    out_ref = ref(x)
    rec.close()
    loss_ref = O.SoftTargetCrossEntropy()(out_ref, tgt)
    loss_ref.backward()
    fix.close()
    for h in handles:
        h.remove()
    assert len(fix.masks) == len(ref.blocks)   # one attn_drop site per block

    ops.dropout_source = fix.source
    ops.mask_source = test_gpu_configs.replay(rec.masks)
    try:
        out = mine(x)
    finally:
        ops.dropout_source = None
        ops.mask_source = None
    loss = SoftTargetCrossEntropy()(out, tgt)
    loss.backward()

    assert elem_err(out, out_ref) < 3e-2 and rms_err(out, out_ref) < 1e-2
    assert abs(loss.item() - loss_ref.item()) < 2e-3 * abs(loss_ref.item()), (loss.item(), loss_ref.item())
    for i, (a, b) in enumerate(zip(acts["mine"], acts["ref"])):
        assert elem_err(a, b) < 3e-2 and rms_err(a, b) < 7e-3, i
    ref_grads = dict(ref.named_parameters())
    for n, p in mine.named_parameters():
        a, b = p.grad, ref_grads[n].grad
        assert a is not None and b is not None, n
        assert rms_err(a, b) < 1.5e-2 and cos_sim(a, b) > 0.999, (n, rms_err(a, b), cos_sim(a, b))


def test_grad_checkpointing_at_448px_gives_the_same_logits(cuda_device):
    """set_grad_checkpointing(True) at N = 785 with attention dropout and DropPath: the re-run forward in the backward uses
    the same masks, so the logits are the same bit for bit.  Above 256 tokens the attention backward red.adds dQ over kv
    tiles in arrival order, so the gradients of a step are not bitwise reproducible (with or without checkpointing); they
    are held to the oracle-parity tolerance instead of the 1e-5 of test_gpu_configs' checkpointing test at N = 197."""
    from vision_transformers_torch_xla_b200 import ops
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model

    dev, B = cuda_device, 2
    torch.manual_seed(0)
    model = create_model("vit_small_patch16_224", img_size=448, attn_drop_rate=0.1, **_KW).to(dev)
    model.train()
    x = torch.randn(B, 3, 448, 448, device=dev)
    tgt = torch.softmax(torch.randn(B, 1000, device=dev), -1)
    masks, drops = {}, {}

    def dp_source(drop_probs, nb, device):
        key = tuple(drop_probs)
        if key not in masks:
            g = torch.Generator().manual_seed(5)
            masks[key] = torch.stack([(torch.rand(nb, generator=g) >= p).float() / (1 - p) for p in drop_probs]).to(device)
        return masks[key]

    def do_source(site, rows, cols, p, device):
        if site not in drops:
            g = torch.Generator().manual_seed(len(drops) + 1)
            drops[site] = (torch.rand(rows, cols, generator=g) >= p).to(torch.uint8).to(device)
        return drops[site]

    def run(ckpt):
        model.set_grad_checkpointing(ckpt)
        model.zero_grad(set_to_none=True)
        ops.mask_source, ops.dropout_source = dp_source, do_source
        try:
            out = model(x)
            SoftTargetCrossEntropy()(out, tgt).backward()
        finally:
            ops.mask_source, ops.dropout_source = None, None
        return out.detach().clone(), {n: p.grad.detach().clone() for n, p in model.named_parameters()}

    out_a, grads_a = run(False)
    out_b, grads_b = run(True)
    model.set_grad_checkpointing(False)
    assert drops, "attention dropout drew no mask"
    assert torch.equal(out_a, out_b)
    for n in grads_a:
        assert rms_err(grads_b[n], grads_a[n]) < 1.5e-2 and cos_sim(grads_b[n], grads_a[n]) > 0.999, (n, rms_err(grads_b[n], grads_a[n]))
