"""tcgen05 attention fwd/bwd vs torch fp32 softmax attention on the same bf16-rounded qkv."""

import pytest
import torch

from conftest import elem_err, rel_err

pytestmark = pytest.mark.gpu


def _ref(qkv, B, N, H, hd, dout=None):
    q, k, v = qkv.float().view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)  # [B,H,N,hd]
    q = q.detach().requires_grad_(True)
    k = k.detach().requires_grad_(True)
    v = v.detach().requires_grad_(True)
    s = (q @ k.transpose(-1, -2)) * (hd ** -0.5)
    lse = torch.logsumexp(s, dim=-1)
    o = torch.softmax(s, dim=-1) @ v
    out = o.transpose(1, 2).reshape(B, N, H * hd)
    if dout is None:
        return out, lse, None
    out.backward(dout.float())
    dqkv = torch.stack([q.grad, k.grad, v.grad], 0).permute(1, 3, 0, 2, 4).reshape(B, N, 3 * H * hd)
    return out, lse, dqkv


# (32, 197, 12) = 384 (b, h) items: more than one item per CTA of the persistent kernels (148 SMs)
@pytest.mark.parametrize("B,N,H", [(2, 128, 2), (2, 197, 3), (3, 198, 12), (1, 64, 1), (2, 256, 2), (1, 577, 4), (1, 300, 2),
                                   (1, 129, 1), (2, 144, 2), (1, 255, 3), (32, 197, 12), (13, 198, 12), (8, 577, 16), (5, 640, 7),
                                   (9, 385, 5), (3, 257, 4)])
def test_attn_fwd(cuda_device, B, N, H, hd=64):
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(0)
    qkv = torch.randn(B, N, 3 * H * hd, device=cuda_device).bfloat16()
    out = torch.full((B, N, H * hd), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    lse = torch.full((B, H, N), float("nan"), device=cuda_device)
    L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5)
    ref, ref_lse, _ = _ref(qkv, B, N, H, hd)
    # narrower heads: a score is a sum of hd (not 64) products, so the same bf16 roundings weigh sqrt(64 / hd) more
    narrow = (64 / hd) ** 0.5 * (1.0 if hd == 64 else 1.15)
    # P is rounded to bf16 before P*V (as in every flash-attention bf16 kernel) and the output is bf16
    assert elem_err(out.float(), ref) < 1e-2 * narrow
    # max|err| / rms: one bf16 rounding of the largest output element alone is 2^-9 * max|ref| (a 10-sigma outlier in a
    # 5M-element tensor), so the bound scales with max|ref| / rms.  Two half ulps: an fp32 result next to a rounding tie
    # lands on the other bf16 neighbour after any change of summation order (torch's own bf16 SDPA shows 2.04 half ulps on
    # the (1, 577, 4) case, tools/attn_check.py); the P rounding underneath is the rest.
    half_ulp_of_max = 2.0 ** -9 * float(ref.detach().abs().max() / ref.detach().pow(2).mean().sqrt())
    assert rel_err(out.float(), ref) < max(3e-2, 2.2 * half_ulp_of_max) * narrow
    # and never worse than 2x the error torch's own bf16 SDPA makes against the same fp32 reference
    q, k, v = qkv.view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
    lib = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, N, H * hd)
    assert rel_err(out.float(), ref) < 2 * rel_err(lib.float(), ref) + 2e-3
    assert rel_err(lse, ref_lse) < 5e-3


@pytest.mark.parametrize("B,N,H", [(2, 128, 2), (2, 197, 3), (3, 198, 12), (1, 64, 1), (2, 256, 2), (1, 100, 2),
                                   (2, 577, 4), (1, 300, 2), (1, 640, 1), (1, 129, 1), (2, 144, 2), (1, 255, 3),
                                   (32, 197, 12), (13, 198, 12)])
def test_attn_bwd(cuda_device, B, N, H, hd=64):
    from vision_transformers_torch_xla_b200 import _lib as L
    torch.manual_seed(1)
    qkv = torch.randn(B, N, 3 * H * hd, device=cuda_device).bfloat16()
    dout = torch.randn(B, N, H * hd, device=cuda_device).bfloat16()
    out = torch.empty((B, N, H * hd), device=cuda_device, dtype=torch.bfloat16)
    lse = torch.empty((B, H, N), device=cuda_device)
    dqkv = torch.full((B, N, 3 * H * hd), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5)
    L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, hd, hd ** -0.5)
    _, _, ref = _ref(qkv, B, N, H, hd, dout)
    d = dqkv.float().view(B, N, 3, H * hd)
    r = ref.view(B, N, 3, H * hd)
    narrow = max(1.0, (64 / hd) ** 0.5)   # see test_attn_fwd
    for i, name in enumerate("qkv"):
        # P and dS are rounded to bf16 before the dV/dK/dQ GEMMs; outputs are bf16
        assert elem_err(d[:, :, i], r[:, :, i]) < 2.5e-2 * narrow, f"d{name}"
        # max|err| / rms grows with the largest element of the tensor (its own bf16 rounding is 2^-9 * max|ref|)
        half_ulp_of_max = 2.0 ** -9 * float(r[:, :, i].abs().max() / r[:, :, i].pow(2).mean().sqrt())
        assert rel_err(d[:, :, i], r[:, :, i]) < max(6e-2, 3 * half_ulp_of_max) * narrow, f"d{name}"


@pytest.mark.parametrize("hd", [48, 32, 16, 56])
@pytest.mark.parametrize("B,N,H", [(3, 197, 3), (2, 100, 2), (2, 577, 3), (40, 197, 5)])
def test_attn_narrow_heads(cuda_device, B, N, H, hd):
    """head_dim < 64 (my_vit_mini: 48, /root/reference/models/my_vit.py:85-95): same kernels, the tensor maps describe
    (head_dim, head slot, token, image) and TMA zero-fills / clips the columns up to the 64-wide tile; all three
    regimes (N <= 128, 128 < N <= 256, N > 256), forward and backward."""
    test_attn_fwd(cuda_device, B, N, H, hd)
    test_attn_bwd(cuda_device, B, N, H, hd)


@pytest.mark.parametrize("hd", [72, 80])
@pytest.mark.parametrize("B,N,H", [(3, 197, 4), (2, 100, 2), (2, 256, 3), (40, 196, 4), (1, 129, 1)])
def test_attn_wide_heads(cuda_device, B, N, H, hd):
    """64 < head_dim <= 80 (my_vit_xs: 72, /root/reference/models/my_vit.py:97-106): every operand takes a second tile
    with the head's columns 64 .. (zero from head_dim on): one more k-step for Q K^T / dO V^T, 80 accumulator columns for
    O / dV / dK / dQ.  N <= 256."""
    test_attn_fwd(cuda_device, B, N, H, hd)
    test_attn_bwd(cuda_device, B, N, H, hd)


def test_attn_unsupported_raises(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    qkv = torch.zeros(1, 16, 3 * 96, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(1, 16, 96, device=cuda_device, dtype=torch.bfloat16)
    lse = torch.zeros(1, 1, 16, device=cuda_device)
    with pytest.raises(L.VitkError):
        L.attn_fwd(qkv, out, lse, 1, 16, 1, 96, 96 ** -0.5)   # wider than a head tile plus its tail
    qkv = torch.zeros(1, 300, 3 * 72, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(1, 300, 72, device=cuda_device, dtype=torch.bfloat16)
    lse = torch.zeros(1, 1, 300, device=cuda_device)
    with pytest.raises(L.VitkError):
        L.attn_fwd(qkv, out, lse, 1, 300, 1, 72, 72 ** -0.5)   # wide heads: N <= 256
