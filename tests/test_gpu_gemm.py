"""tcgen05 GEMM (vitk_gemm_bf16) vs a plain torch fp32 reference on the same bf16-rounded inputs.

Tolerances: fp32 outputs are fp32-accumulate checks (<= 1e-4 of the reference RMS; split-K atomics
and K=3072 accumulate-order noise included); bf16 outputs add one bf16 rounding (<= 6e-3).
"""
import pytest
import torch

from conftest import elem_err, rel_err

pytestmark = pytest.mark.gpu

F32_TOL = 2e-4
BF16_TOL = 6e-3  # elem_err: one bf16 rounding (2^-8) + accumulate-order noise


def _mk(shape, dev, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (128, 256, 128), (300, 256, 768), (256, 192, 192), (200, 128, 256),
                                   (256, 1000, 768), (1576, 576, 192), (4096, 2304, 768), (1000, 768, 3072)])
def test_fprop_f32(cuda_device, M, N, K):
    from vision_transformers_torch_xla_b200 import _lib as L
    a = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((N, K), cuda_device, 0.05, seed=2).bfloat16()
    bias = _mk((N,), cuda_device, seed=3)
    out = torch.full((M, N), float("nan"), device=cuda_device)
    L.gemm(a, w, out, M=M, N=N, K=K, epilogue=L.EPI_F32, bias=bias)
    ref = a.float() @ w.float().t() + bias
    torch.cuda.synchronize()
    assert rel_err(out, ref) < F32_TOL


@pytest.mark.parametrize("block_n", [128, 192, 256])
def test_fprop_block_n_forced(cuda_device, block_n):
    from vision_transformers_torch_xla_b200 import _lib as L
    M, N, K = 384, 768, 320
    a = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((N, K), cuda_device, 0.05, seed=2).bfloat16()
    out = torch.full((M, N), float("nan"), device=cuda_device)
    L.gemm(a, w, out, M=M, N=N, K=K, epilogue=L.EPI_F32, block_n=block_n)
    assert rel_err(out, a.float() @ w.float().t()) < F32_TOL


# bf16 outputs with 16-byte aligned rows leave through TMA as [32 rows][128 B] boxes (N = 200 / 1000: the last box of a row
# is clipped by the tensor map; M = 5000: several tiles per CTA)
@pytest.mark.parametrize("M,N,K", [(394, 768, 768), (5000, 2304, 768), (300, 200, 256), (2049, 1000, 512), (128, 64, 64)])
def test_fprop_bf16_rowscale(cuda_device, M, N, K):
    from vision_transformers_torch_xla_b200 import _lib as L
    a = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((N, K), cuda_device, 0.05, seed=2).bfloat16()
    bias = _mk((N,), cuda_device, seed=3)
    groups = (M + 196) // 197
    rs = torch.tensor([0.0, 1.25, 1.0], device=cuda_device).repeat((groups + 2) // 3)[:groups].contiguous()
    out = torch.full((M, N), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    L.gemm(a, w, out, M=M, N=N, K=K, epilogue=L.EPI_BF16, bias=bias, rowscale=rs, rows_per_group=197)
    ref = (a.float() @ w.float().t() + bias) * rs.repeat_interleave(197)[:M, None]
    assert elem_err(out.float(), ref) < BF16_TOL


def test_fprop_gelu_dual(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    M, N, K = 500, 3072, 768
    a = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((N, K), cuda_device, 0.05, seed=2).bfloat16()
    bias = _mk((N,), cuda_device, seed=3)
    out = torch.empty((M, N), device=cuda_device, dtype=torch.bfloat16)
    aux = torch.empty((M, N), device=cuda_device, dtype=torch.bfloat16)
    L.gemm(a, w, out, M=M, N=N, K=K, epilogue=L.EPI_GELU, bias=bias, aux=aux)
    h = (a.float() @ w.float().t() + bias).requires_grad_(True)
    g = torch.nn.functional.gelu(h)
    g.sum().backward()
    assert elem_err(out.float(), g) < BF16_TOL
    assert elem_err(aux.float(), h.grad) < BF16_TOL  # aux = gelu'(h)


# K <= 1536 takes the TMA residual-ring epilogue (panels prefetched across tiles, TMA stores), larger K the
# register-prefetch one; N = 200 / 1000 end in partial 32-column boxes, M = 5000 / 50432 give every CTA several tiles
@pytest.mark.parametrize("M,N,K", [(394, 768, 3072), (394, 768, 768), (5000, 768, 768), (1000, 384, 384), (300, 200, 256),
                                   (130, 1000, 512), (50432, 768, 768), (2049, 1024, 1024)])
def test_fprop_resid_scales(cuda_device, M, N, K):
    from vision_transformers_torch_xla_b200 import _lib as L
    a = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((N, K), cuda_device, 0.02, seed=2).bfloat16()
    bias = _mk((N,), cuda_device, seed=3)
    resid = _mk((M, N), cuda_device, seed=4)
    groups = (M + 196) // 197
    rs = torch.tensor([1.0 / 0.9, 0.0, 1.0], device=cuda_device).repeat((groups + 2) // 3)[:groups].contiguous()
    cs = _mk((N,), cuda_device, seed=5)
    out = torch.empty((M, N), device=cuda_device)
    L.gemm(a, w, out, M=M, N=N, K=K, epilogue=L.EPI_RESID, bias=bias, resid=resid, rowscale=rs, rows_per_group=197,
           colscale=cs)
    acc = a.float() @ w.float().t() + bias
    ref = resid + rs.repeat_interleave(197)[:M, None] * cs[None, :] * acc
    assert rel_err(out, ref) < F32_TOL
    out2 = torch.empty((M, N), device=cuda_device)
    L.gemm(a, w, out2, M=M, N=N, K=K, epilogue=L.EPI_RESID, bias=bias, resid=resid)
    assert rel_err(out2, resid + acc) < F32_TOL
    # in place on the residual stream (out is resid), the way the block forward calls it; same bits as out of place
    x = resid.clone()
    L.gemm(a, w, x, M=M, N=N, K=K, epilogue=L.EPI_RESID, bias=bias, resid=x)
    assert torch.equal(x, out2)


def test_patch_epilogue(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    Bn, P, D, K, prefix = 3, 196, 192, 768, 1
    a = _mk((Bn * P, K), cuda_device, seed=1).bfloat16()
    w = _mk((D, K), cuda_device, 0.05, seed=2).bfloat16()
    bias = _mk((D,), cuda_device, seed=3)
    pos = _mk((P + prefix, D), cuda_device, seed=4)
    out = torch.zeros((Bn, P + prefix, D), device=cuda_device)
    L.gemm(a, w, out, M=Bn * P, N=D, K=K, epilogue=L.EPI_PATCH, bias=bias, pos=pos, tokens_per_img=P, prefix=prefix)
    ref = torch.zeros_like(out)
    ref[:, prefix:] = (a.float() @ w.float().t() + bias).view(Bn, P, D) + pos[prefix:]
    assert rel_err(out, ref) < F32_TOL


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (394, 768, 2304), (500, 768, 3072), (256, 768, 1000), (300, 384, 1536)])
def test_dgrad_b_mn_major(cuda_device, M, N, K):
    """dX[M, N=in] = dY[M, K=out] @ W[K=out, N=in]: B is W itself, MN-major."""
    from vision_transformers_torch_xla_b200 import _lib as L
    dy = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((K, N), cuda_device, 0.05, seed=2).bfloat16()
    out = torch.empty((M, N), device=cuda_device, dtype=torch.bfloat16)
    L.gemm(dy, w, out, M=M, N=N, K=K, epilogue=L.EPI_BF16, b_mn=True)
    assert elem_err(out.float(), dy.float() @ w.float()) < BF16_TOL


def test_dgrad_dgelu(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    M, N, K = 394, 3072, 768
    dy = _mk((M, K), cuda_device, seed=1).bfloat16()
    w = _mk((K, N), cuda_device, 0.05, seed=2).bfloat16()
    d = _mk((M, N), cuda_device, seed=3).bfloat16()  # gelu'(h) as written by the forward EPI_GELU epilogue
    out = torch.empty((M, N), device=cuda_device, dtype=torch.bfloat16)
    L.gemm(dy, w, out, M=M, N=N, K=K, epilogue=L.EPI_DGELU, b_mn=True, aux=d)
    assert elem_err(out.float(), (dy.float() @ w.float()) * d.float()) < BF16_TOL


@pytest.mark.parametrize("M,N,K,splits", [(128, 256, 64, 1), (768, 768, 1576, 0), (2304, 768, 4000, 0), (1000, 768, 256, 0),
                                          (576, 192, 1576, 3), (768, 3072, 50432, 0)])
def test_wgrad_mn_mn_atomic(cuda_device, M, N, K, splits):
    """dW[M=out, N=in] += dY[K=tokens, M]^T @ X[K=tokens, N]; fp32 red.add with split-K."""
    from vision_transformers_torch_xla_b200 import _lib as L
    dy = _mk((K, M), cuda_device, seed=1).bfloat16()
    x = _mk((K, N), cuda_device, seed=2).bfloat16()
    init = _mk((M, N), cuda_device, seed=3)
    out = init.clone()
    bias_g = torch.full((M,), 0.5, device=cuda_device)
    L.gemm(dy, x, out, M=M, N=N, K=K, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, splits=splits, colsum=bias_g)
    ref = init + dy.float().t() @ x.float()
    assert rel_err(out, ref) < F32_TOL
    # bias gradient fused into the same kernel: column sums of dy via one extra N=16 MMA against ones
    assert rel_err(bias_g, 0.5 + dy.float().sum(0)) < F32_TOL


def test_gemm_rejects_bad_args(cuda_device):
    from vision_transformers_torch_xla_b200 import _lib as L
    a = torch.zeros((128, 64), device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros((128, 12), device=cuda_device)
    outb = torch.zeros((128, 12), device=cuda_device, dtype=torch.bfloat16)
    with pytest.raises(L.VitkError):
        L.gemm(a, a, outb, M=128, N=12, K=64, epilogue=L.EPI_BF16)  # N % 8 != 0 (only the fp32 epilogue is ragged)
    L.gemm(a, a[:12].contiguous(), out, M=128, N=12, K=64, epilogue=L.EPI_F32)
    assert float(out.abs().max()) == 0.0
    with pytest.raises(L.VitkError):
        L.gemm(a, a, out, M=0, N=16, K=64, epilogue=L.EPI_F32)  # empty


@pytest.mark.parametrize("B,C,img,ps,D", [(3, 3, 224, 16, 192), (2, 3, 384, 16, 1024), (64, 3, 224, 16, 768), (1, 3, 32, 16, 64),
                                          (5, 1, 64, 16, 128), (7, 4, 112, 16, 256)])
def test_patch_embed_image_operand(cuda_device, B, C, img, ps, D):
    """im2col-free PatchEmbed (Conv2d k = s = patch, /root/reference/models/vision_transformer.py:552-560): the bf16 NCHW
    image is the GEMM's A operand through a 4-D tensor map (rows (b, gy, gx'), the patch-grid width padded to a multiple of 8), and
    its B operand in the weight gradient.  Against the explicit im2col path (vitk_patchify + the same GEMM), which runs
    the same MMAs in the same order on the same bf16 values, and against conv2d in fp32."""
    from vision_transformers_torch_xla_b200 import _lib as L
    from vision_transformers_torch_xla_b200.ops import _patch_grid_pad
    gh = gw = img // ps
    gwp = _patch_grid_pad(gw)
    P, K, prefix = gh * gw, C * ps * ps, 1
    N = P + prefix
    x = _mk((B, C, img, img), cuda_device, seed=1)
    w = _mk((D, K), cuda_device, 0.03, seed=2).bfloat16()
    bias = _mk((D,), cuda_device, seed=3)
    pos = _mk((N, D), cuda_device, seed=4)
    xb = x.bfloat16()
    geom = (C, img, img, ps, gwp)
    out = torch.full((B, N, D), 7.0, device=cuda_device)
    L.gemm(xb, w, out, M=B * gh * gwp, N=D, K=K, epilogue=L.EPI_PATCH, bias=bias, pos=pos, tokens_per_img=P, prefix=prefix,
           image=("a",) + geom)
    patches = torch.empty((B * P, K), device=cuda_device, dtype=torch.bfloat16)
    L.patchify(x, patches, ps)
    ref = torch.full((B, N, D), 7.0, device=cuda_device)
    L.gemm(patches, w, ref, M=B * P, N=D, K=K, epilogue=L.EPI_PATCH, bias=bias, pos=pos, tokens_per_img=P, prefix=prefix)
    assert torch.equal(out[:, :prefix], ref[:, :prefix]) and float(out[:, 0].min()) == 7.0   # prefix rows untouched
    assert rel_err(out[:, prefix:], ref[:, prefix:]) < 1e-6
    conv = torch.nn.functional.conv2d(xb.float(), w.float().view(D, C, ps, ps), bias, stride=ps).flatten(2).transpose(1, 2) + pos[prefix:]
    assert rel_err(out[:, prefix:], conv) < F32_TOL
    # weight gradient: dW[D, K] += gp^T patches, gp in the padded row order (pad rows zero)
    g = _mk((B, N, D), cuda_device, seed=5)
    gp_pad = torch.full((B * gh * gwp, D), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    dpos = torch.zeros(N, D, device=cuda_device)
    L.embed_bwd(g, gp_pad, dpos, None, None, B, N, D, prefix, gw, gwp)
    v = gp_pad.view(B, gh, gwp, D)
    assert torch.equal(v[:, :, :gw].reshape(B, P, D), g[:, prefix:].bfloat16()) and float(v[:, :, gw:].float().abs().sum()) == 0.0
    dW = torch.zeros(D, K, device=cuda_device)
    db = torch.zeros(D, device=cuda_device)
    L.gemm(gp_pad, xb, dW, M=D, N=K, K=B * gh * gwp, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=db, image=("b",) + geom)
    gp = g[:, prefix:].bfloat16().reshape(B * P, D)
    want = gp.float().t() @ patches.float()
    assert rel_err(dW, want) < F32_TOL
    assert rel_err(db, gp.float().sum(0)) < F32_TOL
