"""Times the GEMM shapes of one training step through the C ABI next to cuBLAS on the same shapes (CUDA events, operand
buffers rotated so that nothing sits in L2 between iterations).

usage: python tools/gemm_bench.py [D ...]            e.g.  python tools/gemm_bench.py 384 768 1024
env:   GB_M (rows, default B*N of the config), GB_ONLY (substring filter, e.g. "qkv fprop"), GB_ITERS (default 20),
       GB_NOLIB=1 (skip the cuBLAS column: for ncu captures)
The cuBLAS column is torch.matmul on the SAME operands with a plain bf16 store (no bias / GELU / residual epilogue) — a
reference point, not part of the product."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

DIMS = [int(a) for a in sys.argv[1:]] or [768]
ONLY = os.environ.get("GB_ONLY", "")
ITERS = int(os.environ.get("GB_ITERS", "20"))
NOLIB = os.environ.get("GB_NOLIB", "0") == "1"
SPLITS = int(os.environ.get("GB_SPLITS", "0"))   # force the split-K factor of the wgrad launches (0 = auto)
BN = int(os.environ.get("GB_BN", "0"))   # force the tile width of the fprop / dgrad launches (128, 192, 256; 0 = auto)
ROWS = {384: 50432, 768: 50432, 1024: 36928, 192: 50432}   # B * N of configs 2, 3, 5 (and ViT-Ti at batch 256)
dev = torch.device("cuda")
torch.manual_seed(0)
R = 3


def timed(fn):
    for _ in range(3):
        fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(ITERS):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS * 1e3   # us


def row(name, flops, fn, lib):
    if ONLY and ONLY not in name:
        return
    us = timed(fn)
    line = f"{name:36s} {us:8.1f} us {flops / us / 1e6:8.1f} TF"
    if not NOLIB and lib is not None:
        ul = timed(lib)
        line += f"   | cuBLAS plain {ul:8.1f} us {flops / ul / 1e6:8.1f} TF   vitk/cuBLAS time {us / ul:5.2f}"
    print(line, flush=True)


for D in DIMS:
    M = int(os.environ.get("GB_M", ROWS.get(D, 50432)))
    F = 4 * D
    print(f"---- D = {D}, F = {F}, M = B*N = {M}  (GB_BN={BN}, GB_SPLITS={SPLITS}) ----")
    xD = [torch.randn(M, D, device=dev).bfloat16() for _ in range(R)]
    xF = [torch.randn(M, F, device=dev).bfloat16() for _ in range(R)]
    x3 = [torch.randn(M, 3 * D, device=dev).bfloat16() for _ in range(R)]
    oF = [torch.empty(M, F, device=dev, dtype=torch.bfloat16) for _ in range(R)]
    aF = [torch.empty(M, F, device=dev, dtype=torch.bfloat16) for _ in range(R)]
    o3 = [torch.empty(M, 3 * D, device=dev, dtype=torch.bfloat16) for _ in range(R)]
    oD = [torch.empty(M, D, device=dev, dtype=torch.bfloat16) for _ in range(R)]
    rD = [torch.randn(M, D, device=dev) for _ in range(R)]
    fD = [torch.empty(M, D, device=dev) for _ in range(R)]
    Wqkv = (torch.randn(3 * D, D, device=dev) * 0.02).bfloat16()
    W1 = (torch.randn(F, D, device=dev) * 0.02).bfloat16()
    W2 = (torch.randn(D, F, device=dev) * 0.02).bfloat16()
    Wp = (torch.randn(D, D, device=dev) * 0.02).bfloat16()
    b3, bF, bD = torch.randn(3 * D, device=dev), torch.randn(F, device=dev), torch.randn(D, device=dev)
    gW1, gW2 = torch.zeros(F, D, device=dev), torch.zeros(D, F, device=dev)
    gWq, gWp = torch.zeros(3 * D, D, device=dev), torch.zeros(D, D, device=dev)
    lW1, lW2 = torch.empty(F, D, device=dev, dtype=torch.bfloat16), torch.empty(D, F, device=dev, dtype=torch.bfloat16)
    lWq, lWp = torch.empty(3 * D, D, device=dev, dtype=torch.bfloat16), torch.empty(D, D, device=dev, dtype=torch.bfloat16)
    mm = torch.matmul

    row("qkv fprop  bias -> bf16", 2 * M * 3 * D * D,
        lambda i: L.gemm(xD[i % R], Wqkv, o3[i % R], M=M, N=3 * D, K=D, epilogue=L.EPI_BF16, bias=b3, block_n=BN),
        lambda i: mm(xD[i % R], Wqkv.t(), out=o3[i % R]))
    row("proj fprop bias + resid f32", 2 * M * D * D,
        lambda i: L.gemm(xD[i % R], Wp, fD[i % R], M=M, N=D, K=D, epilogue=L.EPI_RESID, bias=bD, resid=rD[i % R], block_n=BN),
        lambda i: mm(xD[i % R], Wp.t(), out=oD[i % R]))
    row("fc1 fprop  bias + GELU (2 outs)", 2 * M * F * D,
        lambda i: L.gemm(xD[i % R], W1, oF[i % R], M=M, N=F, K=D, epilogue=L.EPI_GELU, bias=bF, aux=aF[i % R], block_n=BN),
        lambda i: mm(xD[i % R], W1.t(), out=oF[i % R]))
    row("fc2 fprop  bias + resid f32", 2 * M * F * D,
        lambda i: L.gemm(xF[i % R], W2, fD[i % R], M=M, N=D, K=F, epilogue=L.EPI_RESID, bias=bD, resid=rD[i % R], block_n=BN),
        lambda i: mm(xF[i % R], W2.t(), out=oD[i % R]))
    row("fc2 dgrad  x gelu' -> bf16", 2 * M * F * D,
        lambda i: L.gemm(xD[i % R], W2, oF[i % R], M=M, N=F, K=D, epilogue=L.EPI_DGELU, b_mn=True, aux=aF[i % R], block_n=BN),
        lambda i: mm(xD[i % R], W2, out=oF[i % R]))
    row("fc1 dgrad  -> bf16", 2 * M * F * D,
        lambda i: L.gemm(xF[i % R], W1, oD[i % R], M=M, N=D, K=F, epilogue=L.EPI_BF16, b_mn=True, block_n=BN),
        lambda i: mm(xF[i % R], W1, out=oD[i % R]))
    row("qkv dgrad  -> bf16", 2 * M * 3 * D * D,
        lambda i: L.gemm(x3[i % R], Wqkv, oD[i % R], M=M, N=D, K=3 * D, epilogue=L.EPI_BF16, b_mn=True, block_n=BN),
        lambda i: mm(x3[i % R], Wqkv, out=oD[i % R]))
    row("proj dgrad -> bf16", 2 * M * D * D,
        lambda i: L.gemm(xD[i % R], Wp, oD[i % R], M=M, N=D, K=D, epilogue=L.EPI_BF16, b_mn=True, block_n=BN),
        lambda i: mm(xD[i % R], Wp, out=oD[i % R]))
    row("fc1 wgrad  split-K red.add + bias", 2 * M * F * D,
        lambda i: L.gemm(xF[i % R], xD[i % R], gW1, M=F, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=bF, splits=SPLITS),
        lambda i: mm(xF[i % R].t(), xD[i % R], out=lW1))
    row("fc2 wgrad  split-K red.add + bias", 2 * M * F * D,
        lambda i: L.gemm(xD[i % R], xF[i % R], gW2, M=D, N=F, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=bD, splits=SPLITS),
        lambda i: mm(xD[i % R].t(), xF[i % R], out=lW2))
    row("qkv wgrad  split-K red.add + bias", 2 * M * 3 * D * D,
        lambda i: L.gemm(x3[i % R], xD[i % R], gWq, M=3 * D, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=b3, splits=SPLITS),
        lambda i: mm(x3[i % R].t(), xD[i % R], out=lWq))
    row("proj wgrad split-K red.add + bias", 2 * M * D * D,
        lambda i: L.gemm(xD[i % R], xD[(i + 1) % R], gWp, M=D, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=bD, splits=SPLITS),
        lambda i: mm(xD[i % R].t(), xD[(i + 1) % R], out=lWp))
    del xD, xF, x3, oF, aF, o3, oD, rD, fD
    torch.cuda.empty_cache()
