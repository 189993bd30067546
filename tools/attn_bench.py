"""Times the attention forward / backward kernels through the C ABI next to torch's fused SDPA (library) on the same
shapes: the three sequence lengths of the BASELINE configs by default.

usage: python tools/attn_bench.py                      (B, N, H, hd) = (256,197,12,64) (256,198,12,64) (64,577,16,64) (256,197,3,48)
       python tools/attn_bench.py B N H [hd]            one shape (head_dim 64 by default)
       ... --attn-drop P                                 with attention dropout: a keep mask [B, H, N, N] drawn with
                                                         drop probability P feeds the forward and the backward (no SDPA row)
The SDPA rows are F.scaled_dot_product_attention forward and its autograd backward on [B, H, N, hd] views of the same
qkv buffer (whichever backend torch picks on this GPU) — a reference point, not part of the product."""
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

ITERS = int(os.environ.get("GB_ITERS", "10"))
dev = torch.device("cuda")


def timed(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(ITERS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS * 1e3


def run(B, N, H, hd, p_drop=0.0):
    torch.manual_seed(0)
    scale = hd ** -0.5
    qkv = torch.randn(B, N, 3 * H * hd, device=dev).bfloat16()
    dout = torch.randn(B, N, H * hd, device=dev).bfloat16()
    out = torch.empty(B, N, H * hd, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, H, N, device=dev)
    dqkv = torch.empty_like(qkv)
    mask = (torch.rand(B, H, N, N, device=dev) >= p_drop).to(torch.uint8) if p_drop > 0 else None
    drop = dict(keep_mask=mask, keep_scale=1.0 / (1.0 - p_drop))
    f = 4.0 * B * H * N * N * hd
    fwd = timed(lambda: L.attn_fwd(qkv, out, lse, B, N, H, hd, scale, **drop))
    bwd = timed(lambda: L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, hd, scale, **drop))
    if mask is not None or os.environ.get("GB_NOSDPA", "0") == "1":
        print(f"B={B:4d} N={N:4d} H={H:3d} hd={hd:3d}{' drop %.2f' % p_drop if mask is not None else ''} | vitk fwd {fwd:7.1f} us ({f / fwd / 1e6:6.1f} TF)  bwd {bwd:7.1f} us ({2.5 * f / bwd / 1e6:6.1f} TF)", flush=True)
        return
    qkv_g = qkv.clone().requires_grad_(True)
    q, k, v = qkv_g.view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
    lib_fwd = timed(lambda: F.scaled_dot_product_attention(q, k, v))
    o = F.scaled_dot_product_attention(q, k, v)
    go = dout.view(B, N, H, hd).transpose(1, 2)

    def lib_b():
        qkv_g.grad = None
        o.backward(go, retain_graph=True)

    lib_bwd = timed(lib_b)
    print(f"B={B:4d} N={N:4d} H={H:3d} hd={hd:3d} | vitk fwd {fwd:7.1f} us ({f / fwd / 1e6:6.1f} TF)  bwd {bwd:7.1f} us ({2.5 * f / bwd / 1e6:6.1f} TF)"
          f" | torch SDPA fwd {lib_fwd:7.1f} us  bwd {lib_bwd:7.1f} us | vitk / SDPA time: fwd {fwd / lib_fwd:4.2f}  bwd {bwd / lib_bwd:4.2f}",
          flush=True)


args = sys.argv[1:]
p_drop = 0.0
if "--attn-drop" in args:
    i = args.index("--attn-drop")
    p_drop = float(args[i + 1])
    del args[i:i + 2]
if len(args) > 2:
    run(int(args[0]), int(args[1]), int(args[2]), int(args[3]) if len(args) > 3 else 64, p_drop)
else:
    for shape in ((256, 197, 12, 64), (256, 198, 12, 64), (64, 577, 16, 64), (256, 197, 6, 64), (256, 197, 3, 48)):
        run(*shape, p_drop)
