"""Attention and training steps above 640 tokens (fine-tuning at 448 / 512 px), next to torch's SDPA.

usage: python tools/long_seq_bench.py [--out FILE]

Prints the card name and power limit, then
  * attention forward and backward per layer at (B, N, H) = (64, 785, 12), (32, 1025, 12), (16, 1025, 16), head_dim 64,
    without and with an attention-dropout keep mask (p = 0.1), through the C ABI (attn_fwd6 / attn_fwd_stream_kernel /
    attn_bwd_stream_kernel) and as torch SDPA on [B, H, N, hd] views of the same qkv; SDPA with dropout draws its mask
    inside the kernel (dropout_p = 0.1), so its masked row carries no mask tensor;
  * one full training step (forward, backward, AdamW) of ViT-B/16 at 448 px, B = 64, and ViT-L/16 at 512 px, B = 16, with
    drop_path 0.1 as in bench.py.
Every time is a CUDA-event mean over ITERS launches after 3 warm-up launches."""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

ITERS = int(os.environ.get("GB_ITERS", "20"))
dev = torch.device("cuda")
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


def timed(fn, iters=ITERS):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3   # us


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = "power limit unavailable (nvidia-smi)"
    return f"{name}, power limit / max SM clock: {q}"


def attention(B, N, H, hd=64, p=0.1):
    torch.manual_seed(0)
    scale = hd ** -0.5
    qkv = torch.randn(B, N, 3 * H * hd, device=dev).bfloat16()
    dout = torch.randn(B, N, H * hd, device=dev).bfloat16()
    out = torch.empty(B, N, H * hd, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, H, N, device=dev)
    dqkv = torch.empty_like(qkv)
    mask = (torch.rand(B, H, N, N, device=dev) >= p).to(torch.uint8)
    ks = 1.0 / (1.0 - p)
    f = 4.0 * B * H * N * N * hd   # forward FLOPs (backward: 2.5x)
    qkv_g = qkv.clone().requires_grad_(True)
    q, k, v = qkv_g.view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
    go = dout.view(B, N, H, hd).transpose(1, 2)
    for tag, m, dp in (("no mask", None, 0.0), ("keep mask", mask, p)):
        fwd = timed(lambda: L.attn_fwd(qkv, out, lse, B, N, H, hd, scale, keep_mask=m, keep_scale=ks))
        bwd = timed(lambda: L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, hd, scale, keep_mask=m, keep_scale=ks))
        lib_fwd = timed(lambda: F.scaled_dot_product_attention(q, k, v, dropout_p=dp))
        o = F.scaled_dot_product_attention(q, k, v, dropout_p=dp)

        def lib_b():
            qkv_g.grad = None
            o.backward(go, retain_graph=True)

        lib_bwd = timed(lib_b)
        emit(f"attn B={B:3d} N={N:5d} H={H:3d} hd={hd} {tag:9s} | vitk fwd {fwd:8.1f} us ({f / fwd / 1e6:6.1f} TF/s)  "
             f"bwd {bwd:8.1f} us ({2.5 * f / bwd / 1e6:6.1f} TF/s) | torch SDPA fwd {lib_fwd:8.1f} us  bwd {lib_bwd:8.1f} us | "
             f"vitk / SDPA time: fwd {fwd / lib_fwd:4.2f}  bwd {bwd / lib_bwd:4.2f}")
    del mask, qkv_g, o
    torch.cuda.empty_cache()


def train_step(name, img, B, iters=10):
    from vision_transformers_torch_xla_b200 import optim_factory
    from vision_transformers_torch_xla_b200.losses import SoftTargetCrossEntropy
    from vision_transformers_torch_xla_b200.models import create_model

    torch.manual_seed(0)
    model = create_model(name, num_classes=1000, global_pool="avg", drop_path_rate=0.1, img_size=img).to(dev)
    model.train()

    class Args:
        opt, lr, weight_decay, opt_eps, opt_betas = "adamw", 1e-3, 0.05, 1e-8, None

    opt = optim_factory.create_optimizer(Args, model)
    crit = SoftTargetCrossEntropy()
    x = torch.randn(B, 3, img, img, device=dev)
    y = torch.softmax(torch.randn(B, 1000, device=dev), -1)

    def step():
        loss = crit(model(x), y)
        loss.backward()
        opt.step()
        opt.zero_grad()

    ms = timed(step, iters) / 1e3
    N = model.pos_embed.shape[1]
    emit(f"train step {name} img={img} (N={N}) B={B}: {ms:8.2f} ms/step  {B / ms * 1e3:8.1f} img/s  "
         f"(peak memory {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB)")
    del model, opt, x
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the printed lines to this file")
    args = ap.parse_args()
    emit(f"card: {card()}")
    emit(f"torch {torch.__version__}, CUDA events, mean of {ITERS} launches (attention) / 10 steps (training) after 3 warm-ups")
    for shape in ((64, 785, 12), (32, 1025, 12), (16, 1025, 16)):
        attention(*shape)
    train_step("vit_base_patch16_224", 448, 64)
    train_step("vit_large_patch16_384", 512, 16)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
