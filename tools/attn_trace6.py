"""Timeline (SM cycles) of the second work item of CTA 0 of attn_fwd6 (unmasked N > 256): per group and kv step,
when its exps started, when P was written and when the next S was in registers with its maximum known.
usage: attn_trace6.py [B] [N] [H]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
N = int(sys.argv[2]) if len(sys.argv) > 2 else 577
H = int(sys.argv[3]) if len(sys.argv) > 3 else 16
dev = torch.device("cuda")
qkv = torch.randn(B, N, 3 * H * 64, device=dev).bfloat16()
out = torch.empty(B, N, H * 64, device=dev, dtype=torch.bfloat16)
lse = torch.empty(B, H, N, device=dev)
trace = torch.zeros(128, dtype=torch.int64, device=dev)
lib = L.load()
for _ in range(2):
    L.attn_fwd(qkv, out, lse, B, N, H, 64, 0.125)
lib.vitk_debug_set_trace(trace.data_ptr())
L.attn_fwd(qkv, out, lse, B, N, H, 64, 0.125)
torch.cuda.synchronize()
lib.vitk_debug_set_trace(None)
t = trace.cpu().tolist()
ev = []
names = ["exps start", "P written (O rescaled)", "next S in registers, max known"]
for g in (0, 1):
    for i in range(15):
        if t[16 * g + i]:
            ev.append((t[16 * g + i], f"softmax g{g}: step {i // 3} {names[i % 3]}"))
ev.sort()
t0 = ev[0][0] if ev else 0
print(f"B={B} N={N} H={H}")
for v, name in ev:
    print(f"{v - t0:8d}  {name}")
