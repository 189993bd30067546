"""Timeline (SM cycles) of items 2 and 3 of CTA 0 of the warp-specialised attention kernels for 128 < N <= 256 (attn_fwd4 /
attn_bwd4; written for their predecessors attn_fwd3 / attn_bwd3, whose exchange events stay empty).
usage: attn_trace3.py [B] [N] [H]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
N = int(sys.argv[2]) if len(sys.argv) > 2 else 197
H = int(sys.argv[3]) if len(sys.argv) > 3 else 12
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
SM = ["S ready", "max pass done", "max exchanged", "P written", "sum exchanged", "O ready", "O read, slot freed", "O stored"]
MM = ["stage full", "slot free", "S issued", "P ready", "PV issued"]
ev = []
for g in (0, 1):
    for k in (0, 1):
        for e, name in enumerate(SM):
            v = t[16 * g + 8 * k + e]
            if v:
                ev.append((v, f"softmax g{g} item {2 + k}: {name}"))
        for e, name in enumerate(MM):
            v = t[32 + 16 * g + 8 * k + e]
            if v:
                ev.append((v, f"    mma g{g} item {2 + k}: {name}"))
for g in (0, 1):
    for u in range(8):
        v = t[64 + 16 * g + u]
        if v:
            ev.append((v, f"softmax g{g} item 2:        exp unit {u} done"))
ev.sort()
t0 = ev[0][0] if ev else 0
for v, name in ev:
    print(f"{v - t0:8d}  {name}")

# ---- backward (attn_bwd3): item 2 of CTA 0 ----
dout = torch.randn(B, N, H * 64, device=dev).bfloat16()
dqkv = torch.empty_like(qkv)
for _ in range(2):
    L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, 64, 0.125)
trace.zero_()
lib.vitk_debug_set_trace(trace.data_ptr())
L.attn_bwd(qkv, out, dout, lse, dqkv, B, N, H, 64, 0.125)
torch.cuda.synchronize()
lib.vitk_debug_set_trace(None)
t = trace.cpu().tolist()
MMA = ["E1 dV0=,dP00 issued", "E2a dK1+=,dQ1+= (prev) issued", "E2b S10 issued", "E3 dK0=,dQ0=,S01 issued", "E4 dV0+=,dP10 issued",
       "E5 dV1=,dP01 issued", "E6 dK0+=,dQ1=,S11 issued", "E7 dK1=,dQ0+= issued", "E8 dV1+=,dP11 issued", "S00' issued"]
GRP = [[], []]
for j in (0, 1):
    GRP[0] += [f"S_0{j} ready", f"P_0{j} written (+deferred drain)", f"dP_0{j} ready", f"dS_0{j} written"]
    GRP[1] += [f"S_1{j} ready", f"P_1{j} written", f"dP_1{j} ready", f"dS_1{j} written", f"dK_{j} drained"]
ev = []
for i, name in enumerate(MMA):
    if t[i]:
        ev.append((t[i], f"        mma: {name}"))
for w in (0, 1):
    for i, name in enumerate(GRP[w]):
        v = t[32 + 16 * w + i]
        if v:
            ev.append((v, f"group {w}: {name}"))
ev.sort()
print("== attn_bwd3")
t0 = ev[0][0] if ev else 0
for v, name in ev:
    print(f"{v - t0:8d}  {name}")
