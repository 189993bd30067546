"""Where does the attention forward differ from an fp32 reference?  Prints the error of out / lse per 128-row q tile.
usage: attn_check.py B N H [hd]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_transformers_torch_xla_b200 import _lib as L  # noqa: E402

B, N, H = (int(a) for a in sys.argv[1:4])
hd = int(sys.argv[4]) if len(sys.argv) > 4 else 64
dev = torch.device("cuda")
torch.manual_seed(0)
qkv = torch.randn(B, N, 3 * H * hd, device=dev).bfloat16()
out = torch.full((B, N, H * hd), float("nan"), device=dev, dtype=torch.bfloat16)
lse = torch.full((B, H, N), float("nan"), device=dev)
L.attn_fwd(qkv, out, lse, B, N, H, hd, hd ** -0.5)
torch.cuda.synchronize()
q, k, v = qkv.float().view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)
s = (q @ k.transpose(-1, -2)) * hd ** -0.5
ref = (s.softmax(-1) @ v).transpose(1, 2).reshape(B, N, H * hd)
ref_lse = s.logsumexp(-1)
for t in range((N + 127) // 128):
    sl = slice(t * 128, min(N, t * 128 + 128))
    eo = (out[:, sl].float() - ref[:, sl]).abs()
    el = (lse[:, :, sl] - ref_lse[:, :, sl]).abs()
    print(f"q tile {t}: out max err {float(eo.max()):.4g} (nan {int(torch.isnan(eo).sum())})  lse max err {float(el.max()):.4g} (nan {int(torch.isnan(el).sum())})"
          f"  per head out err {[round(float((out[:, sl].float() - ref[:, sl]).abs().view(B, -1, H, hd)[:, :, h].max()), 4) for h in range(H)]}")
rms = ref.pow(2).mean().sqrt()
lib = torch.nn.functional.scaled_dot_product_attention(*qkv.view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)).transpose(1, 2).reshape(B, N, H * hd)
d = (out.float() - ref).abs()
print(f"max/rms {float(d.max() / rms):.4g}  (torch SDPA bf16: {float((lib.float() - ref).abs().max() / rms):.4g})  elem "
      f"{float((d / (ref.abs() + rms)).max()):.4g}  rms err {float(d.pow(2).mean().sqrt() / rms):.4g} (SDPA {float((lib.float() - ref).pow(2).mean().sqrt() / rms):.4g})"
      f"  half ulp of max / rms {float(2.0 ** -9 * ref.abs().max() / rms):.4g}")
