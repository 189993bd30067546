"""Every LayerNorm kernel of csrc/vitk_norm.cu and every kernel of csrc/vitk_elementwise.cu against a float64 reference,
at the shapes and inputs where such kernels go wrong.

LayerNorm.  Each row of ``LN_TABLE`` names the instantiation it must launch as (kind, V, EXACT): ``fwd`` is
``ln_fwd_kernel<V, EXACT>``, ``bwd`` the register-resident ``ln_bwd_kernel<V, false>`` and ``ring`` the shared-memory
ring ``ln_bwd_ring_kernel<V, EXACT>``.  V is the number of float4 vectors per lane (2, 3, 4, 6 or 8) and EXACT means
dim == 128 V, where the column guards are compiled out.  The row runs once under ``torch.profiler``, and the test asserts
that exactly one LayerNorm kernel ran and that it is the row's.  Rows cover:
  * widths: one exact and several inexact widths per V, and the model widths 192 / 288 / 384 / 768 / 1024 buckets;
  * rows 1, 7, 8, 9 (a partial last CTA of 8 warps), 4095 / 4096 / 4097 (the ring threshold), and for the ring
    148 * warps * 5 + 5 rows, so that every warp of a full grid takes at least 5 rows and its 2-stage ring wraps twice;
  * rows with dim % 8 == 4, or ld_dy % 8 == 4, at 4096 rows and more: these must stay on the register kernel;
  * g_in present, absent and equal to g_out; gb_out with a rowscale that has a zero group and rows_per_group not
    dividing rows; dgamma / dbeta accumulating into non-zero values, or NULL; row pitches past dim with NaN in the pad;
    mean / rstd NULL in the forward;
  * ordinary rows, rows whose mean is 10^3 times their standard deviation, constant rows (variance 0, rstd = eps^-1/2)
    and rows scaled by 1e-3 and 1e3.
The backward gets fp32 mean / rstd and bf16 dy as inputs, and the reference uses exactly those values, so the backward
is checked on its own and not through the forward's rounding.

Layout.  Every output is a view into a buffer with a guard row before and after (``guarded`` of
test_gpu_gemm_kernels.py), and pitched outputs have guard columns in their pitch.  What a launch may write starts as NaN
(or as the value it accumulates into); everything else holds a sentinel that must come back bit for bit.

Bounds.  U = 2^-23.  A sum computed as a tree in which no term passes more than h additions is off by at most
h U sum|t| (each addition rounds with a relative error below 2^-24, so h U leaves a factor 2 for the products folded
into the terms).  An element passes when |out - ref| <= (1 + c)(n U mag + extra) + c |ref|, with c = U for fp32 and
c = 2^-8 for bf16 outputs (one rounding to 8 significant bits), and the repository's max/rms <= 2e-4 (fp32) and
elem <= 6e-3 (bf16) metrics hold as well, except max/rms on the cross-entropy gradient: with up to 4096 classes and
logits of scale 30 a row's probability sits on a few classes, the RMS of dlogits is far below its largest elements, and
the __expf error of those elements alone reaches 4e-4 of that RMS on a B200.
  * LayerNorm forward.  A lane adds its 4V terms in V + 2 levels, and the warp shuffle adds 5 more: h = V + 7.  With
    A1 = sum|x|, m and v the exact mean and variance, r = x - m and R = (v + eps)^-1/2:
        e_mu  = h U A1 / D + U |m|                                   (sum, then one division)
        e_q   = D e_mu^2 + (h + 3) U sum (|r| + e_mu)^2              (sum of (x - mu)^2 about the kernel's mu)
        e_var = e_q / D + U (v + e_q / D),   e_t = e_var + U (v + eps + e_var)
        e_R   = 1.01 * R^3 e_t / 2 + 2 U R                           (first order in e_t; rsqrtf is off by <= 2 ulp)
        e_xh  = (e_mu + U (|r| + e_mu)) (R + e_R) + |r| e_R + U |xhat|
    mean is checked against e_mu, rstd against e_R, y against extra = |gamma| e_xh + U |y| (the fma) and c = 2^-8.
  * LayerNorm backward, with a = dy gamma, xhat = (x - mu) rstd from the given mu / rstd (off by <= 3 U |xhat| in
    the kernel), c1 = sum a / D, c2 = sum a xhat / D:
        e_c1 = (h + 3) U sum|a| / D,   e_c2 = (h + 7) U sum|a xhat| / D
        e_t  = e_c1 + |xhat| e_c2 + 6 U (|a| + |c1| + |xhat c2|)     (a - c1 - xhat c2, three roundings)
    g_out = rstd (a - c1 - xhat c2) + g_in has extra = rstd e_t + U |g_out|; gb_out = bf16(s g_out) has
    extra = |s| (rstd e_t + U |g_out|) + U |s g_out| and c = 2^-8.
  * dgamma / dbeta: init + a sum over the rows, added in an order the atomics decide: n = rows + 5 with
    mag = |init| + sum|dy xhat| (the 3 U error of xhat and the fma are in the 5), and n = rows + 1 with
    mag = |init| + sum|dy|.
  * Cross-entropy: __expf(x) is off by at most (2 + 1.173 |x|) ulp and __logf(x) by 2^-21.41 on [0.5, 2], 3 ulp
    elsewhere (CUDA C Programming Guide, intrinsic functions).  Each exponential also carries the error of its argument,
    and results below 2^-126 may flush to 0.  The block reduction adds a thread's 16 terms, then 5 shuffle levels, then
    8 warp partials: h = 28.  ``ce_reference`` carries these first-order errors through the log-sum-exp, the
    per-row loss, the batch mean (n = B + 1) and the gradient.
  * AdamW: a float64 evaluation of the kernel's formula on the fp32 hyperparameters and the fp32 bias corrections the
    host computes in double and rounds once.  Every fp32 operation of the kernel adds one relative U to the bound of
    its result (``adamw_reference``).  shadow must be bf16(p) bit for bit.
  * colsum, embed_bwd's dpos / dprefix, pool_fwd (mode 0): init + a sum of rows terms in any order, n = rows + 2.
  * Single roundings and copies are checked bit for bit against the same roundings done by torch on the CPU side of the
    reference: patchify (bf16 of F.unfold), gp = bf16(g), prefix_rows, scale_cast / rowscale_cast / colscale,
    scale_f32, pool_fwd in mode 1, pool_bwd in mode 1.
On the CPU, ``test_checker_rejects_a_subtly_wrong_result`` shows that these checks reject a LayerNorm variance divided
by D - 1, a last partial column group left at its NaN fill, a dgamma missing one row, a rowscale group off by one row, a
cross-entropy over C - 1 classes, an AdamW bias correction one step off and one changed guard element.  And
``test_every_kernel_is_accounted_for`` checks that every kernel these two files put into libvitk.so is named by a row,
covered by a named test elsewhere, or exempt for a stated reason, so a kernel added later without one fails on any
machine.
"""
import ctypes
import math
import os
import re
import shutil
import subprocess
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

from conftest import report
from test_gpu_gemm_kernels import SENTINEL, U23, Guarded, check, guarded  # noqa: F401  (Guarded: the type of outputs)

U = U23
C_BF16 = 2.0 ** -8
EPS = float(torch.tensor(1e-6, dtype=torch.float32))   # the binding passes eps as a C float
NUM_SMS = 148                                           # B200; only sizes the ring rows, any count is correct
LN_RS_PATTERN = (1.25, 0.0, 1.0 / 0.9)                  # per-sample DropPath scales with a dropped group


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _randn(shape, seed, scale=1.0, dev="cpu"):
    return (torch.randn(shape, generator=_gen(seed), dtype=torch.float64) * scale).float().to(dev)


def _padded(logical, ld, dev, fill=float("nan")):
    rows, cols = logical.shape
    st = torch.full((rows, ld), fill, dtype=logical.dtype, device=dev)
    st[:, :cols] = logical.to(dev)
    return st


def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


# ---------------------------------------------------------------------------------------------------------------------
# LayerNorm table
# ---------------------------------------------------------------------------------------------------------------------
def vbucket(dim):
    v = -(-dim // 128)
    return next(b for b in (2, 3, 4, 6, 8) if v <= b)


def ring_warps(dim):
    """ring_warps() of vitk_norm.cu: the most warps whose 2-stage rings fit 226 KB of shared memory."""
    wmax = 16 if dim <= 512 else 12 if dim <= 768 else 8
    for w in range(wmax, 0, -1):
        if (8 * dim + w * 32 + 127) // 128 * 128 + w * 2 * 10 * dim <= 227 * 1024 - 1024:
            return w
    return 0


@dataclass(frozen=True)
class LnCase:
    kernel: tuple          # (kind, V, EXACT)
    rows: int
    dim: int
    shift: int = 0         # input pattern of row 0 (row r has pattern (r + shift) % 5)
    pitch: bool = False    # ld_x / ld_y / ld_dy / ld_g past dim, with NaN in the input pads
    stats: bool = True     # fwd: mean / rstd written
    g_in: str = "none"     # bwd: none | sep | inplace
    gb: bool = False       # bwd: gb_out written
    rowscale: bool = False
    dgb: bool = True       # bwd: dgamma / dbeta accumulated
    ld_dy4: bool = False   # bwd: ld_dy % 8 == 4

    @property
    def kind(self):
        return self.kernel[0]

    @property
    def ld_x(self):
        return self.dim + 12 if self.pitch else self.dim

    @property
    def ld_y(self):
        return self.dim + 8 if self.pitch else self.dim

    @property
    def ld_dy(self):
        return self.dim + 4 if self.ld_dy4 else self.dim + 8 if self.pitch else self.dim

    @property
    def ld_g(self):
        return self.dim + 4 if self.pitch else self.dim

    @property
    def rpg(self):
        return 5 if self.rows < 64 else 197

    @property
    def id(self):
        k, v, ex = self.kernel
        f = [f"{k}{v}{'T' if ex else 'F'}", f"{self.rows}x{self.dim}", f"p{self.shift % 5}"]
        if self.pitch:
            f.append("pitch")
        if k == "fwd":
            f.append("stats" if self.stats else "nostats")
        else:
            f += [f"gin-{self.g_in}"] + (["gb"] if self.gb else []) + (["rs"] if self.rowscale else []) + \
                 (["dgb"] if self.dgb else []) + (["lddy4"] if self.ld_dy4 else [])
        return "-".join(f)


FWD_WIDTHS = (4, 144, 256, 260, 288, 384, 388, 508, 512, 516, 640, 764, 768, 772, 1020, 1024)
RING_WIDTHS = (144, 256, 288, 384, 504, 512, 640, 768, 1016, 1024)   # dim % 8 == 0; 504 and 1016 reach <4,F> / <8,F>


def _bwd_opts(i):
    return dict(g_in=("sep", "none", "inplace")[i % 3], gb=i % 4 != 3, rowscale=i % 2 == 0, dgb=i % 5 != 4,
                pitch=i % 3 == 1)


def _ln_table():
    rows = []
    k = 0
    for dim in FWD_WIDTHS:
        v = vbucket(dim)
        for r in (1, 7, 8, 9, 4095, 4096, 4097):
            rows.append(LnCase(("fwd", v, dim == 128 * v), r, dim, shift=k, pitch=k % 2 == 1, stats=k % 3 != 2))
            k += 1
    for dim in FWD_WIDTHS:
        v = vbucket(dim)
        counts = (1, 7, 8, 9, 4095) + ((4096, 4097) if dim % 8 == 4 else ())
        for r in counts:
            rows.append(LnCase(("bwd", v, False), r, dim, shift=k, **_bwd_opts(k)))
            k += 1
        if dim % 8 == 0:   # a bf16 dy pitch that is only 8-byte aligned keeps the call off the bulk copies
            rows.append(LnCase(("bwd", v, False), 4097, dim, shift=k, ld_dy4=True, **dict(_bwd_opts(k), pitch=False)))
            k += 1
    for dim in RING_WIDTHS:
        v = vbucket(dim)
        for r in (4096, 4097, NUM_SMS * ring_warps(dim) * 5 + 5):
            rows.append(LnCase(("ring", v, dim == 128 * v), r, dim, shift=k, **_bwd_opts(k)))
            k += 1
    return rows


LN_TABLE = _ln_table()


def ln_inputs(case, dev, seed=0):
    """x [rows, dim] fp32 with the five row patterns, gamma / beta, and for the backward dy (bf16), g_in, the fp32
    statistics of x, the rowscale and the dgamma / dbeta starting values."""
    R, D = case.rows, case.dim
    base = _randn((R, D), seed + 1, 1.0, dev)
    pat = ((torch.arange(R, device=dev) + case.shift) % 5)[:, None]
    x = torch.where(pat == 1, base + 1000.0, base)
    x = torch.where(pat == 2, torch.full_like(base, 3.25), x)          # 3.25 * D sums exactly: variance 0
    x = torch.where(pat == 3, base * 1e-3, x)
    x = torch.where(pat == 4, base * 1e3, x)
    ops = dict(x=x, gamma=(1.0 + _randn((D,), seed + 2, 0.2, dev)), beta=_randn((D,), seed + 3, 0.2, dev))
    if case.kind != "fwd":
        x64 = x.double()
        m = x64.mean(1)
        ops["mean"] = m.float()
        ops["rstd"] = (1.0 / torch.sqrt(((x64 - m[:, None]) ** 2).mean(1) + EPS)).float()
        ops["dy"] = _randn((R, D), seed + 4, 1.0, dev).bfloat16()
        if case.g_in != "none":
            ops["g_in"] = _randn((R, D), seed + 5, 1.0, dev)
        if case.rowscale:
            groups = -(-R // case.rpg)
            ops["rs"] = torch.tensor([LN_RS_PATTERN[g % 3] for g in range(groups)], dtype=torch.float32, device=dev)
        if case.dgb:
            ops["dgamma0"] = _randn((D,), seed + 6, 3.0, dev)
            ops["dbeta0"] = _randn((D,), seed + 7, 3.0, dev)
    return ops


def ln_fwd_reference(case, ops, var_div=None):
    """{name: (ref, mag, n, extra, c)}; ``var_div`` replaces the divisor of the variance (checker self-test only)."""
    x = ops["x"].double()
    D = case.dim
    h = case.kernel[1] + 7
    m = x.mean(1, keepdim=True)
    r = x - m
    v = (r * r).sum(1, keepdim=True) / (var_div or D)
    R = 1.0 / torch.sqrt(v + EPS)
    xh = r * R
    g, b = ops["gamma"].double(), ops["beta"].double()
    y = xh * g + b
    e_mu = h * U * x.abs().sum(1, keepdim=True) / D + U * m.abs()
    e_q = D * e_mu ** 2 + (h + 3) * U * ((r.abs() + e_mu) ** 2).sum(1, keepdim=True)
    e_var = e_q / D + U * (v + e_q / D)
    e_t = e_var + U * (v + EPS + e_var)
    e_R = 1.01 * R ** 3 * e_t / 2 + 2 * U * R
    e_xh = (e_mu + U * (r.abs() + e_mu)) * (R + e_R) + r.abs() * e_R + U * xh.abs()
    res = {"y": (y, 0.0, 0, g.abs() * e_xh + U * y.abs(), C_BF16)}
    if case.stats:
        res["mean"] = (m.flatten(), 0.0, 0, e_mu.flatten(), U)
        res["rstd"] = (R.flatten(), 0.0, 0, e_R.flatten(), U)
    return res


def ln_bwd_reference(case, ops, rs_rows=None, drop_row=None):
    """{name: (ref, mag, n, extra, c)}; ``rs_rows`` / ``drop_row`` perturb the reference (checker self-test only)."""
    D = case.dim
    h = case.kernel[1] + 7
    x, dy = ops["x"].double(), ops["dy"].double()
    mu, R = ops["mean"].double()[:, None], ops["rstd"].double()[:, None]
    g = ops["gamma"].double()
    xh = (x - mu) * R
    a = dy * g
    c1 = a.sum(1, keepdim=True) / D
    c2 = (a * xh).sum(1, keepdim=True) / D
    gi = ops["g_in"].double() if "g_in" in ops else torch.zeros((), dtype=torch.float64, device=x.device)
    go = R * (a - c1 - xh * c2) + gi
    e_c1 = (h + 3) * U * a.abs().sum(1, keepdim=True) / D
    e_c2 = (h + 7) * U * (a * xh).abs().sum(1, keepdim=True) / D
    e_t = e_c1 + xh.abs() * e_c2 + 6 * U * (a.abs() + c1.abs() + (xh * c2).abs())
    e_go = R * e_t + U * go.abs()
    res = {"g_out": (go, 0.0, 0, e_go, U)}
    if case.gb:
        if rs_rows is None:
            rs_rows = ops["rs"].double()[torch.arange(case.rows, device=x.device) // case.rpg] if case.rowscale else \
                torch.ones(case.rows, dtype=torch.float64, device=x.device)
        s = rs_rows[:, None]
        res["gb_out"] = (s * go, 0.0, 0, s.abs() * e_go + U * (s * go).abs(), C_BF16)
    if case.dgb:
        keep = torch.ones((case.rows, 1), dtype=torch.float64, device=x.device)
        if drop_row is not None:
            keep[drop_row] = 0.0
        g0, b0 = ops["dgamma0"].double(), ops["dbeta0"].double()
        res["dgamma"] = (g0 + (keep * dy * xh).sum(0), g0.abs() + (dy * xh).abs().sum(0), case.rows + 5, 0.0, U)
        res["dbeta"] = (b0 + (keep * dy).sum(0), b0.abs() + dy.abs().sum(0), case.rows + 1, 0.0, U)
    return res


def ln_outputs(case, ops, dev):
    R, D = case.rows, case.dim
    o = {}
    if case.kind == "fwd":
        o["y"] = guarded(R, D, case.ld_y, torch.bfloat16, dev)
        if case.stats:
            o["mean"] = guarded(1, R, R, torch.float32, dev)
            o["rstd"] = guarded(1, R, R, torch.float32, dev)
        return o
    o["g_out"] = guarded(R, D, case.ld_g, torch.float32, dev, ops["g_in"] if case.g_in == "inplace" else float("nan"))
    if case.gb:
        o["gb_out"] = guarded(R, D, D, torch.bfloat16, dev)
    if case.dgb:
        o["dgamma"] = guarded(1, D, D, torch.float32, dev, ops["dgamma0"][None, :])
        o["dbeta"] = guarded(1, D, D, torch.float32, dev, ops["dbeta0"][None, :])
    return o


def verify(label, outs, res, no_rms=()):
    """check() of test_gpu_gemm_kernels.py on every output; returns (failures, {name: worst |err| / bound}).  Outputs
    named in ``no_rms`` are held to their element bound alone, without the max/rms metric."""
    fails, margins = [], {}
    for name, (ref, mag, n, extra, c) in res.items():
        g = outs[name]
        ref = ref.reshape(g.rows, g.cols)
        f64 = dict(dtype=torch.float64, device=ref.device)
        f, margin = check(f"{label}:{name}", g, g.index(), ref, torch.as_tensor(mag, **f64).expand_as(ref), n,
                          torch.as_tensor(extra, **f64).expand_as(ref), c)
        if name in no_rms:
            f = [x for x in f if ": max/rms " not in x]
        fails += f
        margins[name] = margin
    return fails, margins


def exact(ref):
    """A result the kernel must produce bit for bit."""
    return (ref.double(), 0.0, 0, 0.0, 0.0)


# ---------------------------------------------------------------------------------------------------------------------
# Kernel names: "ln_fwd_kernel<6, false>", "ln_fwd_kernel<(int)6, (bool)0>" or mangled "ln_fwd_kernelILi6ELb0E"
# ---------------------------------------------------------------------------------------------------------------------
_LN_DEMANGLED = re.compile(r"\b(ln_fwd_kernel|ln_bwd_kernel|ln_bwd_ring_kernel)<([^<>]*)>")
_LN_MANGLED = re.compile(r"(ln_fwd_kernel|ln_bwd_kernel|ln_bwd_ring_kernel)ILi(\d+)ELb([01])E")
_KIND = {"ln_fwd_kernel": "fwd", "ln_bwd_kernel": "bwd", "ln_bwd_ring_kernel": "ring"}


def _targ(tok):
    tok = re.sub(r"^\([a-z ]+\)", "", tok.strip())
    return {"true": 1, "false": 0}[tok] if tok in ("true", "false") else int(tok)


def ln_kernels(text):
    """Every LayerNorm kernel named in `text`, as (kind, V, EXACT) with EXACT a bool."""
    found = []
    for m in _LN_DEMANGLED.finditer(text):
        a = [_targ(t) for t in m.group(2).split(",")]
        found.append((_KIND[m.group(1)], a[0], bool(a[1])))
    for m in _LN_MANGLED.finditer(text):
        found.append((_KIND[m.group(1)], int(m.group(2)), m.group(3) == "1"))
    return found


# ---------------------------------------------------------------------------------------------------------------------
# Cross-entropy and AdamW references (device-agnostic)
# ---------------------------------------------------------------------------------------------------------------------
H_CE = 28
F32_MIN = 2.0 ** -126


def _exp_err(e, arg, arg_err):
    """Bound of |__expf(arg') - exp(arg)| where arg' is off by arg_err (first order, 1 % for the rest)."""
    return 1.01 * e * ((2 + 1.173 * arg.abs() + 1) * U + arg_err) + F32_MIN


def _log_err(s, s_err):
    near = (s >= 0.5) & (s <= 2.0)
    return 1.01 * s_err / s + torch.where(near, torch.full_like(s, 2.0 ** -21.41), 3 * U * torch.log(s).abs())


@dataclass(frozen=True)
class CeCase:
    B: int
    C: int
    mode: str           # hard | smooth | soft | kd
    scale: float = 1.0
    T: float = 1.0
    alpha: float = 0.0

    @property
    def id(self):
        extra = f"-T{self.T:g}-a{self.alpha:g}" if self.mode == "kd" else ""
        return f"B{self.B}-C{self.C}-{self.mode}-s{self.scale:g}{extra}"


def _ce_table():
    modes = [dict(mode="hard"), dict(mode="smooth"), dict(mode="soft"), dict(mode="kd", T=1.0, alpha=0.7),
             dict(mode="kd", T=4.0, alpha=1.0), dict(mode="kd", T=4.0, alpha=0.0), dict(mode="kd", T=1.0, alpha=1.0)]
    rows, k = [], 0
    for C in (1, 2, 255, 256, 257, 1000, 4095, 4096):
        for B in (1, 256, 257, 1000):
            rows.append(CeCase(B, C, scale=(1.0, 5.0, 30.0)[k % 3], **modes[k % len(modes)]))
            k += 1
    return rows


CE_TABLE = _ce_table()


def ce_inputs(case, dev, seed=0):
    B, C = case.B, case.C
    x = _randn((B, C), seed + 1, case.scale, dev)
    x[0, (7 * seed + 3) % C] += 80.0                                   # one row with a +80 outlier
    ops = dict(logits=x)
    if case.mode in ("hard", "smooth"):
        lab = torch.randint(0, C, (B,), generator=_gen(seed + 2))
        lab[0], lab[-1] = 0, C - 1
        ops["labels"] = lab.to(dev)
        ops["smoothing"] = 0.1 if case.mode == "smooth" else 0.0
    else:
        t = torch.rand((B, C), generator=_gen(seed + 3), dtype=torch.float64)
        t = torch.where(t < 0.3, torch.zeros_like(t), t)                # exact zeros
        t[:, 0] += 1e-3
        ops["soft"] = (t / t.sum(1, keepdim=True)).float().to(dev)
        ops["smoothing"] = 0.0
    if case.mode == "kd":
        ops["teacher"] = _randn((B, C), seed + 4, case.scale, dev)
    return ops


def ce_targets(case, ops):
    """The fp32 targets the kernel forms: the soft targets, or off = s / C, on = 1 - s + off in fp32."""
    if "soft" in ops:
        return ops["soft"]
    s = torch.tensor(ops["smoothing"], dtype=torch.float32)
    off = s / case.C
    on = (1.0 - s) + off
    t = torch.full((case.B, case.C), float(off), dtype=torch.float32, device=ops["logits"].device)
    t[torch.arange(case.B, device=t.device), ops["labels"]] = float(on)
    return t


def ce_reference(case, ops, classes=None):
    """{loss, dlogits}; ``classes`` < C evaluates a kernel that misses the last classes (checker self-test only)."""
    C = classes or case.C
    x = ops["logits"].double()[:, :C]
    t = ce_targets(case, ops).double()[:, :C]
    B = case.B
    mx = x.max(1, keepdim=True).values
    e = torch.exp(x - mx)
    se = e.sum(1, keepdim=True)
    d_se = _exp_err(e, x - mx, U * (x - mx).abs()).sum(1, keepdim=True) + H_CE * U * se
    lse = mx + torch.log(se)
    d_lse = _log_err(se, d_se) + U * lse.abs()
    base = -(t * (x - lse)).sum(1, keepdim=True)
    d_base = t.abs().sum(1, keepdim=True) * d_lse + (H_CE + 2) * U * (t * (x - lse)).abs().sum(1, keepdim=True)
    tsum = t.sum(1, keepdim=True)
    d_tsum = H_CE * U * t.abs().sum(1, keepdim=True)
    p = torch.exp(x - lse)
    d_p = _exp_err(p, x - lse, d_lse + U * (x - lse).abs())
    gb = (p * tsum - t) / B
    d_gb = ((d_p * tsum + p * d_tsum) + 2 * U * (p * tsum).abs() + U * (p * tsum - t).abs()) / B + 2 * U * gb.abs()
    if case.mode == "kd":
        T, a = case.T, case.alpha
        z = ops["teacher"].double()[:, :C] / T
        d_z = 2 * U * z.abs()
        zmx = z.max(1, keepdim=True).values
        ez = torch.exp(z - zmx)
        zs = ez.sum(1, keepdim=True)
        d_zs = _exp_err(ez, z - zmx, 2 * d_z + U * (z - zmx).abs()).sum(1, keepdim=True) + H_CE * U * zs
        lse_t = zmx + torch.log(zs)
        d_lse_t = _log_err(zs, d_zs) + d_z.max(1, keepdim=True).values + U * lse_t.abs()
        xs = (x - mx) / T
        es = torch.exp(xs)
        ss = es.sum(1, keepdim=True)
        d_ss = _exp_err(es, xs, 3 * U * xs.abs()).sum(1, keepdim=True) + H_CE * U * ss
        lse_s = mx / T + torch.log(ss)
        d_lse_s = _log_err(ss, d_ss) + 3 * U * (mx / T).abs() + U * lse_s.abs()
        lpt, lps = z - lse_t, x / T - lse_s
        d_lpt = d_z + d_lse_t + U * lpt.abs()
        d_lps = 2 * U * (x / T).abs() + d_lse_s + U * lps.abs()
        pt, ps = torch.exp(lpt), torch.exp(lps)
        d_pt, d_ps = _exp_err(pt, lpt, d_lpt), _exp_err(ps, lps, d_lps)
        kd = (pt * (lpt - lps)).sum(1, keepdim=True)
        d_kd = (d_pt * (lpt - lps).abs() + pt * (d_lpt + d_lps)).sum(1, keepdim=True) + \
            (H_CE + 3) * U * (pt * (lpt - lps)).abs().sum(1, keepdim=True)
        row = (1 - a) * base + a * T * T * kd
        d_row = (1 - a) * d_base + a * T * T * d_kd + 3 * U * ((1 - a) * base.abs() + a * T * T * kd.abs())
        dl = (1 - a) * gb + a * T * (ps - pt) / B
        d_dl = (1 - a) * d_gb + a * T * ((d_ps + d_pt) + U * (ps - pt).abs()) / B + \
            4 * U * ((1 - a) * gb.abs() + a * T * (ps - pt).abs() / B)
    else:
        row, d_row, dl, d_dl = base, d_base, gb, d_gb
    loss = row.sum() / B
    d_loss = d_row.sum() / B + (B + 1) * U * row.abs().sum() / B
    if C < case.C:   # what a kernel that skips the last classes would write there
        dl = torch.cat([dl, torch.zeros((B, case.C - C), dtype=torch.float64, device=dl.device)], 1)
        d_dl = torch.cat([d_dl, torch.zeros_like(dl[:, C:])], 1)
    return {"loss": (loss.reshape(1), 0.0, 0, d_loss.reshape(1), U), "dlogits": (dl, 0.0, 0, d_dl, U)}


@dataclass(frozen=True)
class AdamwCase:
    n: int
    groups: int
    chunk: int
    step: int
    g16: bool = False
    zero_grad: bool = False
    ema: bool = True
    shadow: bool = True

    @property
    def id(self):
        f = [f"n{self.n}", f"g{self.groups}c{self.chunk}", f"step{self.step}"]
        f += [nm for nm, on in (("g16", self.g16), ("zero", self.zero_grad), ("ema", self.ema), ("shadow", self.shadow))
              if on]
        return "-".join(f)


ADAMW_TABLE = [AdamwCase(n, *gc, step, g16=(i % 2 == 1), zero_grad=(i % 3 != 0), ema=(i % 4 != 3), shadow=(i % 5 != 4))
               for i, (n, gc, step) in enumerate((n, gc, s) for n in (4, 1020, 1024, 1028)
                                                 for gc in ((8, 4), (3, 12), (1, 0)) for s in (1, 2, 1000))]
ADAMW_HYPER = dict(beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=0.5, ema_decay=0.99)


def adamw_inputs(case, dev, seed=0):
    n = case.n
    ops = dict(p=_randn((n,), seed + 1, 1.0, dev), m=_randn((n,), seed + 3, 0.1, dev),
               v=_randn((n,), seed + 4, 0.01, dev).abs(), ema=_randn((n,), seed + 5, 1.0, dev))
    g = _randn((n,), seed + 2, 1.0, dev)
    g[: min(n, 4)] = 0.0                                                # v' = b2 v exactly where g = 0
    ops["g"] = g
    if case.g16:
        ops["g16"] = _randn((n,), seed + 6, 1.0, dev).bfloat16()
        ops["gsd"] = torch.tensor([0.75], dtype=torch.float32, device=dev)
    if case.chunk:
        chunks = -(-n // case.chunk)
        ops["cg"] = (torch.arange(chunks) % case.groups).to(torch.uint8).to(dev)
    ops["lrs"] = [1e-3 * (1 + gi) for gi in range(case.groups)]
    ops["wds"] = [0.05 * (gi % 3) for gi in range(case.groups)]
    return ops


def _f32(v):
    return float(torch.tensor(v, dtype=torch.float32))


def adamw_reference(case, ops, step=None):
    """The kernel's formula in float64; ``step`` other than case.step is for the checker self-test only."""
    step = step or case.step
    hp = {k: _f32(v) for k, v in ADAMW_HYPER.items()}
    b1, b2, eps = hp["beta1"], hp["beta2"], hp["eps"]
    inv_bc1 = _f32(1.0 / (1.0 - b1 ** step))
    inv_sqrt_bc2 = _f32(1.0 / math.sqrt(1.0 - b2 ** step))
    dev = ops["p"].device
    n = case.n
    grp = (torch.arange(n, device=dev) // case.chunk).clamp_max(ops["cg"].numel() - 1) if case.chunk else None
    gidx = ops["cg"].long()[grp] if case.chunk else torch.zeros(n, dtype=torch.long, device=dev)
    lr = torch.tensor([_f32(x) for x in ops["lrs"]], dtype=torch.float64, device=dev)[gidx]
    wd = torch.tensor([_f32(x) for x in ops["wds"]], dtype=torch.float64, device=dev)[gidx]
    if case.g16:
        G, gs, k_gs = ops["g16"].double(), hp["grad_scale"] * float(ops["gsd"][0]), 2
    else:
        G, gs, k_gs = ops["g"].double(), hp["grad_scale"], 1
    P, M, V = ops["p"].double(), ops["m"].double(), ops["v"].double()
    gg = G * gs
    e_gg = (k_gs + 1) * U * gg.abs()
    decay = 1.0 - lr * wd
    P1 = P * decay
    e_P1 = 4 * U * P.abs()
    M1 = b1 * M + (1 - b1) * gg
    e_M1 = 3 * U * ((b1 * M).abs() + ((1 - b1) * gg).abs()) + (1 - b1) * e_gg
    V1 = b2 * V + (1 - b2) * gg * gg
    e_V1 = 4 * U * ((b2 * V).abs() + (1 - b2) * gg * gg) + (1 - b2) * 2 * gg.abs() * e_gg * 1.01
    sq = torch.sqrt(V1)
    e_sq = torch.minimum(e_V1 / (2 * sq).clamp_min(1e-300), torch.sqrt(e_V1)) + U * sq
    den = sq * inv_sqrt_bc2 + eps
    e_den = inv_sqrt_bc2 * e_sq + 2 * U * den
    q = M1 / den
    e_q = 1.01 * (e_M1 / den + M1.abs() * e_den / den ** 2) + U * q.abs()
    st = lr * inv_bc1
    P2 = P1 - st * q
    e_P2 = e_P1 + st * (e_q + 2 * U * q.abs()) + U * P2.abs()
    res = {"p": (P2, 0.0, 0, e_P2, U), "m": (M1, 0.0, 0, e_M1, U), "v": (V1, 0.0, 0, e_V1, U)}
    if case.ema:
        d = hp["ema_decay"]
        E = ops["ema"].double()
        E1 = d * E + (1 - d) * P2
        res["ema"] = (E1, 0.0, 0, (1 - d) * e_P2 + 3 * U * ((d * E).abs() + ((1 - d) * P2).abs()), U)
    res["g"] = exact(torch.zeros_like(G) if case.zero_grad else ops["g"])
    return res


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def test_ln_table_rows_are_well_formed():
    """Each row reaches its kernel by the dispatch rule of vitk_layernorm_fwd / _bwd, and every instantiation has rows."""
    for c in LN_TABLE:
        kind, v, ex = c.kernel
        assert v == vbucket(c.dim) and c.dim % 4 == 0 and c.dim <= 1024, c.id
        ring = c.rows >= 4096 and c.dim % 8 == 0 and c.ld_dy % 8 == 0
        if kind == "fwd":
            assert ex == (c.dim == 128 * v), c.id
        elif kind == "bwd":
            assert not ex and not ring, c.id
        else:
            assert ring and ex == (c.dim == 128 * v), c.id
    ids = [c.id for c in LN_TABLE]
    assert len(set(ids)) == len(ids)
    named = {c.kernel for c in LN_TABLE}
    want = {(k, v, e) for k in ("fwd", "ring") for v in (2, 3, 4, 6, 8) for e in (False, True)} | \
        {("bwd", v, False) for v in (2, 3, 4, 6, 8)}
    assert named == want
    for c in LN_TABLE:   # every ring warp wraps twice in the largest row count of each width
        if c.kind == "ring" and c.rows > 4097:
            assert c.rows >= NUM_SMS * ring_warps(c.dim) * 5


def test_ln_kernel_name_parser_reads_every_spelling():
    assert ln_kernels("void (anonymous namespace)::ln_fwd_kernel<6, false>(float const*, long long)") == \
        [("fwd", 6, False)]
    assert ln_kernels("void <unnamed>::ln_bwd_ring_kernel<(int)3, (bool)1>(const __nv_bfloat16 *)") == \
        [("ring", 3, True)]
    assert ln_kernels("void <unnamed>::ln_bwd_kernel<(int)8, (bool)0>(...)") == [("bwd", 8, False)]
    assert ln_kernels("_ZN41_GLOBAL__N__f0_12_vitk_norm_cu_ab13ln_bwd_kernelILi4ELb0EEEvPK") == [("bwd", 4, False)]
    assert ln_kernels("_ZN41_GLOBAL__N__f0_12_vitk_norm_cu_ab18ln_bwd_ring_kernelILi2ELb1EEEvPK") == [("ring", 2, True)]


def test_ce_refuses_more_than_4096_classes():
    """C = 4097 is refused by the entry check, before any CUDA call (the pointers are fake)."""
    from vision_transformers_torch_xla_b200 import _lib

    lib = _lib.load()
    fake = 1 << 20
    rc = lib.vitk_ce_fwd_bwd(fake, None, fake, ctypes.c_float(0.0), None, ctypes.c_float(0.0), ctypes.c_float(1.0), fake,
                             fake, fake, 4, 4097, None)
    assert rc == -1 and b"C=4097" in lib.vitk_last_error()


# Kernels of vitk_norm.cu / vitk_elementwise.cu checked by this file's element-wise tests, and those checked elsewhere.
COVERED_HERE = {
    "ce_kernel": "test_cross_entropy", "mean_rows_kernel": "test_cross_entropy", "adamw_kernel": "test_adamw",
    "colsum_bf16_kernel": "test_colsum", "pool_fwd_kernel": "test_pool", "pool_bwd_kernel": "test_pool",
    "embed_bwd_kernel": "test_embed_bwd", "embed_bwd_pad_kernel": "test_embed_bwd",
    "patchify_kernel<unsigned int>": "test_patchify", "prefix_rows_kernel": "test_prefix_rows",
    "scale_cast_kernel": "test_scale_cast_and_scale_f32", "scale_f32_kernel": "test_scale_cast_and_scale_f32",
    "rowscale_cast_kernel": "test_rowscale_cast", "colscale_bf16_kernel": "test_colscale",
    "layerscale_grad_kernel": "test_layerscale_grad",
}
COVERED_ELSEWHERE = {
    "dropout_mask_kernel": "test_gpu_dropout.py::test_dropout_mask_kernel",
    "mask_mul_kernel<__nv_bfloat16,8>": "test_gpu_dropout.py::test_mask_mul",
    "mask_mul_kernel<float,4>": "test_gpu_dropout.py::test_mask_mul",
    "droppath_masks_kernel": "test_gpu_configs.py::test_droppath_kernel_statistics_and_reproducibility",
    "clip_coef_kernel": "test_gpu_elementwise.py::test_scale_f32_and_clip_coef",
    "mixup_batch_kernel": "test_gpu_mixup.py::test_mixup_matches_oracle_bitwise",
    "mixup_target_kernel": "test_gpu_mixup.py::test_mixup_matches_oracle_bitwise",
    "sumsq_partial_kernel<float>": "test_gpu_elementwise.py::test_sumsq",
    "sumsq_partial_kernel<__nv_bfloat16>": "test_gpu_elementwise.py::test_sumsq",
    "sumsq_final_kernel": "test_gpu_elementwise.py::test_sumsq",
}
EXEMPT = {
    "patchify_kernel<long long>": "taken only for 2^32 or more eight-element vectors: an image batch above 100 GB",
}


def _kernel_key(demangled):
    """'void <unnamed>::mask_mul_kernel<__nv_bfloat16, (int)8>(...)' -> 'mask_mul_kernel<__nv_bfloat16,8>'."""
    s = re.sub(r"\((int|bool|unsigned int)\)", "", demangled)
    s = re.sub(r"^void |<unnamed>::|\(anonymous namespace\)::", "", s.strip())
    m = re.match(r"[A-Za-z_0-9]+(<[^<>]*>)?", s)
    return re.sub(r",\s+", ",", m.group(0)) if m else s


def test_every_kernel_is_accounted_for():
    """Every kernel that vitk_norm.cu and vitk_elementwise.cu put into libvitk.so is named by a row of this file, is
    listed with the test that covers it, or is exempt with its reason."""
    from vision_transformers_torch_xla_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    filt = shutil.which("cu++filt") or os.path.join(os.path.dirname(cuobjdump), "cu++filt")
    if not (os.path.exists(cuobjdump) and os.path.exists(filt)):
        pytest.skip("cuobjdump / cu++filt unavailable")
    out = subprocess.run([cuobjdump, "-elf", _lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump failed: " + out.stderr[-200:])
    mangled = sorted(set(re.findall(r"\.text\.([A-Za-z0-9_]+)", out.stdout)))
    # kernels of an anonymous namespace carry their file's name; the others (global namespace) are all in these files
    ours = [m for m in mangled if "_vitk_norm_cu_" in m or "_vitk_elementwise_cu_" in m or "_GLOBAL__N_" not in m]
    demangled = subprocess.run([filt], input="\n".join(ours), capture_output=True, text=True, check=True).stdout.split("\n")
    ln_named = {c.kernel for c in LN_TABLE}
    missing, counted = [], 0
    for d in demangled[: len(ours)]:
        ln = ln_kernels(d)
        key = _kernel_key(d)
        if ln:
            ok = ln[0] in ln_named
        else:
            ok = key in COVERED_HERE or key in COVERED_ELSEWHERE or key in EXEMPT
        counted += ok
        if not ok:
            missing.append(key if not ln else ln[0])
    print(f"[coverage] {counted} of {len(ours)} kernels of vitk_norm.cu / vitk_elementwise.cu accounted for "
          f"({sum(1 for d in demangled[:len(ours)] if ln_kernels(d))} LayerNorm kernels named by rows, "
          f"{len(COVERED_HERE)} element-wise tests here, {len(COVERED_ELSEWHERE)} elsewhere, {len(EXEMPT)} exempt)")
    assert len(ours) >= 51
    assert not missing, f"kernels without a row, a covering test or an exemption: {missing}"
    keys = {_kernel_key(d) for d in demangled[: len(ours)]}
    stale = (set(COVERED_HERE) | set(COVERED_ELSEWHERE) | set(EXEMPT)) - keys
    assert not stale, f"entries naming kernels that are not built: {sorted(stale)}"


def _finish_fwd(case, ops, res, dev):
    outs = ln_outputs(case, ops, dev)
    outs["y"].view.copy_(res["y"][0].reshape(case.rows, case.dim).to(torch.bfloat16))
    for nm in ("mean", "rstd"):
        if nm in outs:
            outs[nm].view.copy_(res[nm][0].reshape(1, -1).float())
    return outs


def test_checker_rejects_a_subtly_wrong_result():
    """The float64 result rounded to each output type passes; seven subtly wrong results do not."""
    dev = "cpu"
    verdicts = {}

    # LayerNorm forward at an inexact width (the last column group of a lane is partial)
    case = LnCase(("fwd", 4, False), 300, 388, pitch=True)
    ops = ln_inputs(case, dev)
    good = ln_fwd_reference(case, ops)
    assert verify("fwd", _finish_fwd(case, ops, good, dev), good)[0] == []
    verdicts["variance divided by D - 1"] = verify("fwd", _finish_fwd(case, ops, ln_fwd_reference(case, ops, 387), dev),
                                                   good)[0]
    outs = _finish_fwd(case, ops, good, dev)
    outs["y"].view[:, -4:] = float("nan")
    verdicts["last partial column group at its fill"] = verify("fwd", outs, good)[0]
    outs = _finish_fwd(case, ops, good, dev)
    outs["y"].buf[outs["y"].lead + case.dim] = 0.0                      # the first pad element of row 0's pitch
    verdicts["one guard element changed"] = verify("fwd", outs, good)[0]

    # LayerNorm backward with a rowscale
    case = LnCase(("bwd", 6, False), 300, 768, g_in="sep", gb=True, rowscale=True, dgb=True, pitch=True)
    ops = ln_inputs(case, dev)
    good = ln_bwd_reference(case, ops)

    def finish(res):
        outs = ln_outputs(case, ops, dev)
        for nm, (ref, *_r) in res.items():
            outs[nm].view.copy_(ref.reshape(outs[nm].rows, outs[nm].cols).to(outs[nm].buf.dtype))
        return outs

    assert verify("bwd", finish(good), good)[0] == []
    verdicts["dgamma missing one row"] = verify("bwd", finish(ln_bwd_reference(case, ops, drop_row=137)), good)[0]
    shifted = ops["rs"].double()[(torch.arange(case.rows) + 1) // case.rpg]
    verdicts["rowscale group off by one row"] = verify("bwd", finish(ln_bwd_reference(case, ops, rs_rows=shifted)),
                                                       good)[0]

    # cross-entropy with label smoothing
    ce = CeCase(64, 1000, "smooth", 5.0)
    ops = ce_inputs(ce, dev)
    good = ce_reference(ce, ops)

    def ce_outs(res):
        o = {"loss": guarded(1, 1, 1, torch.float32, dev), "dlogits": guarded(ce.B, ce.C, ce.C, torch.float32, dev)}
        for nm in o:
            o[nm].view.copy_(res[nm][0].reshape(o[nm].rows, o[nm].cols).float())
        return o

    assert verify("ce", ce_outs(good), good)[0] == []
    verdicts["cross-entropy over C - 1 classes"] = verify("ce", ce_outs(ce_reference(ce, ops, classes=ce.C - 1)), good)[0]

    # AdamW
    ad = AdamwCase(1028, 8, 4, 2, zero_grad=True)
    ops = adamw_inputs(ad, dev)
    good = adamw_reference(ad, ops)

    def ad_outs(res):
        o = {nm: guarded(1, ad.n, ad.n, torch.float32, dev) for nm in res}
        for nm in o:
            o[nm].view.copy_(res[nm][0].reshape(1, -1).float())
        return o

    assert verify("adamw", ad_outs(good), good)[0] == []
    verdicts["AdamW bias correction one step off"] = verify("adamw", ad_outs(adamw_reference(ad, ops, step=3)), good)[0]

    for what, fails in verdicts.items():
        print(f"[checker] {what}: {fails[0] if fails else 'ACCEPTED'}")
    assert all(verdicts.values()), [w for w, f in verdicts.items() if not f]


# ---------------------------------------------------------------------------------------------------------------------
# GPU: LayerNorm, one launch per row under the profiler
# ---------------------------------------------------------------------------------------------------------------------
def ln_launch(case, ops, outs):
    from vision_transformers_torch_xla_b200 import _lib as L

    dev = ops["x"].device
    x_st = _padded(ops["x"], case.ld_x, dev)
    if case.kind == "fwd":
        L.layernorm_fwd(x_st, ops["gamma"], ops["beta"], outs["y"].view, outs["mean"].view if case.stats else None,
                        outs["rstd"].view if case.stats else None, case.rows, case.dim, EPS, ld_x=case.ld_x,
                        ld_y=case.ld_y)
        return
    dy_st = _padded(ops["dy"], case.ld_dy, dev)
    if case.g_in == "sep":
        g_in = _padded(ops["g_in"], case.ld_g, dev)
    elif case.g_in == "inplace":
        g_in = outs["g_out"].view
    else:
        g_in = None
    L.layernorm_bwd(dy_st, x_st, ops["mean"], ops["rstd"], ops["gamma"], g_in, outs["g_out"].view,
                    outs["gb_out"].view if case.gb else None, ops.get("rs"), case.rpg,
                    outs["dgamma"].view if case.dgb else None, outs["dbeta"].view if case.dgb else None, case.rows,
                    case.dim, ld_x=case.ld_x, ld_dy=case.ld_dy, ld_g=case.ld_g)


@pytest.mark.gpu
@pytest.mark.parametrize("case", LN_TABLE, ids=[c.id for c in LN_TABLE])
def test_layernorm_kernel(cuda_device, case):
    from torch.profiler import ProfilerActivity, profile

    ops = ln_inputs(case, cuda_device)
    # In a long pytest process the profiler now and then returns a trace without the kernel records of a short launch.
    # Such a trace names no LayerNorm kernel at all; the launch is then repeated on fresh outputs (at most twice more),
    # and the outputs checked below are those of the launch whose trace named its kernel.
    for _ in range(3):
        outs = ln_outputs(case, ops, cuda_device)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ln_launch(case, ops, outs)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "ln_" in e.name and "_kernel" in e.name]
        ran = [k for nm in names for k in ln_kernels(nm)]
        if ran:
            break
    assert len(ran) == 1, f"{case.id}: expected one LayerNorm kernel, the profiler saw {names}"
    assert ran[0] == case.kernel, f"{case.id}: ran {ran[0]}, the row names {case.kernel}"
    res = ln_fwd_reference(case, ops) if case.kind == "fwd" else ln_bwd_reference(case, ops)
    fails, margins = verify(case.id, outs, res)
    print(f"[margin] ln_{case.kind}<{case.kernel[1]},{case.kernel[2]}> {case.id}: " +
          " ".join(f"{k}={v:.3f}" for k, v in margins.items()))
    assert not fails, "\n".join(fails)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: element-wise kernels
# ---------------------------------------------------------------------------------------------------------------------
def _margins(family, label, margins):
    print(f"[margin] {family} {label}: " + " ".join(f"{k}={v:.3f}" for k, v in margins.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CE_TABLE, ids=[c.id for c in CE_TABLE])
def test_cross_entropy(cuda_device, case):
    from vision_transformers_torch_xla_b200 import _lib as L

    ops = ce_inputs(case, cuda_device)
    outs = {"loss": guarded(1, 1, 1, torch.float32, cuda_device),
            "dlogits": guarded(case.B, case.C, case.C, torch.float32, cuda_device)}
    scratch = guarded(1, case.B, case.B, torch.float32, cuda_device)
    L.ce_fwd_bwd(ops["logits"], ops.get("soft"), ops.get("labels"), ops["smoothing"], ops.get("teacher"), case.alpha,
                 case.T, outs["loss"].view, outs["dlogits"].view, scratch.view)
    torch.cuda.synchronize()
    guard = torch.ones(scratch.buf.numel(), dtype=torch.bool, device=cuda_device)
    guard[scratch.index()] = False
    assert bool((scratch.buf[guard] == SENTINEL[torch.float32]).all()), "row-loss scratch written out of bounds"
    # dlogits is held to its element bound only: with thousands of classes and logits of scale 30 a row's probability
    # sits on a few classes, the RMS of dlogits falls far below its largest elements, and the __expf error of those
    # elements alone reaches 4e-4 of it (max/rms is a metric for dense outputs)
    fails, margins = verify(case.id, outs, ce_reference(case, ops), no_rms=("dlogits",))
    _margins("ce", case.id, margins)
    report(f"ce {case.id} dlogits", outs["dlogits"].view, ce_reference(case, ops)["dlogits"][0])
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ADAMW_TABLE, ids=[c.id for c in ADAMW_TABLE])
def test_adamw(cuda_device, case):
    from vision_transformers_torch_xla_b200 import _lib as L

    ops = adamw_inputs(case, cuda_device)
    res = adamw_reference(case, ops)
    n = case.n
    outs = {nm: guarded(1, n, n, torch.float32, cuda_device, ops[nm][None, :]) for nm in ("p", "m", "v", "g")}
    if case.ema:
        outs["ema"] = guarded(1, n, n, torch.float32, cuda_device, ops["ema"][None, :])
    shadow = guarded(1, n, n, torch.bfloat16, cuda_device) if case.shadow else None
    hp = ADAMW_HYPER
    L.adamw_flat(outs["p"].view[0], outs["g"].view[0], outs["m"].view[0], outs["v"].view[0],
                 shadow.view[0] if shadow else None, outs["ema"].view[0] if case.ema else None, ops.get("cg"),
                 case.chunk, ops["lrs"], ops["wds"], hp["beta1"], hp["beta2"], hp["eps"], case.step,
                 grad_scale=hp["grad_scale"], ema_decay=hp["ema_decay"], zero_grad=case.zero_grad,
                 g_bf16=ops.get("g16"), grad_scale_dev=ops.get("gsd"))
    torch.cuda.synchronize()
    if shadow is not None:
        outs["shadow"] = shadow
        res["shadow"] = exact(outs["p"].view[0].bfloat16())
    fails, margins = verify(case.id, outs, res)
    _margins("adamw", case.id, margins)
    assert not fails, "\n".join(fails)


COLSUM_TABLE = [(r, c, i % 2 == 1) for i, (r, c) in enumerate(
    [(r, c) for r in (1, 7, 8, 63, 64, 65, 4097) for c in (8, 248, 256, 264, 3072, 4104)] +
    [(100000, c) for c in (8, 264, 4104)])]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,pitch", COLSUM_TABLE, ids=[f"{r}x{c}{'-ld' if p else ''}" for r, c, p in COLSUM_TABLE])
def test_colsum(cuda_device, rows, cols, pitch):
    from vision_transformers_torch_xla_b200 import _lib as L

    x = _randn((rows, cols), 11, 1.0, cuda_device).bfloat16()
    ld = cols + 8 if pitch else cols
    init = _randn((cols,), 12, 10.0, cuda_device)
    out = guarded(1, cols, cols, torch.float32, cuda_device, init[None, :])
    L.colsum_bf16(_padded(x, ld, cuda_device), out.view[0], rows, cols, ld=ld)
    torch.cuda.synchronize()
    x64 = x.double()
    res = {"out": (init.double() + x64.sum(0), init.double().abs() + x64.abs().sum(0), rows + 2, 0.0, U)}
    fails, margins = verify(f"colsum {rows}x{cols}", {"out": out}, res)
    _margins("colsum", f"{rows}x{cols}", margins)
    assert not fails, "\n".join(fails)


POOL_TABLE = [(B, N, D, prefix, mode) for i, (B, D, prefix, N1) in enumerate(
    [(B, D, p, n1) for B, D in ((1, 4), (3, 252), (257, 256), (2, 260), (5, 1024)) for p in (0, 1, 2) for n1 in (1, 7)])
    for N in (prefix + N1,) for mode in (0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,D,prefix,mode", POOL_TABLE, ids=[f"B{b}-N{n}-D{d}-p{p}-m{m}" for b, n, d, p, m in POOL_TABLE])
def test_pool(cuda_device, B, N, D, prefix, mode):
    from vision_transformers_torch_xla_b200 import _lib as L

    x = _randn((B, N, D), 21, 1.0, cuda_device)
    pooled = guarded(B, D, D, torch.float32, cuda_device)
    L.pool_fwd(x, pooled.view, B, N, D, prefix, mode)
    dp = _randn((B, D), 22, 1.0, cuda_device)
    g = guarded(B * N, D, D, torch.float32, cuda_device)
    L.pool_bwd(dp, g.view, B, N, D, prefix, mode)
    torch.cuda.synchronize()
    x64, P = x.double(), N - prefix
    inv = _f32(1.0 / P)
    t = torch.arange(N, device=cuda_device)[None, :, None]
    if mode == 0:
        pres = (x64[:, prefix:].sum(1) * inv, x64[:, prefix:].abs().sum(1) * inv, P + 2, 0.0, U)
        gref = torch.where(t >= prefix, dp.double()[:, None, :] * inv, torch.zeros((), dtype=torch.float64,
                                                                                     device=cuda_device))
        gres = (gref.reshape(B * N, D), gref.abs().reshape(B * N, D), 1, 0.0, U)
    else:
        pres = exact(x[:, 0])
        gres = exact(torch.where(t == 0, dp[:, None, :], torch.zeros((), device=cuda_device)).reshape(B * N, D))
    fails, margins = verify(f"pool B{B} N{N} D{D} p{prefix} m{mode}", {"pooled": pooled, "g": g},
                            {"pooled": pres, "g": gres})
    _margins("pool", f"B{B}-N{N}-D{D}-p{prefix}-m{mode}", margins)
    assert not fails, "\n".join(fails)


EMBED_TABLE = [(B, prefix, lay) for i, (B, prefix) in enumerate((B, p) for B in (1, 31, 32, 33, 64) for p in (0, 1, 2))
               for lay in (("flat", "grid", "padded", "frozen") if i % 3 == 0 else ("flat", "padded"))]


@pytest.mark.gpu
@pytest.mark.parametrize("B,prefix,layout", EMBED_TABLE, ids=[f"B{b}-p{p}-{lay}" for b, p, lay in EMBED_TABLE])
def test_embed_bwd(cuda_device, B, prefix, layout):
    """gp = bf16(g) in the flat or the padded image-operand row order (pad rows zeroed), dpos and the prefix-token
    gradients accumulated over the batch; frozen: no prefix-token gradient at all."""
    from vision_transformers_torch_xla_b200 import _lib as L

    gw, gh, D = 3, 2, 68
    gwp = {"flat": 0, "grid": gw, "padded": gw + 2, "frozen": gw + 2}[layout]
    P = gw * gh
    N = P + prefix
    g = _randn((B, N, D), 31, 1.0, cuda_device)
    rows_gp = B * P if gwp == 0 else B * gh * gwp
    gp = guarded(rows_gp, D, D, torch.bfloat16, cuda_device)
    dpos0, dpre0 = _randn((N, D), 32, 2.0, cuda_device), _randn((2, D), 33, 2.0, cuda_device)
    outs = {"gp": gp, "dpos": guarded(N, D, D, torch.float32, cuda_device, dpos0)}
    frozen = layout == "frozen"
    for j in range(prefix if not frozen else 0):
        outs[f"dprefix{j}"] = guarded(1, D, D, torch.float32, cuda_device, dpre0[j][None, :])
    L.embed_bwd(g, gp.view, outs["dpos"].view, outs["dprefix0"].view[0] if "dprefix0" in outs else None,
                outs["dprefix1"].view[0] if "dprefix1" in outs else None, B, N, D, prefix, gw=gw if gwp else 0, gwp=gwp)
    torch.cuda.synchronize()
    g16 = g[:, prefix:].bfloat16()
    if gwp == 0:
        gp_ref = g16.reshape(B * P, D)
    else:
        gp_ref = torch.zeros((B, gh, gwp, D), dtype=torch.bfloat16, device=cuda_device)
        gp_ref[:, :, :gw] = g16.reshape(B, gh, gw, D)
        gp_ref = gp_ref.reshape(-1, D)
    g64 = g.double()
    res = {"gp": exact(gp_ref),
           "dpos": (dpos0.double() + g64.sum(0), dpos0.double().abs() + g64.abs().sum(0), B + 2, 0.0, U)}
    for j in range(prefix if not frozen else 0):
        res[f"dprefix{j}"] = (dpre0[j].double() + g64[:, j].sum(0), dpre0[j].double().abs() + g64[:, j].abs().sum(0),
                              B + 2, 0.0, U)
    fails, margins = verify(f"embed_bwd B{B} p{prefix} {layout}", outs, res)
    _margins("embed_bwd", f"B{B}-p{prefix}-{layout}", margins)
    assert not fails, "\n".join(fails)


PATCH_TABLE = [(ps, C, gh, gw) for ps in (8, 16, 32) for C in (1, 3) for gh, gw in ((2, 3), (3, 1))]


@pytest.mark.gpu
@pytest.mark.parametrize("ps,C,gh,gw", PATCH_TABLE, ids=[f"ps{p}-C{c}-{h}x{w}" for p, c, h, w in PATCH_TABLE])
def test_patchify(cuda_device, ps, C, gh, gw):
    from vision_transformers_torch_xla_b200 import _lib as L

    B, H, W = 2, gh * ps, gw * ps
    img = _randn((B, C, H, W), 41, 1.0, cuda_device)
    out = guarded(B * gh * gw, C * ps * ps, C * ps * ps, torch.bfloat16, cuda_device)
    L.patchify(img, out.view, ps)
    torch.cuda.synchronize()
    ref = F.unfold(img, ps, stride=ps).transpose(1, 2).reshape(B * gh * gw, C * ps * ps).bfloat16()
    fails, _ = verify(f"patchify ps{ps} C{C}", {"out": out}, {"out": exact(ref)})
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("prefix", [1, 2])
def test_prefix_rows(cuda_device, prefix):
    """x[b, j] = tok[j] + pos[j] for j < prefix; the patch rows stay as they were."""
    from vision_transformers_torch_xla_b200 import _lib as L

    B, N, D = 3, 7, 5
    x0 = _randn((B, N, D), 51, 1.0, cuda_device)
    x0[:, :prefix] = float("nan")
    x = guarded(B * N, D, D, torch.float32, cuda_device, x0.reshape(B * N, D))
    tok, pos = _randn((prefix, D), 52, 1.0, cuda_device), _randn((N, D), 53, 1.0, cuda_device)
    L.prefix_rows(x.view, tok, pos, B, N, D, prefix)
    torch.cuda.synchronize()
    ref = x0.clone()
    ref[:, :prefix] = tok + pos[:prefix]
    fails, _ = verify(f"prefix_rows p{prefix}", {"x": x}, {"x": exact(ref.reshape(B * N, D))})
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 5, 1027])
def test_scale_cast_and_scale_f32(cuda_device, n):
    """bf16(x * s) and x * s, including the scalar tail past the last whole float4."""
    from vision_transformers_torch_xla_b200 import _lib as L

    src = _randn((n,), 61, 3.0, cuda_device)
    s = torch.tensor([0.7], dtype=torch.float32, device=cuda_device)
    outs = {"scaled": guarded(1, n, n, torch.bfloat16, cuda_device), "cast": guarded(1, n, n, torch.bfloat16, cuda_device),
            "x": guarded(1, n, n, torch.float32, cuda_device, src[None, :])}
    L.scale_cast_bf16(src, s, outs["scaled"].view[0])
    L.cast_bf16(src, outs["cast"].view[0])
    L.scale_f32_(outs["x"].view[0], s)
    torch.cuda.synchronize()
    res = {"scaled": exact((src * s).bfloat16()), "cast": exact(src.bfloat16()), "x": exact(src * s)}
    fails, _ = verify(f"scale n{n}", outs, res)
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("n,epg", [(4, 4), (1028, 12), (4096, 100), (394 * 192, 197 * 192)])
def test_rowscale_cast(cuda_device, n, epg):
    """bf16(x * rowscale[i / elems_per_group]) with a zero group, and a last group cut short."""
    from vision_transformers_torch_xla_b200 import _lib as L

    src = _randn((n,), 71, 2.0, cuda_device)
    groups = -(-n // epg)
    rs = torch.tensor([LN_RS_PATTERN[(g + 1) % 3] for g in range(groups)], dtype=torch.float32, device=cuda_device)
    out = guarded(1, n, n, torch.bfloat16, cuda_device)
    L.rowscale_cast_bf16(src, rs, epg, out.view[0])
    torch.cuda.synchronize()
    ref = (src * rs[torch.arange(n, device=cuda_device) // epg]).bfloat16()
    fails, _ = verify(f"rowscale_cast n{n}", {"out": out}, {"out": exact(ref)})
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,dim", [(1, 8), (5, 8), (300, 264), (7, 264)])
def test_colscale(cuda_device, rows, dim):
    from vision_transformers_torch_xla_b200 import _lib as L

    x0 = _randn((rows, dim), 81, 1.0, cuda_device).bfloat16()
    gamma = _randn((dim,), 82, 1.0, cuda_device)
    gamma[1] = 0.0
    x = guarded(rows, dim, dim, torch.bfloat16, cuda_device, x0)
    L.colscale_bf16(x.view, gamma, rows, dim)
    torch.cuda.synchronize()
    fails, _ = verify(f"colscale {rows}x{dim}", {"x": x}, {"x": exact((x0.float() * gamma).bfloat16())})
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 124, 132, 3072])
@pytest.mark.parametrize("bias", [True, False])
def test_layerscale_grad(cuda_device, K, bias):
    """dgamma = (sum_k W dW + b db) / gamma, 0 where gamma = 0; C = 13 channels (not a multiple of the 8 per CTA)."""
    from vision_transformers_torch_xla_b200 import _lib as L

    C = 13
    W, dW = _randn((C, K), 91, 0.05, cuda_device), _randn((C, K), 92, 1.0, cuda_device)
    b, db = (_randn((C,), 93, 1.0, cuda_device), _randn((C,), 94, 1.0, cuda_device)) if bias else (None, None)
    gamma = _randn((C,), 95, 0.1, cuda_device)
    gamma[3] = 0.0
    out = guarded(1, C, C, torch.float32, cuda_device)
    L.layerscale_grad(W, dW, b, db, gamma, out.view[0])
    torch.cuda.synchronize()
    acc = (W.double() * dW.double()).sum(1)
    mag = (W.double() * dW.double()).abs().sum(1)
    if bias:
        acc, mag = acc + b.double() * db.double(), mag + (b.double() * db.double()).abs()
    g = gamma.double()
    nz = g != 0
    ref = torch.where(nz, acc / torch.where(nz, g, 1.0), 0.0)
    extra = torch.where(nz, (K + 3) * U * mag / torch.where(nz, g, 1.0).abs(), 0.0)
    fails, margins = verify(f"layerscale_grad K{K}", {"out": out}, {"out": (ref, 0.0, 0, extra, U)})
    _margins("layerscale_grad", f"K{K}-bias{int(bias)}", margins)
    assert not fails, "\n".join(fails)
