"""Every instantiation of the tcgen05 GEMM (``gemm_kernel<BLOCK_N, A_MN, B_MN, EPI, EW, CTA2>`` in csrc/vitk_gemm.cu)
against a float64 reference, at the tile edges where such kernels go wrong.

Each row of ``TABLE`` names the instantiation it must launch as ``(BLOCK_N, A_MN, B_MN, EPI, EW, CTA2)``.  EPI is the
public epilogue code of include/vitk.h, or one of the internal codes 100 (residual epilogue through a TMA ring) and 101
(bf16 epilogue through TMA).  A row reaches its kernel through ``block_n``, the operand layouts, the epilogue and the
shape; ``torch.profiler`` reports which kernel ran, and the test asserts it is the row's.  ``AUTO`` holds the model's
own shapes with ``block_n = 0`` and pins the automatic tile-width rule the same way.  On the CPU,
``test_table_covers_every_instantiation_in_the_binary`` checks that the rows name exactly the instantiations the
shipped library contains, so a kernel added later without a row fails on any machine.

Layout of every launch:
  * inputs with row pitches past their logical width; the pad holds NaN, so a read past the tensor maps shows up;
  * outputs (and the GELU derivative output and the fused bias gradient) are views into a larger buffer with one guard
    row before and one after, ``ld_out = N + 8`` for bf16 and ``N + 4`` or ``N + 3`` for fp32.  What the launch may
    write is NaN before it (random for the accumulating wgrad epilogue, which reads it), everything else holds a
    sentinel that must come back bit for bit.

Reference: the same bf16 operands in float64; GELU(h) = h Phi(h), GELU'(h) = Phi(h) + h phi(h); the wgrad epilogue is
``init + A^T B`` and its bias gradient ``init + column sums``.

Bounds.  An fp32 sum of n terms t_i, accumulated in any order with any rounding mode, is off by at most
n * 2^-23 * sum |t_i| (one ulp per addition).  A GEMM element adds K products; each epilogue operation (bias, scales,
residual, split-K red.add, ...) adds one more term or rounding.  So every element satisfies
    |out - ref| <= (1 + c) * (n * 2^-23 * mag + extra) + c * |ref|
  * mag = |A| |B|^T with every epilogue term in absolute value (|rowscale * colscale| * (|A||B|^T + |bias|) + ...);
  * n = K plus the roundings of the epilogue (K + 1 for acc + bias, K + splits + 1 for split-K, ...);
  * c = 2^-23 for fp32 outputs, 2^-8 for bf16 outputs (one rounding to 8 significant bits);
  * extra: the GELU evaluation (Abramowitz-Stegun erf, |err| < 1.5e-7, so Phi is off by < 7.5e-8, plus 2^-20 for the
    fp32 polynomial and the approximate exp / reciprocal), and the error of h carried through |GELU'| <= 1.13 and
    |GELU''| <= 0.8.
On top of that the repository's metrics hold (DESIGN.md §2): max/rms <= 2e-4 for fp32 outputs, elem <= 6e-3 for bf16.
``test_checker_rejects_a_subtly_wrong_result`` shows on the CPU that these checks reject a missing k-block, a
rowscale group off by one row, a bias added twice, one changed guard element and one element left at its NaN fill.
"""
import math
import os
import re
import shutil
import subprocess
from dataclasses import dataclass

import pytest
import torch

from conftest import elem_err, rel_err, report

EPI_BF16, EPI_GELU, EPI_RESID, EPI_F32, EPI_DGELU, EPI_ATOMIC, EPI_PATCH = range(7)
RESID_TMA, BF16_TMA = 100, 101
U23 = 2.0 ** -23
F32_TOL = 2e-4     # max/rms, fp32 outputs (DESIGN.md §2)
BF16_TOL = 6e-3    # elem, bf16 outputs
ROWS_PER_GROUP = 197
RS_PATTERN = (1.25, 0.0, 1.0 / 0.9)   # DropPath-like per-sample scales, with a dropped (zero) group
MASK_SCALE = float(torch.tensor(1.0 / 0.9, dtype=torch.float32))   # the binding passes it as a C float
SENTINEL = {torch.float32: 1234.5678, torch.bfloat16: -1056.0}
BITS = {torch.float32: torch.int32, torch.bfloat16: torch.int16}


@dataclass(frozen=True)
class Case:
    kernel: tuple        # (BLOCK_N, A_MN, B_MN, EPI, EW, CTA2) the launch must run
    M: int
    N: int
    K: int
    epi: int             # public epilogue code
    block_n: int = -1    # -1: the row's BLOCK_N; 0: automatic
    bias: bool = True
    rowscale: bool = False
    colscale: bool = False
    mask: bool = False
    inplace: bool = False
    splits: int = 0
    colsum: bool = False
    prefix: int = 0      # PATCH: prefix tokens; M = images * tokens
    tokens: int = 0      # PATCH: tokens per image
    ld_pad: int = -1     # ld_out - N; -1: 8 for bf16 / fp32 with 16-byte rows, 4 for the fp32 epilogue
    lda: int = 0         # 0: logical width rounded up to 8, plus 8 NaN columns
    note: str = ""

    @property
    def a_mn(self):
        return bool(self.kernel[1])

    @property
    def b_mn(self):
        return bool(self.kernel[2])

    @property
    def out_dtype(self):
        return torch.bfloat16 if self.epi in (EPI_BF16, EPI_GELU, EPI_DGELU) else torch.float32

    @property
    def ld_out(self):
        if self.ld_pad >= 0:
            return self.N + self.ld_pad
        return self.N + (4 if self.epi == EPI_F32 else 8)

    @property
    def id(self):
        bn, amn, bmn, epi, ew, cta2 = self.kernel
        flags = [f for f, on in (("bias", self.bias), ("rs", self.rowscale), ("cs", self.colscale), ("mask", self.mask),
                                 ("inplace", self.inplace), ("colsum", self.colsum)) if on]
        if self.epi == EPI_ATOMIC:
            flags.append(f"s{self.splits}")
        if self.epi == EPI_PATCH:
            flags.append(f"P{self.tokens}p{self.prefix}")
        if self.epi == EPI_F32 or self.ld_pad >= 0:
            flags.append(f"ld{self.ld_out}")
        if self.lda:
            flags.append(f"lda{self.lda}")
        if self.block_n == 0:
            flags.append("auto")
        head = f"{bn}.{int(amn)}{int(bmn)}.e{epi}.w{ew}.{'pair' if cta2 else 'one'}"
        return "-".join([head, f"{self.M}x{self.N}x{self.K}"] + flags + ([self.note] if self.note else []))


def _ew(bn, epi):
    return 16 if epi in (EPI_GELU, EPI_DGELU) and bn != 192 else 8


def _bf16(bn):
    return BF16_TMA if bn % 128 == 0 else EPI_BF16


def _resid(bn, K):
    return RESID_TMA if K <= 1536 else EPI_RESID


# ---------------------------------------------------------------------------------------------------------------------
# The table.  Per instantiation five rows touch the edges:
#   M: 1 / 127 / 129 / 255 for a single CTA (128-row tiles), 256 / 257 / 383 / 512 for a CTA pair (256-row tiles);
#   N: whole tiles, a last tile 8 and 72 columns wide (not a multiple of 32), N = 8;
#   K: 8, 24, 72 (k-block tails) and 456 (8 k-blocks: the 6-stage ring wraps);
#   and one row with more tiles than CTAs (more than 148 single CTAs or 74 pairs, some run 3 tiles), so the double-
#   buffered accumulators and the residual prefetch across tiles wrap.
# ---------------------------------------------------------------------------------------------------------------------
WIDTHS = ((128, False), (128, True), (192, False), (192, True), (256, False), (256, True))


def _edges(bn, cta2):
    """(M, N, K) of the five edge rows of a BLOCK_N x (single | pair) kernel."""
    if cta2:
        ms, wide = (256, 383, 512, 257, 2049), bn * 17 + 8        # 2049: 9 row tiles x 18 column tiles = 162 pairs
    else:
        ms, wide = (1, 127, 129, 255, 255), bn * 150 + 8          # 2 x 151 = 302 CTAs
    ns = (2 * bn, bn + 8, 8, 2 * bn + 72, wide)
    ks = (8, 24, 72, 456, 72)
    return list(zip(ms, ns, ks))


def _table():
    rows = []
    for bn, cta2 in WIDTHS:
        e = _edges(bn, cta2)
        # ---- bf16 output: TMA boxes at 128 / 256, staged panels at 192 ----
        for bmn in ((False, True) if (bn, cta2) != (192, True) else (False,)):
            k = (bn, False, bmn, _bf16(bn), 8, cta2)
            for i, (M, N, K) in enumerate(e):
                rows.append(Case(k, M, N, K, EPI_BF16, bias=i != 2, rowscale=i in (1, 3, 4)))
        # ---- GELU (16 epilogue warps except at 192); a keep mask on the 192 rows ----
        k = (bn, False, False, EPI_GELU, _ew(bn, EPI_GELU), cta2)
        for i, (M, N, K) in enumerate(e):
            rows.append(Case(k, M, N, K, EPI_GELU, bias=i != 2, mask=(bn == 192 and i in (1, 3, 4))))
        if bn == 192:   # a dropout mask sends 256-wide GELU tiles to 192
            M, N, K = e[3]
            rows.append(Case(k, M, N, K, EPI_GELU, block_n=256, mask=True, note="256to192"))
        # ---- x GELU' (dgrad, MN-major B) ----
        if (bn, cta2) != (192, True):
            k = (bn, False, True, EPI_DGELU, _ew(bn, EPI_DGELU), cta2)
            for i, (M, N, K) in enumerate(e):
                rows.append(Case(k, M, N, K, EPI_DGELU, bias=False, rowscale=i in (0, 3, 4)))
        # ---- residual through the TMA ring: K <= 1536, aligned resid, no mask (not for single-CTA 256) ----
        if cta2 or bn < 256:
            k = (bn, False, False, RESID_TMA, 8, cta2)
            for i, (M, N, K) in enumerate(e):
                rows.append(Case(k, M, N, K, EPI_RESID, bias=i != 2, rowscale=i in (1, 3, 4), colscale=i in (0, 3, 4),
                                 inplace=i in (2, 4)))
            M, N, _ = e[1]
            rows.append(Case(k, M, N, 1536, EPI_RESID, rowscale=True, colscale=True, note="kmax"))
        # ---- residual, register prefetch: K > 1536 or a keep mask (always for single-CTA 256) ----
        k = (bn, False, False, EPI_RESID, 8, cta2)
        always = bn == 256 and not cta2
        for i, (M, N, K) in enumerate(e):
            mask = not always and i != 3 or always and i == 1
            rows.append(Case(k, M, N, K if (mask or always) else 1544, EPI_RESID, bias=i != 2, rowscale=i in (1, 3, 4),
                             colscale=i in (0, 3, 4), mask=mask, inplace=i in (2, 3)))
        # ---- fp32 output, forward and dgrad layouts; ragged rows (N % 8 != 0 or ld_out % 4 != 0) take scalar stores ----
        for bmn in ((False, True) if (bn, cta2) != (192, True) else (False,)):
            k = (bn, False, bmn, EPI_F32, 8, cta2)
            (m0, n0, k0), (m1, n1, k1), (m2, _, k2), (m3, n3, k3), (m4, n4, k4) = e
            rows += [Case(k, m0, n0, k0, EPI_F32),
                     Case(k, m1, n1, k1, EPI_F32, ld_pad=3),                     # ld_out % 4 != 0
                     Case(k, m2, bn + 4, k2, EPI_F32, bias=False),               # N % 8 != 0
                     Case(k, m3, n3, k3, EPI_F32),
                     Case(k, m4, n4 - 3, k4, EPI_F32, ld_pad=2)]                 # both
        # ---- fused position embedding: M = images * tokens, not a multiple of the tile ----
        k = (bn, False, False, EPI_PATCH, 8, cta2)
        geo = ((86, 3, 1), (196, 2, 2), (73, 7, 1), (257, 1, 2), (196, 11, 1)) if cta2 else \
              ((1, 1, 1), (49, 5, 2), (9, 14, 1), (43, 3, 2), (85, 3, 1))
        for i, ((M, N, K), (P, imgs, prefix)) in enumerate(zip(e, geo)):
            rows.append(Case(k, P * imgs, N, K, EPI_PATCH, bias=i != 2, prefix=prefix, tokens=P))
        # ---- split-K weight gradient, fp32 red.add (not built for 192-wide pairs) ----
        if (bn, cta2) != (192, True):
            for amn in (True, False):
                k = (bn, amn, amn, EPI_ATOMIC, 8, cta2)
                (m0, n0, _), (m1, n1, _), (m2, n2, _), (m3, n3, _), (m4, n4, _) = e
                rows += [Case(k, m0, n0, 8, EPI_ATOMIC, bias=False, splits=1, colsum=amn),
                         Case(k, m1, n1, 456, EPI_ATOMIC, bias=False, splits=3, colsum=amn),     # 8 k-blocks in 3
                         Case(k, m2, n2, 1000, EPI_ATOMIC, bias=False, splits=7, colsum=amn),    # 16 k-blocks in 7
                         Case(k, m3, n3, 72, EPI_ATOMIC, bias=False, splits=5, colsum=amn),      # 2 k-blocks: 5 -> 2
                         Case(k, m4, n4, 456, EPI_ATOMIC, bias=False, splits=0, colsum=amn)]     # automatic
    return rows


def _auto():
    """block_n = 0 at the model's shapes: ViT-Ti / S / B / L (tokens of 4 images of 197) in all three roles, and the
    classifier head of 8 images with 10, 100 and 1000 classes.  The expected kernel follows the tile-width rule of
    vitk_gemm_bf16 (N % 256 == 0 or N > 512 with <= 15 % padding -> 256, else N % 192 -> 192, N % 128 -> 128, else
    the next width up) and the CTA-pair rule of dispatch() (M >= 256; 192-wide pairs only for K-major operands)."""
    T = 4 * 197
    rows = []
    for D, w_d, w_3d, w_4d in ((192, 192, 192, 256), (384, 192, 256, 256), (768, 256, 256, 256), (1024, 256, 256, 256)):
        auto = dict(block_n=0)
        # M = T >= 256: CTA pairs, except 192-wide tiles of the dgrad and wgrad layouts
        rows += [
            # forward: qkv (bf16), proj (residual), fc1 (GELU), fc2 (residual)
            Case((w_3d, 0, 0, _bf16(w_3d), 8, True), T, 3 * D, D, EPI_BF16, **auto, note="qkv"),
            Case((w_d, 0, 0, _resid(w_d, D), 8, True), T, D, D, EPI_RESID, **auto, rowscale=True, colscale=True,
                 note="proj"),
            Case((256, 0, 0, EPI_GELU, 16, True), T, 4 * D, D, EPI_GELU, **auto, note="fc1"),
            Case((w_d, 0, 0, _resid(w_d, 4 * D), 8, True), T, D, 4 * D, EPI_RESID, **auto, rowscale=True,
                 colscale=True, note="fc2"),
            # input gradients: qkv, proj and fc1 (bf16), fc2 (x GELU')
            Case((w_d, 0, 1, _bf16(w_d), 8, w_d != 192), T, D, 3 * D, EPI_BF16, **auto, bias=False, note="qkv"),
            Case((w_d, 0, 1, _bf16(w_d), 8, w_d != 192), T, D, D, EPI_BF16, **auto, bias=False, note="proj"),
            Case((w_d, 0, 1, _bf16(w_d), 8, w_d != 192), T, D, 4 * D, EPI_BF16, **auto, bias=False, note="fc1"),
            Case((256, 0, 1, EPI_DGELU, 16, True), T, 4 * D, D, EPI_DGELU, **auto, bias=False, note="fc2"),
            # weight gradients with the fused bias gradient: dW[out, in] += dY^T X over the tokens
            Case((w_d, 1, 1, EPI_ATOMIC, 8, w_d != 192), 3 * D, D, T, EPI_ATOMIC, **auto, bias=False, colsum=True,
                 note="qkv"),
            Case((w_d, 1, 1, EPI_ATOMIC, 8, w_d != 192), D, D, T, EPI_ATOMIC, **auto, bias=False, colsum=True,
                 note="proj"),
            Case((w_d, 1, 1, EPI_ATOMIC, 8, w_d != 192), 4 * D, D, T, EPI_ATOMIC, **auto, bias=False, colsum=True,
                 note="fc1"),
            Case((w_4d, 1, 1, EPI_ATOMIC, 8, D >= 256), D, 4 * D, T, EPI_ATOMIC, **auto, bias=False, colsum=True,
                 note="fc2"),
            # fp32 input gradient (LinearFn / AttentionFn / MlpFn)
            Case((w_d, 0, 1, EPI_F32, 8, w_d != 192), T, D, 3 * D, EPI_F32, **auto, bias=False, note="qkv"),
        ]
    # a keep mask moves fc1 to 192-wide tiles and the residual epilogues off the TMA ring
    rows += [Case((192, 0, 0, EPI_GELU, 8, True), T, 3072, 768, EPI_GELU, block_n=0, mask=True, note="fc1"),
             Case((256, 0, 0, EPI_RESID, 8, True), T, 768, 768, EPI_RESID, block_n=0, mask=True, rowscale=True,
                  colscale=True, note="proj")]
    # the tile-width rule at its edges: 1152 -> 256 (4.5 tiles), 384 / 576 -> 192, 200 / 1000 -> 256
    rows += [Case((256, 0, 0, BF16_TMA, 8, True), T, 1152, 384, EPI_BF16, block_n=0),
             Case((192, 0, 0, EPI_BF16, 8, True), T, 384, 384, EPI_BF16, block_n=0),
             Case((192, 0, 0, EPI_BF16, 8, True), T, 576, 192, EPI_BF16, block_n=0),
             Case((256, 0, 0, BF16_TMA, 8, True), T, 200, 64, EPI_BF16, block_n=0),
             Case((256, 0, 0, BF16_TMA, 8, True), T, 1000, 64, EPI_BF16, block_n=0)]
    # classifier head, 8 images: logits (ragged fp32 for 10 / 100 classes), the feature gradient with K = C classes and
    # lda = C rounded up to 8 (ops.py pads dlogits to that pitch), and the weight gradient with the bias gradient
    B = 8
    for C, D, w_c, w_d in ((10, 192, 128, 192), (100, 384, 128, 192), (1000, 768, 256, 256)):
        Cp = (C + 7) // 8 * 8
        rows += [Case((w_c, 0, 0, EPI_F32, 8, False), B, C, D, EPI_F32, block_n=0, ld_pad=0, note="head"),
                 Case((w_d, 0, 1, _bf16(w_d), 8, False), B, D, C, EPI_BF16, block_n=0, bias=False, lda=Cp, note="head"),
                 Case((w_d, 1, 1, EPI_ATOMIC, 8, C >= 256), C, D, B, EPI_ATOMIC, block_n=0, bias=False, colsum=True,
                      lda=Cp, note="head")]
    return rows


TABLE = _table()
AUTO = _auto()


# ---------------------------------------------------------------------------------------------------------------------
# Kernel names: demangled by kineto or cu++filt ("gemm_kernel<256, false, ...>" / "gemm_kernel<(int)256, (bool)0, ...>"),
# or still mangled ("gemm_kernelILi256ELb0E...").
# ---------------------------------------------------------------------------------------------------------------------
_DEMANGLED = re.compile(r"gemm_kernel<([^<>]*)>")
_MANGLED = re.compile(r"gemm_kernelILi(\d+)ELb([01])ELb([01])ELi(\d+)ELi(\d+)ELb([01])E")


def _targ(tok):
    tok = re.sub(r"^\([a-z ]+\)", "", tok.strip())   # "(int)256", "(bool)0"
    return {"true": 1, "false": 0}[tok] if tok in ("true", "false") else int(tok)


def kernel_tuples(text):
    """Every gemm_kernel instantiation named in `text`, as (BLOCK_N, A_MN, B_MN, EPI, EW, CTA2) tuples of ints."""
    found = [tuple(_targ(t) for t in m.group(1).split(",")) for m in _DEMANGLED.finditer(text)]
    found += [tuple(int(g) for g in m.groups()) for m in _MANGLED.finditer(text)]
    return [t for t in found if len(t) == 6]


def _norm(kernel):
    return tuple(int(x) for x in kernel)


# ---------------------------------------------------------------------------------------------------------------------
# Operands, guarded outputs, reference and checker (device-agnostic: the checker's self-test runs them on the CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _r8(x):
    return (x + 7) // 8 * 8


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _randn(shape, seed, scale=1.0, dev="cpu"):
    return (torch.randn(shape, generator=_gen(seed)) * scale).to(dev)


def _padded(logical, ld, dev):
    """[rows, ld] storage of a 2-D bf16 operand whose columns past the logical width are NaN; returns (storage, ld)."""
    rows, cols = logical.shape
    st = torch.full((rows, ld), float("nan"), dtype=logical.dtype, device=dev)
    st[:, :cols] = logical
    return st


@dataclass
class Guarded:
    """A flat buffer; `view` is the [rows, cols] window with row pitch `ld` after one leading guard row."""
    buf: torch.Tensor
    view: torch.Tensor
    lead: int
    ld: int
    rows: int
    cols: int

    def index(self, rows=None):
        r = torch.arange(self.rows, device=self.buf.device) if rows is None else rows.to(self.buf.device)
        return (self.lead + r[:, None] * self.ld + torch.arange(self.cols, device=self.buf.device)[None, :]).flatten()


def guarded(rows, cols, ld, dtype, dev, fill=float("nan")):
    align = 16 // torch.tensor([], dtype=dtype).element_size()
    lead = -(-ld // align) * align                      # one guard row, rounded so that the window is 16-byte aligned
    total = lead + rows * ld + ld                       # ... and one guard row after
    buf = torch.full((total,), SENTINEL[dtype], dtype=dtype, device=dev)
    view = buf.as_strided((rows, cols), (ld, 1), lead)
    if isinstance(fill, torch.Tensor):
        view.copy_(fill)
    else:
        view.fill_(fill)
    return Guarded(buf, view, lead, ld, rows, cols)


def make_operands(case, dev, seed=0):
    """Logical operands (A [M, K], B [N, K] bf16, side operands) and their stored layouts."""
    M, N, K = case.M, case.N, case.K
    ops = {}
    a_scale = 1.0 if case.epi != EPI_ATOMIC else 0.5
    ops["A"] = _randn((M, K), seed + 1, a_scale, dev).bfloat16()
    ops["B"] = _randn((N, K), seed + 2, 1.0 / math.sqrt(max(K, 1)), dev).bfloat16()
    if case.a_mn:
        ops["lda"] = case.lda or _r8(M) + 8
        ops["A_st"] = _padded(ops["A"].t().contiguous(), ops["lda"], dev)
    else:
        ops["lda"] = case.lda or _r8(K) + 8
        ops["A_st"] = _padded(ops["A"], ops["lda"], dev)
    if case.b_mn:
        ops["ldb"] = _r8(N) + 8
        ops["B_st"] = _padded(ops["B"].t().contiguous(), ops["ldb"], dev)
    else:
        ops["ldb"] = _r8(K) + 8
        ops["B_st"] = _padded(ops["B"], ops["ldb"], dev)
    if case.bias:
        ops["bias"] = _randn((N,), seed + 3, 1.0, dev)
    if case.rowscale:
        groups = (M + ROWS_PER_GROUP - 1) // ROWS_PER_GROUP
        ops["rs"] = torch.tensor([RS_PATTERN[g % 3] for g in range(groups)], dtype=torch.float32, device=dev)
        ops["rs_rows"] = ops["rs"][torch.arange(M, device=dev) // ROWS_PER_GROUP]
    if case.colscale:
        ops["cs"] = _randn((N,), seed + 4, 0.5, dev)
    if case.mask:
        ops["mask"] = (torch.rand((M, N), generator=_gen(seed + 5)) >= 0.1).to(torch.uint8).to(dev)
    if case.epi == EPI_RESID:
        ops["resid"] = _randn((M, N), seed + 6, 1.0, dev)
    if case.epi == EPI_DGELU:
        ops["aux"] = (_randn((M, N), seed + 7, 0.4, dev) + 0.5).bfloat16()   # gelu'(h) lies in [-0.17, 1.13]
    if case.epi == EPI_PATCH:
        ops["pos"] = _randn((case.tokens + case.prefix, N), seed + 8, 1.0, dev)
    if case.epi == EPI_ATOMIC:
        ops["init"] = _randn((M, N), seed + 9, 1.0, dev)
        if case.colsum:
            ops["cinit"] = _randn((M,), seed + 10, 1.0, dev)
    return ops


def _splits_bound(case):
    kb = -(-case.K // 64)
    return min(case.splits, kb) if case.splits > 0 else min(32, kb)


def _gelu64(h):
    phi_cdf = 0.5 * (1.0 + torch.erf(h / math.sqrt(2.0)))
    pdf = torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)
    return h * phi_cdf, phi_cdf + h * pdf


def reference_rows(case):
    """PATCH: the output row of patch row t = b * P + p is b * (P + prefix) + prefix + p."""
    t = torch.arange(case.M)
    return (t // case.tokens) * (case.tokens + case.prefix) + case.prefix + t % case.tokens


def reference(case, ops):
    """float64 expectation of every written output, with its error budget.

    Returns {name: (ref [rows, cols] or [rows], mag, n, extra, c, written rows or None)}: the bound of an element is
    (1 + c) * (n * 2^-23 * mag + extra) + c * |ref|."""
    A, B = ops["A"].double(), ops["B"].double()
    K = case.K
    acc = A @ B.t()
    mag = A.abs() @ B.abs().t()
    zero = torch.zeros((), dtype=torch.float64, device=acc.device)
    bias = ops["bias"].double() if "bias" in ops else zero
    c_out = 2.0 ** -8 if case.out_dtype == torch.bfloat16 else U23
    rs = ops["rs_rows"].double()[:, None] if "rs_rows" in ops else torch.ones((), dtype=torch.float64, device=acc.device)
    keep = ops["mask"].double() * MASK_SCALE if "mask" in ops else torch.ones((), dtype=torch.float64, device=acc.device)
    res = {}
    if case.epi == EPI_BF16:
        res["out"] = (rs * (acc + bias), rs.abs() * (mag + bias.abs()), K + 2, 0.0, c_out, None)
    elif case.epi == EPI_F32:
        res["out"] = (acc + bias, mag + bias.abs(), K + 1, 0.0, c_out, None)
    elif case.epi == EPI_GELU:
        h = acc + bias
        e_h = (K + 1) * U23 * (mag + bias.abs())
        act, der = _gelu64(h)
        act_x = keep * (1.13 * e_h + h.abs() * (7.5e-8 + 2.0 ** -20)) + U23 * (keep * act).abs()
        der_x = keep * (0.8 * e_h + 7.5e-8 + 2.0 ** -20 * (1.0 + h.abs())) + U23 * (keep * der).abs()
        res["out"] = (keep * act, zero, 0, act_x, c_out, None)
        res["aux"] = (keep * der, zero, 0, der_x, c_out, None)
    elif case.epi == EPI_DGELU:
        d = ops["aux"].double()
        res["out"] = (rs * acc * d, (rs * d).abs() * mag, K + 2, 0.0, c_out, None)
    elif case.epi == EPI_RESID:
        scale = rs * (ops["cs"].double() if "cs" in ops else 1.0) * keep
        r = ops["resid"].double()
        res["out"] = (r + scale * (acc + bias), scale.abs() * (mag + bias.abs()), K + 4, 0.0, c_out, None)
    elif case.epi == EPI_PATCH:
        t = torch.arange(case.M, device=acc.device)
        pos = ops["pos"].double()[case.prefix + t % case.tokens]
        res["out"] = (acc + bias + pos, mag + bias.abs() + pos.abs(), K + 2, 0.0, c_out, reference_rows(case).to(acc.device))
    elif case.epi == EPI_ATOMIC:
        s = _splits_bound(case)
        init = ops["init"].double()
        res["out"] = (init + acc, mag + init.abs(), K + s + 1, 0.0, c_out, None)
        if "cinit" in ops:
            ci = ops["cinit"].double()
            res["colsum"] = (ci + A.sum(1), ci.abs() + A.abs().sum(1), K + s + 16, 0.0, U23, None)
    return res


def check(name, g, idx, ref, mag, n, extra, c):
    """(failures, worst |out - ref| / bound) of guarded output `g`, whose elements `idx` should hold `ref`; `mag` and
    `extra` are float64 tensors shaped like `ref`.  No failures: the guard is intact and every element is in bounds."""
    fails = []
    dt = g.buf.dtype
    guard = torch.ones(g.buf.numel(), dtype=torch.bool, device=g.buf.device)
    guard[idx] = False
    want = torch.tensor([SENTINEL[dt]], dtype=dt).view(BITS[dt]).item()
    gb = g.buf.view(BITS[dt])[guard]
    if not bool((gb == want).all()):
        bad = int((gb != want).sum())
        fails.append(f"{name}: {bad} guard elements changed")
    got = g.buf[idx].double()
    ref, mag, extra = ref.flatten(), mag.flatten(), extra.flatten()
    bound = (1.0 + c) * (n * U23 * mag + extra) + c * ref.abs()
    diff = (got - ref).abs()
    ok = diff <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero().flatten()
        j = int(bad[0])
        fails.append(f"{name}: {bad.numel()} of {ok.numel()} elements outside the bound; first at written element {j}: "
                     f"got {float(got[j])!r} want {float(ref[j])!r} bound {float(bound[j]):.3e}")
    if dt == torch.float32:
        m = rel_err(got, ref)
        if not m <= F32_TOL:
            fails.append(f"{name}: max/rms {m:.3e} > {F32_TOL}")
    else:
        m = elem_err(got, ref)
        if not m <= BF16_TOL:
            fails.append(f"{name}: elem {m:.3e} > {BF16_TOL}")
    margin = float((diff / bound.clamp_min(1e-300)).max()) if ok.all() else float("nan")
    return fails, margin


def outputs(case, ops, dev):
    """The guarded output buffers of a launch, filled as the kernel will find them."""
    o = {}
    rows = case.M if case.epi != EPI_PATCH else (case.M // case.tokens) * (case.tokens + case.prefix)
    if case.epi == EPI_ATOMIC:
        o["out"] = guarded(rows, case.N, case.ld_out, torch.float32, dev, ops["init"])
        if "cinit" in ops:
            o["colsum"] = guarded(1, case.M, case.M, torch.float32, dev, ops["cinit"][None, :])
    elif case.inplace:
        o["out"] = guarded(rows, case.N, case.ld_out, torch.float32, dev, ops["resid"])
    elif case.epi == EPI_PATCH:   # the prefix-token rows are not written: they belong to the guard
        o["out"] = g = guarded(rows, case.N, case.ld_out, torch.float32, dev, SENTINEL[torch.float32])
        g.buf[g.index(reference_rows(case))] = float("nan")
    else:
        o["out"] = guarded(rows, case.N, case.ld_out, case.out_dtype, dev)
    if case.epi == EPI_GELU:
        o["aux"] = guarded(case.M, case.N, case.N + 8, torch.bfloat16, dev)
    return o


def check_case(case, outs, res):
    """Checks every output of one launch against reference(); returns (failures, [(name, written values, ref, margin)])."""
    fails, seen = [], []
    for name, (ref, mag, n, extra, c, orows) in res.items():
        g = outs[name]
        idx = g.index(orows)
        ref = ref.reshape(g.rows if orows is None else orows.numel(), g.cols)
        f64 = dict(dtype=torch.float64, device=ref.device)
        f, margin = check(f"{case.id}:{name}", g, idx, ref, torch.as_tensor(mag, **f64).expand_as(ref), n,
                          torch.as_tensor(extra, **f64).expand_as(ref), c)
        fails += f
        seen.append((name, g.buf[idx], ref.flatten(), margin))
    return fails, seen


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def test_table_rows_are_well_formed():
    """Every row is reachable as written: widths, layouts, epilogue codes and the shape rules of the entry checks."""
    for case in TABLE + AUTO:
        bn, amn, bmn, epi, ew, cta2 = case.kernel
        assert bn in (128, 192, 256) and ew == _ew(bn, case.epi), case.id
        assert case.N % 8 == 0 or case.epi == EPI_F32, case.id
        assert (case.M >= 256) == bool(cta2) or (bn == 192 and not cta2 and (bmn or epi == EPI_ATOMIC)), case.id
        if case.epi == EPI_PATCH:
            assert case.M % case.tokens == 0 and case.M % (256 if cta2 else 128) != 0, case.id
    ids = [c.id for c in TABLE + AUTO]
    assert len(set(ids)) == len(ids)


@pytest.fixture(scope="module")
def libpath():
    from vision_transformers_torch_xla_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    _lib.load()
    return _lib.LIB_PATH


def test_table_covers_every_instantiation_in_the_binary(libpath):
    """The set of kernels the rows name equals the set of gemm_kernel instantiations in libvitk.so."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump unavailable")
    out = subprocess.run([cuobjdump, "-elf", libpath], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump failed: " + out.stderr[-200:])
    text = out.stdout
    filt = shutil.which("cu++filt") or os.path.join(os.path.dirname(cuobjdump), "cu++filt")
    if os.path.exists(filt):
        text = subprocess.run([filt], input=text, capture_output=True, text=True, check=True).stdout
    shipped = set(kernel_tuples(text))
    named = {_norm(c.kernel) for c in TABLE}
    print(f"[coverage] {len(named & shipped)} of {len(shipped)} shipped gemm_kernel instantiations have a row")
    assert len(shipped) >= 1
    assert shipped - named == set(), f"instantiations without a row: {sorted(shipped - named)}"
    assert named - shipped == set(), f"rows naming kernels that are not built: {sorted(named - shipped)}"
    assert {_norm(c.kernel) for c in AUTO} <= shipped


def test_kernel_name_parser_reads_every_spelling():
    assert kernel_tuples("void (anonymous namespace)::gemm_kernel<256, false, true, 101, 8, true>(CUtensorMap_st, "
                         "(anonymous namespace)::GemmParams)") == [(256, 0, 1, 101, 8, 1)]
    assert kernel_tuples("void <unnamed>::gemm_kernel<(int)192, (bool)0, (bool)1, (int)4, (int)8, (bool)0>(...)") == \
        [(192, 0, 1, 4, 8, 0)]
    assert kernel_tuples("_ZN45_GLOBAL__N__0e256d17_12_vitk_gemm_cu_c605168811gemm_kernelILi128ELb1ELb1ELi5ELi8ELb1EEEv14CU") == \
        [(128, 1, 1, 5, 8, 1)]


@pytest.mark.parametrize("epi", [EPI_BF16, EPI_RESID])
def test_checker_rejects_a_subtly_wrong_result(epi):
    """The float64 result rounded to the output type passes; five subtly wrong results do not."""
    bn = 128
    kernel = (bn, False, False, BF16_TMA if epi == EPI_BF16 else RESID_TMA, 8, True)
    case = Case(kernel, 300, 136, 200, epi, rowscale=True, colscale=epi == EPI_RESID)
    ops = make_operands(case, "cpu")

    def run(mut=None, post=None):
        o = dict(ops)
        if mut:
            mut(o)
        res = reference(case, o)
        outs = outputs(case, ops, "cpu")
        outs["out"].view.copy_(res["out"][0].to(case.out_dtype))
        if post:
            post(outs["out"])
        return check_case(case, outs, reference(case, ops))[0]

    assert run() == []

    def drop_kblock(o):
        a = o["A"].clone()
        a[:, 64:128] = 0
        o["A"] = a

    def shift_group(o):
        o["rs_rows"] = o["rs"][(torch.arange(case.M) + 1) // ROWS_PER_GROUP]

    def bias_twice(o):
        o["bias"] = 2 * o["bias"]

    def guard(g):
        g.buf[g.lead - 1] = 0.0

    def nan_left(g):
        g.view[0, case.N - 1] = float("nan")

    for what, mut, post in (("one k-block missing", drop_kblock, None), ("rowscale group off by one", shift_group, None),
                            ("bias added twice", bias_twice, None), ("guard element changed", None, guard),
                            ("element left at its fill", None, nan_left)):
        fails = run(mut, post)
        print(f"[checker] {what}: {fails[0] if fails else 'ACCEPTED'}")
        assert fails, f"the checker accepted a result with {what}"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: one launch per row under the profiler
# ---------------------------------------------------------------------------------------------------------------------
def launch(case, ops, outs):
    from vision_transformers_torch_xla_b200 import _lib as L

    o = outs["out"]
    kw = dict(M=case.M, N=case.N, K=case.K, epilogue=case.epi, a_mn=case.a_mn, b_mn=case.b_mn, lda=ops["lda"],
              ldb=ops["ldb"], ld_out=o.ld, bias=ops.get("bias"), rowscale=ops.get("rs"), rows_per_group=ROWS_PER_GROUP,
              colscale=ops.get("cs"), splits=case.splits, block_n=case.kernel[0] if case.block_n < 0 else case.block_n)
    if "mask" in ops:
        kw.update(mask=ops["mask"], mask_scale=MASK_SCALE)
    if case.epi == EPI_RESID:
        if case.inplace:
            kw.update(resid=o.view, ld_resid=o.ld)
        else:
            r = torch.full((case.M, case.N + 8), float("nan"), device=o.buf.device)
            r[:, :case.N] = ops["resid"]
            kw.update(resid=r, ld_resid=case.N + 8)
    if case.epi == EPI_GELU:
        kw.update(aux=outs["aux"].view, ld_aux=outs["aux"].ld)
    if case.epi == EPI_DGELU:
        kw.update(aux=_padded(ops["aux"], case.N + 8, o.buf.device), ld_aux=case.N + 8)
    if case.epi == EPI_PATCH:
        kw.update(pos=ops["pos"], tokens_per_img=case.tokens, prefix=case.prefix)
    if "colsum" in outs:
        kw.update(colsum=outs["colsum"].view)
    L.gemm(ops["A_st"], ops["B_st"], o.view, **kw)


def _run(case, dev):
    from torch.profiler import ProfilerActivity, profile

    ops = make_operands(case, dev)
    outs = outputs(case, ops, dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        launch(case, ops, outs)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "gemm_kernel" in e.name]
    if not names:
        names = [a.key for a in prof.key_averages() if "gemm_kernel" in a.key for _ in range(a.count)]
    ran = [t for nm in names for t in kernel_tuples(nm)]
    assert len(ran) == 1, f"{case.id}: expected one gemm_kernel launch, the profiler saw {names}"
    assert ran[0] == _norm(case.kernel), f"{case.id}: ran gemm_kernel{ran[0]}, the row names {case.kernel}"
    fails, seen = check_case(case, outs, reference(case, ops))
    for name, got, ref, margin in seen:
        report(f"{case.id}:{name} (|err| / bound {margin:.3f})", got, ref)
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TABLE, ids=[c.id for c in TABLE])
def test_every_instantiation(cuda_device, case):
    _run(case, cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("case", AUTO, ids=[c.id for c in AUTO])
def test_automatic_tile_width_at_model_shapes(cuda_device, case):
    _run(case, cuda_device)
