"""ctypes binding of ``libvitk.so`` (C ABI declared in ``include/vitk.h``).

This is the only place where Python touches the kernel library.  Every wrapper takes torch tensors,
checks device / dtype / contiguity, and passes raw device pointers plus the current CUDA stream
through the C ABI.  There is **no fallback**: if the shared library is missing or a call fails the
wrapper raises, it never routes to PyTorch kernels or to the CPU oracle.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
from ctypes import c_double, POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_uint64, c_void_p
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
#: VITK_LIB: another build of the same sources (A/B experiments); the ABI and build-id checks
#: below still apply (VITK_ALLOW_STALE_LIB=1 for a build with different compile-time flags)
LIB_PATH = os.environ.get("VITK_LIB") or os.path.join(_HERE, "libvitk.so")

EPI_BF16, EPI_GELU, EPI_RESID, EPI_F32, EPI_DGELU, EPI_ATOMIC, EPI_PATCH = range(7)

#: every symbol include/vitk.h declares (tests check the library exports exactly these)
EXPORTED_SYMBOLS = (
    "vitk_abi_version", "vitk_last_error", "vitk_arch", "vitk_gemm_bf16", "vitk_layernorm_fwd",
    "vitk_layernorm_bwd", "vitk_attn_fwd", "vitk_attn_bwd", "vitk_attn_bwd_workspace_bytes", "vitk_patchify", "vitk_prefix_rows",
    "vitk_embed_bwd", "vitk_pool_fwd", "vitk_pool_bwd", "vitk_colsum_bf16", "vitk_ce_fwd_bwd",
    "vitk_scale_cast_bf16", "vitk_rowscale_cast_bf16", "vitk_cast_bf16", "vitk_adamw_flat", "vitk_sumsq",
    "vitk_debug_set_trace", "vitk_mixup_batch", "vitk_mixup_target", "vitk_colscale_bf16", "vitk_layerscale_grad",
    "vitk_build_id", "vitk_droppath_masks", "vitk_scale_f32", "vitk_clip_coef", "vitk_sumsq_bf16", "vitk_sumsq_scratch_floats",
    "vitk_dropout_mask", "vitk_mask_mul_bf16", "vitk_mask_mul_f32",
    "vitk_attn_fwd_dropout", "vitk_attn_bwd_dropout", "vitk_attn_bwd_dropout_workspace_bytes",
)

ABI_VERSION = 5
#: the files whose sha256 csrc/Makefile bakes into the library (same list, same order)
_BUILD_SOURCES = ("csrc/vitk_host.cu", "csrc/vitk_gemm.cu", "csrc/vitk_attn.cu", "csrc/vitk_norm.cu",
                  "csrc/vitk_elementwise.cu", "csrc/vitk_common.cuh", "csrc/vitk_internal.h", "../include/vitk.h")


def source_id(files) -> Optional[str]:
    """sha256 (first 16 hex digits) over the given source files (paths relative to this package), or None if one is missing.
    ``source_id(("csrc/vitk_gemm.cu", "csrc/vitk_common.cuh"))`` identifies the GEMM kernel's sources: an ncu capture of that
    kernel stays valid across builds that only touch other files (profiles/ncu_traffic.json: ``kernel_source_id``)."""
    import hashlib

    h = hashlib.sha256()
    try:
        for rel in files:
            with open(os.path.join(_HERE, rel), "rb") as f:
                h.update(f.read())
    except OSError:
        return None
    return h.hexdigest()[:16]


def source_build_id() -> Optional[str]:
    """sha256 (first 16 hex digits) over the kernel sources next to this package, or None if they are not there."""
    h = hashlib.sha256()
    for rel in _BUILD_SOURCES:
        path = os.path.join(_HERE, rel)
        if not os.path.exists(path):
            return None
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


class GemmArgs(Structure):
    """Mirror of ``struct vitk_gemm_args`` (include/vitk.h)."""

    _fields_ = [
        ("A", c_void_p), ("B", c_void_p), ("lda", c_int64), ("ldb", c_int64),
        ("a_mn_major", c_int32), ("b_mn_major", c_int32),
        ("M", c_int32), ("N", c_int32), ("K", c_int32), ("epilogue", c_int32),
        ("out", c_void_p), ("ld_out", c_int64), ("aux", c_void_p), ("ld_aux", c_int64),
        ("bias", c_void_p), ("resid", c_void_p), ("ld_resid", c_int64),
        ("rowscale", c_void_p), ("rows_per_group", c_int32), ("colscale", c_void_p),
        ("pos", c_void_p), ("tokens_per_img", c_int32), ("prefix", c_int32),
        ("splits", c_int32), ("block_n", c_int32), ("colsum_out", c_void_p),
        ("a_image", c_int32), ("b_image", c_int32),
        ("img_c", c_int32), ("img_h", c_int32), ("img_w", c_int32), ("img_patch", c_int32), ("img_gwp", c_int32),
        ("mask", c_void_p), ("ld_mask", c_int64), ("mask_scale", c_float),
    ]


class VitkError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load libvitk.so (built in-tree by ``__graft_entry__.build()``); raise loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VitkError(
            f"{LIB_PATH} not found: the sm_100a kernel library is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C "
            "vision_transformers_torch_xla_b200/csrc`). There is no CPU/PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.vitk_abi_version.restype = c_int32
    lib.vitk_last_error.restype = c_char_p
    lib.vitk_arch.restype = c_char_p
    if lib.vitk_abi_version() != ABI_VERSION:
        raise VitkError(f"{LIB_PATH} has ABI version {lib.vitk_abi_version()}, this binding needs {ABI_VERSION}: rebuild it "
                        "(`python -c 'import __graft_entry__ as g; g.build()'`)")
    try:
        lib.vitk_build_id.restype = c_char_p
        built = lib.vitk_build_id().decode()
    except AttributeError:
        built = "absent"
    want = source_build_id()
    if want is not None and built != want and os.environ.get("VITK_ALLOW_STALE_LIB", "0") != "1":
        raise VitkError(f"{LIB_PATH} is stale: built from sources {built}, the sources on disk hash to {want}. Rebuild it "
                        "(`python -c 'import __graft_entry__ as g; g.build()'`); set VITK_ALLOW_STALE_LIB=1 to override.")
    lib.vitk_gemm_bf16.argtypes = [POINTER(GemmArgs), c_void_p]
    lib.vitk_layernorm_fwd.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                       c_void_p, c_int64, c_int32, c_float, c_void_p]
    lib.vitk_layernorm_bwd.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int32, c_void_p,
                                       c_void_p, c_int64, c_int32, c_void_p]
    lib.vitk_attn_fwd.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p]
    lib.vitk_attn_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                  c_int32, c_float, c_void_p]
    lib.vitk_attn_bwd_workspace_bytes.argtypes = [c_int32, c_int32, c_int32, c_int32]
    lib.vitk_attn_bwd_workspace_bytes.restype = c_int64
    lib.vitk_patchify.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]
    lib.vitk_prefix_rows.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]
    lib.vitk_embed_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                   c_int32, c_int32, c_void_p]
    lib.vitk_droppath_masks.argtypes = [c_void_p, POINTER(c_float), c_int32, c_int32, c_uint64, c_uint64, c_void_p]
    lib.vitk_scale_f32.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    lib.vitk_clip_coef.argtypes = [c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p]
    lib.vitk_pool_fwd.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]
    lib.vitk_pool_bwd.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]
    lib.vitk_colsum_bf16.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p]
    lib.vitk_ce_fwd_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_float, c_float, c_void_p,
                                    c_void_p, c_void_p, c_int32, c_int32, c_void_p]
    lib.vitk_scale_cast_bf16.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]
    lib.vitk_rowscale_cast_bf16.argtypes = [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]
    lib.vitk_cast_bf16.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    lib.vitk_adamw_flat.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                    c_void_p,
                                    c_int32, c_int32, POINTER(c_float), POINTER(c_float), c_float, c_float, c_float,
                                    c_int64, c_float, c_float, c_int32, c_void_p]
    lib.vitk_sumsq.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]
    lib.vitk_sumsq_bf16.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]
    lib.vitk_sumsq_scratch_floats.restype = c_int32
    lib.vitk_dropout_mask.argtypes = [c_void_p, c_int64, c_float, c_uint64, c_uint64, c_void_p]
    lib.vitk_attn_fwd_dropout.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int32, c_int32, c_int32, c_int32,
                                          c_float, c_void_p]
    lib.vitk_attn_bwd_dropout_workspace_bytes.argtypes = [c_int32, c_int32, c_int32, c_int32]
    lib.vitk_attn_bwd_dropout_workspace_bytes.restype = c_int64
    lib.vitk_attn_bwd_dropout.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int32,
                                          c_int32, c_int32, c_int32, c_float, c_void_p]
    lib.vitk_mask_mul_bf16.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int32, c_float, c_void_p]
    lib.vitk_mask_mul_f32.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int32, c_float, c_void_p]
    lib.vitk_mixup_batch.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_double, c_int32, c_int32, c_int32, c_int32,
                                     c_int32, c_void_p]
    lib.vitk_colscale_bf16.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p]
    lib.vitk_layerscale_grad.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p]
    lib.vitk_mixup_target.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_double, c_double, c_void_p]
    lib.vitk_debug_set_trace.argtypes = [c_void_p]
    lib.vitk_debug_set_trace.restype = None
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("vitk_last_error", "vitk_arch", "vitk_abi_version", "vitk_attn_bwd_workspace_bytes",
                        "vitk_attn_bwd_dropout_workspace_bytes",
                        "vitk_debug_set_trace", "vitk_build_id", "vitk_sumsq_scratch_floats"):
            fn.restype = c_int32
    _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().vitk_last_error().decode("utf-8", "replace")
        raise VitkError(f"{what} failed (status {rc}): {msg}")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype: torch.dtype, name: str) -> None:
    if not t.is_cuda:
        raise VitkError(f"{name}: expected a CUDA tensor (the vitk kernels have no CPU path)")
    if t.dtype != dtype:
        raise VitkError(f"{name}: expected dtype {dtype}, got {t.dtype}")


# ------------------------------------------------------------------------------------------------
# launch counter (bench.py reports how many of OUR kernels ran inside the timed region)
# ------------------------------------------------------------------------------------------------
launch_count = 0
_gemm_timing = None   # list of (flops, start_event, end_event) while bench.py times the GEMM launches
_breakdown = None     # family -> list of (start_event, end_event) for the per-family time table


def _count(n: int = 1) -> None:
    global launch_count
    launch_count += n


def gemm_timing_begin() -> None:
    global _gemm_timing
    _gemm_timing = []


def gemm_timing_end():
    """(total algorithmic flops, total device ms, launches) of the GEMM launches since gemm_timing_begin()."""
    global _gemm_timing
    rec, _gemm_timing = _gemm_timing or [], None
    torch.cuda.synchronize()
    return (sum(r[0] for r in rec), sum(r[1].elapsed_time(r[2]) for r in rec), len(rec))


def gemm_timing_end_by_shape():
    """Like gemm_timing_end(), plus {family: (flops, ms, launches)} per GEMM role / shape."""
    global _gemm_timing
    rec, _gemm_timing = _gemm_timing or [], None
    torch.cuda.synchronize()
    by = {}
    for f, a, b, fam in rec:
        fl, ms, n = by.get(fam, (0.0, 0.0, 0))
        by[fam] = (fl + f, ms + a.elapsed_time(b), n + 1)
    return (sum(v[0] for v in by.values()), sum(v[1] for v in by.values()), len(rec)), by


def breakdown_begin() -> None:
    global _breakdown
    _breakdown = {}


def breakdown_end():
    global _breakdown
    rec, _breakdown = _breakdown or {}, None
    torch.cuda.synchronize()
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in rec.items()}


class _Timed:
    """Brackets one launch with CUDA events on the launching stream when a measurement is active."""

    __slots__ = ("family", "flops", "e0")

    def __init__(self, family: str, flops: float = 0.0):
        self.family, self.flops, self.e0 = family, flops, None

    def __enter__(self):
        if _breakdown is not None or (_gemm_timing is not None and self.flops):
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if self.e0 is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            if _gemm_timing is not None and self.flops:
                _gemm_timing.append((self.flops, self.e0, e1, self.family))
            if _breakdown is not None:
                _breakdown.setdefault(self.family, []).append((self.e0, e1))
        return False


# ------------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------------
def gemm(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, *, M: int, N: int, K: int, epilogue: int,
         a_mn: bool = False, b_mn: bool = False, lda: Optional[int] = None, ldb: Optional[int] = None,
         ld_out: Optional[int] = None, aux: Optional[torch.Tensor] = None, ld_aux: Optional[int] = None,
         bias: Optional[torch.Tensor] = None, resid: Optional[torch.Tensor] = None, ld_resid: Optional[int] = None,
         rowscale: Optional[torch.Tensor] = None, rows_per_group: int = 1,
         colscale: Optional[torch.Tensor] = None, pos: Optional[torch.Tensor] = None,
         tokens_per_img: int = 0, prefix: int = 0, splits: int = 0, block_n: int = 0,
         colsum: Optional[torch.Tensor] = None, image: Optional[tuple] = None,
         mask: Optional[torch.Tensor] = None, mask_scale: float = 1.0) -> None:
    """D[M,N] = opA(a) @ opB(b)^T with a fused epilogue; see ``enum vitk_epilogue`` in include/vitk.h.

    ``mask`` (uint8 [M, N], 1 = keep) with ``mask_scale = 1 / (1 - p)`` is a dropout applied inside the GELU / RESID epilogues.

    ``image = (which, C, H, W, patch, gwp)`` makes operand ``which`` ('a' or 'b') a bf16 NCHW image batch read through TMA
    as its patch matrix (im2col-free; ``struct vitk_gemm_args``: a_image / b_image)."""
    _req(a, torch.bfloat16, "gemm A")
    _req(b, torch.bfloat16, "gemm B")
    args = GemmArgs()
    args.A, args.B = a.data_ptr(), b.data_ptr()
    args.lda = lda if lda is not None else (M if a_mn else K)
    args.ldb = ldb if ldb is not None else (N if b_mn else K)
    args.a_mn_major, args.b_mn_major = int(a_mn), int(b_mn)
    args.M, args.N, args.K, args.epilogue = M, N, K, epilogue
    args.out, args.ld_out = out.data_ptr(), (ld_out if ld_out is not None else N)
    args.aux, args.ld_aux = _ptr(aux), (ld_aux if ld_aux is not None else N)
    args.bias = _ptr(bias)
    args.resid, args.ld_resid = _ptr(resid), (ld_resid if ld_resid is not None else N)
    args.rowscale, args.rows_per_group = _ptr(rowscale), rows_per_group
    if mask is not None:
        _req(mask, torch.uint8, "gemm mask")
        if mask.numel() != M * N:
            raise VitkError(f"gemm mask: expected {M} x {N} keep bytes, got {tuple(mask.shape)}")
        args.mask, args.ld_mask, args.mask_scale = mask.data_ptr(), N, float(mask_scale)
    args.colscale = _ptr(colscale)
    args.pos, args.tokens_per_img, args.prefix = _ptr(pos), tokens_per_img, prefix
    args.splits, args.block_n = splits, block_n
    args.colsum_out = _ptr(colsum)
    if image is not None:
        which, ic, ih, iw, ips, gwp = image
        args.a_image, args.b_image = int(which == "a"), int(which == "b")
        args.img_c, args.img_h, args.img_w, args.img_patch, args.img_gwp = ic, ih, iw, ips, gwp
        if which == "a":
            args.lda = 8      # unused for an image operand (the tensor map comes from the geometry); keeps the checks happy
        else:
            args.ldb = 8
    if colsum is not None:
        _req(colsum, torch.float32, "gemm colsum")
    for t, nm in ((bias, "bias"), (resid, "resid"), (rowscale, "rowscale"), (colscale, "colscale"), (pos, "pos")):
        if t is not None:
            _req(t, torch.float32, f"gemm {nm}")
    if epilogue in (EPI_GELU, EPI_DGELU):
        if aux is None:
            raise VitkError("gemm: the GELU epilogues need the aux (derivative) buffer")
        _req(aux, torch.bfloat16, "gemm aux")
    role = "wgrad" if epilogue == EPI_ATOMIC else ("dgrad" if b_mn else "fprop")
    with _Timed(f"gemm.{role}.epi{epilogue} {M}x{N}x{K}", 2.0 * M * N * K):
        _check(load().vitk_gemm_bf16(ctypes.byref(args), _stream()), "vitk_gemm_bf16")
    _count()


# ------------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------------
def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, y: torch.Tensor,
                  mean: Optional[torch.Tensor], rstd: Optional[torch.Tensor], rows: int, dim: int,
                  eps: float, ld_x: Optional[int] = None, ld_y: Optional[int] = None) -> None:
    _req(x, torch.float32, "layernorm x")
    _req(y, torch.bfloat16, "layernorm y")
    _req(gamma, torch.float32, "layernorm gamma")
    with _Timed("layernorm_fwd"):
        _check(load().vitk_layernorm_fwd(x.data_ptr(), ld_x or dim, gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                         ld_y or dim, _ptr(mean), _ptr(rstd), rows, dim, eps, _stream()),
               "vitk_layernorm_fwd")
    _count()


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, gamma: torch.Tensor,
                  g_in: Optional[torch.Tensor], g_out: torch.Tensor, gb_out: Optional[torch.Tensor],
                  rowscale: Optional[torch.Tensor], rows_per_group: int, dgamma: Optional[torch.Tensor],
                  dbeta: Optional[torch.Tensor], rows: int, dim: int, ld_x: Optional[int] = None,
                  ld_dy: Optional[int] = None, ld_g: Optional[int] = None) -> None:
    _req(dy, torch.bfloat16, "layernorm_bwd dy")
    _req(x, torch.float32, "layernorm_bwd x")
    _req(g_out, torch.float32, "layernorm_bwd g_out")
    with _Timed("layernorm_bwd"):
        _check(load().vitk_layernorm_bwd(dy.data_ptr(), ld_dy or dim, x.data_ptr(), ld_x or dim, mean.data_ptr(),
                                         rstd.data_ptr(), gamma.data_ptr(), _ptr(g_in), g_out.data_ptr(), ld_g or dim,
                                         _ptr(gb_out), _ptr(rowscale), rows_per_group, _ptr(dgamma), _ptr(dbeta), rows,
                                         dim, _stream()), "vitk_layernorm_bwd")
    _count()


# ------------------------------------------------------------------------------------------------
# Attention
# ------------------------------------------------------------------------------------------------
def _req_attn_mask(mask: torch.Tensor, B: int, N: int, H: int) -> None:
    _req(mask, torch.uint8, "attn keep mask")
    if mask.numel() != B * H * N * N:
        raise VitkError(f"attn keep mask: expected {B} x {H} x {N} x {N} keep bytes, got {tuple(mask.shape)}")


def attn_fwd(qkv: torch.Tensor, out: torch.Tensor, lse: torch.Tensor, B: int, N: int, H: int, hd: int,
             scale: float, keep_mask: Optional[torch.Tensor] = None, keep_scale: float = 1.0) -> None:
    """``keep_mask`` (uint8 [B, H, N, N], 1 = keep) with ``keep_scale = 1 / (1 - p)``: attention dropout on the softmax."""
    _req(qkv, torch.bfloat16, "attn qkv")
    _req(out, torch.bfloat16, "attn out")
    _req(lse, torch.float32, "attn lse")
    with _Timed("attn_fwd"):
        if keep_mask is None:
            _check(load().vitk_attn_fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, N, H, hd, scale, _stream()),
                   "vitk_attn_fwd")
        else:
            _req_attn_mask(keep_mask, B, N, H)
            _check(load().vitk_attn_fwd_dropout(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), keep_mask.data_ptr(),
                                                float(keep_scale), B, N, H, hd, scale, _stream()), "vitk_attn_fwd_dropout")
    _count()


def attn_bwd(qkv: torch.Tensor, out: torch.Tensor, dout: torch.Tensor, lse: torch.Tensor, dqkv: torch.Tensor,
             B: int, N: int, H: int, hd: int, scale: float, keep_mask: Optional[torch.Tensor] = None,
             keep_scale: float = 1.0) -> None:
    for t, nm in ((qkv, "qkv"), (out, "out"), (dout, "dout"), (dqkv, "dqkv")):
        _req(t, torch.bfloat16, f"attn_bwd {nm}")
    lib = load()
    ws_bytes = (lib.vitk_attn_bwd_workspace_bytes if keep_mask is None else lib.vitk_attn_bwd_dropout_workspace_bytes)(B, N, H, hd)
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=qkv.device) if ws_bytes > 0 else None
    with _Timed("attn_bwd"):
        if keep_mask is None:
            _check(lib.vitk_attn_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), dqkv.data_ptr(),
                                     _ptr(ws), B, N, H, hd, scale, _stream()), "vitk_attn_bwd")
        else:
            _req_attn_mask(keep_mask, B, N, H)
            _check(lib.vitk_attn_bwd_dropout(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), dqkv.data_ptr(),
                                             _ptr(ws), keep_mask.data_ptr(), float(keep_scale), B, N, H, hd, scale, _stream()),
                   "vitk_attn_bwd_dropout")
    _count()


# ------------------------------------------------------------------------------------------------
# embedding / pooling / reductions
# ------------------------------------------------------------------------------------------------
def patchify(img: torch.Tensor, patches: torch.Tensor, ps: int) -> None:
    _req(img, torch.float32, "patchify img")
    _req(patches, torch.bfloat16, "patchify out")
    B, C, H, W = img.shape
    with _Timed("patchify"):
        _check(load().vitk_patchify(img.data_ptr(), patches.data_ptr(), B, C, H, W, ps, _stream()), "vitk_patchify")
    _count()


def prefix_rows(x: torch.Tensor, tok: torch.Tensor, pos: torch.Tensor, B: int, N: int, D: int, prefix: int) -> None:
    _req(x, torch.float32, "prefix_rows x")
    with _Timed("prefix_rows"):
        _check(load().vitk_prefix_rows(x.data_ptr(), tok.data_ptr(), pos.data_ptr(), B, N, D, prefix, _stream()),
               "vitk_prefix_rows")
    _count()


def embed_bwd(g: torch.Tensor, gp: Optional[torch.Tensor], dpos: Optional[torch.Tensor],
              dprefix0: Optional[torch.Tensor], dprefix1: Optional[torch.Tensor], B: int, N: int, D: int, prefix: int,
              gw: int = 0, gwp: int = 0) -> None:
    """dpos / dprefix0 / dprefix1 are ACCUMULATED into (pos_embed / cls_token / dist_token gradient rows).  ``gw > 0``: gp
    is laid out in the padded row order of an image operand, [B * (P / gw) * gwp, D], pad rows zeroed."""
    _req(g, torch.float32, "embed_bwd g")
    for t in (dpos, dprefix0, dprefix1):
        if t is not None:
            _req(t, torch.float32, "embed_bwd gradient row")
    with _Timed("embed_bwd"):
        _check(load().vitk_embed_bwd(g.data_ptr(), _ptr(gp), _ptr(dpos), _ptr(dprefix0), _ptr(dprefix1), B, N, D, prefix,
                                     gw, gwp, _stream()), "vitk_embed_bwd")
    _count()


def droppath_masks(rs: torch.Tensor, drop_probs, seed: int, offset: int) -> None:
    """rs fp32 [rows, B] <- Bernoulli(1 - p[row]) / (1 - p[row]); one launch for every DropPath of a forward pass."""
    _req(rs, torch.float32, "droppath_masks rs")
    rows, B = rs.shape
    arr = (c_float * rows)(*[float(p) for p in drop_probs])
    with _Timed("droppath_masks"):
        _check(load().vitk_droppath_masks(rs.data_ptr(), arr, rows, B, seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFFFFFFFFFF,
                                          _stream()), "vitk_droppath_masks")
    _count()


def dropout_mask(mask: torch.Tensor, p: float, seed: int, offset: int) -> None:
    """mask uint8 (any shape, contiguous) <- 1 with probability 1 - p, else 0."""
    _req(mask, torch.uint8, "dropout_mask mask")
    with _Timed("dropout_mask"):
        _check(load().vitk_dropout_mask(mask.data_ptr(), mask.numel(), float(p), seed & 0xFFFFFFFFFFFFFFFF,
                                        offset & 0xFFFFFFFFFFFFFFFF, _stream()), "vitk_dropout_mask")
    _count()


def mask_mul_(x: torch.Tensor, mask: torch.Tensor, scale: float, rows: int, cols: int, ld_x: Optional[int] = None) -> None:
    """x[r, c] *= mask[r, c] ? scale : 0 in place (x bf16 or fp32, viewed as [rows, cols] with row pitch ``ld_x``)."""
    _req(mask, torch.uint8, "mask_mul mask")
    if mask.numel() != rows * cols:
        raise VitkError(f"mask_mul: expected {rows} x {cols} keep bytes, got {tuple(mask.shape)}")
    ld = cols if ld_x is None else ld_x
    with _Timed("mask_mul"):
        if x.dtype == torch.bfloat16:
            _req(x, torch.bfloat16, "mask_mul x")
            _check(load().vitk_mask_mul_bf16(x.data_ptr(), ld, mask.data_ptr(), cols, rows, cols, float(scale), _stream()),
                   "vitk_mask_mul_bf16")
        else:
            _req(x, torch.float32, "mask_mul x")
            _check(load().vitk_mask_mul_f32(x.data_ptr(), ld, mask.data_ptr(), cols, rows, cols, float(scale), _stream()),
                   "vitk_mask_mul_f32")
    _count()


def scale_f32_(x: torch.Tensor, scale: torch.Tensor) -> None:
    """x *= scale[0] in place; ``scale`` is a device scalar (no host sync)."""
    _req(x, torch.float32, "scale_f32 x")
    _req(scale, torch.float32, "scale_f32 scale")
    with _Timed("scale_f32"):
        _check(load().vitk_scale_f32(x.data_ptr(), scale.data_ptr(), x.numel(), _stream()), "vitk_scale_f32")
    _count()


def clip_coef(sumsq_t: torch.Tensor, grad_scale: float, max_norm: float, coef: torch.Tensor,
              norm: Optional[torch.Tensor]) -> None:
    for t in (sumsq_t, coef):
        _req(t, torch.float32, "clip_coef")
    with _Timed("clip_coef"):
        _check(load().vitk_clip_coef(sumsq_t.data_ptr(), grad_scale, max_norm, coef.data_ptr(), _ptr(norm), _stream()),
               "vitk_clip_coef")
    _count()


def pool_fwd(x: torch.Tensor, pooled: torch.Tensor, B: int, N: int, D: int, prefix: int, mode: int) -> None:
    _req(x, torch.float32, "pool x")
    with _Timed("pool_fwd"):
        _check(load().vitk_pool_fwd(x.data_ptr(), pooled.data_ptr(), B, N, D, prefix, mode, _stream()), "vitk_pool_fwd")
    _count()


def pool_bwd(dpooled: torch.Tensor, g: torch.Tensor, B: int, N: int, D: int, prefix: int, mode: int) -> None:
    _req(dpooled, torch.float32, "pool_bwd dpooled")
    with _Timed("pool_bwd"):
        _check(load().vitk_pool_bwd(dpooled.data_ptr(), g.data_ptr(), B, N, D, prefix, mode, _stream()), "vitk_pool_bwd")
    _count()


def colsum_bf16(x: torch.Tensor, out: torch.Tensor, rows: int, cols: int, ld: Optional[int] = None) -> None:
    _req(x, torch.bfloat16, "colsum x")
    _req(out, torch.float32, "colsum out")
    with _Timed("colsum_bf16"):
        _check(load().vitk_colsum_bf16(x.data_ptr(), ld or cols, out.data_ptr(), rows, cols, _stream()), "vitk_colsum_bf16")
    _count()


# ------------------------------------------------------------------------------------------------
# loss / casts
# ------------------------------------------------------------------------------------------------
def ce_fwd_bwd(logits: torch.Tensor, soft: Optional[torch.Tensor], labels: Optional[torch.Tensor], smoothing: float,
               teacher: Optional[torch.Tensor], alpha: float, temp: float, loss: torch.Tensor,
               dlogits: torch.Tensor, scratch: torch.Tensor) -> None:
    _req(logits, torch.float32, "ce logits")
    B, C = logits.shape
    if soft is not None:
        _req(soft, torch.float32, "ce soft targets")
    if labels is not None:
        _req(labels, torch.int64, "ce labels")
    if teacher is not None:
        _req(teacher, torch.float32, "ce teacher logits")
    with _Timed("ce_fwd_bwd"):
        _check(load().vitk_ce_fwd_bwd(logits.data_ptr(), _ptr(soft), _ptr(labels), smoothing, _ptr(teacher), alpha, temp,
                                      loss.data_ptr(), dlogits.data_ptr(), scratch.data_ptr(), B, C, _stream()),
               "vitk_ce_fwd_bwd")
    _count(2)


def scale_cast_bf16(src: torch.Tensor, scale: Optional[torch.Tensor], dst: torch.Tensor) -> None:
    _req(src, torch.float32, "scale_cast src")
    _req(dst, torch.bfloat16, "scale_cast dst")
    with _Timed("scale_cast_bf16"):
        _check(load().vitk_scale_cast_bf16(src.data_ptr(), _ptr(scale), dst.data_ptr(), src.numel(), _stream()),
               "vitk_scale_cast_bf16")
    _count()


def rowscale_cast_bf16(src: torch.Tensor, rowscale: Optional[torch.Tensor], elems_per_group: int,
                       dst: torch.Tensor) -> None:
    _req(src, torch.float32, "rowscale_cast src")
    _req(dst, torch.bfloat16, "rowscale_cast dst")
    with _Timed("rowscale_cast_bf16"):
        _check(load().vitk_rowscale_cast_bf16(src.data_ptr(), _ptr(rowscale), elems_per_group, dst.data_ptr(),
                                              src.numel(), _stream()), "vitk_rowscale_cast_bf16")
    _count()


def cast_bf16(src: torch.Tensor, dst: torch.Tensor) -> None:
    scale_cast_bf16(src, None, dst)


# ------------------------------------------------------------------------------------------------
# optimizer
# ------------------------------------------------------------------------------------------------
def adamw_flat(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, shadow: Optional[torch.Tensor],
               ema: Optional[torch.Tensor], chunk_group: Optional[torch.Tensor], chunk: int, lrs, wds, beta1: float,
               beta2: float, eps: float, step: int, grad_scale: float = 1.0, ema_decay: float = 0.0,
               zero_grad: bool = False, g_bf16: Optional[torch.Tensor] = None,
               grad_scale_dev: Optional[torch.Tensor] = None) -> None:
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _req(t, torch.float32, f"adamw {nm}")
    if g_bf16 is not None:
        _req(g_bf16, torch.bfloat16, "adamw g_bf16")
        if g_bf16.numel() != p.numel():
            raise VitkError("adamw: g_bf16 must have as many elements as p")
    if grad_scale_dev is not None:
        _req(grad_scale_dev, torch.float32, "adamw grad_scale_dev")
    n = p.numel()
    ng = len(lrs)
    lr_arr = (c_float * ng)(*[float(x) for x in lrs])
    wd_arr = (c_float * ng)(*[float(x) for x in wds])
    with _Timed("adamw_flat"):
        _check(load().vitk_adamw_flat(p.data_ptr(), g.data_ptr(), _ptr(g_bf16), _ptr(grad_scale_dev), m.data_ptr(),
                                      v.data_ptr(), _ptr(shadow), _ptr(ema), n, _ptr(chunk_group), chunk, ng, lr_arr, wd_arr,
                                      beta1, beta2, eps, step, grad_scale, ema_decay, int(zero_grad), _stream()),
               "vitk_adamw_flat")
    _count()


def sumsq(x: torch.Tensor, out: torch.Tensor) -> None:
    """out[0] += sum(x^2); x fp32 or bf16.  Deterministic (no floating-point atomics): ranks holding the same reduced
    gradient get the same bits."""
    _req(out, torch.float32, "sumsq out")
    if not x.is_cuda or x.dtype not in (torch.float32, torch.bfloat16):
        raise VitkError(f"sumsq x: expected a float32 / bfloat16 CUDA tensor, got {x.dtype} on {x.device}")
    lib = load()
    fn = lib.vitk_sumsq if x.dtype == torch.float32 else lib.vitk_sumsq_bf16
    scratch = torch.empty(lib.vitk_sumsq_scratch_floats(), dtype=torch.float32, device=x.device)
    with _Timed("sumsq"):
        _check(fn(x.data_ptr(), x.numel(), out.data_ptr(), scratch.data_ptr(), _stream()), "vitk_sumsq")
    _count(2)


# ------------------------------------------------------------------------------------------------
# Mixup / CutMix
# ------------------------------------------------------------------------------------------------
def mixup_batch(x: torch.Tensor, lam: float, use_cutmix: bool = False, box=(0, 0, 0, 0)) -> None:
    """In place on fp32 NCHW ``x``: image b mixed with image B-1-b (mixup) or the box copied over (cutmix)."""
    _req(x, torch.float32, "mixup x")
    B, C, H, W = x.shape
    yl, yh, xl, xh = (int(v) for v in box)
    with _Timed("mixup_batch"):
        _check(load().vitk_mixup_batch(x.data_ptr(), B, C, H, W, float(lam), int(use_cutmix), yl, yh, xl, xh, _stream()),
               "vitk_mixup_batch")
    _count()


def mixup_target(labels: torch.Tensor, out: torch.Tensor, lam: float, smoothing: float) -> None:
    _req(labels, torch.int64, "mixup labels")
    _req(out, torch.float32, "mixup targets")
    B, C = out.shape
    with _Timed("mixup_target"):
        _check(load().vitk_mixup_target(labels.data_ptr(), out.data_ptr(), B, C, float(lam), float(smoothing), _stream()),
               "vitk_mixup_target")
    _count()


# ------------------------------------------------------------------------------------------------
# LayerScale (backward side; the forward is the residual GEMM's colscale)
# ------------------------------------------------------------------------------------------------
def colscale_bf16(x: torch.Tensor, gamma: torch.Tensor, rows: int, dim: int) -> None:
    _req(x, torch.bfloat16, "colscale x")
    _req(gamma, torch.float32, "colscale gamma")
    with _Timed("colscale_bf16"):
        _check(load().vitk_colscale_bf16(x.data_ptr(), gamma.data_ptr(), rows, dim, _stream()), "vitk_colscale_bf16")
    _count()


def layerscale_grad(W: torch.Tensor, dW: torch.Tensor, bias: Optional[torch.Tensor], dbias: Optional[torch.Tensor],
                    gamma: torch.Tensor, dgamma: torch.Tensor) -> None:
    for t, nm in ((W, "W"), (dW, "dW"), (gamma, "gamma"), (dgamma, "dgamma")):
        _req(t, torch.float32, f"layerscale_grad {nm}")
    C, K = W.shape
    with _Timed("layerscale_grad"):
        _check(load().vitk_layerscale_grad(W.data_ptr(), dW.data_ptr(), _ptr(bias), _ptr(dbias), gamma.data_ptr(),
                                           dgamma.data_ptr(), C, K, _stream()), "vitk_layerscale_grad")
    _count()
