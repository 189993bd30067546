"""The C-ABI shared library: loads without a GPU, exports every symbol include/vitk.h declares, its argument
struct matches the ctypes mirror, and argument validation fails loudly through the error slot (no compute
call is made here: every call below is rejected before any CUDA work)."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitk.h")


@pytest.fixture(scope="module")
def lib():
    from vision_transformers_torch_xla_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return _lib.load()


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vitk_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(lib):
    from vision_transformers_torch_xla_b200 import _lib

    declared = _declared_symbols()
    assert len(declared) >= 19
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/vitk.h but not exported by libvitk.so"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared, "python binding and header disagree on the symbol list"


def test_abi_version_and_arch(lib):
    from vision_transformers_torch_xla_b200 import _lib

    src = open(HEADER).read()
    assert lib.vitk_abi_version() == _lib.ABI_VERSION == int(re.search(r"#define VITK_ABI_VERSION (\d+)", src).group(1))
    assert lib.vitk_arch() == b"sm_100a"


def test_build_id_ties_the_binary_to_the_sources(lib, monkeypatch, tmp_path):
    """libvitk.so carries the sha256 of the sources it was built from; load() refuses a binary that does not match the
    sources next to it (a stale .so shipped with newer sources would otherwise go unnoticed)."""
    from vision_transformers_torch_xla_b200 import _lib

    lib.vitk_build_id.restype = ctypes.c_char_p
    assert lib.vitk_build_id().decode() == _lib.source_build_id()
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "source_build_id", lambda: "0" * 16)
    with pytest.raises(_lib.VitkError, match="stale"):
        _lib.load()


def test_header_is_plain_c_and_struct_layout_matches_ctypes(tmp_path):
    """include/vitk.h must compile as C (it is the FFI contract) and agree with _lib.GemmArgs."""
    from vision_transformers_torch_xla_b200._lib import GemmArgs

    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vitk.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(vitk_gemm_args), offsetof(vitk_gemm_args, M),'
                   ' offsetof(vitk_gemm_args, out), offsetof(vitk_gemm_args, rowscale), offsetof(vitk_gemm_args, block_n));'
                   'return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    size, off_m, off_out, off_rs, off_bn = map(int, subprocess.run([str(exe)], check=True, capture_output=True,
                                                                   text=True).stdout.split())
    assert size == ctypes.sizeof(GemmArgs)
    assert off_m == GemmArgs.M.offset and off_out == GemmArgs.out.offset
    assert off_rs == GemmArgs.rowscale.offset and off_bn == GemmArgs.block_n.offset


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    """tcgen05.mma -> UTCHMMA, tcgen05.ld -> LDTM, TMA -> UTMALDG must be in the shipped binary."""
    from vision_transformers_torch_xla_b200 import _lib

    out = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG", "UTCBAR"):
        assert mnemonic in out.stdout, mnemonic
    assert "HMMA.16816" not in out.stdout  # no legacy mma.sync tensor path


def test_argument_validation_reports_through_error_slot(lib):
    from vision_transformers_torch_xla_b200._lib import GemmArgs

    args = GemmArgs()
    args.M, args.N, args.K = 0, 16, 64
    rc = lib.vitk_gemm_bf16(ctypes.byref(args), None)
    assert rc < 0 and b"empty problem" in lib.vitk_last_error()
    assert lib.vitk_gemm_bf16(None, None) < 0
    # an epilogue code outside enum vitk_epilogue is refused by the dispatcher; the pointers are fake but 16-byte
    # aligned, so the call gets past the entry checks and still makes no CUDA call
    args = GemmArgs()
    args.A = args.B = args.out = 256
    args.lda = args.ldb = args.ld_out = 64
    args.M, args.N, args.K, args.epilogue = 128, 64, 64, 7
    rc = lib.vitk_gemm_bf16(ctypes.byref(args), None)
    assert rc == -6 and b"epi=7" in lib.vitk_last_error()   # VITK_STATUS_UNSUPPORTED
    rc = lib.vitk_attn_fwd(None, None, None, 1, 16, 1, 96, ctypes.c_float(1.0), None)
    assert rc == -6 and b"head_dim" in lib.vitk_last_error()  # VITK_STATUS_UNSUPPORTED (wider than a head tile + its tail)
    rc = lib.vitk_attn_fwd(None, None, None, 1, 300, 1, 72, ctypes.c_float(1.0), None)
    assert rc == -6 and b"N <= 256" in lib.vitk_last_error()   # heads of 72 / 80: sequences of at most 256 tokens
    rc = lib.vitk_layernorm_fwd(None, 770, None, None, None, 770, None, None, 4, 770, ctypes.c_float(1e-6), None)
    assert rc < 0 and b"multiple of 4" in lib.vitk_last_error()
    rc = lib.vitk_adamw_flat(None, None, None, None, None, None, None, None, 6, None, 64, 1, None, None, ctypes.c_float(0.9),
                             ctypes.c_float(0.999), ctypes.c_float(1e-8), 1, ctypes.c_float(1.0), ctypes.c_float(0.0), 0, None)
    assert rc < 0
    probs = (ctypes.c_float * 2)(0.1, 1.5)
    rc = lib.vitk_droppath_masks(ctypes.c_void_p(16), probs, 2, 4, 0, 0, None)
    assert rc < 0 and b"drop_probs" in lib.vitk_last_error()


@pytest.mark.parametrize("field", ["bias", "colscale", "pos", "resid", "aux"])
def test_gemm_rejects_misaligned_side_operands(lib, field):
    """The epilogues read bias / colscale / pos / resid with float4 loads and aux with 16-byte loads or TMA, so each must be
    16-byte aligned whatever the epilogue.  The call carries epilogue code 7, which the dispatcher refuses ("epi=7") before
    any CUDA call: a missing entry check fails this test instead of launching a kernel on a fake pointer."""
    from vision_transformers_torch_xla_b200._lib import GemmArgs

    args = GemmArgs()
    args.A = args.B = args.out = 256
    args.lda = args.ldb = args.ld_out = args.ld_aux = args.ld_resid = 64
    args.M, args.N, args.K, args.epilogue = 128, 64, 64, 7
    setattr(args, field, 256 + 4)
    rc = lib.vitk_gemm_bf16(ctypes.byref(args), None)
    assert rc == -2, lib.vitk_last_error()   # VITK_STATUS_ALIGN
    assert field.encode() in lib.vitk_last_error()


_FAKE = 1 << 20   # a 16-byte aligned fake device address; no call below reaches a kernel


def _ln_bwd(lib, ptrs):
    p = dict(dy=_FAKE, x=_FAKE, mean=_FAKE, rstd=_FAKE, gamma=_FAKE, g_in=_FAKE, g_out=_FAKE, gb_out=_FAKE, rowscale=None,
             dgamma=_FAKE, dbeta=_FAKE)
    p.update(ptrs)
    return lib.vitk_layernorm_bwd(p["dy"], 768, p["x"], 768, p["mean"], p["rstd"], p["gamma"], p["g_in"], p["g_out"], 768,
                                  p["gb_out"], p["rowscale"], 197, p["dgamma"], p["dbeta"], 0, 768, None)   # rows = 0


def _adamw(lib, ptrs, g_bf16=None, zero_grad=0):
    p = dict(p=_FAKE, g=_FAKE, g_bf16=g_bf16, m=_FAKE, v=_FAKE, shadow=_FAKE, ema=_FAKE)
    p.update(ptrs)
    lr, wd = (ctypes.c_float * 1)(1e-3), (ctypes.c_float * 1)(0.05)
    return lib.vitk_adamw_flat(p["p"], p["g"], p["g_bf16"], None, p["m"], p["v"], p["shadow"], p["ema"], 0, None, 0, 1, lr, wd,
                               ctypes.c_float(0.9), ctypes.c_float(0.999), ctypes.c_float(1e-8), 1, ctypes.c_float(1.0),
                               ctypes.c_float(0.0), zero_grad, None)   # n = 0


def _pool_fwd(lib, ptrs):
    p = dict(x=_FAKE, pooled=_FAKE)
    p.update(ptrs)
    return lib.vitk_pool_fwd(p["x"], p["pooled"], 0, 197, 768, 1, 0, None)   # B = 0


def _pool_bwd(lib, ptrs):
    p = dict(dpooled=_FAKE, g=_FAKE)
    p.update(ptrs)
    return lib.vitk_pool_bwd(p["dpooled"], p["g"], 0, 197, 768, 1, 0, None)   # B = 0


def _embed_bwd(lib, ptrs):
    p = dict(g=_FAKE, gp=_FAKE)
    p.update(ptrs)
    return lib.vitk_embed_bwd(p["g"], p["gp"], _FAKE, _FAKE, None, 0, 197, 768, 1, 14, 16, None)   # B = 0


def _colsum(lib, ptrs):
    p = dict(x=_FAKE)
    p.update(ptrs)
    return lib.vitk_colsum_bf16(p["x"], 768, _FAKE, 0, 768, None)   # rows = 0


# (entry point, pointer, status the call returns with every pointer aligned: 0 = VITK_STATUS_OK, -1 = VITK_STATUS_SHAPE)
_ALIGN_CASES = [(_ln_bwd, nm, 0) for nm in ("x", "g_in", "g_out", "gamma", "dy", "gb_out", "dgamma", "dbeta")] + \
               [(_adamw, nm, 0) for nm in ("p", "g", "g_bf16", "m", "v", "shadow", "ema")] + \
               [(_pool_fwd, "x", -1), (_pool_fwd, "pooled", -1), (_pool_bwd, "dpooled", -1), (_pool_bwd, "g", -1),
                (_embed_bwd, "g", -1), (_embed_bwd, "gp", -1), (_colsum, "x", 0)]


@pytest.mark.parametrize("fn,name,aligned_rc", _ALIGN_CASES,
                         ids=[f"{fn.__name__[1:]}-{nm}" for fn, nm, _ in _ALIGN_CASES])
def test_misaligned_vector_pointers_are_refused(lib, fn, name, aligned_rc):
    """Every pointer the LayerNorm backward, AdamW, pooling, embedding-backward and column-sum kernels access as 16- or
    8-byte vectors is checked before the shape and before the early return of an empty problem.  Each call has rows,
    n or B = 0, so with the check missing it returns VITK_STATUS_OK or a shape error and no kernel ever runs on the fake
    pointer, which is off by 4 bytes."""
    assert fn(lib, {}) == aligned_rc, lib.vitk_last_error()
    rc = fn(lib, {name: _FAKE + 4})
    assert rc == -2, lib.vitk_last_error()   # VITK_STATUS_ALIGN
    assert f": {name} must be".encode() in lib.vitk_last_error()


def test_adamw_ignores_the_alignment_of_a_gradient_it_does_not_touch(lib):
    """With a bf16 gradient and zero_grad off, adamw_flat neither reads nor writes g."""
    assert _adamw(lib, {"g": _FAKE + 4}, g_bf16=_FAKE) == 0, lib.vitk_last_error()
    assert _adamw(lib, {"g": _FAKE + 4}, g_bf16=_FAKE, zero_grad=1) == -2
    assert _adamw(lib, {"g": _FAKE + 4}) == -2


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from vision_transformers_torch_xla_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.VitkError, match="no CPU/PyTorch fallback"):
        _lib.load()
