"""The C-ABI library loads here (no GPU) and exports every symbol include/mmr_b200.h declares; argument
errors are reported through status codes + mmr_last_error; device work fails loudly without a GPU."""
import ctypes as C
import importlib
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "multimodal-rag-for-image-text-search_b200"
native = importlib.import_module(PKG + "._native")


def _declared():
    text = open(os.path.join(ROOT, "include", "mmr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mmr_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_in_tree():
    assert os.path.exists(native.LIB_PATH), "run __graft_entry__.build() first"
    assert os.path.dirname(native.LIB_PATH).startswith(ROOT)


def test_exports_every_declared_symbol():
    handle = C.CDLL(native.LIB_PATH)
    declared = _declared()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/mmr_b200.h but not exported"
    bound = {s[0] for s in native.SYMBOLS}
    assert bound == set(declared), f"binding and header disagree: {bound ^ set(declared)}"
    assert handle.mmr_abi_version() == native.ABI_VERSION


def test_argument_errors_have_messages():
    lib = native.lib()
    out = C.c_void_p()
    assert lib.mmr_index_create(0, 512, 99, 10, None, None, 0, 0, C.byref(out)) == 1  # MMR_ERR_INVALID
    assert b"dtype" in lib.mmr_last_error()
    assert lib.mmr_index_create(0, 500, 0, 0, None, None, 0, 0, C.byref(out)) == 3    # MMR_ERR_UNSUPPORTED
    assert b"384" in lib.mmr_last_error()
    assert lib.mmr_search(None, None, None, 1, 10, None, None, None, 0, None) == 1
    assert lib.mmr_merge_topk(None, None, 0, 1, 10, None, None, None) == 1
    assert lib.mmr_fuse(None, None, 0, None, None, 0, 0, 4, 0.25, None, None, None, None, None, None) == 1
    assert lib.mmr_search_workspace_bytes(None, 1, 10) == 0
    assert lib.mmr_get_option(b"MMR_UMMA_LOCKSTEP") == -1                          # unknown switch
    assert lib.mmr_set_option(b"MMR_UMMA_MODE", b"ts") == 1
    assert b"unknown option" in lib.mmr_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_cpu_fallback():
    lib = native.lib()
    out = C.c_void_p()
    rc = lib.mmr_index_create(0, 512, 0, 0, None, None, 0, 0, C.byref(out))
    assert rc == 2, "without a GPU the library must fail with MMR_ERR_CUDA, not fall back"   # MMR_ERR_CUDA
    pkg = importlib.import_module(PKG)
    with pytest.raises(pkg.NativeError):
        pkg.B200Store()
    with pytest.raises(pkg.NativeError):
        pkg.ResidentIndex(torch.zeros(8, 512, dtype=torch.bfloat16))


def test_encoder_debug_hooks_reject_bad_arguments():
    """mmr_debug_enc_gemm / _attention / _layernorm check every argument before any CUDA call: MMR_ERR_INVALID and a message
    naming what is wrong (the buffers below are never dereferenced)."""
    lib = native.lib()
    buf = (C.c_float * 64)()
    p = C.addressof(buf)                                   # 16-byte aligned, stands in for a device buffer
    odd = p + 2

    def gemm(epi=0, nt=64, fold=0, M=64, N=128, K=64, x=p, src=None, g=None, b=None, ln_out=None, w=p, res=None, o32=p, o16=p):
        return lib.mmr_debug_enc_gemm(epi, nt, fold, M, N, K, x, src, g, b, 1e-5, ln_out, w, None, res, o32, o16, None)

    cases = [
        (dict(epi=4), b"epilogue"), (dict(epi=-1), b"epilogue"),
        (dict(nt=32), b"token tile"), (dict(nt=512), b"token tile"),
        (dict(fold=2), b"fold_ln"),
        (dict(M=0), b"M = 0"),
        (dict(N=192), b"N = 192"), (dict(N=0), b"N = 0"),
        (dict(K=96), b"K = 96"), (dict(K=0), b"K = 0"),
        (dict(w=None), b"W must"), (dict(w=odd), b"W must"),
        (dict(x=None), b"X must"), (dict(x=odd), b"X must"),
        (dict(fold=1, nt=128, K=384, src=p, g=p, b=p), b"64-token tile"),
        (dict(fold=1, K=1536, src=p, g=p, b=p), b"K = 384 or 512"),
        (dict(fold=1, K=384, epi=1, src=p, g=p, b=p, res=p), b"no residual"),
        (dict(fold=1, K=384, g=p, b=p), b"ln_src"),
        (dict(fold=1, K=384, src=p, b=p), b"ln_g"),
        (dict(fold=1, K=384, src=p, g=p), b"ln_b"),
        (dict(fold=1, K=384, src=p, g=p, b=p, ln_out=p), b"alias"),
        (dict(epi=0, o32=None), b"out_f32"),
        (dict(epi=1, res=p, o32=None), b"out_f32"),
        (dict(epi=1, res=None), b"residual"),
        (dict(epi=2, o16=None), b"out_bf16"),
        (dict(epi=3, o16=None), b"out_bf16"),
    ]
    for kw, words in cases:
        assert gemm(**kw) == 1, kw                          # MMR_ERR_INVALID
        assert words in lib.mmr_last_error(), (kw, lib.mmr_last_error())

    def att(tc=0, B=1, S=64, H=384, heads=12, causal=0, qkv=p, mask=None, ctx=p):
        return lib.mmr_debug_enc_attention(tc, B, S, H, heads, causal, qkv, mask, ctx, None)

    cases = [
        (dict(tc=2), b"tensor_cores"), (dict(causal=-1), b"causal"),
        (dict(H=768), b"hidden 768"), (dict(heads=0), b"heads 0"), (dict(heads=4), b"heads 4"), (dict(heads=5), b"heads 5"),
        (dict(B=0), b"B = 0"), (dict(S=0), b"S = 0"), (dict(S=513), b"S = 513"),
        (dict(qkv=None), b"qkv and ctx"), (dict(ctx=None), b"qkv and ctx"), (dict(qkv=odd), b"qkv and ctx"),
    ]
    for kw, words in cases:
        assert att(**kw) == 1, kw
        assert words in lib.mmr_last_error(), (kw, lib.mmr_last_error())
    # head dim 64 on the fp32 kernel ends at 330 tokens (MMR_ERR_UNSUPPORTED, before any CUDA call)
    assert att(S=331, heads=6) == 3 and b"fp32 attention kernel" in lib.mmr_last_error()
    assert att(S=512, H=512, heads=8) == 3 and b"330 tokens at most" in lib.mmr_last_error()

    def ln(H=384, M=4, x=p, g=p, b=p, o32=p, o16=None):
        return lib.mmr_debug_enc_layernorm(H, M, x, g, b, 1e-5, o32, o16, None)

    for kw, words in [(dict(H=256), b"H = 256"), (dict(M=0), b"M = 0"), (dict(x=None), b"NULL"), (dict(g=None), b"NULL"),
                      (dict(b=None), b"NULL"), (dict(o32=None), b"no output")]:
        assert ln(**kw) == 1, kw
        assert words in lib.mmr_last_error(), (kw, lib.mmr_last_error())
