"""Encoder kernels one launch at a time against a float64 reference (mmr_debug_enc_gemm / _attention / _layernorm).

Each hook runs the launch code the forward pass runs.  Every reference is a plain float64 torch computation on the device,
on exactly the inputs the kernel saw: the bf16 X and W of a GEMM, the fp32 qkv of an attention launch (rounded to bf16
first where the tensor-core kernel rounds it).  Tolerances follow from the kernels' arithmetic (u = 2^-24, the fp32 unit
roundoff); each test's docstring gives the derivation.  Bit-identity checks pin the claims the encoders' batch invariance
rests on: the token tile, the ring depth, an aliased residual and a folded LayerNorm never change a result."""
import importlib
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
PKG = "multimodal-rag-for-image-text-search_b200"
U = 2.0 ** -24
EPIS = (0, 1, 2, 3)          # EPI_BIAS_F32, EPI_BIAS_RES_F32, EPI_GELU_BF16, EPI_QUICKGELU_BF16
TILES = (64, 128, 256)


@pytest.fixture(scope="module")
def native():
    n = importlib.import_module(PKG + "._native")
    n.lib()
    return n


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------------------------------------------------- GEMM
def _gemm_inputs(M, N, K, seed):
    """X and W with entries up to +-8 (large products that cancel); every third token row is scaled down so that its
    pre-activation y spans about [-10, 10] (GELU's negative tail, quick-GELU's curved part)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = (torch.rand(M, K, generator=g, device="cuda") * 16 - 8)
    small = torch.arange(M, device="cuda") % 3 == 1
    X[small] *= 1.5 / math.sqrt(K) / 8         # entries within +-1.5 / sqrt(K): std(y) = sqrt(K) (1.5 / sqrt(K)) 8 / 3 = 4
    W = torch.rand(N, K, generator=g, device="cuda") * 16 - 8
    bias = torch.rand(N, generator=g, device="cuda") * 8 - 4
    res = torch.randn(M, N, generator=g, device="cuda") * 50
    return X.to(torch.bfloat16), W.to(torch.bfloat16), bias, res


def _gemm(native, epi, nt, X16, W16, bias, res=None, out32=None, fold=None):
    """One mmr_debug_enc_gemm launch; fold = (ln_src, g, b, eps, ln_out) runs the LayerNorm-folded kernel."""
    M, N, K = (X16.shape[0] if fold is None else fold[0].shape[0]), W16.shape[0], W16.shape[1]
    o32 = out32 if out32 is not None else (torch.full((M, N), float("nan"), device="cuda") if epi in (0, 1) else None)
    o16 = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16) if epi in (2, 3) else None
    if fold is None:
        args = (_p(X16), None, None, None, 0.0, None)
    else:
        src, lg, lb, eps, ln_out = fold
        args = (None, _p(src), _p(lg), _p(lb), eps, _p(ln_out))
    native.check(native.lib().mmr_debug_enc_gemm(epi, nt, 0 if fold is None else 1, M, N, K, *args, _p(W16), _p(bias), _p(res),
                                                 _p(o32), _p(o16), _stream()))
    torch.cuda.synchronize()
    return o32 if epi in (0, 1) else o16


def _act(epi, y):
    if epi == 2:
        return 0.5 * y * (1.0 + torch.special.erf(y / math.sqrt(2.0)))
    if epi == 3:
        return y * torch.sigmoid(1.702 * y)
    return y


def _check_gemm(epi, got, X16, W16, bias, res, what):
    """fp32 outputs: the products of bf16 values are exact in fp32 and the accumulator adds K of them.  Each addition errs
    by less than one ulp of the running sum (2 u relative, whether the tensor core rounds or truncates), and no running sum
    exceeds sum|x w|; then + bias and + residual round once each:
        |got - ref| <= 2 (K + 2) u (|X| |W|^T + |b| + |res|) + 2 u |ref|.
    A dropped 16-wide K step changes y by ~16 / K of sum|x w|, orders of magnitude above this.
    bf16 outputs: y as above (bound_y), the activation's slope is below 1.2, the epilogue's erf (Abramowitz & Stegun
    7.1.26, |error| <= 1.5e-7) and the approximate reciprocal / exp2 units add at most 1e-6 max(1, |y|), and the bf16
    rounding of the result 2^-9 relative (2^-8 leaves room for the rounding of a value already off by bound_y):
        |got - act(ref)| <= 2^-8 |act(ref)| + 1.2 bound_y + 1e-6 max(1, |y|)."""
    Xd, Wd, bd = X16.double(), W16.double(), bias.double()
    y = Xd @ Wd.T + bd
    mag = X16.double().abs() @ W16.double().abs().T + bd.abs()
    K = X16.shape[1]
    if epi == 1:
        y = y + res.double()
        mag = mag + res.double().abs()
    bound_y = 2 * (K + 2) * U * mag + 2 * U * y.abs()
    if epi in (0, 1):
        err = (got.double() - y).abs()
        bound = bound_y
    else:
        ref = _act(epi, y)
        err = (got.double() - ref).abs()
        bound = 2.0 ** -8 * ref.abs() + 1.2 * bound_y + 1e-6 * y.abs().clamp(min=1.0)
    assert torch.isfinite(got.double()).all(), what
    bad = err > bound
    assert not bool(bad.any()), (what, int(bad.sum()), float((err - bound).max()), float(err.max()))


# every (epi, nt) pair meets a K >= 1536 shape with a ragged M, a short-K shape and an edge M (1, 63, 64, 65)
_LONG = [(257, 384, 1536), (1000, 384, 2048), (4097, 384, 1536), (65, 1152, 2048), (255, 2048, 1536), (63, 1536, 2048)]
_SHORT = [(1000, 1152, 384), (4097, 1536, 512), (255, 2048, 384), (257, 384, 512), (1000, 1536, 384), (4097, 1152, 384)]
_EDGE = [(1, 384, 384), (63, 1152, 512), (64, 2048, 384), (65, 1536, 512), (1, 2048, 2048), (64, 384, 1536)]


@pytest.mark.parametrize("epi", EPIS)
@pytest.mark.parametrize("nt", TILES)
def test_gemm_matches_fp64(native, epi, nt):
    i = EPIS.index(epi) * len(TILES) + TILES.index(nt)
    for M, N, K in (_LONG[i % 6], _SHORT[(i + 2) % 6], _EDGE[(i + 4) % 6]):
        X16, W16, bias, res = _gemm_inputs(M, N, K, seed=1000 * i + M)
        got = _gemm(native, epi, nt, X16, W16, bias, res if epi == 1 else None)
        _check_gemm(epi, got, X16, W16, bias, res, (epi, nt, M, N, K))


@pytest.mark.parametrize("epi", EPIS)
def test_gemm_result_does_not_depend_on_token_tile_or_ring_depth(native, epi):
    """The forward pass picks the token tile (64 / 128 / 256) from the pass's token count and the ring depth from
    MMR_ENC_GEMM_SMEM_KB; accumulation runs along K only, so neither may change a bit of any output.  This is what makes
    a query's embedding independent of the micro-batch it rides in.  48 KB gives a 2-stage ring, 210 KB an 8-stage ring at
    the 64-token tile (4 at 256 tokens)."""
    for M, N, K in ((257, 384, 2048), (1000, 1152, 384), (65, 1536, 1536), (4097, 384, 512)):
        X16, W16, bias, res = _gemm_inputs(M, N, K, seed=7 * M + K)
        r = res if epi == 1 else None
        base = _gemm(native, epi, 64, X16, W16, bias, r)
        _check_gemm(epi, base, X16, W16, bias, res, (epi, M, N, K))
        try:
            for kb in (None, "48", "210"):
                native.set_option("MMR_ENC_GEMM_SMEM_KB", kb)
                for nt in TILES:
                    got = _gemm(native, epi, nt, X16, W16, bias, r)
                    assert torch.equal(got, base), (epi, nt, kb, M, N, K, float((got.double() - base.double()).abs().max()))
        finally:
            native.set_option("MMR_ENC_GEMM_SMEM_KB", None)


@pytest.mark.parametrize("nt", TILES)
def test_gemm_residual_in_place_equals_out_of_place(native, nt):
    """EPI_BIAS_RES_F32 with out == residual (the in-place residual stream of the forward pass) loads every residual value
    before its first store: bit-identical to writing a separate buffer."""
    for M, N, K in ((257, 384, 1536), (1000, 512 * 3, 384), (1, 384, 512)):
        X16, W16, bias, res = _gemm_inputs(M, N, K, seed=M + nt)
        apart = _gemm(native, 1, nt, X16, W16, bias, res)
        inplace = res.clone()
        _gemm(native, 1, nt, X16, W16, bias, inplace, out32=inplace)
        assert torch.equal(apart, inplace), (nt, M, N, K)
        _check_gemm(1, inplace, X16, W16, bias, res, (nt, M, N, K))


def _ln_rows(M, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(M, H, generator=g, device="cuda") * 3 + torch.randn(M, 1, generator=g, device="cuda")
    x[1::5] = 100.0 + 0.01 * torch.randn(x[1::5].shape, generator=g, device="cuda")     # cancellation
    rows = torch.arange(3, max(M, 3), 7, device="cuda")                                 # constant rows of dyadic values
    vals = torch.tensor([100.0, -3.5, 0.0, 2.0 ** -20], device="cuda")
    x[rows] = vals[torch.arange(len(rows), device="cuda") % 4][:, None].expand(-1, H)
    lg = torch.randn(H, generator=g, device="cuda") * 0.5 + 1
    lb = torch.randn(H, generator=g, device="cuda") * 0.5
    return x, lg, lb


def _layernorm(native, x, lg, lb, eps, out32=None, bf16=True):
    M, H = x.shape
    o16 = torch.full((M, H), float("nan"), device="cuda", dtype=torch.bfloat16) if bf16 else None
    native.check(native.lib().mmr_debug_enc_layernorm(H, M, _p(x), _p(lg), _p(lb), eps, _p(out32), _p(o16), _stream()))
    torch.cuda.synchronize()
    return o16


@pytest.mark.parametrize("epi", (0, 2, 3))
@pytest.mark.parametrize("K", (384, 512))
def test_gemm_with_folded_layernorm_equals_layernorm_then_gemm(native, epi, K):
    """gemm_wt_kernel<EPI, 64, true> normalises its token tile itself with layernorm_kernel's exact arithmetic: its outputs
    equal layernorm_kernel -> bf16 -> the plain GEMM bit for bit, and ln_out (written by the CTAs of feature tile 0) equals
    the LayerNorm's fp32 output bit for bit.  Without ln_out (the CLIP pre-LN call) nothing else changes."""
    N = 1152 if K == 384 else 2048
    for M in (1, 16, 65, 1000):
        X16, W16, bias, _ = _gemm_inputs(M, N, K, seed=M + K + epi)
        x, lg, lb = _ln_rows(M, K, seed=M * K)
        eps = 1e-12 if K == 384 else 1e-5
        ln32 = torch.empty_like(x)
        ln16 = _layernorm(native, x, lg, lb, eps, out32=ln32)
        sep = _gemm(native, epi, 64, ln16, W16, bias)
        ln_out = torch.full_like(x, float("nan"))
        fused = _gemm(native, epi, 64, None, W16, bias, fold=(x, lg, lb, eps, ln_out))
        assert torch.equal(fused, sep), (epi, K, M)
        assert torch.equal(ln_out, ln32), (epi, K, M)
        fused2 = _gemm(native, epi, 64, None, W16, bias, fold=(x, lg, lb, eps, None))
        assert torch.equal(fused2, sep), (epi, K, M)
        _check_gemm(epi, fused, ln16, W16, bias, None, (epi, K, M))


# -------------------------------------------------------------------------------------------------------- LayerNorm
@pytest.mark.parametrize("H", (384, 512))
@pytest.mark.parametrize("eps", (1e-12, 1e-5))
def test_layernorm_matches_fp64(native, H, eps):
    """layernorm_kernel<H>: warp per row, lane l holds columns 32 i + l; mean = (H/32 sequential adds per lane + a 5-level
    butterfly) / H, so the computed mean is off by at most e_m = (H/32 + 6) u mean|x|; the centred values then carry that
    shift, which the normalisation scales by rstd (this dominates rows with mean 100 and std 0.01); the variance sum, the
    rsqrt (approximate, <= 2 ulp) and the final multiply-adds add a relative (H/32 + 16) u:
        |got - ref| <= |g| rstd e_m + (H/32 + 16) u |g x^| + 2 u |b|.
    Constant rows of dyadic values sum exactly, so their variance is 0 and the output is exactly b.  In place
    (out_f32 == x) and to bf16 (+ 2^-8 |ref| for the rounding)."""
    M = 203
    x, lg, lb = _ln_rows(M, H, seed=H + int(eps * 1e12))
    xd = x.double()
    mean = xd.mean(1, keepdim=True)
    var = ((xd - mean) ** 2).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    xh = (xd - mean) * rstd
    ref = xh * lg.double() + lb.double()
    e_m = (H / 32 + 6) * U * xd.abs().mean(1, keepdim=True)
    bound = lg.double().abs() * rstd * e_m + (H / 32 + 16) * U * (lg.double() * xh).abs() + 2 * U * lb.double().abs()
    inplace = x.clone()
    got16 = _layernorm(native, inplace, lg, lb, eps, out32=inplace)
    for got, b in ((inplace.double(), bound), (got16.double(), bound * (1 + 2.0 ** -8) + 2.0 ** -8 * ref.abs())):
        err = (got - ref).abs()
        assert not bool((err > b).any()), (H, eps, float((err - b).max()))
    const = (x == x[:, :1]).all(1)
    assert int(const.sum()) >= 4
    assert torch.equal(inplace[const], lb.expand(int(const.sum()), H)), "a constant row must normalise to beta exactly"
    assert torch.equal(got16, inplace.to(torch.bfloat16))
    only16 = _layernorm(native, x, lg, lb, eps, out32=None)
    assert torch.equal(only16, got16)


# -------------------------------------------------------------------------------------------------------- attention
S_ALL = (1, 2, 31, 33, 64, 65, 77, 127, 128, 129, 330, 512)


def _qkv(B, S, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B * S, 3 * H, generator=g, device="cuda") * 1.5


def _attention(native, tc, B, S, H, heads, causal, qkv, mask):
    ctx = torch.full((B * S, H), float("nan"), device="cuda", dtype=torch.bfloat16)
    m = None if mask is None else mask.to(device="cuda", dtype=torch.int32).contiguous().reshape(-1)
    native.check(native.lib().mmr_debug_enc_attention(tc, B, S, H, heads, causal, _p(qkv), _p(m), _p(ctx), _stream()))
    torch.cuda.synchronize()
    return ctx


def _attention_ref(tc, B, S, H, heads, causal, qkv, mask):
    """float64 softmax(q k^T / sqrt(DH)) v on the kernel's inputs; a row whose keys are all hidden is 0.  tc: q * scale
    (fp32), k and v rounded to bf16 first, as attention_mma_kernel stages them.  Returns (ref, max|v| of the row's head,
    max_j sum_d |q_d k_d| scale per row)."""
    DH = H // heads
    t = qkv.reshape(B, S, 3, heads, DH).permute(2, 0, 3, 1, 4)                    # [3, B, heads, S, DH]
    scale32 = torch.rsqrt(torch.tensor(float(DH), device="cuda"))
    q, k, v = t[0] * scale32, t[1], t[2]
    if tc:
        q, k, v = (a.to(torch.bfloat16) for a in (q, k, v))
    q, k, v = q.double(), k.double(), v.double()
    s = q @ k.transpose(-1, -2)
    hide = torch.zeros(B, 1, S, S, dtype=torch.bool, device="cuda")
    if mask is not None:
        hide |= (mask.to("cuda") == 0)[:, None, None, :]
    if causal:
        hide |= torch.ones(S, S, dtype=torch.bool, device="cuda").triu(1)
    s = s.masked_fill(hide, -math.inf)
    p = torch.softmax(s, -1).nan_to_num(0.0)
    ref = (p @ v).permute(0, 2, 1, 3).reshape(B * S, H)
    vmax = v.abs().amax(-2, keepdim=True).expand(B, heads, S, DH).permute(0, 2, 1, 3).reshape(B * S, H)
    qk = (q.abs() @ k.abs().transpose(-1, -2)).masked_fill(hide, 0).amax(-1, keepdim=True)
    qk = qk.expand(B, heads, S, DH).permute(0, 2, 1, 3).reshape(B * S, H)
    return ref, vmax, qk


def _check_attention(tc, got, ref, vmax, qk, S, DH, what):
    """With qk = max_j sum_d |q_d k_d| / sqrt(DH) of the row and max|v| over the head's keys (per output dim).
    fp32 kernel: a score is a DH-term fp32 dot product (error <= DH u qk); __expf(x) = ex2.approx(x log2 e) errs by
    (|x| + 4) u relative with |x| <= 2 qk; so every weight is off by a relative (DH + 2) qk u + 4 u, which moves the output by
    at most twice that times max|v|; the normaliser and P.V are fp32 sums of <= S terms (S u each, relative to max|v|);
    the output is rounded to bf16 (2^-9, 2^-8 with room):
        |got - ref| <= 2^-8 |ref| + max|v| u (2 S + 2 (DH + 2) qk + 16).
    Tensor-core kernel (reference on its bf16 q, k, v): the same fp32 terms, plus P rounded to bf16 before P.V (2^-9
    relative per weight while the normaliser keeps the fp32 weights: <= 2^-9 max|v|, 2^-8 with room):
        |got - ref| <= 2^-8 |ref| + 2^-8 max|v| + max|v| u (2 S + 2 (DH + 2) qk + 16)."""
    bound = 2.0 ** -8 * ref.abs() + vmax * U * (2 * S + 2 * (DH + 2) * qk + 16)
    if tc:
        bound = bound + 2.0 ** -8 * vmax
    g = got.double()
    assert torch.isfinite(g).all(), what
    err = (g - ref).abs()
    assert not bool((err > bound).any()), (what, float((err - bound).max()), float(err.max()))


def _masks(B, S, kinds, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.ones(B, S, dtype=torch.int32)
    for b, kind in enumerate(kinds):
        if kind == "tail":
            m[b, max(1, S - S // 3 - 1):] = 0
        elif kind == "left":
            m[b, : S // 3] = 0
        elif kind == "single":
            m[b] = 0
            m[b, int(torch.randint(0, S, (1,), generator=g))] = 1
        elif kind == "dead":
            m[b] = 0
    return m


@pytest.mark.parametrize("tc", (0, 1), ids=("fp32", "tensor_cores"))
@pytest.mark.parametrize("H,heads", ((384, 12), (384, 6), (512, 16), (512, 8)), ids=("h384dh32", "h384dh64", "h512dh32", "h512dh64"))
def test_attention_matches_fp64(native, tc, H, heads):
    """Every sequence length of S_ALL with: no mask (NULL), tail padding, left padding, a single live key, all keys masked
    (output exactly 0, no NaN), and causal (with tail padding and all-masked rows).  Head dim 64 on the fp32 kernel stops at
    330 tokens: 512 is refused with a message instead."""
    DH = H // heads
    for i, S in enumerate(S_ALL):
        if not tc and DH == 64 and S == 512:
            qkv = _qkv(1, S, H, seed=1)
            ctx = torch.empty((S, H), device="cuda", dtype=torch.bfloat16)
            rc = native.lib().mmr_debug_enc_attention(0, 1, S, H, heads, 0, _p(qkv), None, _p(ctx), _stream())
            assert rc == 3 and b"330 tokens at most" in native.lib().mmr_last_error()
            continue
        runs = ((1, 0, None), (3, 0, ("tail", "left", "single")), (3, 1, ("live", "tail", "dead")), (1, 0, ("dead",)))
        for r, (B, causal, kinds) in enumerate(runs):
            qkv = _qkv(B, S, H, seed=100 * i + r + H)
            mask = None if kinds is None else _masks(B, S, kinds, seed=i + r)
            got = _attention(native, tc, B, S, H, heads, causal, qkv, mask)
            ref, vmax, qk = _attention_ref(tc, B, S, H, heads, causal, qkv, mask)
            _check_attention(tc, got, ref, vmax, qk, S, DH, (tc, H, heads, S, B, causal, kinds))
            if kinds is not None:
                for b, kind in enumerate(kinds):
                    if kind == "dead":
                        assert bool((got[b * S:(b + 1) * S] == 0).all()), "all keys masked: the output must be exactly 0"


@pytest.mark.parametrize("tc", (0, 1), ids=("fp32", "tensor_cores"))
@pytest.mark.parametrize("H,heads", ((384, 12), (512, 8)), ids=("dh32", "dh64"))
def test_attention_rows_do_not_depend_on_padding_or_later_tokens(native, tc, H, heads):
    """Bit-identity: a sequence's rows are unchanged when masked keys are appended (padding to a longer neighbour), and
    with causal, row i is unchanged when later tokens are appended (live, unmasked)."""
    DH = H // heads
    for L, S in ((1, 9), (31, 33), (33, 77), (64, 65), (100, 129), (127, 330), (200, 512)):
        if not tc and DH == 64 and S > 330:
            continue
        long = _qkv(1, S, H, seed=L * S + tc)
        short = long[:L].clone()
        alone = _attention(native, tc, 1, L, H, heads, 0, short, None)
        mask = torch.zeros(1, S, dtype=torch.int32)
        mask[0, :L] = 1
        padded = _attention(native, tc, 1, S, H, heads, 0, long, mask)
        assert torch.equal(padded[:L], alone), ("padding", tc, H, L, S)
        alone_c = _attention(native, tc, 1, L, H, heads, 1, short, None)
        longer_c = _attention(native, tc, 1, S, H, heads, 1, long, None)
        assert torch.equal(longer_c[:L], alone_c), ("causal prefix", tc, H, L, S)
