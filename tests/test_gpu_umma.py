"""K2: the tcgen05/TMEM contraction with the fused top-k epilogue (query batches of 3 or more sharing one row range)."""
import importlib

import numpy as np
import pytest
import torch

from oracle import flat_search as ofs
from tests import util

pytestmark = pytest.mark.gpu
PKG = "multimodal-rag-for-image-text-search_b200"


@pytest.fixture(scope="module")
def mmr():
    pkg = importlib.import_module(PKG)
    pkg._native.lib()
    return pkg


def _bf16(x):
    return torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()


@pytest.mark.parametrize("dim", [512, 384])
def test_raw_scores_match_fp32_reference_of_same_inputs(mmr, dim):
    """The tensor-core scores alone (no top-k): bf16 rows x bf16 unit queries, fp32 accumulate, against a plain
    fp32 matmul of the same bf16 values.  Catches descriptor / swizzle / TMEM-layout mistakes directly.
    b <= 128 runs the single-CTA kernel (both operands in shared memory), b = 131 the CTA-pair kernel (query tile in
    tensor memory, tcgen05.mma.cta_group::2)."""
    n = 70_000 + 37           # last tile is partial
    rows = util.unit_rows(n, dim, seed=dim + 1)
    ix = mmr.ResidentIndex.from_f32(rows, dtype="bf16")
    stored = ix.rows.float()
    for b in (1, 5, 128, 131):
        q = util.queries(b, dim) * np.float32(1.7)
        qn = torch.from_numpy(_bf16(np.stack([np.asarray(ofs.normalize(v), np.float32) for v in q]))).cuda()
        for lo, hi in ((0, n), (1000, 1000 + 4099)):
            got = ix.debug_umma_scores(torch.from_numpy(q).cuda(), lo, hi)
            torch.cuda.synchronize()
            want = qn @ stored[lo:hi].T
            assert not torch.isnan(got).any(), "every (query, row) cell must be written"
            err = (got - want).abs().max().item()
            assert err < 3e-6, f"dim {dim} b {b} rows [{lo},{hi}): max err {err}"
    ix.close()


@pytest.mark.parametrize("b", [5, 8, 127, 128, 129, 300])
def test_topk_matches_oracle(mmr, b):
    rows = util.unit_rows(150_000, 512, seed=91, cone=0.3)
    ix = mmr.ResidentIndex.from_f32(rows, dtype="bf16")
    qs = util.queries(b, 512, cone=0.3)
    stored = ofs.bf16_round(rows)
    for k in (10, 50):
        s, r = ix.search(torch.from_numpy(qs).cuda(), k)
        torch.cuda.synchronize()
        assert mmr._native.lib().mmr_last_kernel() == 2, "batches >= 3 over a large range must take the tcgen05 path"
        s, r = s.cpu().numpy(), r.cpu().numpy()
        for j in range(0, b, max(1, b // 16)):
            util.check_topk(s[j], r[j], util.oracle_scores(rows, qs[j]), k, util.TOL_BF16, what=f"K2 b{b} k{k} q{j}")
            # strict: oracle on the stored bf16 rows and the bf16-rounded unit query -> only fp32 summation order differs
            qn = _bf16(np.asarray(ofs.normalize(qs[j]), np.float32))
            full = (stored @ qn).astype(np.float32)
            util.check_topk(s[j], r[j], full, k, 1e-5, what=f"K2 strict b{b} k{k} q{j}")
    ix.close()


def test_k2_equals_k1_on_segments_and_ties(mmr):
    """Same answers from the two kernel families (K1 per group of 4 vs K2), on a tenant segment whose bounds
    are not tile aligned, with exact duplicate rows across tile boundaries."""
    seg = np.array([0, 777, 777 + 100_003, 140_000], dtype=np.int64)
    rows = util.unit_rows(140_000, 384, seed=92)
    q = util.queries(6, 384)
    best = int(np.argmax(rows[seg[1]:seg[2]] @ q[0])) + int(seg[1])
    for p in (seg[1], seg[1] + 127, seg[1] + 128, seg[2] - 1):
        rows[p] = rows[best]
    ix = mmr.ResidentIndex.from_f32(rows, seg_offsets=seg, dtype="bf16")
    qd = torch.from_numpy(q).cuda()
    s2, r2 = ix.search(qd, 12, [1] * 6)
    assert mmr._native.lib().mmr_last_kernel() == 2
    r1 = torch.cat([ix.search(qd[i:i + 2], 12, [1] * 2)[1] for i in (0, 2, 4)])
    assert mmr._native.lib().mmr_last_kernel() == 1
    # ids can differ only through the query's bf16 rounding; the duplicates (exactly equal scores) must be ordered
    want = sorted({int(seg[1]), int(seg[1]) + 127, int(seg[1]) + 128, int(seg[2]) - 1, best})
    assert r2[0][:len(want)].tolist() == want
    assert (s2[0][:len(want)] == s2[0][0]).all()
    assert ((r2 >= seg[1]) & (r2 < seg[2])).all()
    overlap = np.mean([len(set(a.tolist()) & set(b.tolist())) / 12 for a, b in zip(r1.cpu().numpy(), r2.cpu().numpy())])
    assert overlap > 0.9
    ix.close()


def test_fp16_rows_on_tensor_cores(mmr):
    """fp16 storage takes the same tcgen05 path (operand format switch in the instruction descriptor)."""
    rows = util.unit_rows(90_000, 512, seed=93)
    ix = mmr.ResidentIndex.from_f32(rows, dtype="f16")
    stored = ix.rows.float()
    q = util.queries(7, 512)
    qn = torch.from_numpy(np.stack([np.asarray(ofs.normalize(v), np.float32) for v in q])).cuda().half().float()
    got = ix.debug_umma_scores(torch.from_numpy(q).cuda(), 0, 90_000)
    assert (got - qn @ stored.T).abs().max().item() < 3e-6
    s, r = ix.search(torch.from_numpy(q).cuda(), 10)
    assert mmr._native.lib().mmr_last_kernel() == 2
    for j in range(7):
        util.check_topk(s[j].cpu().numpy(), r[j].cpu().numpy(), util.oracle_scores(rows, q[j]), 10, util.TOL_BF16, what=f"f16 q{j}")
    ix.close()


@pytest.mark.parametrize("n", [1, 7, 129, 1000, 4097])
def test_k2_on_tiny_ranges(mmr, n):
    """The kernel family depends on the batch size only, so a 1-row tenant queried by 5 requests also runs on the
    tensor cores: partial tiles, fewer rows than k, TMA boxes hanging over the end of the table."""
    rows = util.unit_rows(n, 512, seed=95)
    ix = mmr.ResidentIndex.from_f32(rows, dtype="bf16")
    q = util.queries(5, 512)
    s, r = ix.search(torch.from_numpy(q).cuda(), 10)
    assert mmr._native.lib().mmr_last_kernel() == 2
    for j in range(5):
        util.check_topk(s[j].cpu().numpy(), r[j].cpu().numpy(), util.oracle_scores(rows, q[j]), 10, util.TOL_BF16, what=f"tiny n{n} q{j}")
    ix.close()


def test_k2_large_batch_parity(mmr):
    """B = 1024 (8 query tiles on CTA pairs, query tile in tensor memory, probe floor): a sample of queries against the oracle."""
    rows = util.unit_rows(300_000, 512, seed=96, cone=0.3)
    ix = mmr.ResidentIndex.from_f32(rows, dtype="bf16")
    q = util.queries(1024, 512, cone=0.3)
    s, r = ix.search(torch.from_numpy(q).cuda(), 10)
    s, r = s.cpu().numpy(), r.cpu().numpy()
    for j in list(range(0, 1024, 37)) + [127, 128, 1023]:
        util.check_topk(s[j], r[j], util.oracle_scores(rows, q[j]), 10, util.TOL_BF16, what=f"B1024 q{j}")
    ix.close()
