"""The e4m3 top-k on the GPU (``Fp8Catalogue``, ``score_topk`` on it, and its two stages alone).

Integer-valued inputs are exact in e4m3 after scaling and every partial sum is exact in fp32, so there
stage 1 must equal the oracle (``tests/oracle_fp8.py``) bit for bit, ties included.  Random inputs check
the accumulation error bound, the ranking, and that re-ranking reproduces the dense fp32 kernel's scores."""
import pytest
import torch

import truth_recommendation_gnn_b200 as trg
from oracle import topk as otopk
from tests import oracle_exclude as oexcl
from tests import oracle_fp8 as o8
from tests.test_gpu_exclude import N_KINDS, _index, _pairs
from truth_recommendation_gnn_b200 import fp8

pytestmark = pytest.mark.gpu

INT64_MAX = torch.iinfo(torch.int64).max


def _ints(b, p, h, seed, ties=False):
    """q in [-3, 3], posts in [0, 2] with 5 % all-zero rows (or every post equal: all scores tie)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randint(-3, 4, (b, h), generator=g).float()
    cat = torch.ones(p, h) if ties else torch.randint(0, 3, (p, h), generator=g).float()
    cat[torch.rand(p, generator=g) < 0.05] = 0
    return q, cat


def _relu_randn(b, p, h, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, h, generator=g).relu(), torch.randn(p, h, generator=g).relu()


# ---- quantiser ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_quantisers_equal_oracle(dev, dtype, monkeypatch):
    monkeypatch.setattr(fp8, "CHUNK_ROWS", 1000)
    g = torch.Generator().manual_seed(1)
    t = (torch.randn(2500, 128, generator=g) * 3).to(dtype)        # 2.5 chunks, both signs
    t[1000, 5] = -40.0                                               # amax in the second chunk, negative
    td = t.to(dev)
    cat = trg.Fp8Catalogue.from_dense(td)
    c8, sc = o8.quantize_table(t)
    assert float(cat.scale) == sc and cat.scale.dim() == 0 and cat.data.dtype == torch.float8_e4m3fn
    assert torch.equal(cat.data.cpu().double(), torch.from_numpy(c8))
    assert cat.dense.data_ptr() == td.data_ptr()                     # the table itself, not a copy
    q = (torch.randn(300, 256, generator=g) * torch.logspace(-6, 6, 300)[:, None]).to(dtype)
    q[3] = 0
    q8, s = fp8.quantize_rows(q.to(dev))
    r8, rs = o8.quantize_rows(q)
    assert torch.equal(s.cpu().double(), torch.from_numpy(rs))
    assert torch.equal(q8.cpu().double(), torch.from_numpy(r8))
    # a shared amax: the scale follows it, not the table
    cat2 = trg.Fp8Catalogue.from_dense(t.to(dev), amax=torch.tensor(1000.0, device=dev))
    c8, sc = o8.quantize_table(t, 1000.0)
    assert float(cat2.scale) == sc and torch.equal(cat2.data.cpu().double(), torch.from_numpy(c8))


# ---- stage 1, integer data: bit for bit ------------------------------------------------------------------
def _stage1_exact(dev, q, cat, k, dtype=torch.float32, pairs=None, n_rows=0, id_offset=0, rows=None):
    ev, ei = o8.stage1_topk(q, cat, k, pairs, id_offset, rows)
    c8 = trg.Fp8Catalogue.from_dense(cat.to(dev, dtype))
    idx = _index(pairs, n_rows, dev) if pairs is not None else None
    gv, gi = fp8._fp8_candidates(q.to(dev, dtype), c8, k, id_offset, exclude=idx,
                                rows=None if rows is None else rows.to(dev))
    assert gv.shape == ev.shape
    assert torch.equal(gi.cpu(), ei)
    assert torch.equal(gv.cpu(), ev.float())
    return gv, gi, c8, idx


@pytest.mark.parametrize("b,p,h,k,ties", [
    (1, 20_000, 128, 1, False), (127, 7001, 128, 7, False), (129, 50_001, 256, 100, False),
    (1000, 3001, 128, 128, False), (5, 60, 128, 100, False), (1, 90, 256, 128, False),
    (64, 200_003, 128, 128, False), (129, 9999, 256, 128, False), (1000, 12_345, 256, 7, False),
    (127, 5000, 128, 100, True), (129, 1000, 256, 1, True)])
def test_stage1_integer_exact(dev, b, p, h, k, ties):
    q, cat = _ints(b, p, h, b * p + h, ties)
    _stage1_exact(dev, q, cat, k)
    if b == 1000:
        _stage1_exact(dev, q, cat, k, torch.bfloat16)


@pytest.mark.parametrize("b,p,h,k", [(1, 20_000, 128, 10), (300, 50_000, 128, 100), (129, 7001, 256, 100),
                                     (5, 7, 128, 10)])
def test_stage1_exclusions_integer_exact(dev, b, p, h, k):
    q, cat = _ints(b, p, h, 7 * b + p)
    off = 7
    pairs, n_rows = _pairs(q, cat, k, off, b + 1)
    gv, gi, _, _ = _stage1_exact(dev, q, cat, k, pairs=pairs, n_rows=n_rows, id_offset=off)
    few = torch.arange(b) % N_KINDS == 4
    if min(k, p) >= 2 and few.any():
        assert (gi.cpu()[few] == -1).any(dim=1).all()


def test_stage1_rows_indirection(dev):
    b, p, h, k = 200, 9000, 128, 50
    q, cat = _ints(b, p, h, 31)
    rows = torch.randint(0, 23, (b,), generator=torch.Generator().manual_seed(32))
    rows[:N_KINDS] = torch.arange(N_KINDS)
    pairs, n_rows = _pairs(q, cat, k, 0, 33, rows=rows)
    _stage1_exact(dev, q, cat, k, pairs=pairs, n_rows=n_rows, rows=rows)


def test_stage1_shards_merge_to_unsharded(dev):
    b, p, h, k = 70, 12_000, 128, 40
    q, cat = _ints(b, p, h, 51)
    pairs, n_rows = _pairs(q, cat, k, 0, 52)
    gv, gi, c8, idx = _stage1_exact(dev, q, cat, k, pairs=pairs, n_rows=n_rows)
    qd, cd = q.to(dev), cat.to(dev)
    amax = fp8.table_amax(cd)
    vs, ids = [], []
    for a, e in [(0, 3000), (3000, 7001), (7001, p)]:
        shard = trg.Fp8Catalogue.from_dense(cd[a:e].contiguous(), amax=amax)
        v, i = fp8._fp8_candidates(qd, shard, k, id_offset=a, exclude=idx)
        vs.append(v)
        ids.append(torch.where(i < 0, torch.full_like(i, INT64_MAX), i))
    mv, mi = trg.topk_merge(torch.cat(vs, 1), torch.cat(ids, 1), 3, k)
    assert torch.equal(mv, gv) and torch.equal(mi, gi)


# ---- stage 1, random data: error bound and ranking ------------------------------------------------------
@pytest.mark.parametrize("h", [128, 256])
def test_stage1_random_error_bound(dev, h):
    b, p, k = 257, 30_001, 128
    q, cat = _relu_randn(b, p, h, h)
    q[:, ::3] *= -1                                        # signed queries
    c8 = trg.Fp8Catalogue.from_dense(cat.to(dev))
    gv, gi = fp8._fp8_candidates(q.to(dev), c8, k)
    gv, gi = gv.cpu().double(), gi.cpu()
    qd, cd = o8.dequantized(q, cat)
    full = qd @ cd.T                                       # fp64 dots of the dequantised inputs
    bound = h * 2.0 ** -24 * (qd.abs() @ cd.abs().T)
    ref = full.gather(1, gi)
    err = (gv - ref).abs()
    assert (err <= bound.gather(1, gi)).all(), f"max error / bound {float((err / bound.gather(1, gi)).max())}"
    assert (gv[:, 1:] <= gv[:, :-1]).all()
    tie = gv[:, 1:] == gv[:, :-1]
    assert (gi[:, 1:][tie] > gi[:, :-1][tie]).all()
    omitted = torch.ones_like(full, dtype=torch.bool)
    omitted.scatter_(1, gi, False)
    slack = 2 * torch.maximum(bound, bound.gather(1, gi[:, -1:]))
    assert not (omitted & (full > gv[:, -1:] + slack)).any()


# ---- stage 2: re-scoring --------------------------------------------------------------------------------
def test_rescore_fp32_equals_dense_kernel(dev):
    b, p, h = 64, 120, 128                                 # P <= 128: the dense kernel returns every post
    q, cat = _relu_randn(b, p, h, 5)
    qd, cd = q.to(dev), cat.to(dev)
    dv, di = trg.score_topk(qd, cd, p)
    by_id = torch.empty_like(dv).scatter_(1, di, dv)       # fp32 kernel score of every (query, post)
    g = torch.Generator().manual_seed(6)
    cand = torch.stack([torch.randperm(p, generator=g)[:90] for _ in range(b)]) + 1000
    rv, ri = fp8.rescore_topk(qd, cd, cand.to(dev), 60, id_offset=1000)
    assert torch.equal(rv, by_id.gather(1, ri - 1000))
    # every candidate: the top 60 of their exact scores, canonical order
    cs = by_id.cpu().gather(1, cand - 1000)
    o = torch.argsort(cand, dim=1)
    cs, cid = cs.gather(1, o), cand.gather(1, o)
    sv, si = torch.sort(cs, dim=1, descending=True, stable=True)
    assert torch.equal(ri.cpu(), cid.gather(1, si)[:, :60]) and torch.equal(rv.cpu(), sv[:, :60])


def test_rescore_bf16_equals_chain_and_skips_invalid(dev):
    b, p, h = 50, 5000, 256
    q, cat = _relu_randn(b, p, h, 8)
    q, cat = q.bfloat16(), cat.bfloat16()
    g = torch.Generator().manual_seed(9)
    cand = torch.stack([torch.randperm(p, generator=g)[:128] for _ in range(b)])
    cand[:, 5] = -1
    cand[:, 9] = p                                         # one past the table
    cand[:, 11] = -7
    cand[3, 4:] = -1                                       # row 3: four valid candidates only
    rv, ri = fp8.rescore_topk(q.to(dev), cat.to(dev), cand.to(dev), 100)
    s = o8.rescore_chain(q, cat, cand)
    o = torch.argsort(torch.where(cand < 0, torch.full_like(cand, INT64_MAX), cand), dim=1)
    s, cid = s.gather(1, o), cand.gather(1, o)
    sv, si = torch.sort(s, dim=1, descending=True, stable=True)
    ei = cid.gather(1, si)[:, :100]
    ei = torch.where(sv[:, :100] == float("-inf"), torch.full_like(ei, -1), ei)
    assert torch.equal(rv.cpu(), sv[:, :100]) and torch.equal(ri.cpu(), ei)
    assert (ri[3, 4:] == -1).all() and (rv[3, 4:] == float("-inf")).all()
    assert not ((ri == p) | (ri == -7)).any()


# ---- end to end -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("b,p,h,k", [(300, 50_000, 128, 100), (129, 7001, 256, 10), (4, 50, 128, 100)])
def test_end_to_end_integer_exact(dev, dtype, b, p, h, k):
    q, cat = _ints(b, p, h, b + p + h)
    qd, cd = q.to(dev, dtype), cat.to(dev, dtype)
    c8 = trg.Fp8Catalogue.from_dense(cd)
    ev, ei = otopk.score_topk(q, cat, k)
    gv, gi = trg.recommend(qd, c8, k=k)
    assert torch.equal(gi.cpu(), ei) and torch.equal(gv.cpu(), ev)
    pairs, n_rows = _pairs(q, cat, k, 0, b)
    xv, xi = oexcl.score_topk_excluding(q, cat, k, pairs)
    idx = _index(pairs, n_rows, dev)
    gv, gi = trg.recommend(qd, c8, k, exclude=idx, rows=torch.arange(b, device=dev))
    assert torch.equal(gi.cpu(), xi) and torch.equal(gv.cpu(), xv)


def test_end_to_end_random_equals_dense_where_candidates_hold_it(dev):
    b, p, h, k = 512, 200_000, 128, 10
    q, cat = _relu_randn(b, p, h, 21)
    qd, cd = q.to(dev), cat.to(dev)
    c8 = trg.Fp8Catalogue.from_dense(cd)
    dv, di = trg.score_topk(qd, cd, k)                     # the dense fp32 kernel
    _, cand = fp8._fp8_candidates(qd, c8)
    held = (di[:, :, None] == cand[:, None, :]).any(-1).all(-1)
    gv, gi = trg.score_topk(qd, c8, k)
    assert held.float().mean() >= 0.95
    assert torch.equal(gv[held], dv[held]) and torch.equal(gi[held], di[held])


def test_end_to_end_shards_with_shared_amax(dev):
    b, p, h, k = 100, 40_000, 256, 50
    q, cat = _ints(b, p, h, 22)
    cat[17_000:] = cat[17_000:].clamp(max=1)               # the second shard alone would get a finer scale
    qd, cd = q.to(dev), cat.to(dev)
    whole = trg.Fp8Catalogue.from_dense(cd)
    gv, gi = trg.score_topk(qd, whole, k)
    amax = torch.maximum(fp8.table_amax(cd[:17_000]), fp8.table_amax(cd[17_000:]))   # the all-reduce (MAX)
    vs, ids = [], []
    for a, e in [(0, 17_000), (17_000, p)]:
        shard = trg.Fp8Catalogue.from_dense(cd[a:e], amax=amax)
        assert torch.equal(shard.scale, whole.scale)
        v, i = trg.recommend(qd, shard, k=k, id_offset=a)
        vs.append(v)
        ids.append(i)
    mv, mi = trg.topk_merge(torch.cat(vs, 1), torch.cat(ids, 1), 2, k)
    assert torch.equal(mv, gv) and torch.equal(mi, gi)


# ---- scale ----------------------------------------------------------------------------------------------
@pytest.mark.timeout(2400)
def test_config5_fp8_stage_integer_exact(dev):
    """4096 queries x 50M posts, K = 100, integer bf16 through the e4m3 stage: ids and values equal an exact
    ranking built from int64 keys (score, then lower id first); the two stages together return the same."""
    B, P, H, K = 4096, 50_000_000, 128, 100
    gen = torch.Generator(device=dev).manual_seed(13)
    q = torch.randint(-3, 4, (B, H), generator=gen, device=dev).to(torch.bfloat16)
    cat = torch.randint(0, 3, (P, H), generator=gen, device=dev, dtype=torch.int8)
    cat[torch.rand(P, generator=gen, device=dev) < 0.05] = 0
    cat = cat.to(torch.bfloat16)
    c8 = trg.Fp8Catalogue.from_dense(cat)
    vals, ids = fp8._fp8_candidates(q, c8, K)
    shift = 1 << 26
    best = torch.full((B, K), -(1 << 62), dtype=torch.int64, device=dev)
    chunk = 500_000
    for a in range(0, P, chunk):
        b = min(a + chunk, P)
        sc = (q.float() @ cat[a:b].float().t()).long()
        key = sc * shift + (shift - 1 - torch.arange(a, b, device=dev))[None, :]
        best = torch.topk(torch.cat([best, key], dim=1), K, dim=1)[0]
        del sc, key
    ref_ids = shift - 1 - (best % shift)
    ref_vals = torch.div(best, shift, rounding_mode="floor").float()
    assert torch.equal(ids, ref_ids)
    assert torch.equal(vals, ref_vals)
    v2, i2 = trg.score_topk(q, c8, K)
    assert torch.equal(i2, ref_ids) and torch.equal(v2, ref_vals)
