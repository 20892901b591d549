"""K5 with per-user exclusions on the GPU (``score_topk(..., exclude=ExclusionIndex)``): both kernels
(fp32 FMA and bf16 tcgen05) on integer-valued inputs, so dot products are exact, ties are massive, and
values AND ids must equal the oracle (``tests/oracle_exclude.py``) bit for bit."""
import pytest
import torch

import truth_recommendation_gnn_b200 as trg
from oracle import topk as otopk
from tests import oracle_exclude as oexcl

pytestmark = pytest.mark.gpu

INT64_MAX = torch.iinfo(torch.int64).max
N_KINDS = 7


def _integer_inputs(b, p, h, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.randint(0, 4, (b, h), generator=g).float()
    cat = torch.randint(0, 3, (p, h), generator=g).float()
    cat[torch.rand(p, generator=g) < 0.05] = 0          # dead-ReLU rows: exact-zero scores
    return q, cat


def _pairs(q, cat, k, id_offset, seed, rows=None):
    """Exclusion (row, global id) pairs; exclusion row r gets kind r % N_KINDS:
    0 nothing (must equal the call without exclusions), 1 ~1 % random posts, 2 its own unfiltered top-k,
    3 that top-k minus one member of the tie at the k-th score, 4 all but fewer than k posts (padded result),
    5 duplicates + ids outside the catalogue, 6 both posts of every 64-post half-tile / 128-post tile (and
    so chunk) boundary, the first and the last post.  Rows of kinds 2-3 are those of query r itself (or of
    the first query mapped to r)."""
    g = torch.Generator().manual_seed(seed)
    b, p = q.size(0), cat.size(0)
    kk = min(k, p)
    rows = torch.arange(b) if rows is None else rows
    n_rows = int(rows.max()) + 1
    first_q = {}
    for i, r in enumerate(rows.tolist()):
        first_q.setdefault(r, i)
    uv, ui = otopk.score_topk(q, cat, kk)                # unfiltered, local ids
    out = []

    def add(r, local):
        local = torch.as_tensor(local, dtype=torch.int64).flatten()
        out.append(torch.stack([torch.full_like(local, r), local + id_offset]))

    bound = torch.arange(0, p + 64, 64)
    bound = torch.cat([bound - 1, bound, torch.tensor([0, p - 1])])
    bound = bound[(bound >= 0) & (bound < p)]
    for r in range(n_rows):
        kind = r % N_KINDS
        i = first_q.get(r)
        if kind == 1:
            add(r, torch.nonzero(torch.rand(p, generator=g) < 0.01).flatten())
        elif kind in (2, 3) and i is not None:
            top = ui[i]
            if kind == 3:
                tie = torch.nonzero(uv[i] == uv[i, -1]).flatten()
                keep = int(tie[torch.randint(0, tie.numel(), (1,), generator=g)])
                top = torch.cat([top[:keep], top[keep + 1:]])
            add(r, top)
        elif kind == 4:
            left = torch.randperm(p, generator=g)[:max(0, kk // 2)]
            mask = torch.ones(p, dtype=torch.bool)
            mask[left] = False
            add(r, torch.nonzero(mask).flatten())
        elif kind == 5:
            x = torch.randint(0, p, (8,), generator=g)
            add(r, torch.cat([x, x, x[:3], torch.tensor([-1, -id_offset - 7, p, p + 100])]))
            if i is not None:
                add(r, ui[i, :2].repeat(3))
        elif kind == 6:
            add(r, bound)
    pairs = torch.cat(out, 1) if out else torch.zeros(2, 0, dtype=torch.int64)
    return pairs, n_rows


def _index(pairs, n_rows, dev):
    """ExclusionIndex through K0; ids below 0 cannot be stored in the COO-built index, so they are dropped
    here (they never match anyway) -- ids past the catalogue are kept."""
    pairs = pairs[:, pairs[1] >= 0]
    num_ids = int(pairs[1].max()) + 1 if pairs.numel() else 1
    return trg.ExclusionIndex.from_edges(pairs.to(dev), n_rows, num_ids)


def _run(dev, q, cat, k, pairs, n_rows, id_offset=0, rows=None, bf16=False):
    ev, ei = oexcl.score_topk_excluding(q, cat, k, pairs, id_offset, rows)
    idx = _index(pairs, n_rows, dev)
    qd, cd = q.to(dev), cat.to(dev)
    if bf16:
        qd, cd = qd.bfloat16(), cd.bfloat16()
    gv, gi = trg.score_topk(qd, cd, k, id_offset, exclude=idx, rows=None if rows is None else rows.to(dev))
    assert gv.shape == ev.shape
    assert torch.equal(gv.cpu(), ev) and torch.equal(gi.cpu(), ei)
    return gv.cpu(), gi.cpu(), qd, cd, idx


def _check_kinds(dev, b, p, h, k, bf16, seed):
    q, cat = _integer_inputs(b, p, h, seed)
    off = 7 if bf16 else 1000
    pairs, n_rows = _pairs(q, cat, k, off, seed)
    gv, gi, qd, cd, _ = _run(dev, q, cat, k, pairs, n_rows, off, bf16=bf16)
    pv, pi = trg.score_topk(qd, cd, k, off)                 # no exclusions at all
    empty = torch.arange(b) % N_KINDS == 0
    assert torch.equal(gv[empty], pv.cpu()[empty]) and torch.equal(gi[empty], pi.cpu()[empty])
    kk = min(k, p)
    few = torch.arange(b) % N_KINDS == 4
    if kk >= 2:
        assert (gi[few] == -1).any(dim=1).all()                   # padded tails
        assert (gv[few][gi[few] == -1] == float("-inf")).all()
    if b == 1:      # a single query row, of every kind in turn
        q, cat = _integer_inputs(N_KINDS, p, h, seed + 1)
        pairs, _ = _pairs(q, cat, k, off, seed + 2)
        for r in range(N_KINDS):
            sel = pairs[:, pairs[0] == r].clone()
            sel[0] = 0
            _run(dev, q[r:r + 1], cat, k, sel, 1, off, bf16=bf16)


@pytest.mark.parametrize("b,p,h,k", [(1, 20_000, 64, 10), (37, 5000, 64, 10), (64, 3000, 128, 100),
                                     (5, 7, 64, 10), (3, 1000, 16, 3), (130, 2500, 256, 128)])
def test_fp32_exclusions_integer_exact(dev, b, p, h, k):
    _check_kinds(dev, b, p, h, k, False, b * p)


@pytest.mark.parametrize("b,p,h,k", [(1, 20_000, 64, 10), (300, 50_000, 128, 100), (129, 7001, 256, 100),
                                     (70, 9000, 192, 100), (4096, 3000, 128, 100), (5, 7, 64, 10),
                                     (64, 200_000, 128, 100)])
def test_bf16_exclusions_integer_exact(dev, b, p, h, k):
    _check_kinds(dev, b, p, h, k, True, b * p + h)


@pytest.mark.parametrize("bf16", [False, True])
def test_rows_indirection_with_repeated_rows(dev, bf16):
    b, p, h, k = 200, 9000, 128, 50
    q, cat = _integer_inputs(b, p, h, 31)
    g = torch.Generator().manual_seed(32)
    rows = torch.randint(0, 23, (b,), generator=g)
    rows[:N_KINDS] = torch.arange(N_KINDS)
    rows[N_KINDS:2 * N_KINDS] = torch.arange(N_KINDS)          # every kind used by two queries at least
    pairs, n_rows = _pairs(q, cat, k, 0, 33, rows=rows)
    gv, gi, qd, cd, idx = _run(dev, q, cat, k, pairs, n_rows, rows=rows, bf16=bf16)
    # queries that share a row with the same embedding get the same answer
    qd2 = torch.cat([qd[:5], qd[:5]])
    r2 = torch.cat([rows[:5], rows[:5]]).to(dev)
    v2, i2 = trg.recommend(qd2, cd, k=k, exclude=idx, rows=r2)
    assert torch.equal(v2[:5], v2[5:]) and torch.equal(i2[:5], i2[5:])
    assert torch.equal(v2[:5].cpu(), gv[:5]) and torch.equal(i2[:5].cpu(), gi[:5])


def test_from_edges_sorted_rows(dev):
    g = torch.Generator().manual_seed(41)
    n_rows, n_ids, e = 300, 5000, 40_000
    row = torch.randint(0, n_rows, (e,), generator=g)
    row[torch.rand(e, generator=g) < 0.3] = 7                    # one long row
    post = torch.randint(0, n_ids, (e,), generator=g)
    post[:1000] = post[1000:2000]                                 # duplicate pairs
    row[:1000] = row[1000:2000]
    idx = trg.ExclusionIndex.from_edges(torch.stack([row, post]).to(dev), n_rows, n_ids)
    rp, ids = idx.rowptr.cpu().long(), idx.ids.cpu().long()
    assert rp[0] == 0 and rp[-1] == e and idx.num_rows == n_rows and ids.numel() == e
    assert torch.equal(rp[1:] - rp[:-1], torch.bincount(row, minlength=n_rows))
    r_of = torch.repeat_interleave(torch.arange(n_rows), rp[1:] - rp[:-1])
    key = r_of * n_ids + ids
    assert (key[1:] >= key[:-1]).all()                            # rows ascending, ids ascending in a row
    assert torch.equal(torch.unique_consecutive(key), torch.unique(row * n_ids + post))
    assert torch.equal(torch.sort(key)[0], torch.sort(row * n_ids + post)[0])   # duplicates kept
    with pytest.raises(IndexError):
        trg.ExclusionIndex.from_edges(torch.stack([row, post]).to(dev), n_rows, n_ids - 1)
    with pytest.raises(IndexError):
        trg.ExclusionIndex.from_edges(torch.stack([row, post]).to(dev), n_rows - 1, n_ids)
    empty = trg.ExclusionIndex.from_edges(torch.zeros(2, 0, dtype=torch.int64, device=dev), 4, 10)
    assert empty.rowptr.tolist() == [0] * 5 and empty.nnz == 0


@pytest.mark.parametrize("bf16", [False, True])
def test_id_offset_shards_merge_to_unsharded(dev, bf16):
    """Each shard scores its own id range against the same (global-id) index; the merged lists, pads
    included, equal the unsharded result."""
    b, p, h, k = 70, 12_000, 128, 40
    q, cat = _integer_inputs(b, p, h, 51)
    pairs, n_rows = _pairs(q, cat, k, 0, 52)
    gv, gi, qd, cd, idx = _run(dev, q, cat, k, pairs, n_rows, bf16=bf16)
    bounds = [(0, 3000), (3000, 7001), (7001, p)]
    vs, ids = [], []
    for a, e in bounds:
        v, i = trg.score_topk(qd, cd[a:e].contiguous(), k, id_offset=a, exclude=idx)
        vs.append(v)
        ids.append(torch.where(i < 0, torch.full_like(i, INT64_MAX), i))   # the merge pads with INT64_MAX
    mv, mi = trg.topk_merge(torch.cat(vs, 1), torch.cat(ids, 1), len(bounds), k)
    assert torch.equal(mv.cpu(), gv) and torch.equal(mi.cpu(), gi)


def test_bf16_large_catalogue_with_exclusions(dev):
    """The 4.2M-post case of the kernel test (tens of thousands of tiles per split, thresholds shared
    across splits) with every kind of exclusion row."""
    b, p, h, k = 9, (1 << 22) + 12_345, 64, 20
    q, cat = _integer_inputs(b, p, h, 99)
    pairs, n_rows = _pairs(q, cat, k, 3, 100)
    _run(dev, q, cat, k, pairs, n_rows, 3, bf16=True)


@pytest.mark.timeout(2400)
def test_config5_excluding_own_top100_integer_exact(dev):
    """4096 queries x 50M posts, K = 100, integer bf16: every row excludes its unfiltered top-100 (ties at
    the 100th score are common) plus 40 random posts.  Exact reference: per chunk, int64 keys
    score * 2^26 + (2^26 - 1 - id), with the keys of excluded pairs pushed below every real key."""
    B, P, H, K, R = 4096, 50_000_000, 128, 100, 40
    gen = torch.Generator(device=dev).manual_seed(12)
    q = torch.randint(0, 4, (B, H), generator=gen, device=dev).to(torch.bfloat16)
    cat = torch.randint(0, 4, (P, H), generator=gen, device=dev, dtype=torch.int8)
    dead = torch.rand(P, generator=gen, device=dev) < 0.05
    cat[dead] = 0
    cat = cat.to(torch.bfloat16)
    _, top = trg.score_topk(q, cat, K)
    rnd = torch.randint(0, P, (B, R), generator=gen, device=dev)
    hist = torch.cat([top, rnd], 1)
    row = torch.arange(B, device=dev)[:, None].expand_as(hist).reshape(-1)
    post = hist.reshape(-1)
    idx = trg.ExclusionIndex.from_edges(torch.stack([row, post]), B, P)
    vals, ids = trg.score_topk(q, cat, K, exclude=idx)
    assert vals.shape == (B, K) and ids.dtype == torch.int64
    shift = 1 << 26
    low = -(1 << 62)
    order = torch.argsort(post)
    s_post, s_row = post[order], row[order]
    best = torch.full((B, K), -1, dtype=torch.int64, device=dev)
    chunk = 500_000
    for a in range(0, P, chunk):
        e = min(a + chunk, P)
        sc = (q.float() @ cat[a:e].float().t()).long()
        key = sc * shift + (shift - 1 - torch.arange(a, e, device=dev))[None, :]
        lo, hi = torch.searchsorted(s_post, torch.tensor([a, e], device=dev)).tolist()
        key[s_row[lo:hi], s_post[lo:hi] - a] = low
        best = torch.topk(torch.cat([best, key], dim=1), K, dim=1)[0]
        del sc, key
    assert (best >= 0).all()
    ref_vals = (best // shift).float()
    ref_ids = shift - 1 - (best % shift)
    assert not (ids[:, :, None] == hist[:, None, :]).any()          # no excluded post comes back
    assert torch.equal(ids, ref_ids)
    assert torch.equal(vals, ref_vals)
