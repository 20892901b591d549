"""Top-k with per-user exclusions, CPU side: the oracle against a per-row loop, the refusal of host
tensors, and the sharded host logic (world-size-2 gloo, oracle compute injected) against the
unsharded oracle, pads included."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import truth_recommendation_gnn_b200 as trg
from oracle import topk as otopk
from tests import oracle_exclude as oexcl
from truth_recommendation_gnn_b200 import _lib
from truth_recommendation_gnn_b200 import dist as tdist


def _loop_reference(q, cat, k, pairs, id_offset=0, rows=None):
    """One Python list per query: admissible (score, id), sorted by (score desc, id asc)."""
    scores = (q @ cat.T).tolist()
    b, p = len(scores), cat.size(0)
    kk = min(k, p)
    excl = set(map(tuple, pairs.t().tolist()))
    vals = torch.full((b, kk), float("-inf"))
    ids = torch.full((b, kk), -1, dtype=torch.int64)
    for i in range(b):
        r = i if rows is None else int(rows[i])
        keep = sorted(((s, j + id_offset) for j, s in enumerate(scores[i]) if (r, j + id_offset) not in excl),
                      key=lambda t: (-t[0], t[1]))[:kk]
        for c, (s, g) in enumerate(keep):
            vals[i, c], ids[i, c] = s, g
    return vals, ids


@pytest.mark.parametrize("id_offset,use_rows", [(0, False), (50, False), (0, True), (1000, True)])
def test_oracle_matches_per_row_loop(id_offset, use_rows):
    g = torch.Generator().manual_seed(5 + id_offset)
    b, p, h, k = 9, 61, 8, 10
    q = torch.randint(0, 3, (b, h), generator=g).float()
    cat = torch.randint(0, 3, (p, h), generator=g).float()      # integer scores: many ties
    n_rows = 6
    rows = torch.randint(0, n_rows, (b,), generator=g) if use_rows else None
    er = torch.randint(0, n_rows if use_rows else b, (300,), generator=g)
    gi = torch.randint(id_offset - 5, id_offset + p + 5, (300,), generator=g)   # some outside the catalogue
    pairs = torch.stack([er, gi])
    # one row loses all but 3 of its posts: padded tail
    last = int(rows[0]) if use_rows else 0
    full = torch.stack([torch.full((p - 3,), last), torch.arange(p - 3) + id_offset])
    pairs = torch.cat([pairs, full, full[:, :5]], 1)                              # duplicates too
    ev, ei = _loop_reference(q, cat, k, pairs, id_offset, rows)
    ov, oi = oexcl.score_topk_excluding(q, cat, k, pairs, id_offset, rows)
    assert torch.equal(ov, ev) and torch.equal(oi, ei)
    assert (oi[0] == -1).sum() >= k - 3
    # no pairs: the plain oracle
    pv, pi = oexcl.score_topk_excluding(q, cat, k, torch.zeros(2, 0, dtype=torch.int64), id_offset, rows)
    sv, si = otopk.score_topk(q, cat, k, id_offset)
    assert torch.equal(pv, sv) and torch.equal(pi, si)


def test_host_tensors_are_refused():
    ei = torch.tensor([[0, 1, 1], [3, 2, 0]])
    with pytest.raises(_lib.TrgError):
        trg.ExclusionIndex.from_edges(ei, 2, 4)
    idx = trg.ExclusionIndex(torch.tensor([0, 1, 3], dtype=torch.int32), torch.tensor([3, 0, 2], dtype=torch.int32), 2)
    with pytest.raises(_lib.TrgError):
        trg.score_topk(torch.zeros(2, 8), torch.zeros(4, 8), 2, exclude=idx)
    with pytest.raises(_lib.TrgError):
        trg.recommend(torch.zeros(2, 8), torch.zeros(4, 8), 2, exclude=idx, rows=torch.tensor([1, 1]))


def test_argument_checks():
    idx = trg.ExclusionIndex(torch.tensor([0, 1, 3], dtype=torch.int32), torch.tensor([3, 0, 2], dtype=torch.int32), 2)
    with pytest.raises(ValueError):
        trg.ExclusionIndex.from_edges(torch.zeros(3, dtype=torch.int64), 2, 4)
    with pytest.raises(TypeError):
        trg.ExclusionIndex(torch.tensor([0, 1, 3]), torch.tensor([3, 0, 2]), 2)
    with pytest.raises(ValueError):
        trg.ExclusionIndex(torch.tensor([0, 3], dtype=torch.int32), torch.tensor([3, 0, 2], dtype=torch.int32), 2)
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("kernel library not built")
    with pytest.raises(ValueError):     # rows without an index
        trg.score_topk(torch.zeros(2, 8), torch.zeros(4, 8), 2, rows=torch.tensor([0, 1]))
    with pytest.raises(ValueError):     # more queries than exclusion rows, no rows= mapping
        trg.score_topk(torch.zeros(3, 8), torch.zeros(4, 8), 2, exclude=idx)
    with pytest.raises(ValueError):     # rows of the wrong length
        trg.score_topk(torch.zeros(2, 8), torch.zeros(4, 8), 2, exclude=idx, rows=torch.tensor([0]))


# ------------------------------------------------------------------ sharded (world size 2, gloo)
B, P, H, K = 7, 53, 8, 10


def _oracle_score_topk(q, cat, k, id_offset=0, exclude=None, rows=None):
    """The kernel's contract on the oracle: ``exclude`` is a [2, E] (row, global id) pair tensor."""
    if exclude is None:
        return otopk.score_topk(q, cat, k, id_offset)
    return oexcl.score_topk_excluding(q, cat, k, exclude, id_offset, rows)


def _oracle_merge(vals, ids, n_lists, k):
    """trg_topk_merge on the oracle: id INT64_MAX is padding, and missing entries come out as -1."""
    k_in = vals.size(1) // n_lists
    mv, mi = otopk.merge_topk([vals[:, i * k_in:(i + 1) * k_in] for i in range(n_lists)],
                              [ids[:, i * k_in:(i + 1) * k_in] for i in range(n_lists)], k)
    return mv, torch.where(mi == torch.iinfo(torch.int64).max, torch.full_like(mi, -1), mi)


def _inputs():
    g = torch.Generator().manual_seed(17)
    q = torch.randint(0, 3, (B, H), generator=g).float()
    cat = torch.randint(0, 3, (P, H), generator=g).float()
    rows = torch.tensor([0, 1, 2, 3, 1, 4, 0])
    er = torch.tensor([0, 2, 4])[torch.randint(0, 3, (60,), generator=g)]     # random history of rows 0, 2, 4
    gi = torch.randint(0, P, (60,), generator=g)
    # row 1 keeps 4 posts (2 per shard), row 3 keeps 1 post in the second shard only: both are padded
    r1 = torch.tensor([j for j in range(P) if j not in (3, 20, 30, 50)])
    r3 = torch.tensor([j for j in range(P) if j != 40])
    pairs = torch.cat([torch.stack([er, gi]), torch.stack([torch.full_like(r1, 1), r1]),
                       torch.stack([torch.full_like(r3, 3), r3])], 1)
    return q, cat, pairs, rows


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        q, cat, pairs, rows = _inputs()
        p0, p1 = rank * P // world, (rank + 1) * P // world
        rv, ri = tdist.recommend_sharded(q, cat[p0:p1].contiguous(), K, p0, _oracle_score_topk, _oracle_merge,
                                         exclude=pairs, rows=rows)
        out.put((rank, rv.numpy().copy(), ri.numpy().copy()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_sharded_recommend_with_exclusions_matches_unsharded():
    world, port = 2, 29500 + os.getpid() % 2000 + 13
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    q, cat, pairs, rows = _inputs()
    ev, ei = oexcl.score_topk_excluding(q, cat, K, pairs, 0, rows)
    assert (ei[1] == -1).sum() == K - 4 and (ei[3] == -1).sum() == K - 1
    assert ei[3, 0] == 40
    for _, rv, ri in res:
        assert torch.equal(torch.from_numpy(rv), ev) and torch.equal(torch.from_numpy(ri), ei)
