"""CPU tests of the oracle itself: restated PyG semantics vs dense-adjacency math, the integer
oracles (torch vs plain C), the committed golden fixtures, and the reference's edge cases."""
import torch
import torch.nn.functional as F

from oracle import cint
from oracle import csr as ocsr
from oracle import sage as osage
from oracle import topk as otopk
from tests.util import golden_graph, load_golden, oracle_model
from truth_recommendation_gnn_b200 import synth


def _dense_sage(x_src, x_dst, ei, w_l, b_l, w_r):
    n_dst, n_src = x_dst.size(0), x_src.size(0)
    a = torch.zeros(n_dst, n_src, dtype=torch.float64)
    for s, d in ei.t().tolist():
        a[d, s] += 1.0                      # duplicates count twice (no coalescing)
    deg = a.sum(1, keepdim=True).clamp(min=1)
    mean = (a / deg) @ x_src.double()
    return mean @ w_l.double().t() + b_l.double() + x_dst.double() @ w_r.double().t()


def test_sage_conv_matches_dense_adjacency():
    g = torch.Generator().manual_seed(7)
    x_src, x_dst = torch.randn(6, 8, generator=g), torch.randn(5, 8, generator=g)
    ei = torch.tensor([[0, 1, 1, 5, 2, 2, 2], [0, 0, 0, 3, 4, 4, 1]])  # dup edges, dst 2 isolated
    w_l, b_l, w_r = torch.randn(4, 8, generator=g), torch.randn(4, generator=g), torch.randn(4, 8, generator=g)
    out = osage.sage_conv(x_src, x_dst, ei, w_l, b_l, w_r)
    ref = _dense_sage(x_src, x_dst, ei, w_l, b_l, w_r)
    assert torch.allclose(out.double(), ref, atol=1e-5)
    # isolated destination: mean is exactly zero -> bias + root term only
    assert torch.allclose(out[2], b_l + x_dst[2] @ w_r.t(), atol=1e-6)


def test_sage_conv_empty_edges_and_no_sources():
    # inference.py:412-419: one user, zero posts, four empty [2,0] edge tensors
    x_user, x_post = torch.randn(1, 8), torch.empty(0, 8)
    empty = torch.empty(2, 0, dtype=torch.long)
    m = osage.WeightedRGCNOracle(4, (8, 8))
    out = m({"user": x_user, "post": x_post},
            {osage.REL_DIRECT: empty, osage.REL_SOCIAL: empty, osage.REL_ENGAGE: empty})
    d, s = m.msg_direct, m.msg_social
    exp = F.relu(1.0 * (d.lin_l.bias + d.lin_r(x_user)) + 0.75 * (s.lin_l.bias + s.lin_r(x_user)))
    assert torch.allclose(out["user"], exp, atol=1e-6)
    assert out["post"].shape == (0, 4)


def test_module_matches_functional_and_keys():
    m = osage.SAGEConvOracle((8, 8), 4)
    assert sorted(m.state_dict().keys()) == ["lin_l.bias", "lin_l.weight", "lin_r.weight"]
    x_src, x_dst = torch.randn(5, 8), torch.randn(3, 8)
    ei = torch.tensor([[0, 4, 2], [1, 1, 0]])
    a = m((x_src, x_dst), ei)
    b = osage.sage_conv(x_src, x_dst, ei, m.lin_l.weight, m.lin_l.bias, m.lin_r.weight)
    assert torch.equal(a, b)


def test_scalar_loss_quirk():
    # train_gnn.py:276-281: pos_loss is a scalar, so (w * pos_loss).mean() == mean(w) * pos_loss
    g = torch.Generator().manual_seed(3)
    u, p = torch.randn(5, 4, generator=g), torch.randn(6, 4, generator=g)
    pos_u, pos_p = torch.tensor([0, 1, 1, 4]), torch.tensor([5, 2, 2, 0])
    neg_p = torch.tensor([1, 1, 3, 4])
    w = torch.zeros(11)
    w[5:] = torch.tensor([1., 3., 1., 3., 1., 1.])
    loss = osage.link_loss(u, p, pos_u, pos_p, neg_p, w, 5)
    ps = (u[pos_u] * p[pos_p]).sum(1)
    ns = (u[pos_u] * p[neg_p]).sum(1)
    exp = w[pos_p + 5].mean() * F.softplus(-ps).mean() + F.softplus(ns).mean()
    assert abs(float(loss) - float(exp)) < 1e-6


def test_csr_oracle_torch_vs_c():
    g = synth.synth_graph(50, 80, 700, 200, 8, seed=5, skew=True)
    for rel, ei in g.edge_index_dict.items():
        n_dst = g.x_dict[rel[2]].size(0)
        rp, col, eid = ocsr.csr_by_dst(ei, n_dst)
        rp2, col2, eid2 = cint.csr_by_dst(ei, n_dst)
        assert torch.equal(rp, rp2) and torch.equal(col, col2) and torch.equal(eid, eid2)
        # structure checks: rows sorted, edge ids ascending inside a row (stability)
        assert int(rp[-1]) == ei.size(1)
        assert torch.equal(ei[1][eid], torch.repeat_interleave(torch.arange(n_dst), rp[1:] - rp[:-1]))
        same_row = ei[1][eid][1:] == ei[1][eid][:-1]
        assert bool(((eid[1:] > eid[:-1]) | ~same_row).all())
    rp, col, eid = ocsr.csr_by_dst(torch.empty(2, 0, dtype=torch.long), 4)
    assert rp.tolist() == [0, 0, 0, 0, 0] and col.numel() == 0


def test_topk_canonical_vs_torch_and_c():
    g = torch.Generator().manual_seed(11)
    scores = torch.randn(6, 200, generator=g)
    vals, ids = otopk.topk_canonical(scores, 10)
    tv, ti = torch.topk(scores, 10)
    assert torch.equal(vals, tv) and torch.equal(ids, ti)   # distinct scores: torch.topk is well defined
    cv, ci = cint.topk_rows(scores, 10)
    assert torch.equal(vals, cv) and torch.equal(ids, ci)
    # ties: values always agree with torch.topk; ids follow (score desc, id asc)
    s = torch.zeros(1, 20)
    s[0, 0] = s[0, 7] = 1.0
    vals, ids = otopk.topk_canonical(s, 5)
    assert torch.equal(vals, torch.topk(s, 5)[0])
    assert ids.tolist() == [[0, 7, 1, 2, 3]]
    cv, ci = cint.topk_rows(s, 5)
    assert torch.equal(ids, ci)
    # K >= n
    vals, ids = otopk.topk_canonical(scores[:, :4], 10)
    assert vals.shape == (6, 4)


def test_topk_sharded_merge_equals_unsharded():
    q, cat = synth.synth_queries(5, 300, 16, zero_frac=0.2)
    vals, ids = otopk.score_topk(q, cat, 10)
    parts = [otopk.score_topk(q, cat[a:b], 10, id_offset=a) for a, b in [(0, 100), (100, 230), (230, 300)]]
    mv, mi = otopk.merge_topk([p[0] for p in parts], [p[1] for p in parts], 10)
    assert torch.equal(ids, mi) and torch.equal(vals, mv)


def test_golden_fixtures_reproduce():
    torch.set_num_threads(1)
    for name in ("tiny_l1", "small_l2", "small_l1_skew"):
        fix = load_golden(name)
        m = fix["meta"]
        g = golden_graph(fix)
        model = oracle_model(m["h"], m["layers"], fix["state_dict"])
        with torch.no_grad():
            out = model(g.x_dict, g.edge_index_dict)
        assert torch.equal(out["user"], fix["out0_user"]) and torch.equal(out["post"], fix["out0_post"])
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        for s in range(m["steps"]):
            loss = osage.train_step(model, opt, g.x_dict, g.edge_index_dict, g.train_edge_index,
                                    g.interaction_type_tensor, m["u"], m["p"], neg_p=fix["neg"][s])
            assert abs(loss - float(fix["losses"][s])) < 1e-6
        for k, v in model.state_dict().items():
            assert torch.allclose(v, fix["state_dict_after"][k], atol=1e-7)
        for rel, c in fix["csr"].items():
            ei = fix["edge_index"][rel]
            rp, col, eid = ocsr.csr_by_dst(ei, g.x_dict[eval(rel)[2]].size(0))
            assert torch.equal(rp.int(), c["rowptr"]) and torch.equal(col.int(), c["col"]) and torch.equal(eid.int(), c["eid"])


def test_stacked_is_composition_of_blocks():
    g = synth.synth_graph(20, 30, 100, 40, 8, seed=1)
    sd = synth.init_state_dict(8, 8, 2, seed=1)
    m2 = oracle_model(8, 2, sd)
    out = m2(g.x_dict, g.edge_index_dict)
    mid = m2.layers[0](g.x_dict, g.edge_index_dict)
    out_b = m2.layers[1](mid, g.edge_index_dict)
    assert torch.equal(out["user"], out_b["user"]) and (out["user"] >= 0).all()


# ------------------------------------------------------------------------------------------------
# pin: the oracle's restatements against the reference's own source, executed
# ------------------------------------------------------------------------------------------------
def _check_oracle_against_reference_run(name, r, m, g, sd, test_edges):
    """``r``: outputs of the reference's WeightedRGCN / train() / evaluate() code (a committed fixture, or a
    live execution).  The oracle must reproduce them BIT FOR BIT: same torch, same ops, same order."""
    from oracle import evaluate as oeval
    model = oracle_model(m["h"], 1, sd)
    with torch.no_grad():
        out = model(g.x_dict, g.edge_index_dict)
    assert torch.equal(out["user"], r["out0_user"]) and torch.equal(out["post"], r["out0_post"]), name
    opt = torch.optim.Adam(model.parameters(), lr=0.001)
    torch.manual_seed(m["seed"])         # the oracle's train_step draws torch.randint like train_gnn.py:272
    for s in range(m["steps"]):
        loss = osage.train_step(model, opt, g.x_dict, g.edge_index_dict, g.train_edge_index,
                                g.interaction_type_tensor, m["u"], m["p"])
        assert loss == float(r["losses"][s]), (name, s, loss, float(r["losses"][s]))
    for n, p in model.named_parameters():
        assert torch.equal(p.grad, r["last_grads"][n]), (name, n)
        assert torch.equal(p.detach(), r["state_dict_after"][n]), (name, n)
    with torch.no_grad():
        out1 = model(g.x_dict, g.edge_index_dict)
    assert torch.equal(out1["user"], r["out1_user"])
    rec, ndcg = oeval.evaluate(test_edges, out1["user"], out1["post"], m["u"], m["k"])
    assert rec == r["recall"] and ndcg == r["ndcg"], (name, rec, ndcg)


def test_oracle_reproduces_reference_executed_fixtures():
    """tests/golden/ref_exec_*.pt hold outputs of the reference's OWN class / function source (pulled from
    the reference's train_gnn.py by name and executed, SAGEConv bound to the oracle's -- see
    tests/golden/make_golden_ref.py).  This pins ``WeightedRGCNOracle``, ``train_step`` / ``link_loss``
    (scalar-loss quirk, randint negatives, Adam) and ``oracle.evaluate`` to the reference itself."""
    torch.set_num_threads(1)
    for name in ("ref_exec_small", "ref_exec_skew"):
        fix = load_golden(name)
        m = fix["meta"]
        g = synth.synth_graph(m["u"], m["p"], m["e_eng"], m["e_soc"], m["h"], seed=0, skew=m["skew"])
        _check_oracle_against_reference_run(name, fix, m, g, fix["state_dict"], fix["test_edges"])
    from oracle import graph_prep as oprep
    from tests.golden.make_golden_ref import synth_activity
    df, u2i, p2i = synth_activity()
    e, a = oprep.build_edge_index_safe(df, u2i, p2i)
    ref = load_golden("ref_exec_edges")
    assert torch.equal(e, ref["engage"]) and torch.equal(a, ref["author"])


def test_committed_fixtures_match_a_live_reference_execution():
    """Where a checkout of the reference project is named by ``TRG_REFERENCE_DIR``, execute its source again
    and check that the committed fixtures are what it produces; skipped without one."""
    import os
    import pytest
    from tests.golden import make_golden_ref as mk
    if not mk.REF or not os.path.exists(os.path.join(mk.REF, "train_gnn.py")):
        pytest.skip("no reference checkout (set TRG_REFERENCE_DIR)")
    torch.set_num_threads(1)
    ns = mk.reference_namespace(osage.SAGEConvOracle)
    name = "ref_exec_small"
    u, p, ee, es, h, steps, seed, n_test, skew = mk.CASES[name]
    fix = load_golden(name)
    g = synth.synth_graph(u, p, ee, es, h, seed=0, skew=skew)
    r = mk.run_reference_case(ns, g, fix["state_dict"], h, steps, seed, test_edges=fix["test_edges"])
    assert torch.equal(r["out0"]["user"], fix["out0_user"])
    assert r["losses"] == [float(x) for x in fix["losses"]]
    for n in r["grads"]:
        assert torch.equal(r["grads"][n], fix["last_grads"][n])
    assert r["recall"] == fix["recall"] and r["ndcg"] == fix["ndcg"]
