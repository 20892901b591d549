"""CPU tests of the host side: the C-ABI library loads and exports every symbol the header
declares, the drop-in modules keep the reference's API contract, and nothing silently falls back
to the CPU."""
import ctypes
import os
import re

import pytest
import torch

import truth_recommendation_gnn_b200 as trg
from truth_recommendation_gnn_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "trg_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(trg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    syms = _declared_symbols()
    assert len(syms) >= 12
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/trg_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "python binding and header disagree"
    assert _lib.load().trg_abi_version() == _lib.ABI_VERSION
    assert _lib.load().trg_csr_workspace_bytes(1000, 100) > 4 * 4 * 1000


def test_no_cpu_fallback():
    conv = trg.SAGEConv((8, 8), 4)
    with pytest.raises(_lib.TrgError):
        conv((torch.zeros(2, 8), torch.zeros(3, 8)), torch.zeros(2, 0, dtype=torch.long))
    with pytest.raises(_lib.TrgError):
        trg.score_topk(torch.zeros(1, 8), torch.zeros(4, 8), 2)
    with pytest.raises(_lib.TrgError):
        trg.build_csr(torch.zeros(3, dtype=torch.long), torch.zeros(3, dtype=torch.long), 2, 2, validate=False)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "truth_recommendation_gnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f


def test_lazy_parameters_and_state_dict_contract():
    # train_gnn.py:206-207: optimizer is built before the first forward on lazily-shaped params
    model = trg.WeightedRGCN(hidden_dim=64)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    ids = [id(p) for p in model.parameters()]
    keys = list(model.state_dict().keys())
    assert keys == [f"{c}.{p}" for c in ("msg_direct", "msg_social", "post_update")
                    for p in ("lin_l.weight", "lin_l.bias", "lin_r.weight")]
    sd = synth.init_state_dict(64, 64)
    model.load_state_dict(sd)                         # strict, materialises in place
    assert ids == [id(p) for p in model.parameters()]
    assert all(torch.equal(model.state_dict()[k], sd[k]) for k in sd)
    assert sum(p.numel() for p in model.parameters()) == 24768   # SURVEY §8 A8
    assert len(opt.param_groups[0]["params"]) == 9
    stacked = trg.StackedWeightedRGCN(32, 3, in_channels=(16, 16))
    assert stacked.layers[0].msg_direct.lin_l.weight.shape == (32, 16)
    assert stacked.layers[2].post_update.lin_r.weight.shape == (32, 32)
    stacked.load_state_dict(synth.init_state_dict(32, 16, 3))


def test_sageconv_rejects_unaccelerated_options():
    with pytest.raises(NotImplementedError):
        trg.SAGEConv((-1, -1), 8, aggr="max")
    with pytest.raises(NotImplementedError):
        trg.SAGEConv((-1, -1), 8, normalize=True)


def test_linear_default_init_matches_torch():
    torch.manual_seed(0)
    a = trg.Linear(16, 8)
    torch.manual_seed(0)
    b = torch.nn.Linear(16, 8)
    assert torch.equal(a.weight, b.weight) and torch.equal(a.bias, b.bias)


def test_synth_is_deterministic_and_in_reference_format():
    g1 = synth.synth_graph(30, 50, 200, 60, 8, seed=0)
    g2 = synth.synth_graph(30, 50, 200, 60, 8, seed=0)
    for k in g1.edge_index_dict:
        assert torch.equal(g1.edge_index_dict[k], g2.edge_index_dict[k])
        assert g1.edge_index_dict[k].dtype == torch.int64 and g1.edge_index_dict[k].shape[0] == 2
    assert torch.equal(g1.edge_index_dict[synth.REL_DIRECT], g1.edge_index_dict[synth.REL_ENGAGE].flip(0))
    assert torch.allclose(g1.x_dict["user"].norm(dim=1), torch.ones(30), atol=1e-6)
    assert g1.mp_edges == 2 * 200 + 60
    w = g1.interaction_type_tensor
    assert w.shape == (80,) and set(w[30:].tolist()) <= {1.0, 3.0} and float(w[:30].abs().sum()) == 0.0


def test_vectorised_graph_prep_matches_reference_loops():
    """§8f N4: vectorised edge-list construction / weight table == the iterrows loops
    (train_gnn.py:40-73, 226-237), including unmapped ids and repeated post ids."""
    import numpy as np
    import pandas as pd
    from oracle import graph_prep as oprep
    from truth_recommendation_gnn_b200 import graph_io
    rng = np.random.default_rng(0)
    users = [f"u{i}" for i in range(40)]
    n = 500
    df = pd.DataFrame({
        "engager": rng.choice(users + ["ghost"], n), "target_user": rng.choice(users + ["nobody"], n),
        "post_id": rng.integers(0, 120, n), "interaction": rng.choice(["QT", "RE", "POST"], n),
        "timestamp": rng.integers(0, 10_000, n)})
    user_to_idx = {u: i for i, u in enumerate(sorted(users))}
    post_to_idx = {i: len(users) + i for i in range(100)}          # posts 100..119 unmapped
    e_ref, a_ref = oprep.build_edge_index_safe(df, user_to_idx, post_to_idx)
    e, a = graph_io.build_edge_index(df, user_to_idx, post_to_idx)
    assert torch.equal(e, e_ref) and torch.equal(a, a_ref) and e.dtype == torch.int64
    train = df[df["post_id"] < 100].sort_values("timestamp").reset_index(drop=True)
    assert torch.equal(graph_io.interaction_type_table(train, post_to_idx), oprep.interaction_type_table(train, post_to_idx))


def test_temporal_split_and_degree_features_match_reference_loops():
    """§8f N4 remainder: chronological 80/10/10 split (train_gnn.py:28-35) and the per-user degree /
    engagement features (build_graph.py:409-429) against their literal loops."""
    import numpy as np
    import pandas as pd
    from oracle import graph_prep as oprep
    from truth_recommendation_gnn_b200 import graph_io
    rng = np.random.default_rng(1)
    users = [f"u{i}" for i in range(50)]
    n = 777
    act = pd.DataFrame({"engager": rng.choice(users + ["ghost"], n), "post_id": rng.integers(0, 90, n),
                        "timestamp": rng.integers(0, 300, n)})            # many equal timestamps
    tr, va, te = graph_io.temporal_split(act)
    tr_r, va_r, te_r = oprep.temporal_split(act)
    for a, b in ((tr, tr_r), (va, va_r), (te, te_r)):
        assert a.equals(b)
    assert len(tr) == int(0.8 * n) and len(tr) + len(va) + len(te) == n
    u2i = {u: i for i, u in enumerate(users)}
    soc = pd.DataFrame({"follower": rng.integers(0, 50, 600), "followee": rng.integers(0, 50, 600)})
    f = graph_io.user_structural_features(soc, act, u2i, 50)
    assert torch.equal(f, oprep.user_structural_features(soc, act, u2i, 50)) and f.dtype == torch.float32


def test_csr_cache_checksum_is_order_sensitive():
    from truth_recommendation_gnn_b200 import graph_io
    ei = torch.tensor([[0, 1, 2, 3], [3, 2, 1, 0]])
    assert graph_io._edge_checksum(ei) != graph_io._edge_checksum(ei.flip(1))
    assert graph_io._edge_checksum(ei) != graph_io._edge_checksum(ei.flip(0))
    assert graph_io._edge_checksum(ei) == graph_io._edge_checksum(ei.clone())
    assert graph_io._edge_checksum(torch.empty(2, 0, dtype=torch.long)) == 0


def test_hetero_inputs_follow_train_gnn_assembly():
    from truth_recommendation_gnn_b200 import graph_io
    nu, np_ = 5, 7
    data = {"num_users": nu, "num_posts": np_, "x": torch.arange((nu + np_) * 4.0).reshape(nu + np_, 4),
            "edge_index_social": torch.tensor([[0, 1, 4], [2, 2, 0]])}
    train_engage = torch.tensor([[0, 3, 4, 9, 2], [nu + 1, nu + 6, nu + 7, nu + 2, nu - 1]])   # 3 invalid rows
    x_dict, ei = graph_io.hetero_inputs(data, train_engage)
    assert x_dict["user"].shape == (nu, 4) and x_dict["post"].shape == (np_, 4)
    assert ei[trg.REL_ENGAGE].tolist() == [[0, 3], [1, 6]]
    assert torch.equal(ei[trg.REL_DIRECT], ei[trg.REL_ENGAGE].flip(0))
    assert torch.equal(ei[trg.REL_SOCIAL], data["edge_index_social"])


def test_negative_share_capacity_covers_randint_modulo_bias():
    """``torch.randint(0, P, (E,))`` (train_gnn.py:272) draws 32 bits and reduces them ``% P``: ids below
    ``2^32 mod P`` are ``1 / floor(2^32 / P)`` more likely.  At config 4 (P = 50M, E = 800M, 8 ranks) that is
    +117 000 entries on a rank's 100M share -- beyond 8 sigma of the binomial count -- and overflowed the
    fixed-capacity selection (found by running config 4; r2).  The capacity must cover the biased expectation."""
    from truth_recommendation_gnn_b200.dist import ShardedGraph
    for P, E, world in ((50_000_000, 800_000_000, 8), (5_000_000, 40_000_000, 8), (70_003, 600_000, 2), (7, 100, 2)):
        sh = ShardedGraph.__new__(ShardedGraph)
        sh.num_posts, sh.n_pos_global, sh.world = P, E, world
        sh.cp = (P + world - 1) // world
        cap = sh.neg_capacity()
        q = 2**32 // P
        worst = E * sh.cp * (q + 1) / 2.0**32                 # expected share of the most favoured rank
        assert cap <= E
        assert cap >= min(E, worst + 7.9 * worst ** 0.5), (P, E, world, cap, worst)
    # the observed overflow: 100 132 949 selected at config 4
    sh.num_posts, sh.n_pos_global, sh.world, sh.cp = 50_000_000, 800_000_000, 8, 6_250_000
    assert sh.neg_capacity() > 100_132_949


def test_bench_reference_arm_line_contract(tmp_path):
    """``bench.py --impl reference`` (run next to the GPU arm): one JSON line on stdout with the
    contract's keys, the SAME ``config`` object the GPU arm prints for that workload, and a ``cpu_baseline``
    describing the run; ``--dump-outputs`` writes the last timed step's loss, parameters and gradients.  Runs
    the tiny workload on the CPU oracle (no GPU involved)."""
    import json
    import os
    import subprocess
    import sys

    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--workload", "tiny", "--steps", "2",
                        "--warmup", "1", "--no-extras", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    sys.path.insert(0, root)
    import bench
    assert d["config"] == bench.config_of("tiny", bench.WORKLOADS["tiny"])      # identical in both arms
    assert d["value"] > 0 and d["steps"] == 2
    w = bench.WORKLOADS["tiny"]
    sd = synth.init_state_dict(w["hidden"], w["hidden"], w["layers"])
    out = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == sorted(["loss"] + [f"{k}.{n}" for k in ("param", "grad") for n in sd])
    assert out["loss"].dtype == np.float64 and out["loss"].shape == () and np.isfinite(out["loss"])
    for n, v in sd.items():
        p, gr = out[f"param.{n}"], out[f"grad.{n}"]
        assert p.dtype == gr.dtype == np.float32 and p.shape == gr.shape == tuple(v.shape)
        assert np.isfinite(gr).all() and not np.array_equal(p, v.numpy()), n     # the steps moved every tensor


def test_bench_refuses_to_run_the_product_without_a_gpu():
    """The GPU arm has no CPU fallback: without a CUDA device it stops with a message, it does not time the oracle."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a machine without a GPU")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--workload", "tiny", "--steps", "1"], capture_output=True,
                       text=True, cwd=root, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)
