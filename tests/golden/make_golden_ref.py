"""Golden vectors produced by EXECUTING THE REFERENCE'S OWN SOURCE (needs a checkout of the reference
project, ``ramkp990/Truth_Recommendation_GNN``, which this repository does not ship):

    TRG_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden_ref.py

The reference's scripts cannot be imported (they load a dataset at import time), so the definitions on
the hot path are pulled out of ``$TRG_REFERENCE_DIR/train_gnn.py`` by name with ``ast`` and executed
unmodified in a namespace that supplies the globals they read:

  * ``class WeightedRGCN``            (train_gnn.py:147-200)
  * ``def train()``                   (train_gnn.py:242-285; its ``torch.randint`` at :272 included)
  * ``def evaluate(...)``             (train_gnn.py:290-367)
  * ``def build_edge_index_safe(...)`` (train_gnn.py:40-73)

The ONE substitution is ``SAGEConv``: ``torch_geometric`` was not available where the fixtures were made,
so the name is bound to ``oracle.sage.SAGEConvOracle``.  Everything else -- the relation
combine, ReLU, scoring, negative sampling, the scalar-loss quirk, BCEWithLogitsLoss, Adam, the evaluation
loop with sklearn's ndcg_score -- is the reference's text running on real torch.  The fixture therefore
pins the oracle's restatements of those functions to the reference itself; only the SAGEConv operator
stays "parity unpinned" (oracle/__init__.py).  No reference source is stored in the fixture or the repo.
"""
import ast
import os
import sys
import types

import numpy as np
import pandas as pd
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import sage as osage  # noqa: E402
from truth_recommendation_gnn_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("TRG_REFERENCE_DIR")


def reference_defs(names, filename="train_gnn.py", ref_dir=REF):
    """{name: code object} of the top-level class / function definitions ``names`` of a reference script."""
    if not ref_dir:
        raise RuntimeError("set TRG_REFERENCE_DIR to a checkout of the reference project")
    path = os.path.join(ref_dir, filename)
    tree = ast.parse(open(path).read(), filename=path)
    out = {}
    for node in tree.body:
        if isinstance(node, (ast.ClassDef, ast.FunctionDef)) and node.name in names:
            mod = ast.Module(body=[node], type_ignores=[])
            out[node.name] = compile(mod, path, "exec")
    missing = set(names) - set(out)
    if missing:
        raise RuntimeError(f"{path}: definitions not found: {sorted(missing)}")
    return out


def reference_namespace(conv_cls, ref_dir=REF):
    """Namespace holding the reference's ``WeightedRGCN``, ``train``, ``evaluate`` and
    ``build_edge_index_safe`` (their own code objects), with ``SAGEConv`` bound to ``conv_cls``."""
    ns = {"torch": torch, "F": F, "SAGEConv": conv_cls, "np": np, "pd": pd, "__name__": "reference_exec"}
    for code in reference_defs({"WeightedRGCN", "train", "evaluate", "build_edge_index_safe"}, ref_dir=ref_dir).values():
        exec(code, ns)
    return ns


def run_reference_case(ns, g, sd, hidden, steps, seed, device="cpu", test_edges=None, K=10):
    """Drive the reference's train() / evaluate() exactly as its script does (train_gnn.py:204-237,
    372-392): module-level globals, Adam(lr=0.001), BCEWithLogitsLoss, ``torch.randint`` negatives."""
    model = ns["WeightedRGCN"](hidden_dim=hidden).to(device)
    gd = g.to(device)
    with torch.no_grad():                      # lazy (-1, -1) convs materialise on the first forward
        model(gd.x_dict, gd.edge_index_dict)
    model.load_state_dict(sd)
    ns.update(model=model, optimizer=torch.optim.Adam(model.parameters(), lr=0.001),
              criterion=torch.nn.BCEWithLogitsLoss(), device=torch.device(device), x_dict=gd.x_dict,
              graph=types.SimpleNamespace(edge_index_dict=gd.edge_index_dict),
              train_edge_index=gd.train_edge_index, num_users=g.num_users, num_posts=g.num_posts,
              interaction_type_tensor=gd.interaction_type_tensor)
    with torch.no_grad():
        out0 = model(gd.x_dict, gd.edge_index_dict)
    torch.manual_seed(seed)                    # train_gnn.py:272 draws from the default generator
    losses = [ns["train"]() for _ in range(steps)]
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    with torch.no_grad():
        out1 = model(gd.x_dict, gd.edge_index_dict)
    res = dict(out0=out0, losses=losses, grads=grads, out1=out1,
               state_dict_after={k: v.detach().clone() for k, v in model.state_dict().items()})
    if test_edges is not None:
        rec, ndcg = ns["evaluate"](test_edges.to(device), out1["user"], out1["post"], K=K)
        res["recall"], res["ndcg"] = float(rec), float(ndcg)
    return res


def synth_test_edges(g, n, seed=9):
    """Held-out engagements in the reference's evaluate() format: row 0 user ids, row 1 GLOBAL post ids."""
    gen = torch.Generator().manual_seed(seed)
    u = torch.randint(0, g.num_users, (n,), generator=gen)
    p = torch.randint(0, g.num_posts, (n,), generator=gen) + g.num_users
    return torch.stack([u, p])


def synth_activity(n_rows=400, n_users=30, n_posts=90, seed=0):
    rng = np.random.default_rng(seed)
    users = [f"u{i}" for i in range(n_users)]
    df = pd.DataFrame({
        "engager": rng.choice(users + ["ghost"], n_rows), "target_user": rng.choice(users + ["nobody"], n_rows),
        "post_id": rng.integers(0, n_posts + 20, n_rows), "interaction": rng.choice(["QT", "RE", "POST"], n_rows),
        "timestamp": rng.integers(0, 10_000, n_rows)})
    user_to_idx = {u: i for i, u in enumerate(sorted(users))}
    post_to_idx = {i: n_users + i for i in range(n_posts)}
    return df, user_to_idx, post_to_idx


CASES = {
    # name: (U, P, E_eng, E_soc, H, steps, seed, n_test, skew)
    "ref_exec_small": (150, 400, 3000, 800, 16, 3, 123, 300, False),
    "ref_exec_skew": (90, 250, 2000, 500, 64, 2, 7, 200, True),
}


def main():
    torch.set_num_threads(1)   # fixed summation order
    ns = reference_namespace(osage.SAGEConvOracle)
    for name, (u, p, ee, es, h, steps, seed, n_test, skew) in CASES.items():
        g = synth.synth_graph(u, p, ee, es, h, seed=0, skew=skew)
        sd = synth.init_state_dict(h, h, 1, seed=1)
        te = synth_test_edges(g, n_test)
        r = run_reference_case(ns, g, sd, h, steps, seed, test_edges=te)
        fix = dict(meta=dict(u=u, p=p, e_eng=ee, e_soc=es, h=h, steps=steps, seed=seed, skew=skew, k=10),
                   state_dict=sd, test_edges=te,
                   out0_user=r["out0"]["user"], out0_post=r["out0"]["post"],
                   losses=torch.tensor(r["losses"], dtype=torch.float64), last_grads=r["grads"],
                   state_dict_after=r["state_dict_after"], out1_user=r["out1"]["user"], out1_post=r["out1"]["post"],
                   recall=r["recall"], ndcg=r["ndcg"])
        path = os.path.join(HERE, name + ".pt")
        torch.save(fix, path)
        print(name, os.path.getsize(path) // 1024, "KiB", "losses", r["losses"], "recall", r["recall"], "ndcg", r["ndcg"])
    # build_edge_index_safe (train_gnn.py:40-73) on a synthetic activity frame
    df, u2i, p2i = synth_activity()
    e, a = ns["build_edge_index_safe"](df, u2i, p2i)
    torch.save(dict(engage=e, author=a), os.path.join(HERE, "ref_exec_edges.pt"))
    print("ref_exec_edges", tuple(e.shape))


if __name__ == "__main__":
    main()
