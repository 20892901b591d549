"""e4m3 top-k against bf16 at config 5: python tools/bench_topk_fp8.py [--repeats N] [--parent-lib SO]

Arms, alternated inside one process (repeat r runs every arm once, then r + 1 ...), each at K = 100 and
K = 10, on config 5 (4096 users x 50M posts, synthetic relu(randn) rows as in ``synth.synth_queries``; the
catalogue does not fit the L2):
  a  bf16 ``score_topk``                         (H = 128 and H = 256)
  b  the e4m3 stage alone, 128 candidates        (H = 128)
  c  both stages: ``score_topk`` on an ``Fp8Catalogue``                (H = 128 and H = 256)
  d  (c) with 40 random history posts per user excluded               (H = 128)
plus the parts of (c): the query quantiser, the re-scoring kernel and the selection (``trg_topk_merge``)
timed alone on the same shapes, and the e4m3 stage keeping only K candidates (what its list length costs).  Recall@K on a 256-query sample against the exact top-K of fp32 copies of
the same tables (fp32 ``score_topk``): (a), the e4m3 stage's own top-K, and (c).

``--parent-lib``: another build of the library (e.g. the parent commit's); bf16 ``trg_score_topk`` of both
libraries is then called side by side on the same inputs (outputs compared bit for bit, times alternated).
Prints the GPU, its power limit and max SM clock, then one JSON line per measurement; ms are per call, CUDA
events around ``iters`` back-to-back calls, the median over repeats."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import truth_recommendation_gnn_b200 as trg  # noqa: E402
from truth_recommendation_gnn_b200 import _lib, fp8, synth  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"
    except (OSError, subprocess.SubprocessError):
        smi = "nvidia-smi unavailable"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


def time_calls(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(arms, iters, repeats):
    for fn in arms.values():      # warm every shape
        fn()
    torch.cuda.synchronize()
    ms = {a: [] for a in arms}
    for _ in range(repeats):
        for a, fn in arms.items():
            ms[a].append(round(time_calls(fn, iters), 4))
    return ms, {a: statistics.median(v) for a, v in ms.items()}


def history(b, n_rand, n_posts, gen, dev):
    hist = torch.randint(0, n_posts, (b, n_rand), generator=gen, device=dev)
    row = torch.arange(b, device=dev)[:, None].expand_as(hist).reshape(-1)
    return trg.ExclusionIndex.from_edges(torch.stack([row, hist.reshape(-1)]), b, n_posts), hist


def recall(found, exact):
    """share of the exact top-K ids (``exact [B, K]``) that are in ``found [B, *]``"""
    return float((exact[:, :, None] == found[:, None, :]).any(-1).float().mean())


def run(h, ks, full, iters, repeats, seed):
    dev = torch.device("cuda")
    b, p = 4096, 50_000_000
    q, cat = synth.synth_queries(b, p, h, seed=seed, device=dev, dtype=torch.bfloat16)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    cat8 = trg.Fp8Catalogue.from_dense(cat)
    s1.record()
    torch.cuda.synchronize()
    build_ms = s0.elapsed_time(s1)
    gen = torch.Generator(device=dev).manual_seed(seed + 1)
    idx, hist = history(b, 40, p, gen, dev)
    results = []
    for k in ks:
        arms = {"a_bf16": lambda: trg.score_topk(q, cat, k),
                "c_fp8_two_stage": lambda: trg.score_topk(q, cat8, k)}
        if full:
            _, cand = fp8._fp8_candidates(q, cat8)
            cv, ci = torch.randn(b, fp8.N_CAND, device=dev), cand.clone()
            arms.update({
                "b_fp8_stage": lambda: fp8._fp8_candidates(q, cat8),
                "part_fp8_stage_at_k": lambda: fp8._fp8_candidates(q, cat8, k),
                "d_fp8_exclude_40": lambda: trg.score_topk(q, cat8, k, exclude=idx),
                "part_query_quantiser": lambda: fp8.quantize_rows(q),
                "part_rescore_and_select": lambda: fp8.rescore_topk(q, cat, cand, k),
                "part_select": lambda: trg.topk_merge(cv, ci, fp8.N_CAND, k),
            })
            _, ids = arms["d_fp8_exclude_40"]()
            assert not (ids[:, :, None] == hist[:, None, :]).any()
        ms, med = alternate(arms, iters, repeats)
        out = {"H": h, "B": b, "P": p, "K": k, "iters_per_repeat": iters, "catalogue_build_ms": round(build_ms, 2),
               "ms": ms, "median_ms": med, "c_over_a": round(med["c_fp8_two_stage"] / med["a_bf16"], 4)}
        if full:
            out["median_ms"]["part_rescore_only"] = round(med["part_rescore_and_select"] - med["part_select"], 4)
            qs = q[:256]
            cat32 = cat.float()
            _, exact = trg.score_topk(qs.float(), cat32, k)
            del cat32
            torch.cuda.empty_cache()
            out["recall_at_k"] = {"a_bf16": recall(trg.score_topk(qs, cat, k)[1], exact),
                                  "fp8_stage_top_k": recall(fp8._fp8_candidates(qs, cat8, k)[1], exact),
                                  "c_fp8_two_stage": recall(trg.score_topk(qs, cat8, k)[1], exact),
                                  "exact_in_fp8_128_candidates": recall(fp8._fp8_candidates(qs, cat8)[1], exact)}
        print(json.dumps(out), flush=True)
        results.append(out)
    del q, cat, cat8
    torch.cuda.empty_cache()
    return results


def parent_ab(path, iters, repeats, seed):
    """bf16 trg_score_topk of this library and of ``path`` on the same config-5 inputs."""
    dev = torch.device("cuda")
    b, p, h = 4096, 50_000_000, 128
    other = ctypes.CDLL(path)
    for name in ("trg_score_topk", "trg_score_topk_workspace_bytes"):
        fn = getattr(other, name)
        fn.restype, fn.argtypes = _lib.SIGNATURES[name]
    q, cat = synth.synth_queries(b, p, h, seed=seed, device=dev, dtype=torch.bfloat16)
    for k in (100, 10):
        ws = torch.empty(int(other.trg_score_topk_workspace_bytes(b, p, h, k)), dtype=torch.uint8, device=dev)
        pv = torch.empty(b, k, device=dev)
        pi = torch.empty(b, k, dtype=torch.int64, device=dev)

        def parent():
            _lib.check(other.trg_score_topk(q.data_ptr(), cat.data_ptr(), b, p, h, _lib.TRG_BF16, k, 0,
                                            pv.data_ptr(), pi.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream()),
                       "parent trg_score_topk")
        parent()
        nv, ni = trg.score_topk(q, cat, k)
        torch.cuda.synchronize()
        same = bool(torch.equal(nv, pv) and torch.equal(ni, pi))
        ms, med = alternate({"parent": parent, "new": lambda: trg.score_topk(q, cat, k)}, iters, repeats)
        print(json.dumps({"ab": "parent_vs_new_bf16", "K": k, "identical_outputs": same, "ms": ms, "median": med}),
              flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--parent-lib", default=None, help="a second libtrg_b200.so to A/B the bf16 path against")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_topk_fp8: no CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    if args.parent_lib:
        parent_ab(args.parent_lib, args.iters, max(args.repeats, 7), 4)
    run(128, (100, 10), True, args.iters, args.repeats, 4)
    run(256, (100, 10), False, args.iters, args.repeats, 5)


if __name__ == "__main__":
    main()
