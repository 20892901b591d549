"""Cost of per-user exclusions in K5: python tools/bench_topk_exclude.py [--repeats N] [--skip-config5]

Four arms, alternated inside one process (repeat r runs a, b, c, d, then r + 1 ...):
  a  no exclusions (``score_topk`` as shipped)
  b  40 random history posts per user
  c  each user's unfiltered top-K plus 40 random posts: every post that would have been returned is
     excluded, the worst case for hand-offs to the selection warps
  d  an index whose rows are all empty: the fixed cost of the kernels with the exclusion test compiled in
at config 5 (4096 users x 50M posts, H = 128, K = 100, bf16 tcgen05; the 12.8 GB catalogue does not fit
the L2) and at the reference's scale (4096 x 20k, H = 64, K = 10, fp32 FMA; the catalogue is L2-resident).
Prints the GPU and its power limit, then one JSON line per scale with every repeat's ms per call."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import truth_recommendation_gnn_b200 as trg  # noqa: E402
from truth_recommendation_gnn_b200 import synth  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"
    except (OSError, subprocess.SubprocessError):
        smi = "nvidia-smi unavailable"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


def history(top, n_rand, n_posts, gen):
    """ExclusionIndex whose row u holds top[u] plus n_rand random posts; also returns the [B, *] ids."""
    rnd = torch.randint(0, n_posts, (top.size(0), n_rand), generator=gen, device=top.device)
    hist = torch.cat([top, rnd], 1)
    row = torch.arange(hist.size(0), device=top.device)[:, None].expand_as(hist).reshape(-1)
    return trg.ExclusionIndex.from_edges(torch.stack([row, hist.reshape(-1)]), hist.size(0), n_posts), hist


def time_calls(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run_scale(name, b, p, h, k, dtype, iters, repeats, seed):
    dev = torch.device("cuda")
    q, cat = synth.synth_queries(b, p, h, seed=seed, device=dev, dtype=dtype)
    gen = torch.Generator(device=dev).manual_seed(seed + 1)
    _, top = trg.score_topk(q, cat, k)
    idx_b, hist_b = history(top[:, :0], 40, p, gen)
    idx_c, hist_c = history(top, 40, p, gen)
    idx_d, _ = history(top[:, :0], 0, p, gen)
    arms = {
        "a_none": lambda: trg.score_topk(q, cat, k),
        "b_40_random": lambda: trg.score_topk(q, cat, k, exclude=idx_b),
        "c_topk_plus_40": lambda: trg.score_topk(q, cat, k, exclude=idx_c),
        "d_empty_index": lambda: trg.score_topk(q, cat, k, exclude=idx_d),
    }
    # sanity: nothing excluded comes back
    for hist, arm in ((hist_b, "b_40_random"), (hist_c, "c_topk_plus_40")):
        _, ids = arms[arm]()
        assert not (ids[:, :, None] == hist[:, None, :]).any(), arm
    for fn in arms.values():      # warm every shape
        fn()
    torch.cuda.synchronize()
    ms = {a: [] for a in arms}
    for _ in range(repeats):
        for a, fn in arms.items():
            ms[a].append(round(time_calls(fn, iters), 4))
    med = {a: statistics.median(v) for a, v in ms.items()}
    out = {"scale": name, "B": b, "P": p, "H": h, "K": k, "dtype": str(dtype).replace("torch.", ""),
           "iters_per_repeat": iters, "ms": ms, "median_ms": med,
           "vs_a": {a: round(med[a] / med["a_none"] - 1, 4) for a in arms}}
    print(json.dumps(out), flush=True)
    del q, cat
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--skip-config5", action="store_true", help="only the reference-scale fp32 arms")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_topk_exclude: no CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    if not args.skip_config5:
        run_scale("config5", 4096, 50_000_000, 128, 100, torch.bfloat16, 3, args.repeats, 4)
    run_scale("reference", 4096, 20_000, 64, 10, torch.float32, 50, args.repeats, 5)


if __name__ == "__main__":
    main()
