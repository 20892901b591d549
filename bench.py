#!/usr/bin/env python
"""Benchmark of the hetero-SAGE hot path (BASELINE.json metric: message-passing edges/s over one
train step, and top-k recs/s, at 1/2/4/8 B200 next to the CPU path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2] [--dump-outputs DIR]

A "step" is the body of the reference's ``train()`` (train_gnn.py:242-285): zero_grad -> forward
-> pos/neg scoring + loss -> backward -> Adam step, full batch.  ``value`` = L * (2*E_eng + E_soc)
/ t_step with everything resident in HBM; ``e2e`` = the same through the public API with this
step's host inputs (the sampled negatives, pinned host memory) copied in and the loss read back
inside the timed region.  Rank 0 prints ONE JSON line.  Besides the headline (BASELINE config 2, strong
scaling over N GPUs) the line carries, as sub-objects, the other configurations BASELINE.json names:

  topk    config 5: 4096 queries x 50M posts, top-100, bf16 -- catalogue sharded over the N GPUs
  cfg3    config 3: the config-2 graph in bf16 (N = 1: one GPU; N > 1: destination-partitioned)
  cfg4    config 4: 10M users / 50M posts / 1B edges, H = 256 bf16, L = 3 -- N = 8 only (generated per shard)
  cfg1    config 1: the reference's own scale, full size, L = 1 literal and L = 2 (N = 1)
  verify  N > 1: parity of the sharded path against the single-GPU path inside this very job

``--impl reference`` times the CPU oracle (the restated reference path; torch_geometric is not installable)
on the host cores: a bounded sample of the headline workload per step (so that K steps end within minutes),
config 1 at full size (like for like with ``cfg1`` above), and the reference's CPU scoring
(inference.py:427-428, batched and the per-user loop).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "message-passing edges/s (train step)"
UNIT = "edges/s"

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (fits one GPU)
    "cfg2": dict(num_users=1_000_000, num_posts=5_000_000, e_eng=40_000_000, e_soc=10_000_000,
                 hidden=128, layers=2, dtype="f32"),
    # configs[2]: same graph in bf16 (multi-GPU scaling config)
    "cfg3": dict(num_users=1_000_000, num_posts=5_000_000, e_eng=40_000_000, e_soc=10_000_000,
                 hidden=128, layers=2, dtype="bf16"),
    # configs[3]: 8 x B200 only; generated per shard on the device (synth.CounterGraph)
    "cfg4": dict(num_users=10_000_000, num_posts=50_000_000, e_eng=800_000_000, e_soc=200_000_000,
                 hidden=256, layers=3, dtype="bf16", counter=True, eager=True, comm="peer-direct"),
    # (config 4 runs the eager step with direct peer loads: the configuration it was validated in at 8 GPUs; its
    # graph-captured / copy-engine-staged form did not finish within the leg's time limit when first tried and
    # there was no 8-GPU time left to find out why)
    # load-balance report (SURVEY §8d): config 2 with Zipf-like destinations, dst = floor(N * u^3)
    "cfg2skew": dict(num_users=1_000_000, num_posts=5_000_000, e_eng=40_000_000, e_soc=10_000_000,
                     hidden=128, layers=2, dtype="f32", skew=True),
    # configs[0]: the reference's own CPU-runnable scale
    "cfg1": dict(num_users=10_000, num_posts=50_000, e_eng=400_000, e_soc=100_000,
                 hidden=64, layers=2, dtype="f32"),
    # 1/8 of config 4 per GPU count 1 (development / 2-GPU checks of the config-4 code path)
    "cfg4mini": dict(num_users=1_250_000, num_posts=6_250_000, e_eng=100_000_000, e_soc=25_000_000,
                     hidden=256, layers=3, dtype="bf16", counter=True, eager=True, comm="peer-direct"),
    "tiny": dict(num_users=2_000, num_posts=8_000, e_eng=60_000, e_soc=15_000,
                 hidden=64, layers=2, dtype="f32"),
}
TOPK = dict(batch=4096, n_post=50_000_000, hidden=128, k=100)      # BASELINE.json configs[4]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


def step_bytes(w, elem):
    """Algorithmic HBM bytes of one train step (SURVEY.md §8d table)."""
    U, P, Ee, Es, H, L = w["num_users"], w["num_posts"], w["e_eng"], w["e_soc"], w["hidden"], w["layers"]
    F, s = H, elem
    rels = [(Ee, P, U), (Es, U, U), (Ee, U, P)]          # (E, N_src, N_dst)
    A = sum(e * (F * s + 4) + 4 * (nd + 1) + nd * F * s for e, ns, nd in rels)
    B = U * (3 * F * s + H * s) + P * (2 * F * s + H * s)
    C = Ee * (3 * H * s + 12)
    D = Ee * (3 * H * s + 12) + (U + P) * H * s
    G = sum(e * (F * s + 4) + 4 * (ns + 1) + ns * F * s + 4 * nd for e, ns, nd in rels)
    return L * (A + B + B) + C + D + (L - 1) * (B + G)


def config_of(name, w):
    """The ``config`` object: identical in the repo arm and the reference arm."""
    return {"workload": f"{name}: {w['num_users']} users / {w['num_posts']} posts / {w['e_eng'] + w['e_soc']} edges, "
                        f"{w['layers']}-layer hetero SAGE hidden={w['hidden']} {w['dtype']}, one full-batch "
                        f"link-pred train step (fwd+loss+bwd+Adam)",
            "mp_edges_per_step": w["layers"] * (2 * w["e_eng"] + w["e_soc"]),
            "l2": "inputs exceed L2 (tables >= 0.5 GB, L2 = 126 MB)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons, pw = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(sm, key=lambda x: x)[len(sm) // 2:] if len(sm) > 3 else sm
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None,
                "sm_mhz_busy_median": statistics.median(busy)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (restated reference path; PyG itself is not installable) on host cores
# ------------------------------------------------------------------------------------------------
def cpu_sample_workload(w):
    """Bounded sample of the workload: same H / L / edge mix / degrees, the graph scaled 1/20 so that one
    oracle step is a few seconds of CPU work (its tables, 150 MB, still exceed the host's caches)."""
    scale = 20 if w["num_users"] >= 1_000_000 else 1
    s = dict(w)
    for k in ("num_users", "num_posts", "e_eng", "e_soc"):
        s[k] = max(w[k] // scale, 1)
    desc = (f"{'1/%d-scale ' % scale if scale > 1 else 'full-size '}graph {s['num_users']} users / {s['num_posts']} posts / "
            f"{s['e_eng'] + s['e_soc']} edges, H={s['hidden']}, L={s['layers']}, fp32, full train step "
            f"(CPU oracle: pure-torch restatement of PyG SAGEConv; torch_geometric is not installable)")
    return s, desc


def step_outputs(loss, model):
    """What one train step hands its caller: the loss, and the model's parameters and gradients as the step
    left them (host float32 / float64 arrays, keyed by the file name ``--dump-outputs`` writes them under)."""
    import numpy as np
    out = {"loss": np.asarray(float(loss), dtype=np.float64)}
    for n, p in model.named_parameters():
        out[f"param.{n}"] = p.detach().float().cpu().numpy()
        if p.grad is not None:
            out[f"grad.{n}"] = p.grad.detach().float().cpu().numpy()
    return out


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, outputs):
    import numpy as np
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_cpu_oracle(w, steps, warmup, sample=True, outputs=None):
    from oracle import sage as osage   # bench.py executes oracle/ only here: the CPU baseline
    from truth_recommendation_gnn_b200 import synth
    s, desc = cpu_sample_workload(w) if sample else (dict(w), "full size")
    g = synth.synth_graph(s["num_users"], s["num_posts"], s["e_eng"], s["e_soc"], s["hidden"], seed=0,
                          skew=w.get("skew", False))
    H, L = s["hidden"], s["layers"]
    model = (osage.WeightedRGCNOracle(H, (H, H)) if L == 1 else osage.StackedWeightedRGCNOracle(H, L, (H, H)))
    model.load_state_dict(synth.init_state_dict(H, H, L))
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    times = []
    for i in range(warmup + steps):
        neg = synth.synth_neg(s["num_posts"], s["e_eng"], i)
        t0 = time.perf_counter()
        loss = osage.train_step(model, opt, g.x_dict, g.edge_index_dict, g.train_edge_index,
                                g.interaction_type_tensor, s["num_users"], s["num_posts"], neg_p=neg)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    if outputs is not None:
        outputs.update(step_outputs(loss, model))
    t = sum(times) / len(times)
    mp = L * (2 * s["e_eng"] + s["e_soc"])
    return dict(value=mp / t, unit=UNIT, cores=torch.get_num_threads(), kind="port", sample=desc,
                ms_per_step=t * 1e3, host_cpus=os.cpu_count())


def cpu_cfg1():
    """BASELINE config 1 at full size on the host cores: the literal L = 1 model and the L = 2 stack."""
    w = WORKLOADS["cfg1"]
    out = {}
    for L in (1, 2):
        r = run_cpu_oracle(dict(w, layers=L), 3, 1, sample=False)
        out[f"L{L}"] = {"edges_per_s": r["value"], "ms_per_step": r["ms_per_step"]}
    out["cores"] = torch.get_num_threads()
    return out


def cpu_topk_baseline(seconds=8.0):
    """The reference's CPU scoring (inference.py:427-428: torch.mm + torch.topk) on the host cores, fp32, on a
    bounded slice of config 5: (a) batched -- 4096 users x a 100k-post slice of the catalogue, top-100;
    (b) the per-user loop the script actually runs -- one [1,H] x [H,P_slice] mm + topk per user.  recs/s are
    scaled to the 50M-post catalogue by posts scored per second (both are linear in the catalogue size)."""
    from truth_recommendation_gnn_b200 import synth
    B, H, K, P = TOPK["batch"], TOPK["hidden"], TOPK["k"], TOPK["n_post"]
    p_slice = 100_000
    q, cat = synth.synth_queries(B, p_slice, H)
    out = {"cores": torch.get_num_threads(), "unit": "recs/s",
           "sample": f"{B} users x {p_slice} posts (1/{P // p_slice} of the config-5 catalogue), H={H}, K={K}, fp32; "
                     f"recs/s scaled to {P} posts by posts scored per second"}
    for name, fn, nq in (("batched", lambda: torch.topk(torch.mm(q, cat.T), K), B),
                         ("per_user_loop", lambda: [torch.topk(torch.mm(q[i:i + 1], cat.T).squeeze(0), K) for i in range(256)], 256)):
        fn()
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds / 2:
            fn()
            n += 1
        dt = (time.perf_counter() - t0) / n
        posts_per_s = nq * p_slice / dt
        out[name] = {"posts_scored_per_s": posts_per_s, "recs_per_s": posts_per_s / P * K,
                     "ms_per_call": dt * 1e3, "users_per_call": nq}
    return out


def run_reference_arm(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    outputs = {} if args.dump_outputs else None
    cb = run_cpu_oracle(w, args.steps, max(args.warmup, 1), outputs=outputs)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, w),
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "each step is a bounded sample of the configured workload (cpu_baseline.sample); cfg1 below is "
                "config 1 at FULL size, like for like with the repo arm's cfg1 object",
    }
    if not args.no_extras:
        line["cfg1"] = cpu_cfg1()
        line["topk"] = cpu_topk_baseline()
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _barrier(world):
    if world > 1:
        torch.distributed.barrier()


def gpu_train_bench(args, w, rank, world, dev, steps, warmup, e2e=True, outputs=None):
    import truth_recommendation_gnn_b200 as trg
    from truth_recommendation_gnn_b200 import _lib, synth
    from truth_recommendation_gnn_b200 import dist as tdist
    from truth_recommendation_gnn_b200 import dist_fused

    dtype = torch.float32 if w["dtype"] == "f32" else torch.bfloat16
    U, P, Ee, Es, H, L = w["num_users"], w["num_posts"], w["e_eng"], w["e_soc"], w["hidden"], w["layers"]
    t_setup0 = time.perf_counter()
    model = trg.WeightedRGCN(H) if L == 1 else trg.StackedWeightedRGCN(H, L)
    model.load_state_dict(synth.init_state_dict(H, H, L))
    model = model.to(dev).to(dtype)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    n_host = 2 if Ee > 100_000_000 else 4
    shard = g = None
    if w.get("counter"):
        cg = synth.CounterGraph(U, P, Ee, Es, H, seed=0)
        if world > 1:
            shard = tdist.ShardedGraph.from_generator(cg, dev, dtype)      # the full graph never exists anywhere
        else:
            g = cg.materialize(dev, dtype)
    else:
        g = synth.synth_graph(U, P, Ee, Es, H, seed=0, device=dev, dtype=dtype, skew=w.get("skew", False))   # same graph on every rank
        if world > 1:
            # destination partition: this rank keeps its rows / edges and drops the full graph
            shard = tdist.ShardedGraph(g.x_dict, g.edge_index_dict, g.train_edge_index,
                                       g.interaction_type_tensor, U, P)
            g = None
    if shard is not None and w.get("comm"):
        shard.comm_mode = w["comm"]
    torch.cuda.empty_cache()
    # this step's input: the sampled negatives (train_gnn.py:272), the SAME full array on every rank; each rank
    # selects its share inside the step (device-side, no host sync)
    neg_dev = [synth.synth_neg(P, Ee, i, device=dev) for i in range(n_host)]
    neg_host = [t.cpu().pin_memory() for t in neg_dev] if e2e else None
    torch.cuda.synchronize()

    # N > 1: the step is replayed from a CUDA graph captured on its first call (the eager step is host-bound at
    # 8 GPUs); TRG_DIST_GRAPH=0 keeps it eager (A/B)
    graphed = (world > 1 and os.environ.get("TRG_DIST_GRAPH", "1") != "0" and os.environ.get("TRG_DIST_TAPE") != "1"
               and not w.get("eager"))
    graphed1 = world == 1 and bool(w.get("cuda_graph"))       # single GPU: config 1 (launch-bound) only

    def step(i, host, eager=False):
        # host: the pinned HOST tensor goes straight into the public API, which copies it in (on a side
        # stream, overlapped with the forward pass: the negatives are first needed by the loss)
        neg = neg_host[i % n_host] if host else neg_dev[i % n_host]
        if world > 1:
            if os.environ.get("TRG_DIST_TAPE") == "1":      # A/B: autograd Functions + blocking collectives
                return tdist.train_step_sharded(model, opt, shard, neg_p_global=neg.to(dev, non_blocking=True),
                                                return_tensor=not host)
            return dist_fused.train_step_sharded_fused(model, opt, shard, neg_p_global=neg, return_tensor=not host,
                                                       cuda_graph=graphed and not eager)
        return trg.train_step(model, opt, g.x_dict, g.edge_index_dict, g.train_edge_index,
                              g.interaction_type_tensor, U, P, neg_p=neg, return_tensor=not host,
                              cuda_graph=graphed1 and not eager)

    for i in range(warmup):
        step(i, False)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup0

    # ---- timed region 1: resident inputs (value) ----
    clocks = ClockSampler(dev.index or 0)
    _lib.PROF.reset()
    _lib.PROF.enabled = not (graphed or graphed1)   # per-kernel CUDA events: inside the timed region when it is eager
    _barrier(world); torch.cuda.synchronize()
    n0 = _lib.launch_count()
    clocks.start()
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host0 = time.perf_counter()
        loss = None
        for i in range(steps):
            loss = step(i, False)
        host_ms = (time.perf_counter() - t_host0) * 1e3 / steps     # CPU time to ENQUEUE one step
        e1.record()
        torch.cuda.synchronize(); _barrier(world)
    finally:
        clk = clocks.stop()       # also on failure: the sampler must not outlive the job
    loss = float(loss)        # now: a graphed step returns its static loss tensor, which later replays overwrite
    n1 = _lib.launch_count()
    _lib.PROF.enabled = False
    ms = e0.elapsed_time(e1) / steps
    prof = _lib.PROF.summary()
    if outputs is not None:       # before the e2e leg, whose steps train the model further
        outputs.update(step_outputs(loss, model))

    # ---- timed region 2: end to end through the public API with host buffers ----
    ms_e2e = None
    if e2e:
        for i in range(2):
            step(i, True)
        _barrier(world); torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            step(i, True)
        e1.record()
        torch.cuda.synchronize(); _barrier(world)
        ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / steps

    launches = n1 - n0
    if graphed or graphed1:
        # the timed region replayed a graph: its kernels are counted from the capture, and the per-kernel
        # breakdown comes from an EAGER pass of the same steps (same kernels, launched one by one)
        launches = steps * (shard._graphed if graphed else model._trg_graphed_step).launches_per_replay
        _lib.PROF.reset()
        _lib.PROF.enabled = True
        for i in range(steps):
            step(i, False, eager=True)
        torch.cuda.synchronize(); _barrier(world)
        _lib.PROF.enabled = False
        prof = _lib.PROF.summary()
    h2d = int(neg_dev[0].numel()) * 8
    if shard is not None and getattr(shard, "_neg_gather", None) is not None:
        h2d = shard._neg_gather.chunk * 8          # this rank uploads its 1/N slice; the rest arrives over NVLink
    if world > 1:
        t = torch.tensor([ms, ms_e2e or 0.0], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), (float(t[1]) if e2e else None)
        c = torch.tensor([launches, h2d], device=dev, dtype=torch.int64)
        torch.distributed.all_reduce(c)
        launches, h2d = int(c[0]), int(c[1])
    mp_edges = L * (2 * Ee + Es)
    mem_gb = torch.cuda.max_memory_allocated(dev) / 2**30
    loss = float(loss)
    if shard is not None and getattr(shard, "_graphed", None) is not None:
        shard._graphed.close()          # the graph holds captured NCCL work: drop it before the group goes away
        shard._graphed = None
    del model, opt, shard, g, neg_dev, neg_host
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return dict(ms=ms, ms_e2e=ms_e2e, mp_edges=mp_edges, prof=prof, launches=launches, clocks=clk, host_ms=host_ms,
                setup_s=setup_s, h2d=h2d, d2h=4 * world, mem_gb=mem_gb, loss=float(loss), graphed=graphed)


def sub_line(name, w, r, world, steps):
    """A secondary configuration's result in the shape of the headline (without the e2e leg)."""
    pk = peaks()
    elem = 4 if w["dtype"] == "f32" else 2
    sb = step_bytes(w, elem)
    return {"config": config_of(name, w), "n_gpus": world, "dtype": w["dtype"], "steps": steps,
            "ms_per_step": r["ms"], "value": r["mp_edges"] / r["ms"] * 1e3, "unit": UNIT,
            "step_roofline": {"algorithmic_bytes_per_step": sb, "per_gpu_achieved_gbs": sb / world / r["ms"] / 1e6,
                              "frac": sb / world / r["ms"] / 1e6 / pk["hbm_gbs"], "roofline_ms": sb / world / pk["hbm_gbs"] / 1e6},
            "kernels_ms_per_step": {k: round(v["ms"] / steps, 3) for k, v in sorted(r["prof"].items())},
            "kernels_gbs": {k: round(v["bytes"] / v["ms"] / 1e6, 1) for k, v in sorted(r["prof"].items()) if v["ms"] > 0},
            "peak_mem_gb": round(r["mem_gb"], 2), "setup_s": round(r["setup_s"], 2), "loss": r["loss"],
            "gpu_launches": r["launches"], "host_enqueue_ms_per_step": round(r["host_ms"], 3)}


def gpu_topk_bench(dev, rank, world, iters=3, outputs=None):
    """Secondary metric: top-k recs/s -- inference.py:427-428 batched, BASELINE config 5 (score all 50M posts per
    user batch of 4096, top-100; bf16 in, fp32 accumulate; tcgen05 + warp-level select).  N > 1: the catalogue is
    sharded by post-id range (each rank holds 50M / N rows), queries replicated, per-shard lists all-gathered and
    merged (``dist.recommend_sharded``); the timed call includes the gather and the merge."""
    import truth_recommendation_gnn_b200 as trg
    from truth_recommendation_gnn_b200 import dist as tdist
    from truth_recommendation_gnn_b200 import synth
    batch, n_post, hidden, k = TOPK["batch"], TOPK["n_post"], TOPK["hidden"], TOPK["k"]
    cp = (n_post + world - 1) // world
    p0, p1 = rank * cp, min((rank + 1) * cp, n_post)
    q, _ = synth.synth_queries(batch, 1, hidden, device=dev, dtype=torch.bfloat16)        # same queries on every rank
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    cat = torch.relu(torch.randn(p1 - p0, hidden, generator=g, device=dev)).to(torch.bfloat16)
    q_host = q.cpu().pin_memory()

    def call(qq):
        if world > 1:
            return tdist.recommend_sharded(qq, cat, k, p0)
        return trg.score_topk(qq, cat, k)

    call(q)
    torch.cuda.synchronize(); _barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        v, i = call(q)
    e1.record()
    torch.cuda.synchronize(); _barrier(world)
    ms = e0.elapsed_time(e1) / iters
    if outputs is not None:
        outputs["topk.values"] = v.float().cpu().numpy()
        outputs["topk.ids"] = i.cpu().double().numpy()      # post ids < 2^53: exact in float64
    # end to end: the query batch comes from pinned host memory, ids + scores go back to the host
    v, i = call(q_host.to(dev, non_blocking=True))     # untimed: first-use host staging buffers
    v, i = v.cpu(), i.cpu()
    _barrier(world)
    t0 = time.perf_counter()
    for _ in range(iters):
        v, i = call(q_host.to(dev, non_blocking=True))
        v, i = v.cpu(), i.cpu()
    ms_e2e = (time.perf_counter() - t0) * 1e3 / iters
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    pk = peaks()
    tf = 2.0 * batch * n_post * hidden / ms / 1e9
    del cat
    torch.cuda.empty_cache()
    return dict(metric="top-k recs/s", value=batch * k / ms * 1e3, unit="recs/s", n_gpus=world,
                users_per_s=batch / ms * 1e3, recs_per_s=batch * k / ms * 1e3, ms_per_batch=ms,
                e2e={"value": batch * k / ms_e2e * 1e3, "unit": "recs/s", "ms_per_batch": ms_e2e,
                     "h2d_bytes_per_step": batch * hidden * 2, "d2h_bytes_per_step": batch * k * 12},
                e2e_recs_per_s=batch * k / ms_e2e * 1e3, e2e_ms_per_batch=ms_e2e,
                roofline=dict(bound="tensor", achieved=tf, per_gpu_achieved=tf / world, peak=pk["bf16_tflops"],
                              unit="TFLOP/s", frac=tf / world / pk["bf16_tflops"], peak_source=pk["source"]),
                config={"workload": f"cfg5: {batch} queries x {n_post} posts, top-{k}, H={hidden}, bf16 in / fp32 accumulate"
                                    + (f", catalogue sharded over {world} GPUs by post-id range" if world > 1 else "")},
                batch=batch, n_post=n_post, hidden=hidden, k=k, dtype="bf16 in / fp32 accumulate",
                kernel="score_topk_tc3_kernel (tcgen05 kind::f16; scan warps read TMEM rows, helper warps keep the "
                       "per-item top-K lists in TMEM and merge them into the rows' global lists under a row lock)")


def gpu_cfg1(dev):
    """BASELINE config 1 at full size on one GPU (the reference's own scale: everything is L2-resident, so this
    is a latency / launch-bound regime, not a roofline one)."""
    out = {}
    a = argparse.Namespace()
    for L in (1, 2):
        for key, graph in ((f"L{L}", False), (f"L{L}_cuda_graph", True)):
            w = dict(WORKLOADS["cfg1"], layers=L, cuda_graph=graph)
            r = gpu_train_bench(a, w, 0, 1, dev, steps=20, warmup=5, e2e=True)
            out[key] = {"edges_per_s": r["mp_edges"] / r["ms"] * 1e3, "ms_per_step": r["ms"],
                        "e2e_edges_per_s": r["mp_edges"] / r["ms_e2e"] * 1e3, "e2e_ms_per_step": r["ms_e2e"],
                        "launches_per_step": r["launches"] / 20, "loss": r["loss"]}
    out["note"] = ("*_cuda_graph: train_step(..., cuda_graph=True) -- the step replayed from a CUDA graph (one launch "
                   "per step); the eager step at this size is bound by the Python launch path")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-topk", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip cfg1 / cfg3 / cfg4 / verify")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, parameters and gradients after the "
                         "step; the top-k leg's scores and ids) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    default_workload = args.workload is None
    if default_workload:
        args.workload = "cfg2"   # the same graph at every N: the driver's scaling ratio compares like with like
    w = WORKLOADS[args.workload]

    if args.impl == "reference":
        run_reference_arm(args, w)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=b200) needs a CUDA device: the hot path has no CPU fallback")
    args.warmup = max(args.warmup, 3)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)

    outputs = {} if args.dump_outputs and rank == 0 else None
    r = gpu_train_bench(args, w, rank, world, dev, args.steps, args.warmup, outputs=outputs)
    if rank == 0:
        print(f"[bench] headline {args.workload} x{world}: {r['ms']:.3f} ms/step, e2e {r['ms_e2e']:.3f}, "
              f"kernels {({k: round(v['ms'] / args.steps, 3) for k, v in sorted(r['prof'].items())})}",
              file=sys.stderr, flush=True)
    extras, errors = {}, {}
    import threading
    build_line = make_line_builder(args, w, r, world, dev, default_workload, extras, errors)

    def emergency(name, limit):
        # a secondary leg that HANGS (a rank died inside a collective, a capture that never ends) must not take
        # the headline with it either: every rank's watchdog fires at the same deadline, rank 0 prints the line
        # with what finished, everybody leaves with exit code 0
        errors[name] = f"no result within {limit:.0f} s: leg abandoned, job ended by the watchdog"
        if rank == 0:
            try:
                print(json.dumps(build_line()), flush=True)
            finally:
                os._exit(0)
        time.sleep(3.0)
        os._exit(0)

    def leg(name, fn, limit=150.0):
        # a secondary leg that fails must not take the headline line with it: the error is reported in its place
        wd = threading.Timer(limit, emergency, args=(name, limit))
        wd.daemon = True
        if world > 1:
            wd.start()
        try:
            extras[name] = fn()
            if rank == 0:           # progress on stderr: a later leg that kills the job does not erase this one
                v = extras[name]
                ms = v[1]["ms"] if isinstance(v, tuple) else (v.get("ms_per_batch") if isinstance(v, dict) else None)
                print(f"[bench] leg {name} done" + (f": {ms:.3f} ms" if ms else ""), file=sys.stderr, flush=True)
        except Exception as e:      # noqa: BLE001
            errors[name] = f"{type(e).__name__}: {e}"[:400]
            torch.cuda.empty_cache()
        finally:
            wd.cancel()

    if not args.no_extras and default_workload:
        sub_steps = min(args.steps, 10)
        if world > 1:
            from truth_recommendation_gnn_b200 import dist_check
            leg("verify", lambda: [dist_check.check_sharded_against_single(dev, dt) for dt in (torch.float32, torch.bfloat16)])
        w3 = WORKLOADS["cfg3"]
        leg("cfg3", lambda: (w3, gpu_train_bench(args, w3, rank, world, dev, sub_steps, 3, e2e=False), sub_steps))
        if world == 8:
            w4 = WORKLOADS["cfg4"]
            leg("cfg4", lambda: (w4, gpu_train_bench(args, w4, rank, world, dev, min(args.steps, 5), 3, e2e=False), min(args.steps, 5)),
                limit=300.0)
    if not args.no_topk:
        leg("topk", lambda: gpu_topk_bench(dev, rank, world, outputs=outputs))

    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(build_line(final=True)))
    if world > 1:
        # teardown must not be able to hang the job after the line is out
        sys.stdout.flush()
        t = threading.Timer(30.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
        t.cancel()


def make_line_builder(args, w, r, world, dev, default_workload, extras, errors):
    def build_line(final=False):
        topk = extras.get("topk")
        pk = peaks()
        elem = 4 if w["dtype"] == "f32" else 2
        value = r["mp_edges"] / r["ms"] * 1e3
        gat = [r["prof"].get(n) for n in ("trg_sage_agg_fwd", "trg_sage_agg_bwd", "trg_gather_wsum")]
        gat = [d for d in gat if d]
        g_bytes, g_ms, g_calls = (sum(d["bytes"] for d in gat), sum(d["ms"] for d in gat), sum(d["calls"] for d in gat))
        achieved = g_bytes / g_ms / 1e6 if g_ms > 0 else 0.0            # GB/s
        traffic = None
        tp = os.path.join(ROOT, "profiles", "gather_traffic.json")
        if world == 1 and os.path.exists(tp):     # one ncu --set full capture of this launch mix on ONE GPU
            traffic = json.load(open(tp)).get(args.workload)
        sb = step_bytes(w, elem)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": config_of(args.workload, w),
            "parallelism": "single GPU" if world == 1 else
                           f"dst-partitioned x{world}: all-gather of user rows per layer, push partial sums reduce-scattered "
                           f"(fp32 transport) by copy-engine pulls + a fused reduce/finish kernel over peer memory, collectives overlapped with kernels (dist_fused); each rank selects its share "
                           f"of the step's negatives inside the timed region"
                           + ("; the whole step is one CUDA-graph replay (kernels_* from an eager pass of the same steps)"
                              if r.get("graphed") else ""),
            "e2e": {"value": r["mp_edges"] / r["ms_e2e"] * 1e3, "unit": UNIT, "ms_per_step": r["ms_e2e"],
                    "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "what": "train_step() via the public API; per step the sampled negatives (int64[E_eng]) are "
                            "copied from pinned host memory (N = 1: the whole array; N > 1: every rank holds the array "
                            "on its host, uploads a 1/N slice and pulls the other slices from its peers over NVLink) "
                            "and loss.item() is read back; graph + "
                            "features stay resident as in the reference (graph.to(device) once, train_gnn.py:211)"},
            "gpu_launches": r["launches"],
            "clocks": r["clocks"],
            "roofline": {"bound": "hbm", "kernel": "gather_reduce (trg_sage_agg_fwd/bwd, trg_gather_wsum)",
                         "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk["source"],
                         "launches": g_calls, "avg_ms_per_launch": g_ms / max(g_calls, 1),
                         "algorithmic_bytes_per_launch": g_bytes / max(g_calls, 1),
                         "share_of_step": g_ms / (r["ms"] * args.steps)},
            "step_roofline": {"algorithmic_bytes_per_step": sb, "achieved_gbs": sb / r["ms"] / 1e6,
                              "per_gpu_achieved_gbs": sb / world / r["ms"] / 1e6,
                              "frac": sb / world / r["ms"] / 1e6 / pk["hbm_gbs"], "roofline_ms": sb / world / pk["hbm_gbs"] / 1e6},
            "kernels_ms_per_step": {k: round(v["ms"] / args.steps, 3) for k, v in sorted(r["prof"].items())},
            "kernels_gbs": {k: round(v["bytes"] / v["ms"] / 1e6, 1) for k, v in sorted(r["prof"].items()) if v["ms"] > 0},
            "setup_s": round(r["setup_s"], 2), "host_enqueue_ms_per_step": round(r["host_ms"], 3), "peak_mem_gb": round(r["mem_gb"], 2),
            "loss": r["loss"],
        }
        if "verify" in extras:
            line["verify"] = extras["verify"]
        for name in ("cfg3", "cfg4"):
            if name in extras:
                wk, rk, st = extras[name]
                line[name] = sub_line(name, wk, rk, world, st)
        if topk is not None:
            line["topk"] = topk
        if errors:
            line["leg_errors"] = errors
        if final and world == 1 and not args.no_extras and default_workload:
            line["cfg1"] = gpu_cfg1(dev)
        if final and not args.no_cpu_baseline and world == 1:
            torch.set_num_threads(os.cpu_count() or 1)
            cb = run_cpu_oracle(w, 2, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            if not args.no_extras and default_workload:
                line["cfg1"]["cpu"] = cpu_cfg1()
                if topk is not None:
                    line["topk"]["cpu_baseline"] = cpu_topk_baseline(6.0)
        return line

    return build_line


if __name__ == "__main__":
    main()
