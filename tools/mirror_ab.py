"""A/B of mirror mode on the benchmark's workload, in one process: the filter step that bench.py times (Adamic-Adar on
the fused K6+K3 kernel + GCN+LinkPredictor on the tensor-core prefilter, same graph, weights and k), run alternately
with ``mirror=False`` (every directed candidate) and ``mirror=True`` (every unordered pair once, list rebuilt).

Reports per arm the median ms per step and the mean phase times, the pairs each arm evaluated, each kernel's achieved
rate against the pairs it actually evaluated (bench.py's roofline entries divide by ``candidates_scored``, the
directed count, so on the mirror path they read about 2x too high), whether both lists of both models are equal
(``torch.equal``), and the card's name, power limit and SM clocks, read in the same run.

    python tools/mirror_ab.py [--workload ppa] [--steps 3] [--warmup 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return dict(zip(q.split(","), [c.strip() for c in r.stdout.strip().split(",")]))
    except Exception as exc:                   # the numbers stay usable without it
        return {"error": repr(exc)}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--workload", default="ppa", choices=["ppa", "collab", "ddi", "small", "tiny"])
    p.add_argument("--steps", type=int, default=3, help="timed steps per arm (alternating)")
    p.add_argument("--warmup", type=int, default=2, help="warm-up steps per arm")
    p.add_argument("--slab-pairs", type=int, default=1 << 27)
    p.add_argument("--out", default=None, help="also write the JSON result here")
    a = p.parse_args()

    import torch
    import bench                                   # the benchmark's workload builder (its stdout goes to stderr)
    from edge_proposal_sets_b200 import _lib, candidates, filter_step

    if not torch.cuda.is_available():
        raise SystemExit("mirror_ab.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    torch.backends.cuda.matmul.allow_tf32 = False
    bargs = argparse.Namespace(scale=1.0, mlp=None, slab_pairs=a.slab_pairs, no_pushdown=False, owners_frac=1.0)
    card_before = card_info()
    wl = bench.Workload(a.workload, bargs, dev, 1)
    adj, x = wl.upload()
    torch.cuda.synchronize()

    def step(mirror, stats=None):
        adj._cache.clear()                         # as bench.py: nothing derived from the graph is reused
        wl.model._h_key = None
        jobs = [filter_step.FilterJob("adamic_ogb", None), filter_step.FilterJob("gcn", wl.model, precision=wl.mlp_arm)]
        return filter_step.filter_topk_multi(jobs, x, adj, k=wl.k, slab_pairs=a.slab_pairs, stats=stats, mirror=mirror)

    arms = {False: dict(ms=[], phases=[], stats=None, outs=None), True: dict(ms=[], phases=[], stats=None, outs=None)}
    for _ in range(a.warmup):
        for m in (False, True):
            step(m)
    for _ in range(a.steps):
        for m in (False, True):
            st = {"time_phases": True}
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs = step(m, st)
            e1.record()
            torch.cuda.synchronize()
            arms[m]["ms"].append(e0.elapsed_time(e1))
            arms[m]["phases"].append(st["phase_ms"])
            arms[m]["stats"], arms[m]["outs"] = st, outs
    card_after = card_info()

    # algorithmic work per step, against the pairs each arm evaluated
    H, L = wl.H, wl.L
    paths_full = int(candidates.two_path_work(adj).sum().item())
    paths_half = int(candidates.half_two_path_work(adj).sum().item())
    report = {"workload": a.workload, "k": wl.k, "n": wl.n, "nnz": adj.nnz, "steps": a.steps, "warmup": a.warmup,
              "card_before": card_before, "card_after": card_after, "arms": {}}
    for m, r in arms.items():
        name = "mirror" if m else "full"
        st = r["stats"]
        P = int(st["pairs_evaluated"])
        ph = {key: statistics.fmean(p.get(key, 0.0) for p in r["phases"]) for key in r["phases"][-1]}
        rates = {}
        if ph.get("mlp"):
            rates["K2 mlp TFLOP/s"] = P * (2 * H * H * (L - 1) + 3 * H) / (ph["mlp"] * 1e-3) / 1e12
        if ph.get("enum_score"):
            rates["K6+K3 enum_score GB/s (8 B per 2-path walked + 44 B per pair)"] = \
                (8 * (paths_half if m else paths_full) + 44 * P) / (ph["enum_score"] * 1e-3) / 1e9
        if ph.get("topk"):
            rates["K4b+K4 topk GB/s (4 B per score read, 2 models)"] = 2 * 4 * P / (ph["topk"] * 1e-3) / 1e9
        report["arms"][name] = {"mirror": st["mirror"], "ms_per_step_median": statistics.median(r["ms"]),
                                "ms_per_step": r["ms"], "phase_ms_mean": ph, "pairs_evaluated": P,
                                "candidates_scored": int(st["candidates_scored"]), "rates": rates,
                                "prefilter": st.get("prefilter"), "prefilter_fallback": st.get("prefilter_fallback")}
    f, h = report["arms"]["full"], report["arms"]["mirror"]
    report["lists_equal"] = {nm: bool(torch.equal(p_, q_)) for nm, p_, q_ in
                             zip(("adamic_ogb", "gcn"), arms[False]["outs"], arms[True]["outs"])}
    report["ratio_ms_per_step"] = h["ms_per_step_median"] / f["ms_per_step_median"]
    report["ratio_phase"] = {key: h["phase_ms_mean"].get(key, 0.0) / v for key, v in f["phase_ms_mean"].items() if v > 0}
    line = json.dumps(report)
    bench.emit(report)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
