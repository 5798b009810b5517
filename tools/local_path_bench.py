"""The Local Path filter on the benchmark's graph, in one process.

1. The full filter job (triangle table, enumerate + score, top-k at the benchmark's k) of `local_path` against the
   `simple` (CN) job, each with mirror mode off and on, run alternately: median ms per step and mean phase times
   (`triangles`, `enum_score`, `topk`, `mirror`).
2. One full slab (the first owner slab of the full stream): the fused LP call against the count-only CN fused call and
   against K3 grouped CN (`ops.cn_aa(grouped_by_v=True)`) on the same slab's pairs, which streams the same N(u) lists
   as the LP walk 3.  Rates in G list elements/s under the pull-work model below, computed from the graph here.
3. The card's name, power limit and SM clocks, read before and after.

Pull-work model (list elements read): the CN fused call walks the owners' 2-paths twice (mark + score); LP walks them
twice and streams N(u) of every candidate u once (walk 3); K3 grouped streams N(u) of every pair and N(v) once per
owner run.

    python tools/local_path_bench.py [--workload ppa] [--steps 2] [--warmup 1] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--workload", default="ppa", choices=["ppa", "collab", "ddi", "small", "tiny"])
    p.add_argument("--steps", type=int, default=2, help="timed steps per job and mirror mode (alternating)")
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--slab-reps", type=int, default=3, help="timed repetitions of each call on the slab")
    p.add_argument("--slab-pairs", type=int, default=1 << 27)
    p.add_argument("--out", default=None, help="also write the JSON result here")
    a = p.parse_args()

    import torch
    import bench
    from mirror_ab import card_info
    from edge_proposal_sets_b200 import _lib, candidates, filter_step, models, ops

    if not torch.cuda.is_available():
        raise SystemExit("local_path_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    bargs = argparse.Namespace(scale=1.0, mlp=None, slab_pairs=a.slab_pairs, no_pushdown=False, owners_frac=1.0)
    card_before = card_info()
    wl = bench.Workload(a.workload, bargs, dev, 1)
    adj, x = wl.upload()
    torch.cuda.synchronize()
    deg = adj.degree().long()
    report = {"workload": a.workload, "k": wl.k, "n": wl.n, "nnz": adj.nnz, "steps": a.steps, "warmup": a.warmup,
              "card_before": card_before,
              "work_model": {"two_paths": int(candidates.two_path_work(adj).sum()),
                             "lp_pull_full": int(candidates.local_path_work(adj).sum()),
                             "lp_pull_half": int(candidates.local_path_work(adj, True).sum()),
                             "triangle_table_k3": int((deg * deg).sum())}}

    # ---- 1. full filter jobs ----
    names = ("simple", "local_path")
    model = {nm: models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=nm) for nm in names}

    def job(nm, mirror, stats=None):
        return filter_step.filter_topk(nm, model[nm], x, adj, k=wl.k, slab_pairs=a.slab_pairs, stats=stats,
                                       mirror=mirror)

    runs = {(nm, m): dict(ms=[], phases=[], stats=None) for nm in names for m in (False, True)}
    for _ in range(a.warmup):
        for key in runs:
            job(*key)
    outs = {}
    for _ in range(a.steps):
        for key, r in runs.items():
            adj._cache.pop("arc_tri", None)                  # the triangle table is part of every LP step
            st = {"time_phases": True}
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[key] = job(*key, stats=st)
            e1.record()
            torch.cuda.synchronize()
            r["ms"].append(e0.elapsed_time(e1))
            r["phases"].append(st["phase_ms"])
            r["stats"] = st
    jobs = {}
    for (nm, m), r in runs.items():
        ph = {key: statistics.fmean(q.get(key, 0.0) for q in r["phases"]) for key in r["phases"][-1]}
        jobs.setdefault(nm, {})["mirror" if m else "full"] = {
            "ms_per_step_median": statistics.median(r["ms"]), "ms_per_step": r["ms"], "phase_ms_mean": ph,
            "mirror": r["stats"]["mirror"], "pairs_evaluated": int(r["stats"]["pairs_evaluated"]),
            "slabs": r["stats"]["slabs"]}
    for nm in names:
        jobs[nm]["lists_equal_mirror_vs_full"] = bool(torch.equal(outs[(nm, False)], outs[(nm, True)]))
    report["jobs"] = jobs
    del outs

    # ---- 2. one full slab ----
    lo, hi, cap = next(filter_step.iter_slabs(adj, 0, adj.n, a.slab_pairs))
    paths = int(candidates.two_path_work(adj)[lo:hi].sum().item())

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.slab_reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts), out

    candidates.arc_triangles(adj)
    t_cn, (e_cn, _, c_cn) = timed(lambda: candidates.two_hop_scored(adj, None, lo, hi, cap=cap, want_count=True))
    N = int(e_cn.shape[1])
    pull = int(deg[e_cn[0].long()].sum().item())
    runs_v = int(torch.unique_consecutive(e_cn[1]).numel())
    pull_v = int(deg[torch.unique_consecutive(e_cn[1]).long()].sum().item())
    t_k3, c_k3 = timed(lambda: ops.cn_aa(adj, e_cn, None, use_values=False, grouped_by_v=True, want_count=True)[1])
    k3_equal = bool(torch.equal(c_k3, c_cn))
    del c_k3
    t_lp, (e_lp, s_lp, c2_lp, c3_lp) = timed(lambda: candidates.two_hop_local_path(adj, lo, hi, cap=cap))
    slab = {"owners": [lo, hi], "cap": int(cap), "candidates": N, "two_paths": paths, "walk3_list_elements": pull,
            "owner_runs": runs_v,
            "cn_fused_count_only": {"ms": t_cn, "G_list_elements_per_s": 2 * paths / t_cn / 1e6},
            "k3_grouped_cn": {"ms": t_k3, "G_list_elements_per_s": (pull + pull_v) / t_k3 / 1e6,
                              "counts_equal_fused": k3_equal},
            "local_path_fused": {"ms": t_lp, "G_list_elements_per_s": (2 * paths + pull) / t_lp / 1e6,
                                 "candidates_equal_cn": bool(torch.equal(e_lp, e_cn)),
                                 "c2_equal_cn": bool(torch.equal(c2_lp, c_cn))},
            "target_ms": t_cn + t_k3, "lp_vs_target": t_lp / (t_cn + t_k3)}
    report["slab"] = slab
    report["card_after"] = card_info()
    line = json.dumps(report)
    bench.emit(report)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
