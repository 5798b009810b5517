"""Distance-3 proposal sets (`filter_topk(..., hops=3)`) against the 2-hop ones, in one process.

1. twitch (the golden graph, a seeded GCN whose logits are spread to mean -2 / std 2) and collab-shape (the benchmark's
   workload and model): the whole-graph GCN job at hops=2 and hops=3, mirror mode on, default (prefilter) arm, run
   alternately: median ms per step, mean phase times, candidates, slabs, and the sum of the slot bounds over the real
   candidate count.  Each hops=3 list is checked against the fp32 arm's list (mirror off).
2. ppa-shape, one full hops=3 slab of owners (the first slab of the full stream): the enumeration call
   (`candidates.three_hop`) against the Local Path fused call on the same owners.  Rates in G list elements/s:
   enumeration = 2 x (2-paths) + sum over the owners' distinct 2-walk ends x of deg x (walk 1 is one pass over the
   2-paths; the freeze re-reads nothing from the graph; counted here by a torch pass over the 2-paths);
   Local Path = 2 x (2-paths) + sum over its candidates u of deg u (as tools/local_path_bench.py).
3. The card's name, power limit and SM clocks, read before and after, in the same process.

    python tools/threehop_bench.py [--steps 3] [--warmup 1] [--out FILE]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _twitch_job(dev):
    from edge_proposal_sets_b200 import candidates, models
    from oracle import gnn as ognn
    from util import golden_graph, spread_linkpred, to_adj
    g = golden_graph("twitch")[2]
    adj = to_adj(g, dev, keep_values=False)
    args = argparse.Namespace(model="gcn", dataset="twitch", num_layers=3, hidden_channels=256, dropout=0.0,
                              use_feature=False, use_learnable_embedding=True)

    class D:
        num_nodes = g.n
        x = None
    mg = models.build_model(args, D, dev)
    mg.load_state_dict(ognn.random_state_dict("gcn", g.n, 0, 256, 3, seed=7))
    mg.eval()
    e = candidates.two_hop(adj)
    spread_linkpred(mg, None, adj, e[:, ::max(e.shape[1] // 1_000_000, 1)].contiguous())
    return adj, None, mg, 100_000


def _jobs(adj, x, model, k, steps, warmup, slab_pairs):
    import torch
    from edge_proposal_sets_b200 import candidates, filter_step

    def run(hops, stats=None, **kw):
        return filter_step.filter_topk("gcn", model, x, adj, k=k, slab_pairs=slab_pairs, stats=stats, hops=hops, **kw)

    runs = {h: dict(ms=[], phases=[], stats=None) for h in (2, 3)}
    for _ in range(warmup):
        for h in runs:
            run(h)
    outs = {}
    for _ in range(steps):
        for h, r in runs.items():
            st = {"time_phases": True}
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[h] = run(h, st)
            e1.record()
            torch.cuda.synchronize()
            r["ms"].append(e0.elapsed_time(e1))
            r["phases"].append(st["phase_ms"])
            r["stats"] = st
    res = {}
    for h, r in runs.items():
        st = r["stats"]
        bound = int(candidates.owner_bounds(adj, st["mirror"], h).sum())
        res[f"hops{h}"] = {"ms_per_step_median": statistics.median(r["ms"]), "ms_per_step": r["ms"],
                           "phase_ms_mean": {key: statistics.fmean(q.get(key, 0.0) for q in r["phases"])
                                             for key in r["phases"][-1]},
                           "mirror": st["mirror"], "hops": st["hops"], "candidates": int(st["candidates_scored"]),
                           "pairs_evaluated": int(st["pairs_evaluated"]), "slabs": st["slabs"],
                           "bound_over_count": bound / max(int(st["pairs_evaluated"]), 1),
                           "prefilter": st.get("prefilter", {}).get("gcn", {}).get("band_occupancy")}
    ref = run(3, precision="fp32", mirror=False)
    res["hops3_equals_fp32_arm_full"] = bool(torch.equal(outs[3], ref))
    res["hops3_list_rows_outside_2hop"] = int(k - _in_two_hop(adj, outs[3]))
    return res


def _in_two_hop(adj, lst):
    """Rows of a proposal list that are 2-hop candidates (|N(u) & N(v)| > 0)."""
    from edge_proposal_sets_b200 import ops
    e = torch_edges(lst)
    return int((ops.cn_aa(adj, e, None, use_values=False, grouped_by_v=False, want_count=True)[1] > 0).sum())


def torch_edges(lst):
    import torch
    return torch.stack([lst[:, 0].int(), lst[:, 1].int()]).contiguous()


def _two_walk_end_degrees(adj, lo, hi):
    """sum over owners v in [lo, hi) of sum_{x in distinct 2-walk ends of v} deg x, and the 2-path count."""
    import torch
    rp, col = adj.rowptr.long(), adj.col.long()
    deg = rp[1:] - rp[:-1]
    ks = col[rp[lo]:rp[hi]]
    owner = torch.repeat_interleave(torch.arange(lo, hi, device=col.device), deg[lo:hi])
    lens = deg[ks]
    starts = torch.repeat_interleave(rp[ks], lens)
    pos = torch.arange(int(lens.sum()), device=col.device) - torch.repeat_interleave(torch.cumsum(lens, 0) - lens, lens)
    ends = col[starts + pos]
    key = torch.unique(torch.repeat_interleave(owner, lens) * adj.n + ends)
    return int(deg[key % adj.n].sum()), int(lens.sum())


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=3, help="timed steps per hops value (alternating)")
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--slab-reps", type=int, default=3, help="timed repetitions of each call on the ppa slab")
    p.add_argument("--slab-pairs", type=int, default=1 << 27)
    p.add_argument("--out", default=None, help="also write the JSON result here")
    a = p.parse_args()

    import torch
    import bench
    from mirror_ab import card_info
    from edge_proposal_sets_b200 import _lib, candidates, filter_step

    if not torch.cuda.is_available():
        raise SystemExit("threehop_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    report = {"card_before": card_info(), "steps": a.steps, "warmup": a.warmup, "slab_pairs": a.slab_pairs}
    bargs = argparse.Namespace(scale=1.0, mlp=None, slab_pairs=a.slab_pairs, no_pushdown=False, owners_frac=1.0)

    # ---- 1. whole-graph GCN jobs ----
    adj, x, mg, k = _twitch_job(dev)
    report["twitch"] = dict(n=adj.n, nnz=adj.nnz, k=k, **_jobs(adj, x, mg, k, a.steps, a.warmup, a.slab_pairs))
    del adj, x, mg
    wl = bench.Workload("collab", bargs, dev, 1)
    adj, x = wl.upload()
    torch.cuda.synchronize()
    report["collab"] = dict(n=wl.n, nnz=adj.nnz, k=wl.k, **_jobs(adj, x, wl.model, wl.k, a.steps, a.warmup,
                                                                  a.slab_pairs))
    del wl, adj, x
    torch.cuda.empty_cache()

    # ---- 2. ppa-shape, one full hops=3 slab ----
    wl = bench.Workload("ppa", bargs, dev, 1)
    adj, _ = wl.upload()
    torch.cuda.synchronize()
    lo, hi, cap = next(filter_step.iter_slabs(adj, 0, adj.n, a.slab_pairs, hops=3))

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

    t3, e3 = timed(lambda: candidates.three_hop(adj, lo, hi, cap=cap))
    N3 = int(e3.shape[1])
    walk3, paths = _two_walk_end_degrees(adj, lo, hi)
    del e3
    candidates.arc_triangles(adj)
    t_lp, r_lp = timed(lambda: candidates.two_hop_local_path(adj, lo, hi))
    deg = adj.degree().long()
    lp_pull = int(deg[r_lp[0][0].long()].sum())
    N2 = int(r_lp[0].shape[1])
    del r_lp
    el3, el_lp = 2 * paths + walk3, 2 * paths + lp_pull
    report["ppa_slab"] = {
        "n": adj.n, "nnz": adj.nnz, "owners": [lo, hi], "cap_hops3": int(cap), "candidates_hops3": N3,
        "candidates_hops2": N2, "two_paths": paths, "walk3_list_elements": walk3,
        "three_hop_enum": {"ms": t3, "list_elements": el3, "G_list_elements_per_s": el3 / t3 / 1e6},
        "local_path_fused": {"ms": t_lp, "list_elements": el_lp, "G_list_elements_per_s": el_lp / t_lp / 1e6},
        "per_element_vs_lp": (t3 / el3) / (t_lp / el_lp)}
    report["ppa_full_hops3_job"] = "not measured"
    report["card_after"] = card_info()
    bench.emit(report)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(json.dumps(report) + "\n")


if __name__ == "__main__":
    main()
