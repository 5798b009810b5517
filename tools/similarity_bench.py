"""The degree-normalised similarity filters on the benchmark's graph, in one process.

1. The full filter job (enumerate, score, top-k at the benchmark's k) of every similarity model against the `simple`
   (CN) and `adamic_ogb` jobs, each with mirror mode off and on, run alternately: median ms per step and mean phase
   times (`enum_score`, `topk`, `mirror`).
2. One full slab of the job (the first owner slab, ~125 M candidates on the ppa shape): the fused epilogue
   (`two_hop_scored(kind=...)`) against a torch composition (CN counts from the fused kernel, degrees gathered,
   formula in torch ops) and against the count-only CN call, with bit equality of fused and composition.
   Rates: G candidates/s, and GB/s under the traffic model stated in the output.
3. The card's name, power limit and SM clocks, read before and after.

    python tools/similarity_bench.py [--workload ppa] [--steps 2] [--warmup 1] [--out FILE]
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

KINDS = ("jaccard", "sorensen", "salton", "hub_promoted", "hub_depressed", "leicht_holme_newman",
         "preferential_attachment")


def torch_similarity(torch, c, a, b, kind):
    """The kernels' operation sequence (include/eps.h, EPS_SCORE_*) in torch ops, from int64 c, a, b."""
    if kind == "preferential_attachment":
        return (a * b).float()
    if kind in ("salton", "leicht_holme_newman"):
        ab = a.double() * b.double()
        q = c.double() / (torch.sqrt(ab) if kind == "salton" else ab)
        return torch.where(ab == 0, torch.zeros_like(q), q).float()
    num = c
    if kind == "jaccard":
        den = a + b - c
    elif kind == "sorensen":
        num, den = 2 * c, a + b
    elif kind == "hub_promoted":
        den = torch.minimum(a, b)
    else:
        den = torch.maximum(a, b)
    q = num.float() / den.float()
    return torch.where(den == 0, torch.zeros_like(q), q)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--workload", default="ppa", choices=["ppa", "collab", "ddi", "small", "tiny"])
    p.add_argument("--steps", type=int, default=2, help="timed steps per job and mirror mode (alternating)")
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--slab-reps", type=int, default=5, help="timed repetitions of each call on the slab")
    p.add_argument("--slab-pairs", type=int, default=1 << 27)
    p.add_argument("--out", default=None, help="also write the JSON result here")
    a = p.parse_args()

    import torch
    import bench
    from mirror_ab import card_info
    from edge_proposal_sets_b200 import _lib, candidates, filter_step, models

    if not torch.cuda.is_available():
        raise SystemExit("similarity_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    bargs = argparse.Namespace(scale=1.0, mlp=None, slab_pairs=a.slab_pairs, no_pushdown=False, owners_frac=1.0)
    card_before = card_info()
    wl = bench.Workload(a.workload, bargs, dev, 1)
    adj, x = wl.upload()
    torch.cuda.synchronize()
    report = {"workload": a.workload, "k": wl.k, "n": wl.n, "nnz": adj.nnz, "steps": a.steps, "warmup": a.warmup,
              "card_before": card_before}

    # ---- 1. full filter jobs ----
    names = ("simple", "adamic_ogb") + KINDS
    model = {nm: (None if nm == "adamic_ogb" else
                  models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=nm)) for nm in names}

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
            "mirror": r["stats"]["mirror"], "pairs_evaluated": int(r["stats"]["pairs_evaluated"])}
    for nm in names:
        jobs[nm]["lists_equal_mirror_vs_full"] = bool(torch.equal(outs[(nm, False)], outs[(nm, True)]))
    cn = jobs["simple"]
    for nm in names:
        for arm in ("full", "mirror"):
            e_cn = cn[arm]["phase_ms_mean"].get("enum_score", 0.0)
            jobs[nm][arm]["enum_score_vs_cn"] = jobs[nm][arm]["phase_ms_mean"].get("enum_score", 0.0) / e_cn if e_cn else None
    report["jobs"] = jobs

    # ---- 2. one full slab: fused epilogue vs torch composition ----
    lo, hi, cap = next(filter_step.iter_slabs(adj, 0, adj.n, a.slab_pairs))
    deg = adj.degree().long()
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

    def composition(kind):
        e, _, c = candidates.two_hop_scored(adj, None, lo, hi, cap=cap, want_count=True)
        return e, torch_similarity(torch, c.long(), deg[e[0].long()], deg[e[1].long()], kind)

    t_cn, (e_cn, _) = timed(lambda: candidates.two_hop_scored(adj, None, lo, hi, cap=cap))
    N = int(e_cn.shape[1])
    del e_cn
    # traffic of the fused call: the 2-path walk reads 4 B of `col` per 2-path twice (mark + score); per candidate the
    # walk writes u and the count into the padded slot (8 B), the compaction reads them (8 B) and writes u, v, score
    # (12 B); a similarity kind adds deg u (two 4 B rowptr loads, L2-resident) = 28 B + 8 B
    model_txt = "8 B per 2-path walked + 28 B per candidate (+ 8 B of rowptr for deg u with a similarity kind)"
    slab = {"owners": [lo, hi], "cap": int(cap), "candidates": N, "two_paths": paths, "traffic_model": model_txt,
            "cn_count_only": {"ms": t_cn, "G_candidates_per_s": N / t_cn / 1e6,
                              "GB_per_s": (8 * paths + 28 * N) / t_cn / 1e6}}
    for kind in KINDS:
        t_f, (e_f, s_f) = timed(lambda: candidates.two_hop_scored(adj, None, lo, hi, cap=cap, kind=kind))
        t_c, (e_c, s_c) = timed(lambda: composition(kind))
        slab[kind] = {"fused_ms": t_f, "torch_composition_ms": t_c, "fused_vs_cn": t_f / t_cn,
                      "G_candidates_per_s": N / t_f / 1e6, "GB_per_s": (8 * paths + 36 * N) / t_f / 1e6,
                      "bit_equal": bool(torch.equal(e_f, e_c) and torch.equal(s_f.view(torch.int32),
                                                                               s_c.view(torch.int32)))}
        del e_f, s_f, e_c, s_c
    report["slab"] = slab
    report["card_after"] = card_info()
    line = json.dumps(report)
    bench.emit(report)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
