#!/usr/bin/env python
"""Per-node proposal budgets on the bench workload: the cost of ``filter_topk_multi(..., per_node=m)`` next to the
global job in the same process, and K4c (``ops.segment_topk``) against the torch composition it replaces.

    python tools/pernode_bench.py [--workload ppa] [--m 10 100] [--k 4000000]

Same graph, models and jobs as bench.py (``bench.Workload``: Adamic-Adar on the fused K6+K3 path and the GCN filter
on the tensor-core prefilter).  Prints ONE JSON line with, per (m, K in {k, None}): the per-node phase in ms per slab,
the whole job in ms and candidates/s, the bytes model of K4c (4 B read per candidate + 12 B written per survivor, per
job) against the HBM peak, the survivors and the GCN pool; the owners' candidate-count distribution; the torch
composition (two stable sorts + rank-within-owner) on one full slab with a bit-identity check; GPU name and power
limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (keeps fd 1 for the result line, see bench.emit)

HBM_PEAK = 7.7e12          # B/s, B200 data sheet (one GPU)


def gpu_info():
    import torch
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def run_job(wl, adj, x, k, m):
    import torch
    from edge_proposal_sets_b200 import filter_step
    adj._cache.clear()
    wl.model._h_key = None
    jobs = [filter_step.FilterJob("adamic_ogb", None), filter_step.FilterJob("gcn", wl.model, precision=wl.mlp_arm)]
    st = {"time_phases": True}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = filter_step.filter_topk_multi(jobs, x, adj, k=k, slab_pairs=wl.args.slab_pairs, stats=st, per_node=m,
                                        owners=wl.owners)
    b.record()
    torch.cuda.synchronize()
    return out, st, a.elapsed_time(b)


def torch_baseline(adj, slab_pairs, m):
    """One full slab (the first): AA scores + owner offsets, K4c vs two stable torch sorts + rank-within-owner."""
    import torch
    from edge_proposal_sets_b200 import candidates, filter_step, ops
    lo, hi, cap = next(filter_step.iter_slabs(adj, 0, adj.n, slab_pairs))
    t = filter_step.heuristic_table("adamic_ogb", adj)
    edges, score, off = candidates.two_hop_scored(t[0], t[1], lo, hi, sigmoid=t[2], cap=cap, use_values=t[3],
                                                  want_offsets=True)
    M = score.numel()
    cnt = off[1:] - off[:-1]
    seg = torch.repeat_interleave(torch.arange(cnt.numel(), device=score.device), cnt)

    def composed():
        o1 = torch.sort(score, descending=True, stable=True).indices
        owner = seg[o1]
        o2 = torch.sort(owner, stable=True).indices
        rank = torch.arange(M, device=score.device) - off[owner[o2]]
        keep = torch.sort(o1[o2[rank < m]]).values
        return keep

    def timed(fn, reps=3):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        fn()
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(reps):
            r = fn()
        ev[1].record()
        torch.cuda.synchronize()
        return r, ev[0].elapsed_time(ev[1]) / reps

    keep, ms_torch = timed(composed)
    (e2, s2, _), ms_k4c = timed(lambda: ops.segment_topk(score, edges, off, m))
    identical = bool(torch.equal(e2[0], edges[0][keep]) and torch.equal(e2[1], edges[1][keep])
                     and torch.equal(s2.view(torch.int32), score[keep].view(torch.int32)))
    return dict(m=m, slab_candidates=int(M), slab_owners=int(hi - lo), torch_ms=ms_torch, k4c_ms=ms_k4c,
                speedup=ms_torch / ms_k4c if ms_k4c > 0 else None, bit_identical=identical,
                k4c_bytes_model_tb_s=(4 * M + 12 * s2.numel()) / (ms_k4c * 1e-3) / 1e12)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--workload", default="ppa", choices=["ppa", "collab", "ddi", "small", "tiny"])
    p.add_argument("--m", type=int, nargs="+", default=[10, 100])
    p.add_argument("--k", type=int, default=None, help="the K of the K-limited runs (default: bench.py's k)")
    p.add_argument("--slab-pairs", type=int, default=1 << 27)
    p.add_argument("--scale", type=float, default=1.0)
    p.add_argument("--owners-frac", type=float, default=1.0)
    a = p.parse_args()
    import numpy as np
    import torch
    from edge_proposal_sets_b200 import _lib, candidates
    _lib.load()
    dev = torch.device("cuda:0")
    wargs = argparse.Namespace(scale=a.scale, mlp=None, owners_frac=a.owners_frac, slab_pairs=a.slab_pairs,
                               no_pushdown=False)
    wl = bench.Workload(a.workload, wargs, dev, 1)
    k = a.k or wl.k
    adj, x = wl.upload()
    info = gpu_info()
    cnt = candidates.owner_counts(adj).double()
    dist = dict(owners=int(cnt.numel()), mean=float(cnt.mean()), p99=float(torch.quantile(cnt[::max(1, cnt.numel() // 1_000_000)], 0.99)),
                max=int(cnt.max()), candidates=int(cnt.sum()))
    run_job(wl, adj, x, k, None)                                  # warm-up: every kernel and shape of both modes
    run_job(wl, adj, x, k, a.m[0])
    _, st_g, ms_g = run_job(wl, adj, x, k, None)
    cand = st_g["candidates_scored"]
    rows = []
    for m in a.m:
        for kk in (k, None):
            out, st, ms = run_job(wl, adj, x, kk, m)
            ph = st["phase_ms"]
            surv = st["per_node"]["survivors"]
            pn_ms = ph.get("per_node", 0.0)
            bytes_model = 2 * 4 * cand + 12 * sum(surv)
            rows.append(dict(m=m, k=kk, ms_job=ms, candidates_per_s=cand / (ms * 1e-3), slabs=st["slabs"],
                             per_node_ms=pn_ms, per_node_ms_per_slab=pn_ms / max(st["slabs"], 1),
                             added_vs_global_ms=ms - ms_g, global_topk_phase_ms=st_g["phase_ms"].get("topk", 0.0),
                             per_node_topk_phase_ms=ph.get("topk", 0.0), rescore_ms=ph.get("rescore", 0.0),
                             survivors=surv, gcn_pool=st.get("prefilter", {}).get("gcn", {}).get("pool"),
                             prefilter_fallback=st.get("prefilter_fallback"), rows=[int(o.shape[0]) for o in out],
                             k4c_bytes_model=bytes_model,
                             k4c_share_of_hbm_peak=(bytes_model / (pn_ms * 1e-3)) / HBM_PEAK if pn_ms > 0 else None))
            del out
            torch.cuda.empty_cache()
    base = [torch_baseline(adj, a.slab_pairs, m) for m in a.m]
    bench.emit(dict(tool="pernode_bench", workload=a.workload, gpu=info, k=k, candidates=cand,
                    global_job=dict(ms_job=ms_g, candidates_per_s=cand / (ms_g * 1e-3), phase_ms=st_g["phase_ms"]),
                    per_node=rows, segment_sizes=dist, torch_composition_one_slab=base,
                    hbm_peak_tb_s=HBM_PEAK / 1e12))


if __name__ == "__main__":
    main()
