#!/usr/bin/env python
"""bench.py — candidate pairs scored / second on the ogbl-ppa shape (BASELINE.json metric).

One STEP = the WHOLE filter job (/root/reference/filter.py:92-166) of the graph, through the product call
``filter_step.filter_topk_multi`` — the call filter.py makes — for the two filter models BASELINE.json names:

  GCN embeddings once (gcn_norm + L x [cuBLAS x·W row blocks + K1 SpMM]; row-sharded + all-gathered when N > 1)
  for every owner slab of the graph (all 576,289 owners, 8.26 G candidates on the ppa shape):
      K6+K3 fused, one pass : candidates + Adamic-Adar score of every candidate
      K2 tcgen05            : GCN+LinkPredictor score of every candidate (fp16 operands: the prefilter)
      K4b + K4              : threshold push-down + running top-k (exact list for AA, tolerance band for GCN)
  fp32 re-scoring of the GCN band (K2 FFMA arm) -> the fp32 arm's exact top-k; one stable sort per list
  [N > 1: owners sharded by 2-path work, global k-th score exchanged, lists merged (NCCL)]

`value` = candidates of the graph / device time of the step (every candidate is scored by BOTH filter models),
strong scaling: the same job on N GPUs.  Nothing is cached between steps.  `e2e` = the same call with HOST
inputs: graph, features and weights uploaded from pinned memory and both [k,3] lists copied back, every step.

  python bench.py [--gpus N --steps K --warmup W] [--workload ppa|collab|ddi|small|tiny] [--dump-outputs DIR]
  python bench.py --impl reference ...     # the reference's CPU path (oracle port) on host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: keep a private handle to it and point fd 1 at stderr, so that
# nothing a library prints (NCCL's version banner, torchrun notices) can land next to the result
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict) -> None:
    _RESULT_OUT.write(json.dumps(line) + "\n")
    _RESULT_OUT.flush()


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="ppa", choices=["ppa", "collab", "ddi", "small", "tiny"])
    p.add_argument("--slab-pairs", type=int, default=1 << 27, help="candidate capacity of one owner slab")
    p.add_argument("--owners-frac", type=float, default=1.0,
                   help="score only the first fraction of the owners (debug / profiling runs; 1.0 = the whole graph)")
    p.add_argument("--mlp", default=None, choices=[None, "prefilter", "fp32", "f16"],
                   help="K2 arm of the GCN filter: prefilter = tcgen05 (fp16 operands) scores + fp32 re-scoring of the band "
                        "(default; the fp32 arm's exact list), f16 = tensor-core scores only, fp32 = FFMA arm")
    p.add_argument("--scale", type=float, default=1.0, help="shrink the synthetic graph (debug only)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extras", action="store_true",
                   help="skip the ddi / collab shape lines, the library baseline and the multi-GPU self-check")
    p.add_argument("--no-pushdown", action="store_true", help="K4 select over every slab instead of K4b push-down (A/B)")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the proposal lists of the last timed step to DIR/<filter model>.npy (float32 rows u, v, "
                        "score; lists over their share of 60 MiB cut to rows at fixed seeded positions), so that two "
                        "builds can be compared output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl != "b200":
        p.error("--dump-outputs writes the b200 arm's outputs")
    return a


# ------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------

MODEL_CFG = {  # builder's choice for ppa (the reference has no ppa defaults, SURVEY A.8)
    "ppa": dict(layers=3, hidden=256, k=4_000_000),        # submit_job.py:210
    "collab": dict(layers=3, hidden=256, k=200_000),       # models.py:712-721, submit_job.py:202
    "ddi": dict(layers=2, hidden=256, k=530_000),          # models.py:685-694, submit_job.py:194
    "small": dict(layers=3, hidden=256, k=20_000), "tiny": dict(layers=2, hidden=64, k=500),
}


def build_host_inputs(workload, scale=1.0):
    """Synthetic graph of the named shape + seeded random-init weights, as host tensors."""
    import torch
    from edge_proposal_sets_b200 import synth
    t0 = time.time()
    s = synth.make_shape(workload, scale)
    ei = synth.undirected_edge_index(s["train_edges"])
    cfg = MODEL_CFG[workload]
    n, H, L = s["n"], cfg["hidden"], cfg["layers"]
    g = torch.Generator().manual_seed(1234)
    feat = 0 if s["x"] is None else s["x"].shape[1]
    f_in = H + feat
    sd = {"emb.weight": torch.randn(n, H, generator=g)}
    for i in range(L):
        ic = f_in if i == 0 else H
        a = (6.0 / (ic + H)) ** 0.5
        sd[f"gnn.convs.{i}.weight"] = (torch.rand(ic, H, generator=g) * 2 - 1) * a
        sd[f"gnn.convs.{i}.bias"] = (torch.rand(H, generator=g) * 2 - 1) * 0.05
    # LinkPredictor: random weights at the scale of a TRAINED filter model.  With nn.Linear's default init the
    # pair-dependent signal (|h_u * h_v| ~ 1e-3 after three GCN layers) drowns in the hidden biases: every
    # candidate of the graph scores 0.4869 +- 1e-4 (measured), the top-k boundary sits in a spike of ~4e9
    # near-equal scores and neither a reduced-precision prefilter nor the ordering itself means anything.
    # Hidden layers: He-uniform weights, zero biases (ReLU keeps the signal's scale); the output layer is
    # rescaled on the device so that the logits have mean -2 and std 2 (``Workload.calibrate_model``), the
    # score spread of a trained link predictor.  Work per candidate is unchanged.
    for i in range(L):
        oc = 1 if i == L - 1 else H
        b = (6.0 / H) ** 0.5 if i < L - 1 else 1.0 / H ** 0.5
        sd[f"linkpred.lins.{i}.weight"] = (torch.rand(oc, H, generator=g) * 2 - 1) * b
        sd[f"linkpred.lins.{i}.bias"] = torch.zeros(oc)
    host = dict(n=n, H=H, L=L, feat=feat, edge_index=torch.from_numpy(ei), workload=workload,
                edge_weight=None if s["edge_weight"] is None else torch.from_numpy(np.concatenate([s["edge_weight"]] * 2)),
                x=None if s["x"] is None else torch.from_numpy(s["x"]), sd=sd,
                dataset="collab" if s["edge_weight"] is not None else workload, gen_s=time.time() - t0)
    return host


def workload_text(workload: str, k: int, slab_pairs: int) -> str:
    return (f"{workload}-shape FULL filter job: GCN embeddings once, every owner of the graph enumerated in slabs of "
            f"<= {slab_pairs} candidates, every candidate scored by Adamic-Adar (fused K6+K3) and GCN+LinkPredictor "
            f"(tcgen05), top-{k} proposal list of each")


# ------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------

class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# the reference's CPU path (oracle port), bounded sample
# ------------------------------------------------------------------------------------------

_G = {}


def _aa_worker(sl):
    from oracle import heuristics as oh
    return oh.aa_scipy(_G["g"], _G["cand"][:, sl[0]:sl[1]], 2000)


def cpu_reference_pass(host, owners, seconds_budget, procs):
    """One pass of the reference's CPU filter step over `owners` (a small owner range):
    scipy A@A candidate enumeration (filter.py:96-109), adamic_utils.AA-style scipy scoring fanned
    out over `procs` processes (scipy itself is single-threaded), torch-CPU LinkPredictor with all
    threads on embeddings computed once, torch CPU sort (filter.py:160).  Returns timings."""
    import multiprocessing as mp
    import torch
    from oracle import gnn as ognn, graph as og, heuristics as oh
    g = _G["g"]
    lo, hi = owners
    t0 = time.time()
    A = g.to_scipy()
    sub = (A @ A[:, lo:hi]).tocsc()
    sub.sort_indices()
    rows = sub.indices.astype(np.int64)
    cols = np.repeat(np.arange(lo, hi, dtype=np.int64), np.diff(sub.indptr))
    keep = rows != cols
    keys = np.repeat(np.arange(g.n, dtype=np.int64), np.diff(g.rowptr)) * g.n + g.col
    k = rows * g.n + cols
    pos = np.minimum(np.searchsorted(keys, k), keys.size - 1)
    keep &= keys[pos] != k
    cand = np.stack([rows[keep], cols[keep]])
    t_cand = time.time() - t0
    M = cand.shape[1]
    _G["cand"] = cand
    t0 = time.time()
    if procs > 1 and M > 20000:
        step = (M + procs - 1) // procs
        with mp.get_context("fork").Pool(procs) as pool:
            aa = np.concatenate(pool.map(_aa_worker, [(i, min(i + step, M)) for i in range(0, M, step)]))
    else:
        aa = oh.aa_scipy(g, cand, 2000)
    t_aa = time.time() - t0
    t0 = time.time()
    h = _G["h"]
    with torch.no_grad():
        sc = ognn.linkpred_forward(h, cand, host["sd"], host["L"], torch.float32)
    t_mlp = time.time() - t0
    t0 = time.time()
    torch.from_numpy(aa).sort(descending=True)
    sc.sort(descending=True)
    t_sort = time.time() - t0
    return dict(pairs=M, t_cand=t_cand, t_aa=t_aa, t_mlp=t_mlp, t_sort=t_sort,
                total=t_cand + t_aa + t_mlp + t_sort)


def cpu_setup(host):
    import torch
    from oracle import gnn as ognn, graph as og
    ei = host["edge_index"].numpy()
    w = np.ones(ei.shape[1], np.float32) if host["edge_weight"] is None else host["edge_weight"].numpy()
    g = og.add_edges(host["dataset"], ei, w, np.zeros((2, 0), np.int64), host["n"])
    _G["g"] = g
    t0 = time.time()
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        xin = ognn.link_gnn_input(host["sd"], host["x"])
        _G["h"] = ognn.gcn_forward(g, xin, host["sd"], host["L"], torch.float32)
    return time.time() - t0


def cpu_pick_owners(host, seconds_budget):
    """Size the owner sample so one pass costs roughly `seconds_budget` on this host."""
    g = _G["g"]
    deg = np.diff(g.rowptr)
    work = np.add.reduceat(deg[g.col], g.rowptr[:-1][deg > 0]) if g.nnz else np.zeros(0)
    w_full = np.zeros(g.n); w_full[deg > 0] = work
    # the whole CPU pass (scipy A@A + scipy AA + torch MLP + sort) costs ~1.5 us per 2-path on this
    # class of host (measured); size the owner sample to the time budget
    budget = seconds_budget / 1.5e-6
    cs = np.cumsum(w_full)
    hi = int(np.searchsorted(cs, budget)) + 1
    return 0, max(1, min(hi, g.n))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    host = build_host_inputs(args.workload, args.scale)
    embed_s = cpu_setup(host)
    procs = os.cpu_count()
    owners = cpu_pick_owners(host, max(args.cpu_seconds / 3, 1.0))
    for _ in range(args.warmup):
        r = cpu_reference_pass(host, owners, args.cpu_seconds, procs)
        if r["total"] > 3 * args.cpu_seconds:      # keep the whole run within minutes
            owners = (owners[0], max(owners[0] + 1, owners[0] + (owners[1] - owners[0]) // 2))
    tot_pairs, tot_t, last = 0, 0.0, None
    for _ in range(args.steps):
        last = cpu_reference_pass(host, owners, args.cpu_seconds, procs)
        tot_pairs += last["pairs"]; tot_t += last["total"]
    value = tot_pairs / tot_t
    cfg = MODEL_CFG[args.workload]
    line = {
        "impl": "reference", "metric": "candidate pairs scored/sec (CN/AA + GCN+LinkPredictor filter step)",
        "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the B200 arm's workload; each reference step is a BOUNDED SAMPLE of it (cpu_baseline.sample): the same
        # graph, models and per-candidate work, but only the candidates of `sample_owners` — the whole job
        # (8.26 G candidates on ppa) would take the CPU path several hours
        "config": {"workload": workload_text(args.workload, cfg["k"], args.slab_pairs),
                   "n": host["n"], "nnz": int(host["edge_index"].shape[1]),
                   "gnn": f"gcn L={cfg['layers']} H={cfg['hidden']} F_in={cfg['hidden'] + host['feat']}",
                   "sample_owners": [owners[0], owners[1]], "same_config_as_b200_arm": False,
                   "why": "bounded sample of the same workload (rate per candidate; the job itself is not finished)"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": procs, "kind": "port",
                         "sample": f"{last['pairs']} candidates of owners [{owners[0]},{owners[1]}) per step; "
                                   f"scipy A@A enumeration + scipy AA x{procs} procs + torch-CPU MLP + torch sort; "
                                   f"GCN embeddings once ({embed_s:.1f}s, not counted)",
                         "breakdown_s": {k: last[k] for k in ("t_cand", "t_aa", "t_mlp", "t_sort")}},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------

class Workload:
    """One synthetic shape on this rank's GPU: pinned host inputs, upload(), and the step."""

    def __init__(self, name, args, dev, world, pin=True):
        import torch
        from edge_proposal_sets_b200 import graph as pg, models
        self.name, self.args, self.dev, self.world = name, args, dev, world
        host = build_host_inputs(name, args.scale)
        self.host = host
        n, H, L = host["n"], host["H"], host["L"]
        self.n, self.H, self.L = n, H, L
        self.k = MODEL_CFG[name]["k"]
        pinf = (lambda t: t.pin_memory()) if pin else (lambda t: t)
        ew = host["edge_weight"] if host["edge_weight"] is not None else torch.ones(host["edge_index"].shape[1])
        adj0 = pg.add_edges(host["dataset"], host["edge_index"].to(dev), ew.to(dev),
                            torch.zeros([2, 0], dtype=torch.long, device=dev), n)
        # rows of the node features / embedding table this rank's share of the row-sharded GNN reads (a function of
        # the graph alone: models._ConvStack.embed_rows cuts the same ranges)
        self.rank = int(os.environ.get("RANK", "0")) if world > 1 else 0
        from edge_proposal_sets_b200 import parallel as _par
        rb = _par.row_partition(adj0.gcn_norm()[0], n, world)
        self.rows = (rb[self.rank], rb[self.rank + 1])
        self.h_rowptr, self.h_col = pinf(adj0.rowptr.cpu()), pinf(adj0.col.cpu())
        self.h_val = None if adj0.val is None else pinf(adj0.val.cpu())
        self.h_x = None if host["x"] is None else pinf(host["x"])
        self.h_sd = {k: pinf(v.contiguous()) for k, v in host["sd"].items()}
        del adj0
        torch.cuda.empty_cache()
        self.mlp_arm = args.mlp or os.environ.get("EPS_BENCH_MLP", "prefilter")
        margs = argparse.Namespace(model="gcn", dataset=name, num_layers=L, hidden_channels=H, dropout=0.0,
                                   use_feature=host["x"] is not None, use_learnable_embedding=True,
                                   mlp_precision=self.mlp_arm)

        class D:
            num_nodes = n
            x = host["x"]
        self.model = models.build_model(margs, D, dev)        # parameter storage; every upload() refills it
        self.model.eval()
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.calibrate_model()
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in [self.h_rowptr, self.h_col] +
                             ([self.h_val] if self.h_val is not None else []) +
                             ([self.h_x] if self.h_x is not None else []) + list(self.h_sd.values()))
        self.owners = None if args.owners_frac >= 1.0 else (0, max(1, int(n * args.owners_frac)))
        # end-to-end upload at N > 1: the whole graph, but only this rank's ROW SHARD of the node-indexed inputs
        frac = (self.rows[1] - self.rows[0]) / max(n, 1)
        node_indexed = ([self.h_x] if self.h_x is not None else []) + [v for k_, v in self.h_sd.items() if k_ == "emb.weight"]
        full_nodes = sum(t.numel() * t.element_size() for t in node_indexed)
        self.h2d_bytes_sharded = int(self.h2d_bytes - full_nodes + full_nodes * frac) if world > 1 else self.h2d_bytes

    def calibrate_model(self):
        """Rescale the output layer so that the fp32 logits of ~10^6 candidates have mean -2, std 2 (see
        build_host_inputs).  Deterministic: same graph, same seeds, same sample on every rank."""
        import torch
        from edge_proposal_sets_b200 import candidates, ops
        adj, x = self.upload()
        h = self.model.embed(x, adj)
        bounds = torch.cumsum(candidates.owner_bounds(adj), 0)
        v_hi = int(torch.searchsorted(bounds, torch.tensor(1 << 20, device=self.dev)).item())
        edges = candidates.two_hop(adj, 0, max(v_hi, 1))
        lins = self.model.linkpred.lins
        logit = ops.linkpred_mlp(h, edges, [l.weight for l in lins], [l.bias for l in lins], "fp32", sigmoid=False)
        mean, std = float(logit.double().mean().item()), float(logit.double().std().item())
        scale = 2.0 / max(std, 1e-30)
        wl, bl = f"linkpred.lins.{self.L - 1}.weight", f"linkpred.lins.{self.L - 1}.bias"
        self.h_sd[wl].mul_(scale)
        self.h_sd[bl].copy_((self.h_sd[bl] - mean) * scale - 2.0)
        self.host["sd"][wl], self.host["sd"][bl] = self.h_sd[wl].clone(), self.h_sd[bl].clone()
        self.model_scale = dict(sample=int(edges.shape[1]), logit_mean_before=mean, logit_std_before=std, scale=scale)
        self.model._h_key = None

    def upload(self, shard: bool = False):
        """H2D of everything the public call takes (graph first; features + weights on a copy stream).
        ``shard`` (the end-to-end loop at N > 1): of the node-indexed inputs — features and the embedding table —
        only the rows this rank's share of the row-sharded GNN reads (``self.rows``) are copied; the other rows of
        the device buffers are never read by this rank (embed_rows slices before it computes)."""
        import torch
        from edge_proposal_sets_b200 import graph as pg
        dev = self.dev
        adj = pg.SparseAdj(self.h_rowptr.to(dev, non_blocking=True), self.h_col.to(dev, non_blocking=True),
                           None if self.h_val is None else self.h_val.to(dev, non_blocking=True), self.n)
        part = shard and self.world > 1
        lo, hi = self.rows
        self.copy_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.copy_stream), torch.no_grad():
            x = None
            if self.h_x is not None:
                if part:
                    x = torch.empty(self.h_x.shape, dtype=self.h_x.dtype, device=dev)
                    x[lo:hi].copy_(self.h_x[lo:hi], non_blocking=True)
                else:
                    x = self.h_x.to(dev, non_blocking=True)
            for k_, p_ in self.model.state_dict().items():
                if part and k_ == "emb.weight":
                    p_[lo:hi].copy_(self.h_sd[k_][lo:hi], non_blocking=True)
                else:
                    p_.copy_(self.h_sd[k_], non_blocking=True)
        torch.cuda.current_stream().wait_stream(self.copy_stream)
        return adj, x

    def step(self, adj, x, stats=None, distributed=None):
        """The filter job through the product call; returns [AA list, GCN list] ([k,3] each)."""
        from edge_proposal_sets_b200 import filter_step
        adj._cache.clear()                                    # nothing derived from the graph is reused
        self.model._h_key = None                              # no embedding cache across steps
        jobs = [filter_step.FilterJob("adamic_ogb", None),
                filter_step.FilterJob("gcn", self.model, precision=self.mlp_arm)]
        dist_on = (self.world > 1) if distributed is None else distributed
        return filter_step.filter_topk_multi(jobs, x, adj, k=self.k, slab_pairs=self.args.slab_pairs,
                                             distributed=dist_on, stats=stats, pushdown=not self.args.no_pushdown,
                                             owners=self.owners)


def measure(wl: Workload, steps: int, warmup: int, rank: int, world: int, e2e_steps: int, sampler=None):
    """Warm-up, K device-timed steps (barrier + sync both sides, max over ranks), then the e2e loop."""
    import torch
    import torch.distributed as dist
    from edge_proposal_sets_b200 import ops
    dev = wl.dev
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    adj, x = wl.upload()
    torch.cuda.synchronize()
    for _ in range(max(warmup, 3)):
        outs = wl.step(adj, x)
    ops.LAUNCHES["n"] = 0
    ops.KERNEL_EVENTS = {}
    if sampler is not None:
        sampler.start()
    all_stats = []
    barrier()
    t0, t1 = ev(), ev()
    t0.record()
    for _ in range(steps):
        st = {"time_phases": True}
        outs = wl.step(adj, x, st)
        all_stats.append(st)
    t1.record()
    barrier()
    kev, ops.KERNEL_EVENTS = ops.KERNEL_EVENTS, None
    launches = ops.LAUNCHES["n"]
    ms_total = t0.elapsed_time(t1)
    tmax = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    cand = torch.tensor([float(all_stats[-1]["candidates_scored"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(cand, op=dist.ReduceOp.SUM)
    ms_step = float(tmax.item()) / steps
    total_pairs = float(cand.item())
    phase_ms = {}
    for st in all_stats:
        for k_, v in st["phase_ms"].items():
            phase_ms[k_] = phase_ms.get(k_, 0.0) + v / steps
    spmm_ms = [a_.elapsed_time(b_) for a_, b_ in kev.get("spmm_csr", [])]

    # ---- end to end through the public call with HOST buffers ----
    out_host = [torch.empty((wl.k, 3), dtype=torch.float32).pin_memory() for _ in range(2)]

    def e2e_step():
        a, xx = wl.upload(shard=True)
        res = wl.step(a, xx)
        for o, r in zip(out_host, res):
            o[: r.shape[0]].copy_(r, non_blocking=True)
        torch.cuda.current_stream().synchronize()             # the caller holds the result on the host
        return res

    e2e = None
    if e2e_steps > 0:
        e2e_step()
        barrier()
        w0 = time.perf_counter()
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record()
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)   # D2H syncs: wall clock is the honest one
        tm = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e = {"value": total_pairs * e2e_steps / (float(tm.item()) * 1e-3), "unit": "pairs/s",
               "h2d_bytes_per_step": wl.h2d_bytes_sharded, "d2h_bytes_per_step": 2 * wl.k * 12, "steps": e2e_steps,
               "ms_per_step": float(tm.item()) / e2e_steps,
               "note": "per step and per rank: pinned-host graph + features + weights -> device, the product call, "
                       "both [k,3] lists -> pinned host" +
                       ("; N > 1: every rank uploads the whole graph and the dense weights but only its row shard of the "
                        "node features and of the embedding table (the rows its share of the row-sharded GNN reads)"
                        if world > 1 else "")}
    return dict(ms_step=ms_step, total_pairs=total_pairs, phase_ms=phase_ms, stats=all_stats[-1], launches=launches,
                spmm_ms=spmm_ms, e2e=e2e, outs=outs, adj=adj, x=x)


def dump_outputs(outs, out_dir, budget=60 << 20):
    """``outs`` (Workload.step's [k,3] lists: u, v, score) -> out_dir/<filter model>.npy, float32.  A list larger than
    its share of ``budget`` bytes keeps the rows at a seeded sample of positions, ascending: the same positions in
    every run of the same arguments, so that the files of two builds compare row for row."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(("adamic_ogb", "gcn"), outs):
        a = t.float().cpu().numpy()
        rows = budget // len(outs) // (a.shape[1] * a.itemsize)
        if a.shape[0] > rows:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def library_baseline(wl: Workload, adj, x, k):
    """SURVEY §2.1's bar, same box: the library kernels the reference reaches — ATen index_select + mul,
    cuBLAS Linear, relu, sigmoid (models.py:478-485,506) in fp32 (TF32 off, the reference default) and in bf16
    autocast-style, and torch.topk / torch.sort for the ordering (filter.py:160) — on one slab of this graph."""
    import torch
    from edge_proposal_sets_b200 import candidates
    model = wl.model
    h = model.embed(x, adj)
    bounds = torch.cumsum(candidates.owner_bounds(adj), 0)
    v_hi = int(torch.searchsorted(bounds, torch.tensor(min(wl.args.slab_pairs, 1 << 26), device=wl.dev)).item())
    edges = candidates.two_hop(adj, 0, max(v_hi, 1))
    M = edges.shape[1]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    out = {"slab_candidates": int(M)}
    lins = model.linkpred.lins
    B = 1 << 20                                               # 16x the reference's largest batch (64K, models.py:685-694)
    nb = min(8, max(1, M // B))
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        hh = h.to(dt)
        Ws = [(l.weight.to(dt), l.bias.to(dt)) for l in lins]

        def run(lo):
            e = edges[:, lo:lo + B].long()
            z = hh[e[0]] * hh[e[1]]
            for w, b in Ws[:-1]:
                z = torch.relu(torch.nn.functional.linear(z, w, b))
            return torch.sigmoid(torch.nn.functional.linear(z, Ws[-1][0], Ws[-1][1]))
        run(0); run(0)
        a, b_ = ev(), ev()
        a.record()
        for i in range(nb):
            run((i * B) % max(M - B, 1))
        b_.record()
        torch.cuda.synchronize()
        out[f"torch_eager_{name}_mlp_pairs_per_s"] = nb * min(B, M) / (a.elapsed_time(b_) * 1e-3)
    sc = model.linkpred.score_pairs(h, edges, "f16")
    kk = min(k, M)
    for name, fn in (("torch_topk", lambda: torch.topk(sc, kk)), ("torch_sort_stable", lambda: torch.sort(sc, descending=True, stable=True))):
        fn()
        a, b_ = ev(), ev()
        a.record()
        fn()
        b_.record()
        torch.cuda.synchronize()
        out[f"{name}_ms_per_slab"] = a.elapsed_time(b_)
    from edge_proposal_sets_b200 import ops
    ops.topk_edges(edges, sc, kk)
    a, b_ = ev(), ev()
    a.record()
    ops.topk_edges(edges, sc, kk)
    b_.record()
    torch.cuda.synchronize()
    out["eps_topk_k4_ms_per_slab"] = a.elapsed_time(b_)
    for prec in ("f16", "fp32"):
        mm = M if prec == "f16" else min(M, 1 << 23)
        e_ = edges[:, :mm].contiguous()
        model.linkpred.score_pairs(h, e_, prec)
        a, b_ = ev(), ev()
        a.record()
        model.linkpred.score_pairs(h, e_, prec)
        b_.record()
        torch.cuda.synchronize()
        out[f"eps_k2_{prec}_pairs_per_s"] = mm / (a.elapsed_time(b_) * 1e-3)
    out["note"] = ("same slab, same box: eager = index_select x2 + mul + (Linear, relu) x (L-1) + Linear + sigmoid in batches of "
                   "2^20 pairs (the reference uses <= 2^16); K4 vs torch.topk / stable torch.sort of the slab's scores")
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from edge_proposal_sets_b200 import _lib, candidates

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    torch.backends.cuda.matmul.allow_tf32 = False          # reference default: fp32 SGEMM

    wl = Workload(args.workload, args, dev, world)
    n, H, L, k = wl.n, wl.H, wl.L, wl.k
    sampler = ClockSampler(local) if rank == 0 else None
    res = measure(wl, args.steps, args.warmup, rank, world, e2e_steps=min(args.steps, 5), sampler=sampler)
    clocks = sampler.stop() if sampler is not None else None
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(res["outs"], args.dump_outputs)
    adj, x = res["adj"], res["x"]
    st = res["stats"]
    phase_ms = res["phase_ms"]
    slabs = st["slabs"]
    M_rank = st["candidates_scored"]

    # ---- multi-GPU self-check: the merged lists == the single-GPU lists, bit for bit ----
    verified = None
    if world > 1 and not args.no_extras:
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        if rank == 0:
            single = wl.step(adj, x, distributed=False)
            ok = all(torch.equal(a, b) for a, b in zip(single, res["outs"]))
            flag.fill_(1 if ok else 2)
            del single
        dist.broadcast(flag, 0)
        verified = bool(int(flag.item()) == 1)

    # ---- the other BASELINE shapes, same product call, same N (strong scaling) ----
    shapes = {}
    if args.workload == "ppa" and not args.no_extras and args.owners_frac >= 1.0:
        for nm in ("ddi", "collab"):
            w2 = Workload(nm, args, dev, world, pin=False)
            r2 = measure(w2, 5, 3, rank, world, e2e_steps=0)
            ok2 = None
            if world > 1:
                flag = torch.zeros(1, dtype=torch.int32, device=dev)
                if rank == 0:
                    single = w2.step(r2["adj"], r2["x"], distributed=False)
                    flag.fill_(1 if all(torch.equal(a, b) for a, b in zip(single, r2["outs"])) else 2)
                dist.broadcast(flag, 0)
                ok2 = bool(int(flag.item()) == 1)
            shapes[nm] = {"value": r2["total_pairs"] / (r2["ms_step"] * 1e-3), "unit": "pairs/s", "ms_per_step": r2["ms_step"],
                          "candidates": r2["total_pairs"], "k": w2.k, "n": w2.n, "nnz": int(w2.h_col.numel()),
                          "phase_ms_rank0": r2["phase_ms"], "prefilter": r2["stats"].get("prefilter"),
                          "multi_gpu_verified": ok2, "steps": 5, "warmup": 3}
            del w2, r2
            torch.cuda.empty_cache()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        tc_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "measured (MEASURED_PEAKS.json, sustained bf16 / copy bandwidth)" if peaks else "fallback (B200_PROFILING.md)"
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload, {})
        except Exception:
            pass

        def roof_entry(kernel, bound, work, ms, launches_, tkey, note=None, extra=None):
            """work = algorithmic bytes / flops of ALL launches of the step on this rank; ms = their summed time."""
            peak = hbm_peak if bound == "hbm" else tc_peak
            ach = work / (ms * 1e-3) / (1e9 if bound == "hbm" else 1e12) if ms > 0 else 0.0
            e = {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak,
                 "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": ach / peak,
                 "traffic": traffic.get(tkey), "peak_source": peak_src,
                 ("algorithmic_bytes_per_launch" if bound == "hbm" else "algorithmic_flops_per_launch"): work / max(launches_, 1),
                 "ms_per_launch": ms / max(launches_, 1), "launches_per_step": launches_}
            if note:
                e["note"] = note
            if extra:
                e.update(extra)
            return e

        # algorithmic work of this rank's owner range (SURVEY §8d)
        lo_o, hi_o = st["owners"]
        deg = adj.degree().long()
        work2 = candidates.two_path_work(adj)
        twopaths = int(work2[lo_o:hi_o].sum().item())
        weighted = adj.val is not None
        # the fused K6+K3 kernel walks the owners' 2-paths twice (mark, score): 2 x 4 B per 2-path (+ 4 B value when
        # weighted); per candidate the padded slot (u 4 B, fixed-point sum 8 B zero + 8 B RED) and the compaction
        # (12 B read, 12 B written: u, v, score)
        fused_bytes = (12 if weighted else 8) * twopaths + 44 * M_rank
        # SURVEY's pair-by-pair figure 4(d_u+d_v)+12 for the same candidates: sum over owners v of
        # [#cand(v) * d_v + sum of d_u over its candidates]; the second term is bounded by the 2-path walk and is
        # sampled on the first slab instead of being enumerated again
        mlp_flops = M_rank * (2 * H * H * (L - 1) + 3 * H)
        nnz_hat = int(wl.h_col.numel()) + n
        spmm_bytes = 4 * (n + 1) + 8 * nnz_hat + 4 * H * nnz_hat + 4 * n * H          # gather model, per layer, whole graph
        fused_key = "enum_score" if "enum_score" in phase_ms else "enum"
        n_models = 2
        roofs = {}
        if "mlp" in phase_ms:
            arm = wl.mlp_arm
            roofs["mlp"] = roof_entry(
                "linkpred_fp32_kernel (K2 fp32 arm, FFMA-bound)" if arm == "fp32" else "linkpred_tc3_kernel (K2 tcgen05, cta_group::2)",
                "tensor", mlp_flops, phase_ms["mlp"], slabs, "linkpred_tc3",
                "phase = the kernel (+ bf16 table and weight images, built once per step); flops = 2H^2(L-1)+3H per candidate")
        roofs["enum_score"] = roof_entry(
            "twohop_score_kernel + twohop_compact_kernel (K6+K3 fused, one pass)", "hbm", fused_bytes, phase_ms.get(fused_key, 0.0),
            slabs, "twohop_onepass",
            "bytes = the kernel's OWN traffic model: 8 B per 2-path (two walks; 12 B weighted) + 44 B per candidate "
            "(padded slot, fixed-point accumulator, compaction); latency / L2-atomic bound, not HBM bound")
        roofs["topk"] = roof_entry(
            "threshold_count/write (K4b) + topk_hist/count/write (K4), both models", "hbm",
            n_models * (4 * M_rank + 12 * k * slabs), phase_ms.get("topk", 0.0), n_models * slabs, "topk",
            "algorithmic bytes = one read of the slab's scores + 12 B per kept row per select (SURVEY 8d); K4b reads the "
            "scores twice, K4 runs over the survivors only; the phase includes the final sorts")
        dom = max(roofs, key=lambda p: roofs[p]["ms_per_launch"] * roofs[p]["launches_per_step"])
        roof = roofs[dom]
        other = [roofs[p] for p in roofs if p != dom]
        if res["spmm_ms"]:
            per_step = len(res["spmm_ms"]) // args.steps
            frac_rows = 1.0 / world
            other.append(roof_entry("spmm_csr_kernel (K1)", "hbm", spmm_bytes * frac_rows * per_step,
                                    float(np.sum(res["spmm_ms"])) / args.steps, per_step, "spmm_csr",
                                    "gather model 4(n+1)+8nnz+4F*nnz+4nF (SURVEY 8d) of this rank's row shard; rows that hit "
                                    "in L2 let it exceed the HBM peak"))
        value = res["total_pairs"] / (res["ms_step"] * 1e-3)
        line = {
            "metric": "candidate pairs scored/sec (CN/AA + GCN+LinkPredictor filter step)",
            "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": res["ms_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None,
            "dtype": {"prefilter": "f16-operand tcgen05 prefilter (f32 accumulate) + f32 re-score: f32-exact lists", "f16": "f16(mlp operands)/f32",
                      "fp32": "f32"}[wl.mlp_arm],
            "data": "synthetic graph (seeded Chung-Lu of the named shape); seeded random weights, LinkPredictor at a "
                    "trained model's score spread (He-uniform hidden layers, output layer rescaled to logit mean -2 / std 2)",
            "config": {"workload": workload_text(args.workload, k, args.slab_pairs), "model_scale": wl.model_scale,
                       "n": n, "nnz": int(wl.h_col.numel()), "graph_total_candidates": int(res["total_pairs"]),
                       "candidates_rank0": int(M_rank), "slabs_rank0": slabs, "owners_rank0": st["owners"],
                       "owners_frac": args.owners_frac, "gnn": f"gcn L={L} H={H} F_in={H + wl.host['feat']}",
                       "mlp_arm": wl.mlp_arm, "k": k, "slab_pairs": args.slab_pairs, "pushdown": not args.no_pushdown,
                       "parallelism": f"owner ranges by 2-path work x{world}; embeddings row-sharded + all-gathered; "
                                      "k-th score exchange + list merge" if world > 1 else "single GPU",
                       "l2": "inputs larger than L2 (CSR 170 MB + embeddings 590 MB + >= 1 GB of pairs per slab); no flush needed"
                       if (n * H * 4) > 200e6 else "graph + embeddings smaller than L2: effective (cache-resident) bandwidth"},
            "detail": {"phase_ms_rank0": phase_ms,
                       "pairs_per_s_by_phase_rank0": {p: M_rank / (v * 1e-3) for p, v in phase_ms.items() if v > 0 and p in ("enum_score", "enum", "mlp", "topk")},
                       "prefilter": st.get("prefilter"), "prefilter_fallback": st.get("prefilter_fallback"),
                       "topk_identical_to_fp32": (wl.mlp_arm == "prefilter" and "prefilter_fallback" not in st) or wl.mlp_arm == "fp32",
                       "pushdown_survivors_rank0": st.get("pushdown_survivors"),
                       "multi_gpu_verified": verified, "shapes": shapes},
            "roofline": roof,
            "roofline_other": other,
            "e2e": res["e2e"],
            "gpu_launches": res["launches"],
            "clocks": clocks,
        }
        if world == 1 and not args.no_extras:
            try:
                line["detail"]["library_baseline"] = library_baseline(wl, adj, x, k)
                lb = line["detail"]["library_baseline"]
                roofs_mlp = roofs.get("mlp")
                if roofs_mlp:
                    lb["eps_step_mlp_pairs_per_s"] = M_rank / (phase_ms["mlp"] * 1e-3)
            except Exception as exc:
                line["detail"]["library_baseline"] = {"failed": repr(exc)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                embed_s = cpu_setup(wl.host)
                owners = cpu_pick_owners(wl.host, args.cpu_seconds / 2)
                r = cpu_reference_pass(wl.host, owners, args.cpu_seconds, os.cpu_count())
                line["cpu_baseline"] = {
                    "value": r["pairs"] / r["total"], "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
                    "sample": f"{r['pairs']} candidates of owners [{owners[0]},{owners[1]}): scipy A@A enumeration, "
                              f"scipy AA (adamic_utils.AA formulation) x{os.cpu_count()} procs, torch-CPU fp32 LinkPredictor, "
                              f"torch sort; GCN embeddings computed once ({embed_s:.1f}s, not counted)",
                    "breakdown_s": {kk: r[kk] for kk in ("t_cand", "t_aa", "t_mlp", "t_sort")}}
            except Exception as exc:  # the baseline must never take the bench line down
                line["cpu_baseline"] = {"value": None, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
                                        "sample": f"failed: {exc!r}"}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
