"""The filter step: score every 2-hop non-edge with the filter model, keep the k best.

B200-native restatement of the body of /root/reference/filter.py:92-166:

  reference                                         here
  ---------                                         ----
  A2 = adj@adj on one CPU thread, scipy masking     K6 one-pass bitmap enumeration per owner slab
  for batch in DataLoader(range(N), B):             one K2 / K3 launch per slab
      model(x, edges, adj)   # GNN re-run per batch   embeddings computed once (LinkGNN.embed)
      cat([edges.t(), score]).cpu()                   scores stay on the device
  all_scores[:,2].sort(descending=True)  # CPU      K4 radix-select + K4b threshold push-down + one stable sort
  torch.save([N,3])                                 [k,3] float32 (k = N keeps the full list)

Slabs: owners are cut into contiguous ranges whose candidate BOUND is at most ``slab_pairs``
(``iter_slabs``); every slab is folded into the running proposal set (``RunningTopK``) — positions in
the concatenation of the slabs preserve the global candidate order, so the final stable sort equals a
single global stable sort.  Multi-GPU: each rank takes a contiguous owner range
(parallel.partition_by_work), the GNN embeddings are computed row-sharded and all-gathered
(models._ConvStack.embed_rows) and the per-rank lists are merged after an exchange of the global k-th
score (parallel.merge_topk).
"""
from __future__ import annotations

from typing import Iterator, Optional, Tuple

import torch

from . import adamic_utils, candidates, ops, parallel
from .graph import SparseAdj, add_edges
from .models import GNN_MODELS, LinkGNN


def score_edges(model_name: str, model, x, adj: SparseAdj, edges: torch.Tensor,
                grouped_by_v: bool = True, ra_adj: Optional[SparseAdj] = None) -> torch.Tensor:
    """Scores of ``edges [2,M]`` under the filter model (/root/reference/filter.py:113-142)."""
    if model_name in GNN_MODELS:
        assert isinstance(model, LinkGNN)
        h = model.embed(x, adj)
        return model.linkpred.score_pairs(h, edges)
    if model_name in ("simple", "adamic"):
        model.grouped_by_v = grouped_by_v
        return model(x, edges, adj)
    if model_name == "adamic_ogb":
        return adamic_utils.AA(adamic_utils.get_A(adj, adj.n), edges, grouped_by_v=grouped_by_v)[0]
    if model_name == "resource_allocation":
        A = ra_adj if ra_adj is not None else adj
        return ops.cn_aa(A, edges, A.ra_weights(), use_values=True, grouped_by_v=grouped_by_v)
    raise ValueError(f"model {model_name!r} is not a filter model on this path")


def same_structure(a: SparseAdj, b: SparseAdj) -> bool:
    """True when two unweighted adjacencies hold the same entries (e.g. the RA graph rebuilt from
    the raw train split, filter.py:130-139, when no proposal edges were added)."""
    return (a is b) or (a.val is None and b.val is None and a.n == b.n and a.nnz == b.nnz
                        and bool(torch.equal(a.rowptr, b.rowptr)) and bool(torch.equal(a.col, b.col)))


def heuristic_table(model_name: str, adj: SparseAdj, ra_adj: Optional[SparseAdj] = None):
    """(graph, weight table, sigmoid, use_values) of a heuristic filter model when it can take the fused
    enumerate+score kernel (K6+K3, candidates.two_hop_scored): the scoring graph IS the graph whose 2-hop
    neighbourhood defines the candidates and, if weighted (collab), its values are bitwise symmetric.
    ``None`` otherwise (RA on a rebuilt multigraph) -> two_hop + ops.cn_aa."""
    if not candidates.values_symmetric(adj):
        return None
    if model_name == "simple":
        return adj, None, False, True                        # models.py:536-542 (weighted on collab)
    if model_name == "adamic":
        return adj, adj.adamic_weights(), True, False        # models.py:544-554 (indices only)
    if model_name == "adamic_ogb":
        return adj, adj.aa_ogb_weights(), False, True        # adamic_utils.py:13-25 (values of A)
    if model_name == "resource_allocation" and adj.val is None and (ra_adj is None or same_structure(ra_adj, adj)):
        return adj, adj.ra_weights(), False, True            # train_and_eval.py:195-216
    return None


def ra_graph_from_train_edges(train_edges: torch.Tensor, num_nodes: int) -> SparseAdj:
    """filter.py:130-139: A rebuilt from the raw train split, both directions, duplicate pairs
    SUMMED into integer weights (scipy csr_matrix constructor semantics)."""
    e = train_edges.reshape(-1, 2).long()
    both = torch.cat([e, e.flip(1)], 0).t()
    n = int(num_nodes)
    key = both[0] * n + both[1]
    ukey, cnt = torch.unique(key, sorted=True, return_counts=True)
    row = torch.div(ukey, n, rounding_mode="floor")
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=e.device)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    val = cnt.float()
    return SparseAdj(rowptr.int(), (ukey - row * n).int(), None if bool((cnt == 1).all()) else val, n)


def iter_slabs(adj: SparseAdj, v_lo: int, v_hi: int, slab_pairs: int) -> Iterator[Tuple[int, int, int]]:
    """Yield (lo, hi, cap) owner ranges whose candidate count is at most ``cap <= slab_pairs``
    (a single owner whose bound exceeds that gets a slab of its own).  ``cap`` is the sum of the
    per-owner upper bounds (candidates.owner_bounds) — it sizes the one-pass kernel's outputs, so no
    count pass over the graph is needed to plan the slabs."""
    if v_hi <= v_lo:
        return
    cs = torch.cumsum(candidates.owner_bounds(adj)[v_lo:v_hi], 0).cpu()
    lo = 0
    n_own = v_hi - v_lo
    base = 0
    while lo < n_own:
        hi = int(torch.searchsorted(cs, torch.tensor(base + slab_pairs), right=True).item())
        hi = max(hi, lo + 1)
        hi = min(hi, n_own)
        end = int(cs[hi - 1])
        yield v_lo + lo, v_lo + hi, end - base
        base = end
        lo = hi


def owner_cost(adj: SparseAdj, jobs) -> torch.Tensor:
    """Per-owner cost estimate that the multi-GPU owner ranges are balanced on.  Enumeration (K6) costs the owner's
    2-paths; scoring a candidate with a GNN filter model (K2) costs ~8 x a 2-path visit (measured on the ppa shape:
    0.218 ns per candidate against 0.029 ns per 2-path), and the candidate count is bounded by the owner's slot size
    (candidates.owner_bounds).  Balancing on 2-paths alone left the ranks with few hubs 5 % more candidates and the
    others waiting at the merge (N = 4: 33 ms of a 615 ms step)."""
    work = candidates.two_path_work(adj).double()
    if any((j.name if hasattr(j, "name") else j[0]) in GNN_MODELS for j in jobs):
        work = work + 8.0 * candidates.owner_bounds(adj).double()
    return work


class PrefilterToleranceError(RuntimeError):
    """The fp16 tensor-core scores left their stated tolerance band around the fp32 scores; the
    caller re-runs on the fp32 arm (``filter_topk`` does)."""


# Tolerance of the prefilter.  How far the tensor-core scores (fp16 operands) sit from the fp32 scores depends
# on the model: on benign weights |s16 - s32| <= ~2e-4 (tests/test_gpu_mlp_tc.py), on the bench's deliberately
# ill-conditioned model (zero hidden biases, output layer scaled 470x: logits are differences of large terms)
# ~1e-3.  The prefilter therefore CALIBRATES its tolerance per job — PREFILTER_SAFETY x the largest deviation seen
# on ~2.6e5 candidates of the first slab (its best-scoring ones and a strided sample), capped by PREFILTER_TOL —
# and VERIFIES it on the final pool (every candidate next to the boundary is re-scored in fp32 anyway); see
# ``filter_topk_multi``.  A factor 2 over the maximum of 2.6e5 samples: for rounding noise (sums of ~10^5 independent
# roundings) the maximum over 2.6e5 draws sits near 4.6 sigma, so 2x is ~9 sigma — out of reach of 10^10 candidates.
PREFILTER_TOL = 1e-2                   # ceiling: beyond this the arm is not a usable prefilter
PREFILTER_SAFETY = 2.0
PREFILTER_TOL_FLOOR = 2e-5            # below this the sample statistic is the fp32 arm's own rounding noise (its error vs fp64 is ~1e-5)
PREFILTER_CAL_SAMPLE = 1 << 17        # top-scoring + strided candidates of the first slab, each
PREFILTER_POOL_CAP = 1 << 27          # pool entries beyond which the band is called too wide (-> fp32 arm)


class _Phases:
    """CUDA-event stop-watch for the phases of the filter step (bench.py reads ``stats['phase_ms']``)."""

    def __init__(self, on: bool):
        self.on, self.marks = on, []
        self.mark(None)

    def mark(self, name):
        if self.on:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.marks.append((name, e))

    def totals(self):
        out = {}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out


class RunningTopK:
    """The proposal set while owner slabs stream by, as SoA (u, v int32, score fp32) in CANDIDATE ORDER
    (= the reference's column-major order, which is the tie rule of the final sort).

    Exact mode (``margin=None``): the state is exactly the k best candidates seen so far.  Until the list
    is full a slab is folded in by K4's radix select over (state ++ slab); from then on K4b pushes the
    k-th score down into the slab — only elements STRICTLY better survive one ordered compaction (a slab
    tie at the k-th score comes later in candidate order than the list's own ties, so it can never
    displace one) — and the select runs over (state ++ survivors).  ``result`` sorts once (stable, score
    descending).  Equal to one global stable sort of all candidates, bit for bit (tests/test_gpu_topk.py).

    Band mode (``margin > 0``, the tensor-core prefilter): the state is the POOL of every candidate whose score
    is >= (k-th best score seen so far) - margin; the k-th score only rises, so nothing dropped could
    re-enter.  ``pool`` returns it for the fp32 re-scoring (``filter_topk_multi``)."""

    def __init__(self, k: Optional[int], margin: Optional[float] = None, pushdown: bool = True):
        self.k = k                      # None: keep every candidate, like the reference
        self.margin = margin
        self.pushdown = pushdown        # False: K4 select over every slab (the pre-K4b path, kept for A/B)
        self.u = self.v = self.score = None
        self.kth_key = None             # order key of the current k-th score (device), once the list is full
        self.seen = 0
        self.survivors = 0              # slab elements that passed the push-down (statistic)
        self._pending = 0
        self.overflow = False           # band mode: the pool outgrew PREFILTER_POOL_CAP (band too wide)

    @property
    def size(self) -> int:
        return 0 if self.score is None else self.score.numel()

    def _append(self, pu, pv, score, clone=False):
        if self.score is None:
            self.u, self.v, self.score = (pu.clone(), pv.clone(), score.clone()) if clone else (pu, pv, score)
        else:
            self.u, self.v = torch.cat([self.u, pu]), torch.cat([self.v, pv])
            self.score = torch.cat([self.score, score])

    def rethreshold(self) -> None:
        """Band mode: recompute the k-th key over the pool and drop what fell out of the band."""
        if self.margin is None or self.k is None or self.size < self.k:
            return
        self.kth_key = ops.kth_key(self.score, self.k)
        self.u, self.v, self.score = ops.threshold_compact(self.score, torch.stack([self.u, self.v]), self.kth_key,
                                                           self.margin, inclusive=True)
        self._pending = 0
        if self.size > max(PREFILTER_POOL_CAP, 4 * self.k):
            # nearly every candidate lies inside the band: the prefilter cannot prune this model's scores.
            # Keep the state bounded and let the caller fall back (decided collectively at the end).
            self.overflow = True
            self.u, self.v, self.score = self.u[:self.k].clone(), self.v[:self.k].clone(), self.score[:self.k].clone()

    def update(self, edges: torch.Tensor, score: torch.Tensor) -> None:
        M = score.numel()
        if M == 0:
            return
        self.seen += M
        if self.overflow:
            return
        pu, pv = ops._pairs(edges)
        score = score.contiguous().float()
        have = self.size
        band = self.margin is not None
        if self.k is None or have + M <= self.k:             # everything survives: plain append
            self._append(pu, pv, score, clone=True)
            if band and self.k is not None and self.size == self.k:
                self.rethreshold()
            return
        if self.kth_key is not None and (self.pushdown or band):
            # the list is full: push its k-th score down into the slab (K4b)
            su, sv, ss = ops.threshold_compact(score, edges, self.kth_key, self.margin or 0.0, inclusive=band)
            c = ss.numel()
            self.survivors += c
            if c == 0:
                return
            if band:
                self._append(su, sv, ss)
                self._pending += c
                if self._pending * 8 >= self.k:
                    self.rethreshold()
                return
            idx, sc, self.kth_key = ops.topk_select2(self.score, ss, self.k, want_kth_key=True)
            self.u, self.v = ops.gather_pairs2((self.u, self.v), (su, sv), idx)
            self.score = sc
            return
        if band:                                             # the slab that fills the pool
            self._append(pu, pv, score, clone=True)
            self.rethreshold()
            return
        # exact mode, list not yet full (or push-down switched off): K4 select over (list ++ slab)
        kk = min(self.k, have + M)
        prune = self.kth_key if (have == kk and self.kth_key is not None) else None
        idx, sc, kth = ops.topk_select2(self.score, score, kk, prune_key=prune, want_kth_key=True)
        self.u, self.v = ops.gather_pairs2(None if self.score is None else (self.u, self.v), (pu, pv), idx)
        self.score = sc
        self.kth_key = kth if kk == self.k else None

    def pool(self):
        """Band mode: (edges int32 [2,P], score fp32 [P]) of the final pool, candidate order."""
        self.rethreshold()
        if self.score is None:
            return None, None
        return torch.stack([self.u, self.v]), self.score

    def result(self, device=None) -> torch.Tensor:
        if self.score is None or self.score.numel() == 0:
            return torch.empty((0, 3), dtype=torch.float32, device=device)
        k = self.score.numel() if self.k is None else min(self.k, self.score.numel())
        return ops.topk_edges(torch.stack([self.u, self.v]), self.score, k)


class FilterJob:
    """One filter model of a ``filter_topk_multi`` call: ``name`` in models.SUPPORTED_MODELS, the model
    object (``LinkGNN`` / ``CommonNeighborsPredictor``), optionally the rebuilt RA graph (filter.py:130-139)
    and, for the GNN models, the K2 arm:

      ``"fp32"``       reference arithmetic on FFMA for every candidate;
      ``"f16"``        the tcgen05 arm alone (fp16 operands; alias "bf16", its round-1 name) — list approximately
                       the fp32 one;
      ``"prefilter"``  the tcgen05 arm as a PREFILTER and the fp32 arm on its survivors: the fp32 arm's
                       exact proposal list at tensor-core speed (default)."""

    def __init__(self, name: str, model, ra_adj: Optional[SparseAdj] = None, precision: Optional[str] = None):
        self.name, self.model, self.ra_adj = name, model, ra_adj
        if precision is None and name in GNN_MODELS:
            precision = getattr(model.linkpred, "precision", None) or "prefilter"
        self.precision = precision


def tc_arm_supported(model) -> bool:
    """Shapes the tcgen05 arm is built for (csrc/linkpred_tc.cu): >= 2 layers, H in {64, 128, 256}, and at
    H = 256 at most 3 layers (the hidden layers' weights stay resident in shared memory)."""
    lp = model.linkpred
    H, L = lp.lins[0].in_features, len(lp.lins)
    return L >= 2 and H in (64, 128, 256) and not (H == 256 and L > 3)


@torch.no_grad()
def filter_topk_multi(jobs, x, adj: SparseAdj, k: Optional[int] = None, slab_pairs: int = 1 << 27,
                      distributed: bool = False, stats: Optional[dict] = None, pushdown: bool = True,
                      owners: Optional[Tuple[int, int]] = None, per_node: Optional[int] = None):
    """``_filter_multi`` (see there) with the prefilter's safety net: when a job's tensor-core scores leave the
    calibrated tolerance, or its band cannot prune, the call is repeated with that job on the fp32 arm."""
    jobs = [j if isinstance(j, FilterJob) else FilterJob(*j) for j in jobs]
    try:
        return _filter_multi(jobs, x, adj, k, slab_pairs, distributed, stats, pushdown, owners, per_node)
    except PrefilterToleranceError as exc:
        import warnings
        warnings.warn(f"{exc}; re-running the filter step on the fp32 arm")
        for j in jobs:
            if j.precision == "prefilter":
                j.precision = "fp32"
        if stats is not None:
            stats["prefilter_fallback"] = str(exc)
        return _filter_multi(jobs, x, adj, k, slab_pairs, distributed, stats, pushdown, owners, per_node)


@torch.no_grad()
def _filter_multi(jobs, x, adj: SparseAdj, k: Optional[int] = None, slab_pairs: int = 1 << 27,
                  distributed: bool = False, stats: Optional[dict] = None, pushdown: bool = True,
                  owners: Optional[Tuple[int, int]] = None, per_node: Optional[int] = None):
    """The filter step for several filter models over ONE enumeration of the 2-hop candidates: a list of
    sorted proposal lists (float32 ``[k,3]`` rows (u, v, score) on the device; score descending, ties by
    the reference's candidate order), one per job.  ``k=None`` keeps every candidate like the reference.

    GNN jobs with ``precision="prefilter"``: every candidate is scored by the tcgen05 arm (fp16 operands)
    and the running pool keeps all candidates whose tensor-core score s16 is within ``2 * tol`` of the running k-th
    best such score T16.  With |s16 - s32| <= tol for every pair, the k candidates with the best s16 all
    have s32 >= T16 - tol, so a candidate with s16 < T16 - 2 tol (hence s32 < T16 - tol) cannot be among the
    k best by s32: the pool contains the fp32 arm's top-k.  The pool (~k candidates) is then re-scored by
    the fp32 arm and sorted — the result is the fp32 arm's list bit for bit.  ``tol`` is calibrated on the
    first slab (``_calibrate``: PREFILTER_SAFETY x the largest deviation over ~2.6e5 candidates, at most the
    kernel's stated PREFILTER_TOL) and checked again on the pool — millions of pairs next to the boundary;
    a violation, or a band so wide that it cannot prune, raises ``PrefilterToleranceError``
    (``filter_topk_multi`` then re-runs the call with the job on the fp32 arm).

    ``owners=(lo, hi)`` restricts the candidates to those owned by v in [lo, hi) (a sample of the job).

    ``per_node=m`` (per-node proposal budgets): only the m best candidates (u, v) of every owner v — score
    descending, ties by u ascending — take part; the list is then ordered by the same rule and cut to k (``k=None``
    keeps every owner's m).  The budget is per v, the second column of a row: keeping (u, v) in v's list says nothing
    about (v, u) in u's list (``add_edges`` symmetrises the graph, so either adds the undirected edge).  An owner's
    candidates are contiguous inside one slab, so K4c (``ops.segment_topk``) selects them slab by slab and its
    survivors, still in candidate order, feed the unchanged running top-k.  With m >= every owner's candidate count
    the result is the global list.  GNN jobs on the prefilter: per slab, the band select keeps every candidate whose
    tensor-core score s16 is >= (its owner's m-th best s16) - 2 tol; the pool is re-scored in fp32, the tolerance
    verified on it, and the exact per-owner select runs on the fp32 scores.  Sound because, with |s16 - s32| <= tol
    for every pair, an owner's j-th best s32 is >= its j-th best s16 - tol for every j <= m (its j best candidates by
    s16 all have s32 >= that value): a candidate with s16 < S16_m - 2 tol has s32 < S16_m - tol <= S32_m, strictly
    below the owner's m-th best fp32 score, so it cannot be among the owner's exact m best.  No band is exchanged or
    pruned across owners (each rank's per-owner lists are complete), and the prefilter stays on with ``k=None``:
    the n * m budget bounds the pool."""
    rank, world = parallel.world_info() if distributed else (0, 1)
    if per_node is not None and int(per_node) < 1:
        raise ValueError(f"per_node must be >= 1 (got {per_node})")
    m = None if per_node is None else int(per_node)
    if world > 1 and k is None:
        raise ValueError("distributed filter needs a proposal size k")
    jobs = [j if isinstance(j, FilterJob) else FilterJob(*j) for j in jobs]
    ph = _Phases(stats is not None and bool(stats.get("time_phases")))
    o_lo, o_hi = (0, adj.n) if owners is None else (max(int(owners[0]), 0), min(int(owners[1]), adj.n))
    v_lo, v_hi = o_lo, o_hi
    if world > 1:
        bounds = parallel.partition_by_work(owner_cost(adj, jobs)[o_lo:o_hi], world)
        v_lo, v_hi = o_lo + bounds[rank], o_lo + bounds[rank + 1]
    # per job: scoring plan + running proposal set
    plans = []
    fused_job = None
    for j in jobs:
        if j.name in GNN_MODELS:
            assert isinstance(j.model, LinkGNN)
            prec = j.precision
            if prec in ("prefilter", "f16", "bf16", "tc") and not tc_arm_supported(j.model):
                prec = "fp32"                                # shapes the tcgen05 arm is not built for (H=300)
            if prec == "prefilter" and k is None and m is None:
                prec = "fp32"                                # keeping every candidate: nothing to prefilter
            h = j.model.embed(x, adj, distributed=world > 1)
            band = prec == "prefilter" and m is None
            plans.append(dict(kind="gnn", prec=prec, h=h, ctx=None if prec == "fp32" else j.model.linkpred.tc_context(h),
                              tol=None, cal=None, pn_kept=0,
                              pool=dict(e=[], s=[], cnt=[], size=0, owners=0, budget=None, overflow=False)
                              if (prec == "prefilter" and m is not None) else None,
                              run=RunningTopK(k, 2.0 * PREFILTER_TOL if band else None, pushdown)))
        else:
            table = heuristic_table(j.name, adj, j.ra_adj)
            if table is not None and fused_job is None:
                fused_job = len(plans)
            plans.append(dict(kind="heuristic", table=table, pn_kept=0, pool=None, run=RunningTopK(k, None, pushdown)))
    ph.mark("embed")
    n_slabs = 0
    n_cand = 0
    for lo, hi, cap in iter_slabs(adj, v_lo, v_hi, slab_pairs):
        n_slabs += 1
        scores = {}
        offsets = None
        if fused_job is not None:
            # CN / AA / RA are the values of A@A: one walk over the owners' 2-paths yields the
            # candidates and their scores together (bit-identical to scoring the pairs with K3)
            t = plans[fused_job]["table"]
            r = candidates.two_hop_scored(t[0], t[1], lo, hi, sigmoid=t[2], cap=cap, use_values=t[3],
                                          want_offsets=m is not None)
            edges, scores[fused_job] = r[0], r[1]
            offsets = r[2] if m is not None else None
            ph.mark("enum_score")
        else:
            r = candidates.two_hop(adj, lo, hi, cap=cap, want_offsets=m is not None)
            edges, offsets = r if m is not None else (r, None)
            ph.mark("enum")
        if edges.shape[1] == 0:
            continue
        n_cand += edges.shape[1]
        for i, (j, p) in enumerate(zip(jobs, plans)):
            if i in scores:
                continue
            if p["kind"] == "gnn":
                scores[i] = (j.model.linkpred.score_pairs(p["h"], edges, "fp32") if p["prec"] == "fp32"
                             else p["ctx"].score(edges))
                ph.mark("mlp")
                if p["prec"] == "prefilter" and p["tol"] is None:
                    _calibrate(j.model, p, edges, scores[i], world)
                    ph.mark("calibrate")
            else:
                scores[i] = score_edges(j.name, j.model, x, adj, edges, True, j.ra_adj)
                ph.mark("score")
        if m is None:
            for i, p in enumerate(plans):
                p["run"].update(edges, scores[i])
            ph.mark("topk")
        else:
            _per_node_slab(plans, edges, scores, offsets, m, hi - lo, ph)
        del edges, scores, offsets
    out = []
    for j, p in zip(jobs, plans):
        run = p["run"]
        if p["kind"] == "gnn" and p["prec"] == "prefilter" and p["tol"] is None:
            _calibrate(j.model, p, None, None, world)        # this rank owned no candidates: still one collective
        if p["pool"] is not None:
            res, info = _rescore_pool_per_node(j.model, p["h"], p["pool"], k, m, world, p["tol"], p["cal"])
            if stats is not None:
                stats.setdefault("prefilter", {})[j.name] = info
            ph.mark("rescore")
        elif p["kind"] == "gnn" and p["prec"] == "prefilter":
            res, info = _rescore_pool(j.model, p["h"], run, k, world, p["tol"], p["cal"])
            if stats is not None:
                stats.setdefault("prefilter", {})[j.name] = info
            ph.mark("rescore")
        else:
            res = run.result(adj.device)
            ph.mark("topk")
        if world > 1:
            res = parallel.merge_topk(res, k)
            ph.mark("merge")
        out.append(res)
    if stats is not None:
        stats["candidates_scored"] = (plans[0]["run"].seen if m is None else n_cand) if plans else 0
        if m is not None:
            stats["per_node"] = dict(m=m, survivors=[p["pn_kept"] for p in plans])
        stats["slabs"] = n_slabs
        stats["owners"] = [v_lo, v_hi]
        stats["pushdown_survivors"] = [p["run"].survivors for p in plans]
        if ph.on:
            torch.cuda.synchronize()
            stats["phase_ms"] = ph.totals()
    return out


def _per_node_slab(plans, edges, scores, offsets, m: int, n_owners: int, ph) -> None:
    """Per-node mode, one slab: K4c per job — the exact per-owner top-m, or for a prefilter job the band of every
    owner's m-th tensor-core score, appended to the job's pool — then the exact survivors into the running top-k."""
    kept = []
    for i, p in enumerate(plans):
        pool = p["pool"]
        if pool is not None and pool["overflow"]:
            kept.append(None)
            continue
        margin = None if pool is None else 2.0 * p["tol"]
        kept.append(ops.segment_topk(scores[i], edges, offsets, m, margin=margin))
        p["pn_kept"] += kept[-1][1].numel()
        if pool is not None:
            b = torch.clamp(offsets[1:] - offsets[:-1], max=m).sum()     # this slab's exact budget, on the device
            pool["budget"] = b if pool["budget"] is None else pool["budget"] + b
    ph.mark("per_node")
    for p, kp in zip(plans, kept):
        if kp is None:
            continue
        e, s, off = kp
        pool = p["pool"]
        if pool is None:
            p["run"].update(e, s)
            continue
        pool["e"].append(e)
        pool["s"].append(s)
        pool["cnt"].append(off[1:] - off[:-1])
        pool["size"] += s.numel()
        pool["owners"] += n_owners
        if pool["size"] > max(PREFILTER_POOL_CAP, 4 * m * pool["owners"]):
            # the band holds more than 4x every owner's budget: it cannot prune (decided collectively at the end)
            pool.update(e=[], s=[], cnt=[], overflow=True)
    ph.mark("topk")


def _rescore_pool_per_node(model, h, pool, k: Optional[int], m: int, world: int, tol: float, cal=None):
    """Per-node prefilter epilogue: fp32 scores of the pool, tolerance check on it, exact per-owner top-m of the fp32
    scores (K4c over the pool's owner segments), then the first k rows by score.  No exchange between ranks but the
    decision flags: owners are partitioned, so every rank's pool holds its owners' complete bands."""
    dev = h.device
    margin = 2.0 * tol
    P = pool["size"] if not pool["overflow"] else 0
    budget = 0 if pool["budget"] is None else int(pool["budget"].item())
    overflow = pool["overflow"] or P > max(PREFILTER_POOL_CAP, 4 * budget)
    info = dict(m=int(m), k=None if k is None else int(k), pool=int(pool["size"]), budget=budget, tol=tol,
                margin=margin, tol_ceiling=PREFILTER_TOL, calibration=cal, band_occupancy=float(P) / max(budget, 1))
    res = torch.empty((0, 3), dtype=torch.float32, device=dev)
    flags = torch.zeros(2, dtype=torch.float32, device=dev)       # [max deviation on the pool, pool overflow]
    if P and not overflow:
        edges, s16, cnt = torch.cat(pool["e"], 1), torch.cat(pool["s"]), torch.cat(pool["cnt"])
        s32 = model.linkpred.score_pairs(h, edges, "fp32")
        flags[0] = (s32 - s16).abs().max()
        off = torch.zeros(cnt.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(cnt, 0, out=off[1:])
        e, s, _ = ops.segment_topk(s32, edges, off, m)
        res = ops.topk_edges(e, s, s.numel() if k is None else min(int(k), s.numel()))
    pool.update(e=[], s=[], cnt=[])
    flags[1] = 1.0 if overflow else 0.0
    if world > 1:                                            # every rank must take the same decision
        torch.distributed.all_reduce(flags, op=torch.distributed.ReduceOp.MAX)
    info["max_abs_dev_tc_vs_fp32"] = float(flags[0].item())
    if float(flags[1].item()) > 0:
        raise PrefilterToleranceError(f"the per-node prefilter band (margin {margin:.2e}) holds more than "
                                      f"{max(PREFILTER_POOL_CAP, 4 * budget)} candidates: this model's scores are too "
                                      "close together for a reduced-precision prefilter")
    if not info["max_abs_dev_tc_vs_fp32"] <= tol:
        raise PrefilterToleranceError(f"tensor-core prefilter scores deviate {info['max_abs_dev_tc_vs_fp32']:.3e} from fp32 "
                                      f"on the pool (> calibrated tolerance {tol:.2e})")
    return res, info


def _calibrate(model, plan, edges, s16, world: int) -> None:
    """Prefilter tolerance of this job: PREFILTER_SAFETY x the largest |s16 - s32| over the best-scoring and a
    strided sample of the first slab's candidates, within [PREFILTER_TOL_FLOOR, PREFILTER_TOL]; the same value
    on every rank (max).  Sets the margin of the job's running pool."""
    h = plan["h"]
    e_cal = torch.zeros(1, dtype=torch.float32, device=h.device)
    n_cal = 0
    if s16 is not None and s16.numel():
        M = s16.numel()
        top = ops.topk(s16, min(PREFILTER_CAL_SAMPLE, M))[0]
        step = max(M // PREFILTER_CAL_SAMPLE, 1)
        idx = torch.cat([top, torch.arange(0, M, step, device=h.device)])
        n_cal = idx.numel()
        s32 = model.linkpred.score_pairs(h, edges[:, idx].contiguous(), "fp32")
        e_cal = (s32 - s16[idx]).abs().max().reshape(1)
    if world > 1:
        torch.distributed.all_reduce(e_cal, op=torch.distributed.ReduceOp.MAX)
    e = float(e_cal.item())
    plan["cal"] = dict(sample=int(n_cal), max_abs_dev=e, safety=PREFILTER_SAFETY)
    plan["tol"] = min(max(PREFILTER_SAFETY * e, PREFILTER_TOL_FLOOR), PREFILTER_TOL)
    plan["run"].margin = 2.0 * plan["tol"]


def _rescore_pool(model, h, run: RunningTopK, k: int, world: int, tol: float, cal=None):
    """Prefilter epilogue: fp32 scores of the pool, tolerance check, exact top-k of the fp32 scores."""
    edges, s16 = run.pool()
    dev = h.device
    margin = 2.0 * tol
    pool_local = 0 if s16 is None else s16.numel()
    if world > 1:
        # the global k-th tensor-core score bounds every rank's pool from below (it is >= each local k-th)
        if s16 is None:
            s16 = torch.empty(0, dtype=torch.float32, device=dev)
            edges = torch.empty((2, 0), dtype=torch.int32, device=dev)
        gkey = parallel.global_kth_key(s16, k)
        u, v, s16 = ops.threshold_compact(s16, edges, gkey, margin, inclusive=True)
        edges = torch.stack([u, v])
    P = 0 if s16 is None else s16.numel()
    info = dict(k=int(k), pool=int(P), pool_before_exchange=int(pool_local), tol=tol, margin=margin,
                tol_ceiling=PREFILTER_TOL, calibration=cal, band_occupancy=float(P) / max(int(k), 1))
    res = torch.empty((0, 3), dtype=torch.float32, device=dev)
    flags = torch.zeros(2, dtype=torch.float32, device=dev)       # [max deviation on the pool, pool overflow]
    if P and not run.overflow:
        s32 = model.linkpred.score_pairs(h, edges, "fp32")
        flags[0] = (s32 - s16).abs().max()
        res = ops.topk_edges(edges, s32, min(int(k), P))
    flags[1] = 1.0 if run.overflow else 0.0
    if world > 1:                                            # every rank must take the same decision
        torch.distributed.all_reduce(flags, op=torch.distributed.ReduceOp.MAX)
    info["max_abs_dev_tc_vs_fp32"] = float(flags[0].item())
    if float(flags[1].item()) > 0:
        raise PrefilterToleranceError(f"the prefilter band (margin {margin:.2e}) holds more than "
                                      f"{max(PREFILTER_POOL_CAP, 4 * int(k))} candidates: this model's scores are too "
                                      "close together for a reduced-precision prefilter")
    if not info["max_abs_dev_tc_vs_fp32"] <= tol:
        raise PrefilterToleranceError(f"tensor-core prefilter scores deviate {info['max_abs_dev_tc_vs_fp32']:.3e} from fp32 "
                                      f"on the pool (> calibrated tolerance {tol:.2e})")
    return res, info


@torch.no_grad()
def filter_topk(model_name: str, model, x, adj: SparseAdj, k: Optional[int] = None,
                slab_pairs: int = 1 << 27, distributed: bool = False, ra_adj: Optional[SparseAdj] = None,
                stats: Optional[dict] = None, precision: Optional[str] = None,
                owners: Optional[Tuple[int, int]] = None, per_node: Optional[int] = None) -> torch.Tensor:
    """Sorted proposal list of one filter model, float32 ``[k,3]`` rows (u, v, score) on the device: score
    descending, ties by the reference's candidate order.  ``k=None`` keeps every candidate like the
    reference.  ``precision`` (GNN models): see ``FilterJob``; default = the model's ``linkpred.precision``.
    ``per_node=m``: only the m best candidates of every owner v (see ``_filter_multi``)."""
    job = FilterJob(model_name, model, ra_adj, precision)
    return filter_topk_multi([job], x, adj, k, slab_pairs, distributed, stats, owners=owners, per_node=per_node)[0]


def load_extra_edges(path: str, num_sorted_edge: int) -> torch.Tensor:
    """filter.py:82 / rank.py:294: the first ``num_sorted_edge`` rows of a saved sorted list."""
    t = torch.load(path)
    extra = t[:num_sorted_edge, :2].t().long()
    assert extra.size(0) == 2 and extra.size(1) == num_sorted_edge
    return extra
