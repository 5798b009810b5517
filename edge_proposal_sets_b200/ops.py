"""Python-side operators over the C ABI (include/eps.h).  All tensors are CUDA tensors; torch is
used for allocation and the current stream only.  Nothing here computes on the CPU: a CPU tensor
or a missing library raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import (EPS_CN_GROUPED_BY_V, EPS_CN_SIGMOID, EPS_MLP_FP32, EPS_MLP_REUSE_WORKSPACE, EPS_MLP_TC_F16,
                   EPS_REDUCE_MEAN, EPS_REDUCE_SUM, EpsError, check)
from .graph import SparseAdj


# kernels launched through this module since the counter was last reset (bench.py reports it)
LAUNCHES = {"n": 0}
# optional per-kernel CUDA-event timing on the launching stream: set KERNEL_EVENTS to a dict and every
# wrapped call appends (start, end) events under its kernel name (bench.py reads them after a sync)
KERNEL_EVENTS = None
_TOPK_LAUNCHES = 22      # 3 hist + 3 pick + count + scan + write + 4 x (hist, scan, scatter) + finalize
_SELECT_LAUNCHES = 10    # 3 hist + 3 pick + count + scan + write + finalize


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise EpsError("edge_proposal_sets_b200 kernels need CUDA tensors (no CPU fallback)")


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _event_pair(name: str):
    if KERNEL_EVENTS is None:
        return None
    pair = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    pair[0].record()
    KERNEL_EVENTS.setdefault(name, []).append(pair)
    return pair


def _pairs(edges: torch.Tensor):
    """[2,M] (any int dtype) -> two contiguous int32 rows."""
    if edges.dim() != 2 or edges.shape[0] != 2:
        raise EpsError("edges must have shape [2, M]")
    e = edges if edges.dtype == torch.int32 else edges.to(torch.int32)
    if e.shape[1] and e.stride(1) != 1:
        e = e.contiguous()                # rows of a [2,N] view of a wider buffer are already contiguous
    return e[0], e[1]


def spmm_csr(rowptr: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], x: torch.Tensor,
             reduce: str = "sum", bias: Optional[torch.Tensor] = None, relu: bool = False,
             out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """K1.  y = reduce_j val_ij * x[col_j]  (+bias)(relu)."""
    _need_cuda(rowptr, col, val, x, bias)
    lib = _lib.load()
    x = x.contiguous().float()
    n_rows = rowptr.numel() - 1
    F = x.shape[1]
    y = out if out is not None else torch.empty((n_rows, F), dtype=torch.float32, device=x.device)
    ws = _ws(lib.eps_spmm_workspace_bytes(), x.device)
    red = {"sum": EPS_REDUCE_SUM, "add": EPS_REDUCE_SUM, "mean": EPS_REDUCE_MEAN}[reduce]
    bias = None if bias is None else bias.contiguous().float()
    ev = _event_pair("spmm_csr")
    check(lib.eps_spmm_csr_f32(_ptr(rowptr), _ptr(col), _ptr(val), _ptr(x), _ptr(y), n_rows, F, red,
                               _ptr(bias), int(relu), _ptr(ws), ws.numel(), _stream()), "eps_spmm_csr_f32")
    if ev is not None:
        ev[1].record()
    LAUNCHES["n"] += 1
    return y


def pair_hadamard(h: torch.Tensor, edges: torch.Tensor) -> torch.Tensor:
    """K7 forward: z0[b,:] = h[u_b,:] * h[v_b,:] for edges [2,B] -> fp32 [B,H] (training-mode input of the MLP)."""
    _need_cuda(h, edges)
    lib = _lib.load()
    h = h.contiguous().float()
    pu, pv = _pairs(edges)
    M = pu.numel()
    out = torch.empty((M, h.shape[1]), dtype=torch.float32, device=h.device)
    check(lib.eps_pair_hadamard_f32(_ptr(h), h.shape[0], h.shape[1], _ptr(pu), _ptr(pv), M, _ptr(out), _stream()),
          "eps_pair_hadamard_f32")
    LAUNCHES["n"] += 1
    return out


def pair_hadamard_bwd(h: torch.Tensor, edges: torch.Tensor, dz: torch.Tensor) -> torch.Tensor:
    """K7 backward: dh[u_b] += dz[b] * h[v_b], dh[v_b] += dz[b] * h[u_b] -> fp32 [n,H]."""
    _need_cuda(h, edges, dz)
    lib = _lib.load()
    h = h.contiguous().float()
    dz = dz.contiguous().float()
    pu, pv = _pairs(edges)
    M = pu.numel()
    dh = torch.zeros_like(h)
    check(lib.eps_pair_hadamard_bwd_f32(_ptr(h), h.shape[0], h.shape[1], _ptr(pu), _ptr(pv), M, _ptr(dz), _ptr(dh),
                                        _stream()), "eps_pair_hadamard_bwd_f32")
    LAUNCHES["n"] += 1
    return dh


def cn_aa(adj: SparseAdj, edges: torch.Tensor, wtable: Optional[torch.Tensor] = None,
          use_values: bool = True, sigmoid: bool = False, grouped_by_v: bool = False,
          want_count: bool = False, kind: Optional[str] = None):
    """K3.  score[i] = sum_{k in N(u)&N(v)} a_u (a_v w_k); optional exact int32 counts.  ``kind`` (a name of
    ``_lib.SCORE_KINDS``, e.g. "jaccard"): the degree-normalised similarity of the count and the degrees instead
    (structure only: needs ``wtable=None`` and no sigmoid, ignores edge values)."""
    _need_cuda(adj.col, edges, wtable)
    lib = _lib.load()
    from .candidates import check_fixed_point_range, similarity_flags
    kind_flags = similarity_flags(adj, kind)
    if kind_flags and (wtable is not None or sigmoid):
        raise EpsError(f"cn_aa: the {kind} score takes no weight table and no sigmoid")
    if kind_flags:
        use_values = False
    check_fixed_point_range(adj, wtable, use_values)
    pu, pv = _pairs(edges)
    M = pu.numel()
    score = torch.empty(M, dtype=torch.float32, device=adj.device)
    count = torch.empty(M, dtype=torch.int32, device=adj.device) if want_count else None
    val = adj.val if use_values else None
    flags = (EPS_CN_SIGMOID if sigmoid else 0) | (EPS_CN_GROUPED_BY_V if grouped_by_v else 0) | kind_flags
    ws = _ws(lib.eps_cn_aa_workspace_bytes(), adj.device)
    check(lib.eps_cn_aa(_ptr(adj.rowptr), _ptr(adj.col), _ptr(val), _ptr(wtable), adj.n, _ptr(pu), _ptr(pv),
                        M, flags, _ptr(score), _ptr(count), _ptr(ws), ws.numel(), _stream()), "eps_cn_aa")
    LAUNCHES["n"] += 1 if M else 0
    return (score, count) if want_count else score


def local_path(adj: SparseAdj, edges: torch.Tensor, want_counts: bool = False):
    """Local Path index of arbitrary pairs (eps_local_path_pairs): score fp32 [M] (+ c2, c3 int32 [M] with
    ``want_counts``), the same bits as the fused filter kernel (``candidates.two_hop_local_path``) on the same pair.
    A pair costs sum_{j in N(u)} deg j: meant for evaluation sets.  The pairs are run sorted by v (one N(v) bitmap
    per run) and the results put back in input order.  Structure only; the graph must be structurally symmetric."""
    from .candidates import require_symmetric
    require_symmetric(adj, "local_path")
    _need_cuda(adj.col, edges)
    lib = _lib.load()
    pu, pv = _pairs(edges)
    M = pu.numel()
    dev = adj.device
    score = torch.empty(M, dtype=torch.float32, device=dev)
    c2 = torch.empty(M, dtype=torch.int32, device=dev) if want_counts else None
    c3 = torch.empty(M, dtype=torch.int32, device=dev) if want_counts else None
    if M:
        order = torch.argsort(pv, stable=True)
        su, sv = pu[order].contiguous(), pv[order].contiguous()
        ss = torch.empty_like(score)
        s2 = torch.empty(M, dtype=torch.int32, device=dev) if want_counts else None
        s3 = torch.empty(M, dtype=torch.int32, device=dev) if want_counts else None
        ws = _ws(lib.eps_local_path_pairs_workspace_bytes(), dev)
        ev = _event_pair("local_path_pairs")
        check(lib.eps_local_path_pairs(_ptr(adj.rowptr), _ptr(adj.col), adj.n, _ptr(su), _ptr(sv), M, 0, _ptr(ss),
                                       _ptr(s2), _ptr(s3), _ptr(ws), ws.numel(), _stream()), "eps_local_path_pairs")
        if ev is not None:
            ev[1].record()
        LAUNCHES["n"] += 1
        score[order] = ss
        if want_counts:
            c2[order] = s2
            c3[order] = s3
    return (score, c2, c3) if want_counts else score


# K2 arms: "fp32" = FFMA (reference arithmetic); "f16" = tcgen05 tensor cores, fp16 operands / fp32 accumulate
# ("tc" and the round-1 name "bf16" are aliases)
MLP_PRECISIONS = {"fp32": EPS_MLP_FP32, "f16": EPS_MLP_TC_F16, "tc": EPS_MLP_TC_F16, "bf16": EPS_MLP_TC_F16}


def linkpred_mlp(h: torch.Tensor, edges: torch.Tensor, weights: Sequence[torch.Tensor],
                 biases: Sequence[torch.Tensor], precision: str = "fp32", sigmoid: bool = True) -> torch.Tensor:
    """K2.  sigmoid(MLP(h[u] * h[v])) for every pair."""
    _need_cuda(h, edges, *weights, *biases)
    lib = _lib.load()
    h = h.contiguous().float()
    pu, pv = _pairs(edges)
    M = pu.numel()
    L = len(weights)
    Ws = [w.contiguous().float() for w in weights]
    bs = [b.contiguous().float() for b in biases]
    n, H = h.shape
    for l, w in enumerate(Ws):
        want = (1 if l == L - 1 else H, H)
        if tuple(w.shape) != want:
            raise EpsError(f"linkpred layer {l}: weight shape {tuple(w.shape)} != {want}")
    prec = MLP_PRECISIONS[precision]
    Wp = (C.c_void_p * L)(*[w.data_ptr() for w in Ws])
    bp = (C.c_void_p * L)(*[b.data_ptr() for b in bs])
    score = torch.empty(M, dtype=torch.float32, device=h.device)
    ws = _ws(lib.eps_linkpred_workspace_bytes(n, H, L, M, prec), h.device)
    check(lib.eps_linkpred_mlp(_ptr(h), n, H, _ptr(pu), _ptr(pv), M, Wp, bp, L, prec, int(sigmoid),
                               _ptr(score), _ptr(ws), ws.numel(), _stream()), "eps_linkpred_mlp")
    LAUNCHES["n"] += ((5 if M >= 2 * n else 4) if prec == EPS_MLP_TC_F16 else 1) if M else 0
    return score


def tc_scale(h: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor]):
    """Host restatement of the tensor-core arm's power-of-two scale (csrc/linkpred_tc.cu tc_scale_kernel), for
    tests and diagnostics: ``(hscale, S)`` with S = hscale^2 = 4^a, a = floor(log2(2^15 / worst) / 2), where
    ``worst`` is the largest worst-case magnitude among the Hadamard products (max|h|^2) and the hidden layers'
    outputs (B_l = max row L1 norm of W_l * B_{l-1} + max|b_l|)."""
    import math
    bound = float(h.abs().max().item()) ** 2
    worst = bound
    for w, b in zip(weights[:-1], biases[:-1]):
        bound = float(w.double().abs().sum(1).max().item()) * bound + float(b.abs().max().item())
        worst = max(worst, bound)
    a = 0
    if 0.0 < worst < 1e300:
        a = int(math.floor(math.log2(32768.0 / worst) * 0.5))
    a = max(-40, min(40, a))
    return 2.0 ** a, 4.0 ** a


class LinkpredTC:
    """K2's tcgen05 arm bound to ONE embedding matrix and ONE set of weights for a series of calls (the ~100
    owner slabs of a filter job): the scale, the fp16 copy of ``h`` and the packed weight images live in a workspace this
    object owns and are built by the first long call only (EPS_MLP_REUSE_WORKSPACE afterwards).  ``h`` and the
    weights are held by reference and must not be modified while the object is in use.  Same scores, bit for
    bit, as ``linkpred_mlp(..., precision="f16")``."""

    def __init__(self, h: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor]):
        _need_cuda(h, *weights, *biases)
        self.h = h.contiguous().float()
        self.Ws = [w.detach().contiguous().float() for w in weights]
        self.bs = [b.detach().contiguous().float() for b in biases]
        self.ws = None
        self.prepared = False

    def score(self, edges: torch.Tensor, sigmoid: bool = True) -> torch.Tensor:
        lib = _lib.load()
        n, H = self.h.shape
        L = len(self.Ws)
        pu, pv = _pairs(edges)
        M = pu.numel()
        if M < 2 * n:                      # short list: no fp16 table in the workspace, nothing to reuse
            return linkpred_mlp(self.h, edges, self.Ws, self.bs, "f16", sigmoid)
        if self.ws is None:                # on the table path the size depends on (n, H, L) only
            self.ws = _ws(lib.eps_linkpred_workspace_bytes(n, H, L, M, EPS_MLP_TC_F16), self.h.device)
        Wp = (C.c_void_p * L)(*[w.data_ptr() for w in self.Ws])
        bp = (C.c_void_p * L)(*[b.data_ptr() for b in self.bs])
        score = torch.empty(M, dtype=torch.float32, device=self.h.device)
        prec = EPS_MLP_TC_F16 | (EPS_MLP_REUSE_WORKSPACE if self.prepared else 0)
        check(lib.eps_linkpred_mlp(_ptr(self.h), n, H, _ptr(pu), _ptr(pv), M, Wp, bp, L, prec, int(sigmoid),
                                   _ptr(score), _ptr(self.ws), self.ws.numel(), _stream()), "eps_linkpred_mlp")
        LAUNCHES["n"] += 1 if self.prepared else 5
        self.prepared = True
        return score


def topk(score: torch.Tensor, k: int):
    """K4.  (idx int64 [k], score fp32 [k]) ordered score-descending, ties by position ascending."""
    _need_cuda(score)
    lib = _lib.load()
    score = score.contiguous().float()
    M = score.numel()
    k = min(int(k), M)
    if k <= 0:
        return (torch.empty(0, dtype=torch.int64, device=score.device),
                torch.empty(0, dtype=torch.float32, device=score.device))
    idx = torch.empty(k, dtype=torch.int32, device=score.device)   # uint32 payload
    out = torch.empty(k, dtype=torch.float32, device=score.device)
    ws = _ws(lib.eps_topk_workspace_bytes(M, k), score.device)
    check(lib.eps_topk_f32(_ptr(score), M, k, _ptr(idx), _ptr(out), _ptr(ws), ws.numel(), _stream()),
          "eps_topk_f32")
    LAUNCHES["n"] += _TOPK_LAUNCHES
    return idx.long() & 0xFFFFFFFF, out


def topk_edges(edges: torch.Tensor, score: torch.Tensor, k: int) -> torch.Tensor:
    """filter.py:119,160-161 restricted to the first k rows: float32 [k,3] = (u, v, score)."""
    _need_cuda(edges, score)
    lib = _lib.load()
    pu, pv = _pairs(edges)
    score = score.contiguous().float()
    M = score.numel()
    k = min(int(k), M)
    out = torch.empty((k, 3), dtype=torch.float32, device=score.device)
    if k == 0:
        return out
    idx = torch.empty(k, dtype=torch.int32, device=score.device)
    sc = torch.empty(k, dtype=torch.float32, device=score.device)
    ws = _ws(lib.eps_topk_workspace_bytes(M, k), score.device)
    check(lib.eps_topk_f32(_ptr(score), M, k, _ptr(idx), _ptr(sc), _ptr(ws), ws.numel(), _stream()),
          "eps_topk_f32")
    check(lib.eps_pack_edges(_ptr(pu), _ptr(pv), _ptr(idx), _ptr(sc), k, _ptr(out), _stream()),
          "eps_pack_edges")
    LAUNCHES["n"] += _TOPK_LAUNCHES + 1
    return out


def topk_select2(score_a: Optional[torch.Tensor], score_b: torch.Tensor, k: int,
                 prune_key: Optional[torch.Tensor] = None, want_kth_key: bool = False):
    """K4 steps 1-3 over the virtual concatenation ``score_a ++ score_b``: (virtual positions int32 [k]
    ascending, scores fp32 [k]) of the k best, ties by position.  No sort (see ``RunningTopK``).
    ``prune_key`` (int32 [1] device: the k-th key returned by the previous call whose result is
    ``score_a``) lets pass 0 skip elements that are already out; ``want_kth_key`` returns this call's."""
    _need_cuda(score_a, score_b, prune_key)
    lib = _lib.load()
    Ma = 0 if score_a is None else score_a.numel()
    Mb = score_b.numel()
    assert (score_a is None or (score_a.dtype == torch.float32 and score_a.is_contiguous())) \
        and score_b.dtype == torch.float32 and score_b.is_contiguous()
    k = min(int(k), Ma + Mb)
    idx = torch.empty(k, dtype=torch.int32, device=score_b.device)
    out = torch.empty(k, dtype=torch.float32, device=score_b.device)
    kth = torch.empty(1, dtype=torch.int32, device=score_b.device) if want_kth_key else None
    if k == 0:
        return (idx, out, kth) if want_kth_key else (idx, out)
    ws = _ws(lib.eps_topk_workspace_bytes(Ma + Mb, k), score_b.device)
    check(lib.eps_topk_select2_f32(_ptr(score_a), Ma, _ptr(score_b), Mb, k, _ptr(prune_key), _ptr(kth), _ptr(idx),
                                   _ptr(out), _ptr(ws), ws.numel(), _stream()), "eps_topk_select2_f32")
    LAUNCHES["n"] += _SELECT_LAUNCHES
    return (idx, out, kth) if want_kth_key else (idx, out)


def kth_key(score: torch.Tensor, k: int) -> torch.Tensor:
    """Order key (int32 [1], device) of the k-th best score: the three histogram passes of K4 only."""
    _need_cuda(score)
    lib = _lib.load()
    M = score.numel()
    assert score.dtype == torch.float32 and score.is_contiguous() and 1 <= k <= M
    kth = torch.empty(1, dtype=torch.int32, device=score.device)
    ws = _ws(lib.eps_topk_workspace_bytes(M, k), score.device)
    check(lib.eps_topk_select2_f32(None, 0, _ptr(score), M, k, None, _ptr(kth), None, None, _ptr(ws), ws.numel(),
                                   _stream()), "eps_topk_select2_f32")
    LAUNCHES["n"] += 6
    return kth


def key_to_score(key) -> float:
    """Host value of the score an order key stands for (the inverse of K4's key map)."""
    import numpy as np
    kk = int(key.item() if hasattr(key, "item") else key) & 0xFFFFFFFF
    asc = ~kk & 0xFFFFFFFF
    bits = (asc ^ 0x80000000) if asc >> 31 else (~asc & 0xFFFFFFFF)
    return float(np.array([bits], dtype=np.uint32).view(np.float32)[0])


def score_to_key(score: float) -> int:
    """K4's order key of a score (ascending key == descending score, -0.0 folded into +0.0)."""
    import numpy as np
    b = int((np.array([score], dtype=np.float32) + np.float32(0.0)).view(np.uint32)[0])
    asc = b ^ (0xFFFFFFFF if b >> 31 else 0x80000000)
    return ~asc & 0xFFFFFFFF


def key_tensor(key: int, device) -> torch.Tensor:
    """A uint32 order key as the int32 [1] device tensor the kernels read."""
    key = int(key) & 0xFFFFFFFF
    return torch.tensor([key - 2**32 if key >= 2**31 else key], dtype=torch.int32, device=device)


def threshold_compact(score: torch.Tensor, edges: Optional[torch.Tensor], bound_key: torch.Tensor,
                      margin: float = 0.0, inclusive: bool = False, want_pos: bool = False):
    """K4b.  The elements of ``score`` that beat the running k-th score (``bound_key``), in position order:
    ``(u, v, score)`` int32/int32/fp32 (+ positions with ``want_pos``; ``edges=None`` skips the pairs).
    ``inclusive=False``: strictly better; ``inclusive=True``: ``score >= s_k - margin``.
    One host sync (the survivor count sizes the outputs)."""
    _need_cuda(score, edges, bound_key)
    lib = _lib.load()
    M = score.numel()
    dev = score.device
    assert score.dtype == torch.float32 and score.is_contiguous() and bound_key.dtype == torch.int32
    pu = pv = None
    if edges is not None:
        pu, pv = _pairs(edges)
        assert pu.numel() == M
    nt = int(lib.eps_threshold_tiles(M))
    off = torch.empty(nt + 1, dtype=torch.int32, device=dev)
    ws = _ws(lib.eps_threshold_workspace_bytes(M), dev)
    check(lib.eps_threshold_count(_ptr(score), M, _ptr(bound_key), float(margin), int(inclusive), _ptr(off), _ptr(ws),
                                  ws.numel(), _stream()), "eps_threshold_count")
    LAUNCHES["n"] += 2 if M else 0
    c = int(off[-1].item()) & 0xFFFFFFFF
    ou = torch.empty(c if pu is not None else 0, dtype=torch.int32, device=dev)
    ov = torch.empty(c if pu is not None else 0, dtype=torch.int32, device=dev)
    osc = torch.empty(c, dtype=torch.float32, device=dev)
    opos = torch.empty(c, dtype=torch.int32, device=dev) if want_pos else None
    if c:
        check(lib.eps_threshold_write(_ptr(score), _ptr(pu), _ptr(pv), M, _ptr(bound_key), float(margin), int(inclusive),
                                      _ptr(off), _ptr(ou) if pu is not None else None,
                                      _ptr(ov) if pu is not None else None, _ptr(osc), _ptr(opos), _stream()),
              "eps_threshold_write")
        LAUNCHES["n"] += 1
    return (ou, ov, osc, opos) if want_pos else (ou, ov, osc)


def gather_pairs2(pairs_a, pairs_b, idx: torch.Tensor):
    """(u, v) int32 [k] each of the virtual positions ``idx`` over pair segments a ++ b; a segment is
    a (u, v) tuple of int32 vectors or ``None``."""
    lib = _lib.load()
    k = idx.numel()
    dev = idx.device
    ou = torch.empty(k, dtype=torch.int32, device=dev)
    ov = torch.empty(k, dtype=torch.int32, device=dev)
    ua, va = (None, None) if pairs_a is None else pairs_a
    ub, vb = (None, None) if pairs_b is None else pairs_b
    Ma = 0 if ua is None else ua.numel()
    check(lib.eps_gather_pairs2(_ptr(ua), _ptr(va), Ma, _ptr(ub), _ptr(vb), _ptr(idx), k, _ptr(ou), _ptr(ov),
                                _stream()), "eps_gather_pairs2")
    LAUNCHES["n"] += 1 if k else 0
    return ou, ov


def segment_topk(score: torch.Tensor, edges: torch.Tensor, offsets: torch.Tensor, m: int,
                 margin: Optional[float] = None):
    """K4c.  Per-segment top-m of ``score`` with segments ``offsets`` (int64 [S+1], device; an owner slab's
    per-owner offsets): ``(edges int32 [2,R], score fp32 [R], kept offsets int64 [S+1])``, the survivors in
    position order.  ``margin=None``: the m best of every segment (score descending, ties by position); a number:
    every element with score >= (the segment's m-th best score) - margin (the prefilter band, bounded like K4b's
    ``threshold_compact``).  One host sync (the survivor count sizes the outputs)."""
    _need_cuda(score, edges, offsets)
    lib = _lib.load()
    m = int(m)
    if m < 1:
        raise EpsError(f"segment_topk: m must be >= 1 (got {m})")
    dev = score.device
    score = score.contiguous().float()
    M = score.numel()
    pu, pv = _pairs(edges)
    if pu.numel() != M:
        raise EpsError(f"segment_topk: {pu.numel()} pairs for {M} scores")
    if offsets.dim() != 1 or offsets.numel() < 1:
        raise EpsError("segment_topk: offsets must be a 1-D tensor of n_seg + 1 entries")
    off = offsets.contiguous().to(torch.int64)
    n_seg = off.numel() - 1
    kept32 = torch.empty(n_seg + 1, dtype=torch.int32, device=dev)     # uint32 payload
    ws = _ws(lib.eps_segment_topk_workspace_bytes(n_seg), dev)
    band = margin is not None
    ev = _event_pair("segment_topk")
    check(lib.eps_segment_topk_select(_ptr(score), M, _ptr(off), n_seg, m, float(margin or 0.0), int(band),
                                      _ptr(kept32), _ptr(ws), ws.numel(), _stream()), "eps_segment_topk_select")
    LAUNCHES["n"] += (3 + (2 if n_seg + 1 > 8192 else 0)) if n_seg else 0
    kept = kept32.long() & 0xFFFFFFFF
    R = int(kept[-1].item())
    out = torch.empty((2, R), dtype=torch.int32, device=dev)
    osc = torch.empty(R, dtype=torch.float32, device=dev)
    if R:
        check(lib.eps_segment_topk_write(_ptr(score), _ptr(pu), _ptr(pv), M, _ptr(off), n_seg, _ptr(kept32),
                                         _ptr(out[0]), _ptr(out[1]), _ptr(osc), _ptr(ws), ws.numel(), _stream()),
              "eps_segment_topk_write")
        LAUNCHES["n"] += 1
    if ev is not None:
        ev[1].record()
    return out, osc, kept
