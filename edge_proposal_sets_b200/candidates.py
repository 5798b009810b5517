"""2-hop candidate enumeration (K6) — the GPU replacement for /root/reference/filter.py:96-109.

``two_hop(adj)`` returns the reference's ``all_edges`` as int32 ``[2, N]`` on the device, in the
reference's column-major order (sorted by (all_edges[1], all_edges[0])).  ``owner_counts`` /
``two_hop(adj, v_lo, v_hi)`` work on a contiguous owner range so callers can stream slabs of a
graph whose full candidate list would not fit (ogbl-ppa scale) or shard owners across GPUs.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import EPS_CN_SIGMOID, EpsError, check
from .graph import SparseAdj
from .ops import _need_cuda, _ptr, _stream, _ws


def owner_counts(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None) -> torch.Tensor:
    """#candidates of every owner v in [v_lo, v_hi) as int64."""
    _need_cuda(adj.col)
    lib = _lib.load()
    v_hi = adj.n if v_hi is None else v_hi
    counts = torch.zeros(max(v_hi - v_lo, 0), dtype=torch.int32, device=adj.device)
    if v_hi <= v_lo:
        return counts.long()
    ws = _ws(lib.eps_twohop_workspace_bytes(), adj.device)
    check(lib.eps_twohop_candidates(_ptr(adj.rowptr), _ptr(adj.col), adj.n, v_lo, v_hi, None, _ptr(counts),
                                    None, None, _ptr(ws), ws.numel(), _stream()), "eps_twohop_candidates")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 1 if v_hi > v_lo else 0
    return counts.long() & 0xFFFFFFFF


def owner_bounds(adj: SparseAdj) -> torch.Tensor:
    """Upper bound of every owner's candidate count, int64 [n]: a candidate of v is the end point of
    a 2-path from v (<= #2-paths) and is neither v nor a neighbour of v: <= n - |N(v) U {v}|, i.e.
    n - 1 - deg v, or n - deg v when v carries a self loop (add_edges keeps them; v is then in N(v)).
    Torch ops only; sizes the outputs of the one-pass kernel and cuts owner ranges into slabs / GPU shards."""
    if "owner_bounds" not in adj._cache:
        deg = adj.degree().long()
        rp = adj.rowptr.long()
        # self loop of v <=> v occurs in its own (sorted) row: one vectorised binary search over the column array
        ar = torch.arange(adj.n, device=adj.device)
        key = adj.row() * adj.n + adj.col.long() if adj.nnz < (1 << 22) else None
        if key is not None:
            pos = torch.searchsorted(key, ar * adj.n + ar).clamp_(max=max(adj.nnz - 1, 0))
            loop = (key[pos] == ar * adj.n + ar).long() if adj.nnz else torch.zeros_like(deg)
        else:
            loop = torch.ones_like(deg)                 # large graphs: the looser n - deg for everyone
        adj._cache["owner_bounds"] = torch.minimum(two_path_work(adj), (adj.n - 1 - deg + loop).clamp_(min=0))
    return adj._cache["owner_bounds"]


def check_fixed_point_range(adj: SparseAdj, wtable, use_values: bool) -> None:
    """The exact pair-score accumulator (csrc/eps_common.cuh: 64-bit fixed point, 38 fractional bits) holds
    |sum| < 2^25.  A score is a sum of at most max_deg terms a_u * (a_v * w_k), and a common neighbour k has
    degree >= 2, so max_deg * max|a|^2 * max_{deg k >= 2} |w_k| bounds it.  Checked once per (graph, table);
    raises instead of letting the integer sums wrap."""
    key = ("fx_ok", None if wtable is None else (wtable.data_ptr(), wtable._version), bool(use_values))
    if key not in adj._cache:
        deg = adj.degree()
        dmax = float(deg.max().item()) if adj.n else 0.0
        amax = float(adj.val.abs().max().item()) if (use_values and adj.val is not None and adj.nnz) else 1.0
        wmax = 1.0
        if wtable is not None and adj.n:
            w = wtable.abs()[deg >= 2]
            wmax = float(w.max().item()) if w.numel() else 0.0
        adj._cache[key] = dmax * amax * amax * wmax
    bound = adj._cache[key]
    if not bound < 2.0 ** 25:
        raise EpsError(f"pair scores may reach {bound:.3g} >= 2^25, outside the exact fixed-point accumulator of the "
                       "CN/AA kernels (csrc/eps_common.cuh); rescale the edge weights or the weight table")


def values_symmetric(adj: SparseAdj) -> bool:
    """True when A[u,k] == A[k,u] bit for bit (always, for ``add_edges`` graphs with integer-valued
    weights: both directions receive the same exact sum).  Checked once per graph."""
    if adj.val is None:
        return True
    if "val_sym" not in adj._cache:
        from .autograd import transposed_values
        adj._cache["val_sym"] = bool(torch.equal(transposed_values(adj.rowptr, adj.col, adj.val, adj.n), adj.val))
    return adj._cache["val_sym"]


def _onepass(adj: SparseAdj, wtable, v_lo: int, v_hi: int, bounds, sigmoid: bool, want_score: bool, want_count: bool,
             cap: int | None = None, val: torch.Tensor | None = None):
    """eps_twohop_onepass: (edges int32 [2,N] view, score | None, count | None, offsets int64 [n_own+1]).
    ``bounds``: per-owner upper bounds of the candidate counts (default ``owner_bounds``); ``cap``: their
    sum when the caller already knows it (filter_step.iter_slabs) — saves a host sync."""
    lib = _lib.load()
    dev = adj.device
    n_own = v_hi - v_lo
    if n_own <= 0:
        z = torch.zeros(1, dtype=torch.int64, device=dev)
        return (torch.empty((2, 0), dtype=torch.int32, device=dev),
                torch.empty(0, dtype=torch.float32, device=dev) if want_score else None,
                torch.empty(0, dtype=torch.int32, device=dev) if want_count else None, z)
    if bounds is None:
        bounds = owner_bounds(adj)[v_lo:v_hi]
    boff = torch.zeros(n_own + 1, dtype=torch.int64, device=dev)
    torch.cumsum(bounds, 0, out=boff[1:])
    cap = int(boff[-1].item()) if cap is None else int(cap)
    if cap >= 2**31:
        raise EpsError(f"up to {cap} candidates in one slab; split the owner range (see filter_step.iter_slabs)")
    buf = torch.empty((2, max(cap, 1)), dtype=torch.int32, device=dev)
    score = torch.empty(max(cap, 1), dtype=torch.float32, device=dev) if want_score else None
    count = torch.empty(max(cap, 1), dtype=torch.int32, device=dev) if want_count else None
    offsets = torch.empty(n_own + 1, dtype=torch.int64, device=dev)
    wt = None if wtable is None else wtable.contiguous().float()
    ws = _ws(lib.eps_twohop_onepass_workspace_bytes(cap, n_own), dev)
    check(lib.eps_twohop_onepass(_ptr(adj.rowptr), _ptr(adj.col), _ptr(val), _ptr(wt), adj.n, v_lo, v_hi, _ptr(boff), cap,
                                 EPS_CN_SIGMOID if sigmoid else 0, _ptr(buf[0]), _ptr(buf[1]), _ptr(score),
                                 _ptr(count), _ptr(offsets), _ptr(ws), ws.numel(), _stream()), "eps_twohop_onepass")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 3
    N = int(offsets[-1].item())                 # the one host sync of the slab (sizes the later launches)
    if N > cap:
        raise EpsError(f"eps_twohop_onepass: an owner's candidates exceed the caller's bound (N={N}, cap={cap})")
    return (buf[:, :N], None if score is None else score[:N], None if count is None else count[:N], offsets)


def two_hop(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None, counts: torch.Tensor | None = None,
            cap: int | None = None, want_offsets: bool = False):
    """(u, v) candidate list of owners [v_lo, v_hi): int32 [2, N], column-major reference order.
    ``counts`` (from ``owner_counts``) selects the two-pass kernels; without it the one-pass kernel
    runs (no count pass) and the result is a [2, N] view of a buffer sized by the owner_bounds sum
    (``cap`` = that sum, when the caller already has it on the host).  ``want_offsets`` returns
    ``(edges, offsets)``: offsets int64 [v_hi - v_lo + 1], owner v's candidates are
    ``edges[:, offsets[v - v_lo]:offsets[v - v_lo + 1]]`` (the segments of ``ops.segment_topk``)."""
    _need_cuda(adj.col)
    lib = _lib.load()
    v_hi = adj.n if v_hi is None else v_hi
    if counts is None:
        # one pass: padded per-owner slots sized by owner_bounds, compacted by the finalize pass
        r = _onepass(adj, None, v_lo, v_hi, None, False, False, False, cap)
        return (r[0], r[3]) if want_offsets else r[0]
    offsets = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=adj.device)
    torch.cumsum(counts, 0, out=offsets[1:])
    N = int(offsets[-1].item())
    if N >= 2**31:
        raise EpsError(f"{N} candidates in one slab; split the owner range (see filter_step.iter_slabs)")
    edges = torch.empty((2, N), dtype=torch.int32, device=adj.device)
    if N == 0:
        return (edges, offsets) if want_offsets else edges
    ws = _ws(lib.eps_twohop_workspace_bytes(), adj.device)
    check(lib.eps_twohop_candidates(_ptr(adj.rowptr), _ptr(adj.col), adj.n, v_lo, v_hi, _ptr(offsets), None,
                                    _ptr(edges[0]), _ptr(edges[1]), _ptr(ws), ws.numel(), _stream()),
          "eps_twohop_candidates")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 1
    return (edges, offsets) if want_offsets else edges


def two_hop_scored(adj: SparseAdj, wtable: torch.Tensor | None = None, v_lo: int = 0, v_hi: int | None = None,
                   counts: torch.Tensor | None = None, sigmoid: bool = False, want_count: bool = False,
                   cap: int | None = None, use_values: bool = True, want_offsets: bool = False):
    """K6+K3 fused: the candidates of owners [v_lo, v_hi) AND their heuristic scores from one walk
    over the owners' 2-paths (``wtable=None`` -> CN count, else sum of ``wtable[k]`` over the common
    neighbours: AA with 1/log deg, RA with 1/deg).  Returns ``(edges int32 [2,N], score fp32 [N])``
    (+ ``count int32 [N]`` with ``want_count``); scores are bit-identical to ``ops.cn_aa`` on the
    same pairs.  A weighted adjacency (collab, ``use_values``) contributes A[u,k]*(A[v,k]*wtable[k]) per
    2-path on the one-pass kernel; ``use_values=False`` ignores the values ('adamic', models.py:544-554).
    Without ``counts`` the one-pass kernel runs: no count pass, outputs are views of buffers sized by
    the owner_bounds sum of the range.  ``want_offsets`` appends the per-owner offsets (int64
    [v_hi - v_lo + 1], as in ``two_hop``) to the returned tuple."""
    _need_cuda(adj.col, wtable)
    val = adj.val if use_values else None
    check_fixed_point_range(adj, wtable, use_values)
    if val is not None and (counts is not None or not values_symmetric(adj)):
        raise EpsError("two_hop_scored: a weighted adjacency takes the one-pass kernel (no `counts`) and needs "
                       "bitwise symmetric values; otherwise score with two_hop + ops.cn_aa")
    lib = _lib.load()
    v_hi = adj.n if v_hi is None else v_hi
    if counts is None:
        edges, score, count, offsets = _onepass(adj, wtable, v_lo, v_hi, None, sigmoid, True, want_count, cap, val)
        out = (edges, score, count) if want_count else (edges, score)
        return out + (offsets,) if want_offsets else out
    offsets = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=adj.device)
    torch.cumsum(counts, 0, out=offsets[1:])
    N = int(offsets[-1].item())
    if N >= 2**31:
        raise EpsError(f"{N} candidates in one slab; split the owner range (see filter_step.iter_slabs)")
    edges = torch.empty((2, N), dtype=torch.int32, device=adj.device)
    score = torch.empty(N, dtype=torch.float32, device=adj.device)
    count = torch.empty(N, dtype=torch.int32, device=adj.device) if want_count else None
    if N:
        wt = None if wtable is None else wtable.contiguous().float()
        ws = _ws(lib.eps_twohop_scored_workspace_bytes(N), adj.device)
        check(lib.eps_twohop_scored(_ptr(adj.rowptr), _ptr(adj.col), _ptr(wt), adj.n, v_lo, v_hi, _ptr(offsets), N,
                                    EPS_CN_SIGMOID if sigmoid else 0, _ptr(edges[0]), _ptr(edges[1]), _ptr(score),
                                    _ptr(count), _ptr(ws), ws.numel(), _stream()), "eps_twohop_scored")
        from . import ops as _ops
        _ops.LAUNCHES["n"] += 2
    out = (edges, score, count) if want_count else (edges, score)
    return out + (offsets,) if want_offsets else out


def two_path_work(adj: SparseAdj) -> torch.Tensor:
    """Per-owner work estimate sum_{k in N(v)} deg(k) (the 2-path count), used to cut owner ranges
    into equal-work slabs / GPU shards (SURVEY §8e).  Torch ops only; device-agnostic."""
    if "two_path_work" not in adj._cache:
        deg = adj.degree().long()
        cs = torch.zeros(adj.nnz + 1, dtype=torch.int64, device=adj.device)
        torch.cumsum(deg[adj.col.long()], 0, out=cs[1:])          # segment sums by row: no atomics
        rp = adj.rowptr.long()
        adj._cache["two_path_work"] = cs[rp[1:]] - cs[rp[:-1]]
    return adj._cache["two_path_work"]
