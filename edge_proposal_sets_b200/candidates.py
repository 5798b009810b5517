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
from ._lib import EPS_CN_GROUPED_BY_V, EPS_CN_SIGMOID, EPS_SCORE_KIND_SHIFT, EPS_TWOHOP_UPPER, SCORE_KINDS, EpsError, check
from .graph import SparseAdj
from .ops import _need_cuda, _ptr, _stream, _ws


def owner_counts(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None) -> torch.Tensor:
    """#candidates of every owner v in [v_lo, v_hi) as int64: the differences of the one-pass offsets, enumerated in
    owner ranges of at most 2^27 bounded candidates (filter_step.iter_slabs), so a large graph needs no buffer of all
    its candidates."""
    from .filter_step import iter_slabs
    _need_cuda(adj.col)
    v_hi = adj.n if v_hi is None else v_hi
    parts = [torch.zeros(0, dtype=torch.int64, device=adj.device)]
    for lo, hi, cap in iter_slabs(adj, v_lo, v_hi, 1 << 27):
        parts.append(two_hop(adj, lo, hi, cap=cap, want_offsets=True)[1].diff())
    return torch.cat(parts)


def owner_bounds(adj: SparseAdj, upper: bool = False, hops: int = 2) -> torch.Tensor:
    """Upper bound of every owner's candidate count, int64 [n]: a candidate of v is the end point of
    a 2-path from v (<= #2-paths) and is neither v nor a neighbour of v: <= n - |N(v) U {v}|, i.e.
    n - 1 - deg v, or n - deg v when v carries a self loop (add_edges keeps them; v is then in N(v)).
    Torch ops only; sizes the outputs of the one-pass kernel and cuts owner ranges into slabs / GPU shards.
    ``upper``: the bound of the half candidates u > v (``half_bounds``).  ``hops=3``: the distance-3 candidates
    (``three_hop``), whose 2- and 3-walk counts add ``local_path_work`` (the 3-walks) to the first term."""
    if hops == 3:
        key = ("three_hop_bounds", bool(upper))
        if key not in adj._cache:
            owner_bounds(adj, upper)                      # caches the second term ("free" / "half_free")
            walks = (half_two_path_work(adj) if upper else two_path_work(adj)) + local_path_work(adj)
            adj._cache[key] = torch.minimum(walks, adj._cache["half_free" if upper else "free"])
        return adj._cache[key]
    if hops != 2:
        raise ValueError(f"hops must be 2 or 3 (got {hops})")
    if upper:
        return half_bounds(adj)
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
        adj._cache["free"] = (adj.n - 1 - deg + loop).clamp_(min=0)
        adj._cache["owner_bounds"] = torch.minimum(two_path_work(adj), adj._cache["free"])
    return adj._cache["owner_bounds"]


def _mirror_search(adj: SparseAdj):
    """(key, mirror, pos): key = row * n + col of every entry (int64 [nnz], ascending: rows are stored in order with
    sorted columns), mirror = col * n + row, pos = the first key > mirror.  Keys are integers, so pos is also the first
    key >= k * n + v + 1 for the entry (v, k), i.e. where the suffix of N(k) above v starts; and (k, v) is an entry
    exactly when key[pos - 1] == mirror.  One search serves the symmetry check and the half bounds."""
    if "mirror_search" not in adj._cache:
        row, col = adj.row(), adj.col.long()
        key = row * adj.n + col
        mirror = col * adj.n + row
        adj._cache["mirror_search"] = (key, mirror, torch.searchsorted(key, mirror, right=True))
    return adj._cache["mirror_search"]


def half_bounds(adj: SparseAdj) -> torch.Tensor:
    """Upper bound of every owner's count of HALF candidates u > v (the upper-triangle mode of the one-pass kernel),
    int64 [n]: min(#2-paths v - k - u with u > v, (n - 1 - v) - |N(v) & (v, n)|).  The 2-path term is
    sum_{k in N(v)} |N(k) & (v, n)|; one searchsorted of k * n + v + 1 over the sorted entry keys gives each
    |N(k) & (v, n)| (``_mirror_search``).  With the full bound every slab of the half stream would be about half empty."""
    if "half_bounds" not in adj._cache:
        n = adj.n
        rp = adj.rowptr.long()
        if adj.nnz == 0:
            adj._cache["half_bounds"] = torch.zeros(n, dtype=torch.int64, device=adj.device)
            adj._cache["half_two_path_work"] = adj._cache["half_bounds"]
            adj._cache["half_free"] = (n - 1 - torch.arange(n, device=adj.device)).clamp_(min=0)
            return adj._cache["half_bounds"]
        key, _, pos = _mirror_search(adj)
        # entry (v, k): the suffix of N(k) above v starts at the first key >= k * n + v + 1
        suffix = rp[adj.col.long() + 1] - pos
        cs = torch.zeros(adj.nnz + 1, dtype=torch.int64, device=adj.device)
        torch.cumsum(suffix, 0, out=cs[1:])
        paths = cs[rp[1:]] - cs[rp[:-1]]
        ar = torch.arange(n, device=adj.device)
        above = rp[1:] - torch.searchsorted(key, ar * n + ar + 1)          # |N(v) & (v, n)|
        adj._cache["half_two_path_work"] = paths
        adj._cache["half_free"] = (n - 1 - ar - above).clamp_(min=0)
        adj._cache["half_bounds"] = torch.minimum(paths, adj._cache["half_free"])
    return adj._cache["half_bounds"]


def structurally_symmetric(adj: SparseAdj) -> bool:
    """True when (u, k) is an entry exactly when (k, u) is (``add_edges`` graphs always are) and no entry repeats: then
    u is a candidate of v exactly when v is a candidate of u.  Checked once per graph."""
    if "struct_sym" not in adj._cache:
        ok = True
        if adj.nnz:
            key, mirror, pos = _mirror_search(adj)
            ok = bool(torch.equal(key[(pos - 1).clamp_(min=0)], mirror)) and bool((key[1:] > key[:-1]).all())
        adj._cache["struct_sym"] = ok
    return adj._cache["struct_sym"]


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


def similarity_flags(adj: SparseAdj, kind: str | None) -> int:
    """The flag bits of a similarity kind (``_lib.SCORE_KINDS``; ``None`` -> 0) for ``adj``.  The kernels divide
    integers held in fp32, exact only below 2^24: raises when 2 * max degree >= 2^24 (a + b could reach it).  The
    degree is checked once per graph."""
    if kind is None:
        return 0
    if kind not in SCORE_KINDS:
        raise EpsError(f"unknown similarity kind {kind!r} (known: {', '.join(SCORE_KINDS)})")
    if "max_degree" not in adj._cache:
        adj._cache["max_degree"] = int(adj.degree().max().item()) if adj.n else 0
    if not 2 * adj._cache["max_degree"] < 2 ** 24:
        raise EpsError(f"max degree {adj._cache['max_degree']}: deg u + deg v may reach 2^24, beyond the integers fp32 "
                       f"holds exactly; the {kind} kernels cannot score this graph exactly")
    return SCORE_KINDS[kind] << EPS_SCORE_KIND_SHIFT


def values_symmetric(adj: SparseAdj) -> bool:
    """True when A[u,k] == A[k,u] bit for bit (always, for ``add_edges`` graphs with integer-valued
    weights: both directions receive the same exact sum).  Checked once per graph."""
    if adj.val is None:
        return True
    if "val_sym" not in adj._cache:
        from .autograd import transposed_values
        adj._cache["val_sym"] = bool(torch.equal(transposed_values(adj.rowptr, adj.col, adj.val, adj.n), adj.val))
    return adj._cache["val_sym"]


def _slot_offsets(bounds: torch.Tensor, cap: int | None):
    """(boff, cap): the padded slot offsets of the one-pass entry points (exclusive prefix of the per-owner ``bounds``,
    int64 [n_own + 1]) and their total, which sizes the outputs (``cap``, when the caller already has it on the host,
    saves a sync)."""
    boff = torch.zeros(bounds.numel() + 1, dtype=torch.int64, device=bounds.device)
    torch.cumsum(bounds, 0, out=boff[1:])
    cap = int(boff[-1].item()) if cap is None else int(cap)
    if cap >= 2**31:
        raise EpsError(f"up to {cap} candidates in one slab; split the owner range (see filter_step.iter_slabs)")
    return boff, cap


def _compact_size(offsets: torch.Tensor, cap: int, what: str) -> int:
    """N = offsets[-1], the one host sync of a one-pass call (it sizes the later launches); raises when an owner's
    candidates exceeded its bound (the kernel then poisons N instead of overrunning the slot)."""
    N = int(offsets[-1].item())
    if N > cap:
        raise EpsError(f"{what}: an owner's candidates exceed the caller's bound (N={N}, cap={cap})")
    return N


def _onepass(adj: SparseAdj, wtable, v_lo: int, v_hi: int, bounds, sigmoid: bool, want_score: bool, want_count: bool,
             cap: int | None = None, val: torch.Tensor | None = None, upper: bool = False, kind_flags: int = 0):
    """eps_twohop_onepass: (edges int32 [2,N] view, score | None, count | None, offsets int64 [n_own+1]).
    ``bounds``: per-owner upper bounds of the candidate counts (default ``owner_bounds(adj, upper)``); ``cap``: their
    sum when the caller already knows it (filter_step.iter_slabs) — saves a host sync.  ``upper``: only the
    candidates u > v of every owner v (EPS_TWOHOP_UPPER).  ``kind_flags``: a similarity kind (``similarity_flags``)."""
    lib = _lib.load()
    dev = adj.device
    n_own = v_hi - v_lo
    if n_own <= 0:
        z = torch.zeros(1, dtype=torch.int64, device=dev)
        return (torch.empty((2, 0), dtype=torch.int32, device=dev),
                torch.empty(0, dtype=torch.float32, device=dev) if want_score else None,
                torch.empty(0, dtype=torch.int32, device=dev) if want_count else None, z)
    if bounds is None:
        bounds = owner_bounds(adj, upper)[v_lo:v_hi]
    boff, cap = _slot_offsets(bounds, cap)
    buf = torch.empty((2, max(cap, 1)), dtype=torch.int32, device=dev)
    score = torch.empty(max(cap, 1), dtype=torch.float32, device=dev) if want_score else None
    count = torch.empty(max(cap, 1), dtype=torch.int32, device=dev) if want_count else None
    offsets = torch.empty(n_own + 1, dtype=torch.int64, device=dev)
    wt = None if wtable is None else wtable.contiguous().float()
    ws = _ws(lib.eps_twohop_onepass_workspace_bytes(cap, n_own), dev)
    check(lib.eps_twohop_onepass(_ptr(adj.rowptr), _ptr(adj.col), _ptr(val), _ptr(wt), adj.n, v_lo, v_hi, _ptr(boff), cap,
                                 (EPS_CN_SIGMOID if sigmoid else 0) | (EPS_TWOHOP_UPPER if upper else 0) | kind_flags,
                                 _ptr(buf[0]), _ptr(buf[1]), _ptr(score),
                                 _ptr(count), _ptr(offsets), _ptr(ws), ws.numel(), _stream()), "eps_twohop_onepass")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 3
    N = _compact_size(offsets, cap, "eps_twohop_onepass")
    return (buf[:, :N], None if score is None else score[:N], None if count is None else count[:N], offsets)


def two_hop(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None, cap: int | None = None,
            want_offsets: bool = False, upper: bool = False):
    """(u, v) candidate list of owners [v_lo, v_hi): int32 [2, N], column-major reference order, from the one-pass
    kernel (no count pass): a [2, N] view of a buffer sized by the owner_bounds sum (``cap`` = that sum, when the caller
    already has it on the host).  ``want_offsets`` returns ``(edges, offsets)``: offsets int64 [v_hi - v_lo + 1], owner
    v's candidates are ``edges[:, offsets[v - v_lo]:offsets[v - v_lo + 1]]`` (the segments of ``ops.segment_topk``).
    ``upper``: only the candidates u > v of every owner v — each unordered pair once on a structurally symmetric graph;
    ``cap`` is then the sum of ``half_bounds``."""
    _need_cuda(adj.col)
    v_hi = adj.n if v_hi is None else v_hi
    r = _onepass(adj, None, v_lo, v_hi, None, False, False, False, cap, upper=upper)
    return (r[0], r[3]) if want_offsets else r[0]


def two_hop_scored(adj: SparseAdj, wtable: torch.Tensor | None = None, v_lo: int = 0, v_hi: int | None = None,
                   sigmoid: bool = False, want_count: bool = False, cap: int | None = None, use_values: bool = True,
                   want_offsets: bool = False, upper: bool = False, kind: str | None = None):
    """K6+K3 fused: the candidates of owners [v_lo, v_hi) AND their heuristic scores from one walk
    over the owners' 2-paths (``wtable=None`` -> CN count, else sum of ``wtable[k]`` over the common
    neighbours: AA with 1/log deg, RA with 1/deg).  Returns ``(edges int32 [2,N], score fp32 [N])``
    (+ ``count int32 [N]`` with ``want_count``); scores are bit-identical to ``ops.cn_aa`` on the
    same pairs.  A weighted adjacency (collab, ``use_values``) contributes A[u,k]*(A[v,k]*wtable[k]) per
    2-path; ``use_values=False`` ignores the values ('adamic', models.py:544-554).  One-pass kernel, no count
    pass: outputs are views of buffers sized by the owner_bounds sum of the range.  ``want_offsets`` appends the
    per-owner offsets (int64 [v_hi - v_lo + 1], as in ``two_hop``) to the returned tuple.  ``upper``: as in ``two_hop``.
    ``kind`` (a name of ``_lib.SCORE_KINDS``, e.g. "jaccard"): a degree-normalised similarity of the exact count and
    the degrees of both ends instead (include/eps.h, EPS_SCORE_*): structure only, so needs ``wtable=None`` and no
    sigmoid, and ignores edge values.  ``kind="local_path"``: the Local Path index (``two_hop_local_path``; the count is
    c2)."""
    if kind == LOCAL_PATH:
        if wtable is not None or sigmoid:
            raise EpsError("two_hop_scored: the local_path score takes no weight table and no sigmoid")
        e, s, c2, _, off = two_hop_local_path(adj, v_lo, v_hi, cap, upper, want_offsets=True)
        out = (e, s, c2) if want_count else (e, s)
        return out + (off,) if want_offsets else out
    _need_cuda(adj.col, wtable)
    kind_flags = similarity_flags(adj, kind)
    if kind_flags and (wtable is not None or sigmoid):
        raise EpsError(f"two_hop_scored: the {kind} score takes no weight table and no sigmoid")
    if kind_flags:
        use_values = False
    val = adj.val if use_values else None
    check_fixed_point_range(adj, wtable, use_values)
    if val is not None and not values_symmetric(adj):
        raise EpsError("two_hop_scored: a weighted adjacency needs bitwise symmetric values; otherwise score with "
                       "two_hop + ops.cn_aa")
    v_hi = adj.n if v_hi is None else v_hi
    edges, score, count, offsets = _onepass(adj, wtable, v_lo, v_hi, None, sigmoid, True, want_count, cap, val,
                                            upper, kind_flags)
    out = (edges, score, count) if want_count else (edges, score)
    return out + (offsets,) if want_offsets else out


def half_two_path_work(adj: SparseAdj) -> torch.Tensor:
    """``two_path_work`` of the upper-triangle mode: the 2-paths v - k - u with u > v of every owner (the first term of
    ``half_bounds``); low ids carry most of it."""
    if "half_two_path_work" not in adj._cache:
        half_bounds(adj)
    return adj._cache["half_two_path_work"]


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


# ---------------------------------------------------------------------------------------------
# Local Path index: LP(u, v) = (A^2)_uv + 1e-3 (A^3)_uv (include/eps.h, eps_local_path_*)
# ---------------------------------------------------------------------------------------------
LOCAL_PATH = "local_path"


def require_symmetric(adj: SparseAdj, what: str) -> None:
    """The Local Path kernels count 3-paths through the candidate relation, which needs a structurally symmetric graph
    (``structurally_symmetric``, checked once per graph): raises before anything is launched otherwise."""
    if not structurally_symmetric(adj):
        raise EpsError(f"{what}: the local_path score needs a structurally symmetric adjacency ((u, k) stored exactly "
                       "when (k, u) is, no repeated entry); add_edges graphs are")


def arc_triangles(adj: SparseAdj) -> torch.Tensor:
    """tri int32 [nnz]: tri[p] = |N(v) & N(k)| for the stored arc p = (v, k), i.e. the exact K3 counts of the pairs
    (k, v) (grouped by v: rows are stored in order).  Structure only.  Built once per graph."""
    if "arc_tri" not in adj._cache:
        _need_cuda(adj.col)
        lib = _lib.load()
        tri = torch.empty(adj.nnz, dtype=torch.int32, device=adj.device)
        if adj.nnz:
            row = adj.row().to(torch.int32)
            ws = _ws(lib.eps_cn_aa_workspace_bytes(), adj.device)
            check(lib.eps_cn_aa(_ptr(adj.rowptr), _ptr(adj.col), None, None, adj.n, _ptr(adj.col), _ptr(row), adj.nnz,
                                EPS_CN_GROUPED_BY_V, None, _ptr(tri), _ptr(ws), ws.numel(), _stream()), "eps_cn_aa")
            from . import ops as _ops
            _ops.LAUNCHES["n"] += 1
        adj._cache["arc_tri"] = tri
    return adj._cache["arc_tri"]


def local_path_work(adj: SparseAdj, upper: bool = False) -> torch.Tensor:
    """Per-owner pull work of the Local Path walk 3, int64 [n]: sum_{k in N(v)} sum_{u in N(k)} deg u (two products of A
    with the degrees; a candidate reached by several 2-paths counts once per 2-path, so this bounds the work of its
    N(u) stream).  ``upper``: only the end points u > v.  Torch ops only; device-agnostic."""
    key = ("lp_work", bool(upper))
    if key not in adj._cache:
        deg = adj.degree().long()
        rp = adj.rowptr.long()
        cs = torch.zeros(adj.nnz + 1, dtype=torch.int64, device=adj.device)
        if adj.nnz:
            torch.cumsum(deg[adj.col.long()], 0, out=cs[1:])            # prefix of deg u over the entries
        if upper and adj.nnz:
            _, _, pos = _mirror_search(adj)                             # entry (v, k): N(k) above v starts at pos
            per_entry = cs[rp[adj.col.long() + 1]] - cs[pos]
        else:
            per_entry = (cs[rp[1:]] - cs[rp[:-1]])[adj.col.long()]      # sum_{u in N(k)} deg u
        ce = torch.zeros(adj.nnz + 1, dtype=torch.int64, device=adj.device)
        if adj.nnz:
            torch.cumsum(per_entry, 0, out=ce[1:])
        adj._cache[key] = ce[rp[1:]] - ce[rp[:-1]]
    return adj._cache[key]


def _lp_ctas(device) -> int:
    """Per-CTA scratch areas handed to eps_local_path_onepass and eps_threehop_onepass: every CTA that can be resident
    (<= 4 per SM at 512 threads)."""
    return 4 * torch.cuda.get_device_properties(device).multi_processor_count


def two_hop_local_path(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None, cap: int | None = None,
                       upper: bool = False, want_offsets: bool = False):
    """The candidates of owners [v_lo, v_hi) with their Local Path scores from one fused walk
    (eps_local_path_onepass): ``(edges int32 [2,N], score fp32 [N], c2 int32 [N], c3 int32 [N])`` (+ offsets int64
    [v_hi - v_lo + 1] with ``want_offsets``), candidates in the order of ``two_hop``.  c2 = |N(u) & N(v)|,
    c3 = (A^3)_uv, score = fp32(c2 + 1e-3 * c3) rounded once from fp64.  ``upper`` / ``cap``: as in ``two_hop``.
    Structure only (edge values ignored); raises on a graph that is not structurally symmetric."""
    require_symmetric(adj, "two_hop_local_path")
    _need_cuda(adj.col)
    lib = _lib.load()
    dev = adj.device
    v_hi = adj.n if v_hi is None else v_hi
    n_own = v_hi - v_lo
    if n_own <= 0:
        z = torch.zeros(1, dtype=torch.int64, device=dev)
        i0 = torch.empty(0, dtype=torch.int32, device=dev)
        out = (torch.empty((2, 0), dtype=torch.int32, device=dev), torch.empty(0, dtype=torch.float32, device=dev), i0, i0)
        return out + (z,) if want_offsets else out
    tri = arc_triangles(adj)
    boff, cap = _slot_offsets(owner_bounds(adj, upper)[v_lo:v_hi], cap)
    if "max_bound" not in adj._cache:
        adj._cache["max_bound"] = int(owner_bounds(adj).max().item()) if adj.n else 0
    max_count, ctas = adj._cache["max_bound"], _lp_ctas(dev)
    buf = torch.empty((2, max(cap, 1)), dtype=torch.int32, device=dev)
    score = torch.empty(max(cap, 1), dtype=torch.float32, device=dev)
    c2 = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    c3 = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    offsets = torch.empty(n_own + 1, dtype=torch.int64, device=dev)
    ws = _ws(lib.eps_local_path_onepass_workspace_bytes(cap, n_own, max_count, ctas), dev)
    check(lib.eps_local_path_onepass(_ptr(adj.rowptr), _ptr(adj.col), _ptr(tri), adj.n, v_lo, v_hi, _ptr(boff), cap,
                                     max_count, ctas, EPS_TWOHOP_UPPER if upper else 0, _ptr(buf[0]), _ptr(buf[1]),
                                     _ptr(score), _ptr(c2), _ptr(c3), _ptr(offsets), _ptr(ws), ws.numel(), _stream()),
          "eps_local_path_onepass")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 6
    N = _compact_size(offsets, cap, "eps_local_path_onepass")
    out = (buf[:, :N], score[:N], c2[:N], c3[:N])
    return out + (offsets,) if want_offsets else out


# ---------------------------------------------------------------------------------------------
# Distance-3 candidates: the ends of 2- and 3-walks (include/eps.h, eps_threehop_onepass)
# ---------------------------------------------------------------------------------------------
def three_hop(adj: SparseAdj, v_lo: int = 0, v_hi: int | None = None, cap: int | None = None,
              want_offsets: bool = False, upper: bool = False):
    """The distance-<= 3 candidates of owners [v_lo, v_hi): every u with (A^2)_uv + (A^3)_uv > 0 that is neither v nor
    a neighbour of v, as int32 [2, N] in the column-major order of ``two_hop`` (whose list is a subset).  Enumeration
    only, one fused walk per owner (eps_threehop_onepass); ``cap`` / ``want_offsets`` / ``upper`` as in ``two_hop``,
    with the bounds of ``owner_bounds(adj, upper, hops=3)``.  Structure only (edge values ignored)."""
    _need_cuda(adj.col)
    lib = _lib.load()
    dev = adj.device
    v_hi = adj.n if v_hi is None else v_hi
    n_own = v_hi - v_lo
    if n_own <= 0:
        e = torch.empty((2, 0), dtype=torch.int32, device=dev)
        return (e, torch.zeros(1, dtype=torch.int64, device=dev)) if want_offsets else e
    boff, cap = _slot_offsets(owner_bounds(adj, upper, hops=3)[v_lo:v_hi], cap)
    if "max_two_walk_ends" not in adj._cache:                # distinct 2-walk ends: <= #2-walks and <= n
        adj._cache["max_two_walk_ends"] = int(two_path_work(adj).clamp(max=adj.n).max().item()) if adj.n else 0
    max_ends, ctas = adj._cache["max_two_walk_ends"], _lp_ctas(dev)
    buf = torch.empty((2, max(cap, 1)), dtype=torch.int32, device=dev)
    offsets = torch.empty(n_own + 1, dtype=torch.int64, device=dev)
    ws = _ws(lib.eps_threehop_onepass_workspace_bytes(cap, n_own, max_ends, ctas), dev)
    check(lib.eps_threehop_onepass(_ptr(adj.rowptr), _ptr(adj.col), adj.n, v_lo, v_hi, _ptr(boff), cap, max_ends, ctas,
                                   EPS_TWOHOP_UPPER if upper else 0, _ptr(buf[0]), _ptr(buf[1]), _ptr(offsets),
                                   _ptr(ws), ws.numel(), _stream()), "eps_threehop_onepass")
    from . import ops as _ops
    _ops.LAUNCHES["n"] += 6
    N = _compact_size(offsets, cap, "eps_threehop_onepass")
    return (buf[:, :N], offsets) if want_offsets else buf[:, :N]
