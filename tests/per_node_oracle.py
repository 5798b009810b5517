"""Oracle of the per-node proposal budgets (``filter_step._filter_multi(per_node=m)``, ``filter.py
--per_node_topk``), in numpy on top of the global ordering of ``oracle.ranking``."""
from __future__ import annotations

import numpy as np

from oracle.ranking import stable_order_desc


def per_node_topk(all_edges: np.ndarray, score: np.ndarray, m: int, k: int | None = None) -> np.ndarray:
    """Per-node proposal budgets: the m best candidates (u, v) of every owner v = all_edges[1] (score descending,
    ties by candidate order), ordered by the global rule (stable descending sort) and cut to the first k rows.
    float32 ``[rows,3]`` like ``sorted_edges``: a stable descending sort of all candidates, a mask of
    rank-within-owner < m, then the first k."""
    e = np.asarray(all_edges)
    order = stable_order_desc(score)
    owner = e[1, order].astype(np.int64)
    by_owner = np.argsort(owner, kind="stable")              # within an owner: the sorted order
    so = owner[by_owner]
    start = np.r_[0, np.flatnonzero(np.diff(so)) + 1] if so.size else np.zeros(0, np.int64)
    first = np.repeat(start, np.diff(np.r_[start, so.size]))
    rank = np.empty(order.size, dtype=np.int64)
    rank[by_owner] = np.arange(order.size) - first
    order = order[rank < int(m)]
    if k is not None:
        order = order[:k]
    out = np.empty((order.shape[0], 3), dtype=np.float32)
    out[:, 0] = e[0, order]
    out[:, 1] = e[1, order]
    out[:, 2] = np.asarray(score, dtype=np.float32)[order]
    return out
