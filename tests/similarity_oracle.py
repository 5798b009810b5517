"""Oracle of the degree-normalised similarity scores (``jaccard`` ... ``preferential_attachment``; include/eps.h
EPS_SCORE_*), in numpy on top of the common-neighbour counts of ``oracle.heuristics``."""
from __future__ import annotations

import numpy as np

from oracle.graph import CSR, two_hop_candidates
from oracle.heuristics import cn_count_pairs

SIMILARITY_KINDS = ("jaccard", "sorensen", "salton", "hub_promoted", "hub_depressed", "leicht_holme_newman",
                    "preferential_attachment")


def similarity_pairs(g: CSR, edges: np.ndarray, kind: str, counts: np.ndarray | None = None) -> np.ndarray:
    """Degree-normalised similarity of pairs ``edges[2,B]`` (include/eps.h, EPS_SCORE_*), fp32, by the operation
    sequence the kernels use: c = |N(u) & N(v)| (``cn_count_pairs``, or ``counts`` when the caller has them, e.g. the
    A@A values of ``oracle.graph.two_hop_candidates`` on the unweighted structure), a = |N(u)|, b = |N(v)| (stored
    lists, self loops included, values ignored)."""
    e = np.asarray(edges, dtype=np.int64)
    deg = np.diff(g.rowptr).astype(np.int64)
    c = cn_count_pairs(g, e) if counts is None else counts
    return similarity_from_counts(np.asarray(c, dtype=np.int64), deg[e[0]], deg[e[1]], kind)


def similarity_from_counts(c: np.ndarray, a: np.ndarray, b: np.ndarray, kind: str) -> np.ndarray:
    """The score of count c and degrees a, b (int64 arrays).  jaccard / sorensen / hub_promoted / hub_depressed: ONE
    fp32 division of integers exact in fp32 (correctly rounded); salton / leicht_holme_newman: the fp64 expression
    rounded once to fp32; preferential_attachment: the int64 product rounded once to fp32.  A zero denominator gives 0."""
    assert 2 * int(max(a.max(initial=0), b.max(initial=0))) < 2 ** 24
    if kind == "preferential_attachment":
        return (a * b).astype(np.float32)
    if kind in ("salton", "leicht_holme_newman"):
        ab = a.astype(np.float64) * b.astype(np.float64)
        den = np.sqrt(ab) if kind == "salton" else ab
        with np.errstate(divide="ignore", invalid="ignore"):
            q = c.astype(np.float64) / den
        return np.where(ab == 0, 0.0, q).astype(np.float32)
    num = c
    if kind == "jaccard":
        den = a + b - c
    elif kind == "sorensen":
        num, den = 2 * c, a + b
    elif kind == "hub_promoted":
        den = np.minimum(a, b)
    elif kind == "hub_depressed":
        den = np.maximum(a, b)
    else:
        raise ValueError(f"unknown similarity kind {kind!r}")
    with np.errstate(divide="ignore", invalid="ignore"):
        q = num.astype(np.float32) / den.astype(np.float32)
    return np.where(den == 0, np.float32(0), q).astype(np.float32)


def candidates_with_counts(g: CSR):
    """(candidates int64 [2,N] in the reference's order, their exact common-neighbour counts): the A@A values of the
    unweighted structure of ``g``."""
    ones = CSR(g.rowptr, g.col, np.ones(g.nnz, np.float32), g.n)
    cand, vals = two_hop_candidates(ones, return_values=True)
    return cand, np.rint(vals).astype(np.int64)
