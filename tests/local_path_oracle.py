"""Oracle of the Local Path index (``local_path``; include/eps.h eps_local_path_*) in numpy / scipy:
c2 = (A^2)_uv, c3 = (A^3)_uv on the stored structure (self loops included, edge values ignored) and
score = fp32(c2 + 1e-3 * c3), the fp64 product and sum each rounded once (no FMA), then rounded to fp32."""
from __future__ import annotations

import numpy as np
import scipy.sparse as ssp

from oracle.graph import CSR

LP_EPS = 1e-3


def structure(g: CSR) -> ssp.csr_matrix:
    return ssp.csr_matrix((np.ones(g.nnz, np.int64), g.col.astype(np.int64), g.rowptr.astype(np.int64)),
                          shape=(g.n, g.n))


def local_path_score(c2: np.ndarray, c3: np.ndarray) -> np.ndarray:
    return (np.asarray(c2, np.int64).astype(np.float64) + LP_EPS * np.asarray(c3, np.int64).astype(np.float64)
            ).astype(np.float32)


def local_path_counts(g: CSR, edges: np.ndarray, block_bytes: int = 1 << 27):
    """(c2, c3) int64 of the pairs ``edges[2,B]``: columns of A^2 and A^3 = A @ A^2 in dense blocks of owners v."""
    e = np.asarray(edges, dtype=np.int64)
    A = structure(g)
    A2 = (A @ A).tocsc()
    c2 = np.zeros(e.shape[1], np.int64)
    c3 = np.zeros(e.shape[1], np.int64)
    if e.shape[1] == 0:
        return c2, c3
    B = max(1, block_bytes // (8 * max(g.n, 1)))
    order = np.argsort(e[1], kind="stable")
    vs = e[1][order]
    for v0 in range(0, g.n, B):
        a, b = np.searchsorted(vs, [v0, v0 + B])
        if a == b:
            continue
        sel = order[a:b]
        blk = A2[:, v0:v0 + B]
        c2[sel] = blk.toarray()[e[0][sel], e[1][sel] - v0]
        c3[sel] = (A @ blk).toarray()[e[0][sel], e[1][sel] - v0]
    return c2, c3


def local_path_pairs(g: CSR, edges: np.ndarray):
    """(score fp32, c2, c3) of the pairs ``edges[2,B]``."""
    c2, c3 = local_path_counts(g, edges)
    return local_path_score(c2, c3), c2, c3
