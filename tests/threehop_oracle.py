"""Oracle of the distance-3 candidates (``candidates.three_hop``; include/eps.h eps_threehop_onepass) in numpy / scipy:
the candidates of owner v are the u with (A^2 + A^3)[v, u] > 0 that are neither v nor stored in row v (self loops
included, edge values ignored), in column-major order (v ascending, then u ascending).  Row v of A^2 + A^3 is column v
of the transposed matrices, so for the symmetric graphs ``add_edges`` builds this is scipy's (A@A + A@A@A) > 0 minus A
and the diagonal, read CSC -> COO.  Computed in dense blocks of owners."""
from __future__ import annotations

import numpy as np
import scipy.sparse as ssp

from oracle.graph import CSR


def _blocks(g: CSR, v_lo: int, v_hi: int, block: int):
    """Yield (v0, mask bool [b, n]): the candidate rows of owners v0 .. v0 + b - 1."""
    A = ssp.csr_matrix((np.ones(g.nnz, np.float32), g.col.astype(np.int64), g.rowptr.astype(np.int64)),
                       shape=(g.n, g.n))
    At = A.T.tocsr()
    for v0 in range(v_lo, v_hi, block):
        v1 = min(v0 + block, v_hi)
        R = A[v0:v1].toarray()                       # rows of A (entries are 1: no cancellation in the sums below)
        R2 = (At @ R.T).T                            # R @ A
        R3 = (At @ R2.T).T                           # R @ A @ A
        M = (R2 + R3) > 0
        M[R > 0] = False                             # neighbours of v
        M[np.arange(v1 - v0), np.arange(v0, v1)] = False
        yield v0, M


def three_hop_candidates(g: CSR, v_lo: int = 0, v_hi: int | None = None, block: int = 256) -> np.ndarray:
    """int32 [2, N] (u, v) candidates of owners [v_lo, v_hi) in column-major order."""
    v_hi = g.n if v_hi is None else v_hi
    out = [np.zeros((2, 0), np.int32)]
    for v0, M in _blocks(g, v_lo, v_hi, block):
        vv, uu = np.nonzero(M)                       # row-major: v ascending, then u ascending
        out.append(np.stack([uu.astype(np.int32), (vv + v0).astype(np.int32)]))
    return np.concatenate(out, 1)


def three_hop_counts(g: CSR, upper: bool = False, block: int = 256) -> np.ndarray:
    """int64 [n]: every owner's number of candidates (``upper``: only those u > v)."""
    out = np.zeros(g.n, np.int64)
    for v0, M in _blocks(g, 0, g.n, block):
        if upper:
            M &= np.arange(g.n)[None, :] > np.arange(v0, v0 + M.shape[0])[:, None]
        out[v0:v0 + M.shape[0]] = M.sum(1)
    return out
