"""Generate tests/golden/{twitch,fb}.npz (graph split, whole-set checksums) and {twitch,fb}_sample.npz
(the reference's scores on a seeded sample of candidates) by EXECUTING the reference.

TEST INFRASTRUCTURE — see ``oracle/__init__.py``.  Run from the repo root:

    python -m oracle.make_golden            # needs /root/reference (read-only)

What is pinned (SURVEY §8c):
  * the bundled twitch / fb graphs with the reference's seeded split
    (/root/reference/twitch/data.py:39-64, fb/data.py same code): train edges are
    stored as a uint16 array so the fixture travels to the GPU box;
  * candidate enumeration order + count (filter.py:96-109 through scipy, A.6);
  * ``adamic_utils.AA`` outputs (the real function, via ``refshim``) on a
    seeded sample of candidates + whole-set checksums;
  * ``train_and_eval.resource_allocation`` outputs on the same sample;
  * CN = (A@A) values scipy computes at filter.py:98;
  * the exact CN top-k proposal list (ties by candidate index) as a sha256.
"""
from __future__ import annotations

import hashlib
import os
import random
import sys
import time

import numpy as np
import pandas as pd

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import graph as og, heuristics as oh, ranking as orank, refshim  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

DATASETS = {
    "twitch": ("twitch/musae_DE_edges.csv", 9498),
    "fb": ("fb/musae_facebook_edges.csv", 22470),
}


def seeded_train_split(csv_rel: str):
    """twitch/data.py:39-64 — sort endpoints, drop self loops, random.seed(42) shuffle, first 80%."""
    random.seed(42)
    np.random.seed(42)
    data = pd.read_csv(os.path.join(refshim.REFERENCE_ROOT, csv_rel))
    edges = data.values.tolist()
    edges = [list(sorted([int(e[0]), int(e[1])])) for e in edges]
    edges = [e for e in edges if e[0] < e[1]]
    n = len(edges)
    random.shuffle(edges)
    train = np.asarray(edges[: int(0.8 * n)], dtype=np.int64)
    valid = np.asarray(edges[int(0.8 * n): int(0.9 * n)], dtype=np.int64)
    test = np.asarray(edges[int(0.9 * n):], dtype=np.int64)
    return train, valid, test


def to_undirected(train: np.ndarray, n: int) -> np.ndarray:
    """torch_geometric.utils.to_undirected (twitch/data.py:116): both directions, coalesced, sorted."""
    r = np.concatenate([train[:, 0], train[:, 1]])
    c = np.concatenate([train[:, 1], train[:, 0]])
    key = np.unique(r * n + c)
    return np.stack([key // n, key % n])


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    assert refshim.available(), "needs /root/reference"
    os.makedirs(OUT, exist_ok=True)
    for name, (csv_rel, n) in DATASETS.items():
        t0 = time.time()
        train, valid, test = seeded_train_split(csv_rel)
        assert train.max() < 65536
        ei = to_undirected(train, n)
        g = og.add_edges(name, ei, np.ones(ei.shape[1], np.float32), np.zeros((2, 0), np.int64), n)
        assert og.degree_sorted_is_valid(g)
        A = g.to_scipy()

        # candidate order: the reference's scipy walk vs the oracle restatement
        ref_c, ref_vals = refshim.reference_candidates(A)
        cand, cn_vals = og.two_hop_candidates(g, return_values=True)
        assert ref_c.shape == cand.shape and np.array_equal(ref_c, cand), "candidate order mismatch"
        assert np.array_equal(ref_vals, cn_vals)
        N = cand.shape[1]
        print(f"{name}: n={n} nnz={g.nnz} candidates={N}  ({time.time()-t0:.1f}s)")

        # the real reference AA on ALL candidates (single-thread scipy)
        t1 = time.time()
        aa_all = refshim.reference_AA(A, cand)
        t_aa = time.time() - t1
        print(f"   reference AA on all candidates: {t_aa:.1f}s = {N/t_aa/1e6:.2f} M pairs/s (1 core)")

        rng = np.random.default_rng(7)
        samp = np.unique(np.concatenate([
            np.arange(0, min(N, 3000)), np.arange(max(N - 3000, 0), N),
            rng.choice(N, size=34000, replace=False)]))
        s_edges = cand[:, samp]
        ra_s = refshim.reference_RA(A.astype(np.int64), s_edges)

        k = 50000
        cn_order = orank.stable_order_desc(cn_vals.astype(np.float32))[:k]
        topk_cn = np.stack([cand[0, cn_order], cand[1, cn_order]], 1).astype(np.int32)

        np.savez_compressed(
            os.path.join(OUT, f"{name}.npz"),
            n=np.int64(n),
            train_edges=train.astype(np.uint16),
            valid_edges=valid.astype(np.uint16),
            test_edges=test.astype(np.uint16),
            num_candidates=np.int64(N),
            cand_sha256=np.array(sha(cand.astype(np.int32))),
            sum_cn=np.int64(cn_vals.astype(np.int64).sum()),
            sum_aa=np.float64(aa_all.astype(np.float64).sum()),
            max_cn=np.int64(cn_vals.max()),
            topk_k=np.int64(k),
            topk_cn_sha256=np.array(sha(topk_cn)),
            topk_cn_head=topk_cn[:64],
            topk_cn_tail=topk_cn[-64:],
            ref_aa_pairs_per_s_1core=np.float64(N / t_aa),
        )
        np.savez_compressed(
            os.path.join(OUT, f"{name}_sample.npz"),
            sample_index=samp.astype(np.int64),
            sample_edges=s_edges.astype(np.int32),
            sample_cn=cn_vals[samp].astype(np.int32),
            sample_aa=aa_all[samp].astype(np.float32),
            sample_ra=ra_s.astype(np.float32),
        )
        print(f"   wrote {name}.npz, {name}_sample.npz  sum_cn={int(cn_vals.sum())} max_cn={int(cn_vals.max())}")


if __name__ == "__main__":
    main()
