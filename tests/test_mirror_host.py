"""Mirror mode on the host: the reconstruction of the full proposal list from the half top-k
(filter_step.mirror_topk) against brute force, the half-candidate bounds, the symmetry check and the guards that
keep a call on the full path, and the ABI of the upper-triangle flag (no device needed)."""
import os
import re
import sys

import numpy as np
import pytest
import torch

from oracle import graph as og, ranking as orank

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _select(edges, score, k):
    """ops.topk_edges' contract (score descending, ties by position) on the CPU."""
    return torch.from_numpy(orank.sorted_edges(edges.numpy(), score.numpy(), k))


def _random_symmetric_job(rng, n, density, levels):
    """Candidate list in column-major order (sorted by (v, u)) of a random symmetric relation without diagonal, and
    scores of a symmetric matrix with few distinct values (long tie runs)."""
    mask = np.triu(rng.random((n, n)) < density, 1)
    mask = mask | mask.T
    S = rng.integers(0, levels, (n, n)).astype(np.float32) / np.float32(levels)
    S = np.triu(S, 1)
    S = S + S.T
    v, u = np.nonzero(mask.T)                    # rows of mask.T are owners v: (v, u) ascending
    cand = np.stack([u, v])
    return cand, S[u, v].astype(np.float32)


@pytest.mark.parametrize("seed", range(24))
def test_mirror_topk_equals_full_list(seed):
    from edge_proposal_sets_b200 import filter_step
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 40))
    cand, score = _random_symmetric_job(rng, n, float(rng.uniform(0.05, 0.9)), int(rng.integers(1, 6)))
    half = cand[0] > cand[1]
    C_ = cand.shape[1]
    for k in sorted({1, 2, 3, 5, max(C_ // 3, 1), max(C_ - 1, 1), C_, C_ + 7}):
        want = orank.sorted_edges(cand, score, k)
        half_top = torch.from_numpy(orank.sorted_edges(cand[:, half], score[half], k))
        got = filter_step.mirror_topk(half_top, k, n, select=_select)
        assert np.array_equal(got.numpy(), want), (seed, n, k)


def test_mirror_topk_empty():
    from edge_proposal_sets_b200 import filter_step
    e = torch.empty((0, 3), dtype=torch.float32)
    assert filter_step.mirror_topk(e, 10, 5, select=_select).shape == (0, 3)


def _adj(name="small"):
    from util import synth_graph, to_adj
    s, ei, w, g = synth_graph(name)
    return g, to_adj(g, "cpu")


def test_half_bounds_hold_and_halve_the_slots():
    from edge_proposal_sets_b200 import candidates
    g, adj = _adj()
    cand = og.two_hop_candidates(g)
    up = cand[0] > cand[1]
    cnt = np.bincount(cand[1][up], minlength=g.n)
    hb = candidates.owner_bounds(adj, upper=True).numpy()
    assert (hb >= cnt).all()
    assert 2 * hb.sum() <= candidates.owner_bounds(adj).sum().item() * 1.05
    # the 2-path term counts exactly the 2-paths v - k - u with u > v
    rp, col = g.rowptr, g.col
    paths = np.zeros(g.n, np.int64)
    for v in range(g.n):
        for k in col[rp[v]:rp[v + 1]]:
            paths[v] += int((col[rp[k]:rp[k + 1]] > v).sum())
    assert np.array_equal(candidates.half_two_path_work(adj).numpy(), paths)


def test_structural_symmetry_check():
    from edge_proposal_sets_b200 import candidates
    from edge_proposal_sets_b200.graph import SparseAdj
    g, adj = _adj("tiny")
    assert candidates.structurally_symmetric(adj)
    one_way = SparseAdj(torch.tensor([0, 1, 1, 1], dtype=torch.int32), torch.tensor([1], dtype=torch.int32), None, 3)
    assert not candidates.structurally_symmetric(one_way)
    dup = SparseAdj(torch.tensor([0, 2, 4], dtype=torch.int32), torch.tensor([1, 1, 0, 0], dtype=torch.int32), None, 2)
    assert not candidates.structurally_symmetric(dup)          # a repeated entry is not a plain symmetric graph
    loops = SparseAdj(torch.tensor([0, 2, 3], dtype=torch.int32), torch.tensor([0, 1, 0], dtype=torch.int32), None, 2)
    assert candidates.structurally_symmetric(loops)


def test_guards_route_to_the_full_path():
    from edge_proposal_sets_b200 import filter_step
    from edge_proposal_sets_b200.graph import SparseAdj
    g, adj = _adj("tiny")
    FJ = filter_step.FilterJob
    gnn = FJ("gcn", None, precision="fp32")
    aa = FJ("adamic_ogb", None)
    assert filter_step.mirror_eligible([aa, gnn], adj, 100)
    assert filter_step.mirror_eligible([FJ("simple", None), FJ("resource_allocation", None)], adj, 100)
    assert not filter_step.mirror_eligible([aa, gnn], adj, None)                     # k=None
    assert not filter_step.mirror_eligible([aa, gnn], adj, 100, owners=(0, 10))      # owner subset
    assert not filter_step.mirror_eligible([aa, gnn], adj, 100, per_node=3)          # per-node budgets
    one_way = SparseAdj(torch.tensor([0, 1, 1, 1], dtype=torch.int32), torch.tensor([1], dtype=torch.int32), None, 3)
    assert not filter_step.mirror_eligible([gnn], one_way, 100)                      # asymmetric adjacency
    # weighted graph: the value-weighted heuristics are not bit-symmetric, the index-only one and the GNN are
    w = SparseAdj(adj.rowptr, adj.col, torch.full((adj.nnz,), 2.0), adj.n)
    assert not filter_step.mirror_eligible([aa, gnn], w, 100)
    assert not filter_step.mirror_eligible([FJ("simple", None)], w, 100)
    assert filter_step.mirror_eligible([FJ("adamic", None), gnn], w, 100)
    # RA on a rebuilt graph with other entries is scored pair by pair (not the fused kernel): full path
    other = SparseAdj(torch.tensor([0] + [0] * adj.n, dtype=torch.int32), torch.zeros(0, dtype=torch.int32), None, adj.n)
    assert not filter_step.mirror_eligible([FJ("resource_allocation", None, other)], adj, 100)
    # mirror=True insists: a call that cannot take the half path says so before any kernel runs
    with pytest.raises(ValueError, match="mirror=True"):
        filter_step.filter_topk("adamic_ogb", None, None, adj, k=None, mirror=True)


def test_cost_model_balances_half_work():
    from edge_proposal_sets_b200 import candidates, filter_step, parallel
    g, adj = _adj()
    jobs = [filter_step.FilterJob("gcn", None, precision="fp32")]
    full = filter_step.owner_cost(adj, jobs)
    half = filter_step.owner_cost(adj, jobs, upper=True)
    assert half.sum() < full.sum()
    b = parallel.partition_by_work(half, 2)
    assert b[1] < parallel.partition_by_work(full, 2)[1]      # low ids carry most of the half work
    lo, hi = half[:b[1]].sum().item(), half[b[1]:].sum().item()
    assert abs(lo - hi) <= half.max().item() + 1e-9


def test_upper_flag_abi():
    from edge_proposal_sets_b200 import _lib
    h = open(os.path.join(ROOT, "include", "eps.h")).read()
    assert int(re.search(r"#define EPS_TWOHOP_UPPER (\d+)", h).group(1)) == _lib.EPS_TWOHOP_UPPER
    assert int(re.search(r"#define EPS_VERSION (\d+)", h).group(1)) == _lib.EPS_VERSION == 203
    assert _lib.EPS_TWOHOP_UPPER & (_lib.EPS_CN_SIGMOID | _lib.EPS_CN_GROUPED_BY_V) == 0
    lib = _lib.load()
    assert lib.eps_version() == 203
