"""Distance-3 candidates on the host: the scipy oracle against brute-force walks and BFS distances, its counts on the
golden graphs, the per-owner bounds against the real counts, the 2-hop set as a subset, the ``--hops`` option, the
refusal of heuristic jobs at hops=3, and the argument checks of eps_threehop_onepass (all without a device)."""
import ctypes as C
import importlib.util
import os
from collections import deque
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from similarity_oracle import candidates_with_counts
from threehop_oracle import three_hop_candidates, three_hop_counts
from util import csr_from_undirected, golden_graph, tiny_graphs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _random_graph(seed, n=70, m=120):
    """Random undirected graph with self loops, a hub (node 0) and isolated nodes (the last three)."""
    rng = np.random.default_rng(seed)
    e = [(int(a), int(b)) for a, b in rng.integers(0, n - 3, (m, 2)) if a != b]
    e += [(int(x), int(x)) for x in rng.choice(n - 3, 5, replace=False)]
    e += [(0, int(u)) for u in range(5, n - 3, 4)]
    return csr_from_undirected(n, np.unique(np.sort(np.asarray(e), 1), axis=0))


def _graphs():
    out = {name: csr_from_undirected(n, e) for name, (n, e) in tiny_graphs().items()}
    # bipartite: a 6-cycle plus a pendant path (distance-2 pairs have no 3-walk and vice versa), isolated node 9
    out["bipartite10"] = csr_from_undirected(10, np.array([[0, 1], [1, 2], [2, 3], [3, 4], [4, 5], [5, 0], [5, 6],
                                                           [6, 7], [7, 8]]))
    out["loops6"] = csr_from_undirected(6, np.array([[0, 0], [0, 1], [1, 2], [2, 2], [3, 4], [5, 5]]))
    for s in range(3):
        out[f"random{s}"] = _random_graph(s)
    return out


def _lists(g):
    return [g.col[g.rowptr[i]:g.rowptr[i + 1]].tolist() for i in range(g.n)]


@pytest.mark.parametrize("name", list(_graphs()))
def test_oracle_against_walks_and_bfs(name):
    g = _graphs()[name]
    nb = _lists(g)
    want = []
    for v in range(g.n):
        e2 = {u for k in nb[v] for u in nb[k]}                    # 2-walk ends
        e3 = {u for j in e2 for u in nb[j]}                       # 3-walk ends
        cand = (e2 | e3) - set(nb[v]) - {v}
        dist = {v: 0}                                             # BFS: the same set is distance 2 or 3
        q = deque([v])
        while q:
            x = q.popleft()
            for y in nb[x]:
                if y not in dist:
                    dist[y] = dist[x] + 1
                    q.append(y)
        assert cand == {u for u, d in dist.items() if d in (2, 3)}, (name, v)
        want += [(u, v) for u in sorted(cand)]
    got = three_hop_candidates(g, block=3)
    assert got.dtype == np.int32 and np.array_equal(got.T, np.asarray(want, np.int64).reshape(-1, 2)), name
    assert np.array_equal(three_hop_counts(g, block=4), np.bincount(got[1], minlength=g.n))
    assert np.array_equal(three_hop_counts(g, upper=True), np.bincount(got[1][got[0] > got[1]], minlength=g.n))
    lo, hi = g.n // 3, g.n - 1
    part = three_hop_candidates(g, lo, hi)
    assert np.array_equal(part, got[:, (got[1] >= lo) & (got[1] < hi)])
    if name == "bipartite10":                                     # the union matters: each parity misses pairs
        assert (2, 0) in map(tuple, got.T) and (3, 0) in map(tuple, got.T)


def _adj(g):
    from edge_proposal_sets_b200.graph import SparseAdj
    return SparseAdj(torch.from_numpy(g.rowptr.astype(np.int32)), torch.from_numpy(g.col.astype(np.int32)), None, g.n)


def _check_bounds(g, full, half):
    from edge_proposal_sets_b200 import candidates
    adj = _adj(g)
    bf = candidates.owner_bounds(adj, hops=3).numpy()
    bh = candidates.owner_bounds(adj, True, hops=3).numpy()
    assert (bf >= full).all() and (bh >= half).all()
    # hops=2 keeps its bounds; hops=3 never bounds below them
    assert (bf >= candidates.owner_bounds(adj).numpy()).all() and (bh >= candidates.owner_bounds(adj, True).numpy()).all()
    return bf, bh


@pytest.mark.parametrize("name", list(_graphs()))
def test_bounds_and_two_hop_subset_small(name):
    g = _graphs()[name]
    got = three_hop_candidates(g)
    full = np.bincount(got[1], minlength=g.n)
    half = np.bincount(got[1][got[0] > got[1]], minlength=g.n)
    _check_bounds(g, full, half)
    two, _ = candidates_with_counts(g)
    k3 = set(map(tuple, got.T.tolist()))
    assert set(map(tuple, two.T.tolist())) <= k3


@pytest.fixture(scope="module")
def golden():
    out = {}
    for name in ("twitch", "fb"):
        g = golden_graph(name)[2]
        out[name] = (g, three_hop_counts(g), three_hop_counts(g, upper=True))
    return out


@pytest.mark.timeout(900)
@pytest.mark.parametrize("name,total", [("twitch", 75_622_132), ("fb", 37_114_296)])
def test_golden_counts_bounds_and_subset(golden, name, total):
    g, full, half = golden[name]
    assert int(full.sum()) == total and 2 * int(half.sum()) == total    # a symmetric relation
    bf, bh = _check_bounds(g, full, half)
    two, _ = candidates_with_counts(g)
    assert (np.bincount(two[1], minlength=g.n) <= full).all()
    # the 2-hop list is a subset, owner by owner, on a slice of owners (the whole list is checked on the GPU)
    lo, hi = 100, 400
    k3 = three_hop_candidates(g, lo, hi)
    t2 = two[:, (two[1] >= lo) & (two[1] < hi)]
    key3 = k3[1].astype(np.int64) * g.n + k3[0]
    assert np.isin(t2[1].astype(np.int64) * g.n + t2[0], key3).all()


def _cli(name):
    spec = importlib.util.spec_from_file_location(f"{name}_cli", os.path.join(ROOT, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_hops_option():
    f = _cli("filter")
    base = ["--dataset", "twitch", "--model", "gcn", "--checkpoint", "twitch_gcn||0|0.pt"]
    assert f.parse_args(base).hops == 2
    assert f.parse_args(base + ["--hops", "3"]).hops == 3
    for bad in ("1", "4", "x"):
        with pytest.raises(SystemExit):
            f.parse_args(base + ["--hops", bad])


def test_heuristic_jobs_refused_at_hops3():
    from edge_proposal_sets_b200 import candidates, filter_step, models
    adj = _adj(_random_graph(0))
    cn = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="simple")
    gnn = SimpleNamespace(linkpred=SimpleNamespace(precision="fp32"))    # never embedded: the check comes first
    for names in (["simple"], ["local_path"], ["jaccard"], ["gcn", "adamic"], ["sage", "resource_allocation"]):
        jobs = [(nm, gnn if nm in models.GNN_MODELS else cn) for nm in names]
        with pytest.raises(ValueError, match="hops=3 takes GNN filter models only"):
            filter_step.filter_topk_multi(jobs, None, adj, k=5, hops=3)
    with pytest.raises(ValueError, match="hops=3 takes GNN"):
        filter_step.filter_topk("simple", cn, None, adj, k=5, hops=3)
    for hops in (1, 4):
        with pytest.raises(ValueError, match="hops must be 2 or 3"):
            filter_step.filter_topk("gcn", gnn, None, adj, k=5, hops=hops)
        with pytest.raises(ValueError, match="hops must be 2 or 3"):
            candidates.owner_bounds(adj, hops=hops)


def test_owner_cost_hops3():
    from edge_proposal_sets_b200 import candidates, filter_step
    adj = _adj(_random_graph(1))
    for upper in (False, True):
        two = filter_step.owner_cost(adj, [("gcn", None)], upper)
        three = filter_step.owner_cost(adj, [("gcn", None)], upper, hops=3)
        b2, b3 = candidates.owner_bounds(adj, upper).double(), candidates.owner_bounds(adj, upper, 3).double()
        want = two + 8.0 * (b3 - b2) + candidates.local_path_work(adj, upper).double()
        assert torch.allclose(three, want, rtol=0, atol=0)


def test_entry_point_rejects_arguments_without_a_device():
    from edge_proposal_sets_b200 import _lib
    lib = _lib.load()
    d = C.c_void_p(16)                                   # never dereferenced
    ws = lib.eps_threehop_onepass_workspace_bytes(3, 5, 7, 2)
    assert ws >= 512 + 3 * 4 + 2 * 7 * 4
    assert lib.eps_threehop_onepass_workspace_bytes(-1, -1, -1, -1) == lib.eps_threehop_onepass_workspace_bytes(0, 0, 0, 0)

    def onepass(rowptr=d, col=d, n=10, lo=0, hi=5, boff=d, cap=3, me=7, ctas=2, flags=0, pu=d, pv=d, off=d, w=d, wb=ws):
        return lib.eps_threehop_onepass(rowptr, col, n, lo, hi, boff, cap, me, ctas, flags, pu, pv, off, w, wb, None)

    for kw, msg in ((dict(rowptr=None), b"null"), (dict(col=None), b"null"), (dict(boff=None), b"null"),
                    (dict(off=None), b"null"), (dict(n=0), b"bad owner range"), (dict(hi=11), b"bad owner range"),
                    (dict(lo=5), b"bad owner range"), (dict(lo=-1), b"bad owner range"),
                    (dict(cap=-1), b"bad owner range"), (dict(cap=1 << 31), b"bad owner range"),
                    (dict(me=-1), b"bad max_ends"), (dict(me=1 << 31), b"bad max_ends"), (dict(ctas=0), b"bad max_ends"),
                    (dict(pu=None), b"missing pair output"), (dict(pv=None), b"missing pair output"),
                    (dict(flags=_lib.EPS_CN_SIGMOID), b"unknown flag bits"), (dict(flags=1 << 8), b"unknown flag bits"),
                    (dict(flags=_lib.EPS_TWOHOP_UPPER | 2), b"unknown flag bits")):
        assert onepass(**kw) == -1 and msg in lib.eps_last_error(), kw
    assert onepass(wb=ws - 1) == -3 and b"workspace too small" in lib.eps_last_error()
    assert onepass(w=None) == -3
    assert _lib.EPS_VERSION == 203 and lib.eps_version() == 203
