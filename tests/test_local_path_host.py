"""The Local Path index on the host: the numpy / scipy oracle against brute-force 3-walk counts, the c3 <= nnz bound,
the identity the fused kernel computes c3 by, the per-owner work estimate against brute force, the model table and
CLI, the symmetric-graph guard and the argument checks of the new entry points (all without a device)."""
import argparse
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

from local_path_oracle import local_path_counts, local_path_pairs, local_path_score
from oracle import graph as og
from similarity_oracle import candidates_with_counts
from util import csr_from_undirected, golden_graph, tiny_graphs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dense(g):
    A = np.zeros((g.n, g.n), np.int64)
    rows = np.repeat(np.arange(g.n), np.diff(g.rowptr))
    A[rows, g.col] = 1
    return A


def _random_graph(seed, n=60, m=150, loops=6, hub=True):
    """Random undirected graph with self loops, a hub (node 0), a dense corner and isolated nodes (the last three)."""
    rng = np.random.default_rng(seed)
    e = [(int(a), int(b)) for a, b in rng.integers(0, n - 3, (m, 2)) if a != b]
    e += [(int(x), int(x)) for x in rng.choice(n - 3, loops, replace=False)]
    if hub:
        e += [(0, int(u)) for u in range(1, n - 3, 2)]
    e += [(a, b) for a in range(n - 12, n - 5) for b in range(a + 1, n - 5)]
    return csr_from_undirected(n, np.unique(np.sort(np.asarray(e), 1), axis=0))


def _graphs():
    out = {name: csr_from_undirected(n, e) for name, (n, e) in tiny_graphs().items()}
    for s in range(3):
        out[f"random{s}"] = _random_graph(s)
    return out


@pytest.mark.parametrize("name", list(_graphs()))
def test_oracle_against_brute_force_walks(name):
    g = _graphs()[name]
    A = _dense(g)
    adj = [set(np.flatnonzero(A[i]).tolist()) for i in range(g.n)]
    uu, vv = np.meshgrid(np.arange(g.n), np.arange(g.n))
    e = np.stack([uu.ravel(), vv.ravel()])                # every pair: isolated ends, u == v and edges included
    c2, c3 = local_path_counts(g, e, block_bytes=8 * g.n * 7)   # several owner blocks
    w2 = np.zeros((g.n, g.n), np.int64)
    w3 = np.zeros((g.n, g.n), np.int64)
    for u in range(g.n):                                  # walks u - j - v and u - j - i - v, one by one
        for j in adj[u]:
            for v in adj[j]:
                w2[u, v] += 1
            for i in adj[j]:
                for v in adj[i]:
                    w3[u, v] += 1
    assert np.array_equal(c2, w2[e[0], e[1]]) and np.array_equal(c3, w3[e[0], e[1]])
    assert np.array_equal(w3, A @ A @ A)
    s = local_path_pairs(g, e)[0]
    assert np.array_equal(s, (c2 + 1e-3 * c3).astype(np.float32))
    assert c3.max(initial=0) <= g.nnz                     # c3 <= sum_{j in N(u)} deg j <= nnz


def test_score_rounding():
    c2 = np.array([0, 1, 13, 7, 2**20, 3], np.int64)
    c3 = np.array([0, 1, 999, 2**31 - 1, 12345, 3], np.int64)
    s = local_path_score(c2, c3)
    for a, b, x in zip(c2, c3, s):
        want = np.float32(np.float64(a) + np.float64(1e-3) * np.float64(b))    # two RN fp64 operations, then fp32
        assert x.view(np.uint32) == want.view(np.uint32)
    assert s[0] == 0.0 and s[1] == np.float32(1.001)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_fused_identity_and_bound(seed):
    """The kernel's decomposition on the candidates of every owner: c3(u, v) = sum_{j in N(u) & C(v)} c2(j, v) +
    sum_{k in N(u) & N(v)} tri(v, k), tri(v, k) = |N(v) & N(k)|."""
    g = _random_graph(seed, n=80, m=260)
    A = _dense(g)
    A2, A3 = A @ A, A @ A @ A
    cand, cnt = candidates_with_counts(g)
    assert np.array_equal(cnt, A2[cand[0], cand[1]])
    cset = [set() for _ in range(g.n)]
    for u, v in cand.T:
        cset[v].add(int(u))
    nb = [set(np.flatnonzero(A[i]).tolist()) for i in range(g.n)]
    for u, v in cand.T:
        t1 = sum(A2[j, v] for j in nb[u] & cset[v])
        t2 = sum(len(nb[v] & nb[k]) for k in nb[u] & nb[v])
        assert t1 + t2 == A3[u, v], (u, v)
    assert A3.max() <= g.nnz


def test_oracle_on_golden_sample():
    z, ei, g = golden_graph("fb")
    rng = np.random.default_rng(2)
    e = np.concatenate([z["sample_edges"][:, rng.choice(z["sample_edges"].shape[1], 300, replace=False)],
                        rng.integers(0, g.n, (2, 100))], 1).astype(np.int64)
    c2, c3 = local_path_counts(g, e)
    A = og.CSR(g.rowptr, g.col, np.ones(g.nnz, np.float32), g.n).to_scipy().astype(np.int64).tocsr()
    for i in range(0, e.shape[1], 37):
        u, v = e[:, i]
        row_u = A[u].toarray().ravel()
        col_v = (A @ A[:, v]).toarray().ravel()
        assert c2[i] == int(row_u @ A[:, v].toarray().ravel()) and c3[i] == int(row_u @ col_v)


def _adj(g):
    from edge_proposal_sets_b200.graph import SparseAdj
    return SparseAdj(torch.from_numpy(g.rowptr.astype(np.int32)), torch.from_numpy(g.col.astype(np.int32)), None, g.n)


@pytest.mark.parametrize("seed", [0, 1])
def test_local_path_work_against_brute_force(seed):
    from edge_proposal_sets_b200 import candidates, filter_step
    g = _random_graph(seed)
    adj = _adj(g)
    nb = [g.col[g.rowptr[i]:g.rowptr[i + 1]].tolist() for i in range(g.n)]
    deg = np.diff(g.rowptr)
    full = [sum(deg[u] for k in nb[v] for u in nb[k]) for v in range(g.n)]
    half = [sum(deg[u] for k in nb[v] for u in nb[k] if u > v) for v in range(g.n)]
    assert candidates.local_path_work(adj).tolist() == full
    assert candidates.local_path_work(adj, upper=True).tolist() == half
    for upper in (False, True):
        base = filter_step.owner_cost(adj, [("simple", None)], upper)
        lp = filter_step.owner_cost(adj, [("simple", None), ("local_path", None)], upper)
        assert torch.equal(lp - base, torch.tensor(half if upper else full, dtype=torch.float64))


def _cli(name):
    spec = importlib.util.spec_from_file_location(f"{name}_cli", os.path.join(ROOT, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_cli_and_model_table():
    from edge_proposal_sets_b200 import filter_step, models
    kind = "local_path"
    assert kind in models.HEURISTIC_MODELS and kind in models.SUPPORTED_MODELS and kind not in models.SIMILARITY_MODELS
    a = _cli("filter").parse_args(["--dataset", "twitch", "--model", kind, "--checkpoint", "twitch_lp||0|0.pt",
                                   "--topk", "100000"])
    assert a.model == kind and a.topk == 100000
    r = _cli("rank").parse_args(["--dataset", "twitch", "--model", kind, "--sorted_edge_path", "x.pt",
                                 "--num_sorted_edge", "100000", "--runs", "1"])
    assert r.model == kind
    for dataset in ("ddi", "collab", "ppa", "twitch", "fb", "email", "reddit"):
        ns = argparse.Namespace(dataset=dataset, model=kind, num_layers=None, hidden_channels=None, dropout=None,
                                batch_size=None, lr=None, epochs=None, use_feature=True, use_learnable_embedding=True)
        d = models.default_model_configs(ns)
        assert d.use_feature is False and d.use_learnable_embedding is False and d.num_layers is None
    ns = argparse.Namespace(model=kind, use_learnable_embedding=False, use_feature=False, hidden_channels=None,
                            num_layers=None, dropout=None)
    m = models.build_model(ns, None, "cpu")
    assert isinstance(m, models.CommonNeighborsPredictor) and m.type == kind
    assert sum(p.numel() for p in m.parameters()) == 0
    # katz is unchanged: accepted by the predictor, scores nothing
    assert models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="katz")(None, None, None) is None
    # the fused plan on any graph, mirror mode on structurally symmetric ones (weighted too)
    g = _random_graph(0)
    adj = _adj(g)
    assert filter_step.heuristic_table(kind, adj) == (adj, None, False, False, kind)
    from edge_proposal_sets_b200.graph import SparseAdj
    wadj = SparseAdj(adj.rowptr, adj.col, torch.full((adj.nnz,), 3.0), adj.n)
    job = filter_step.FilterJob(kind, m)
    assert filter_step.mirror_eligible([job], adj, 10) and filter_step.mirror_eligible([job], wadj, 10)
    assert not filter_step.mirror_eligible([job], adj, 10, per_node=3)


def _asym():
    from edge_proposal_sets_b200.graph import SparseAdj
    return SparseAdj(torch.tensor([0, 2, 3, 3], dtype=torch.int32), torch.tensor([1, 2, 2], dtype=torch.int32), None, 3)


def test_asymmetric_graph_is_refused_before_any_launch():
    from edge_proposal_sets_b200 import _lib, candidates, filter_step, models, ops
    adj = _asym()
    m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="local_path")
    with pytest.raises(_lib.EpsError, match="structurally symmetric"):
        candidates.two_hop_local_path(adj)
    with pytest.raises(_lib.EpsError, match="structurally symmetric"):
        ops.local_path(adj, torch.tensor([[0], [2]]))
    with pytest.raises(_lib.EpsError, match="structurally symmetric"):
        filter_step.filter_topk("local_path", m, None, adj, k=2)
    with pytest.raises(_lib.EpsError, match="structurally symmetric"):
        candidates.two_hop_scored(adj, kind="local_path")


def test_second_local_path_job_is_refused():
    from edge_proposal_sets_b200 import candidates, filter_step, models
    adj = _adj(_random_graph(1))
    m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="local_path")
    with pytest.raises(ValueError, match="at most one local_path"):
        filter_step.filter_topk_multi([("local_path", m), ("simple", m), ("local_path", m)], None, adj, k=5)
    with pytest.raises(candidates.EpsError, match="no weight table"):
        candidates.two_hop_scored(adj, torch.ones(adj.n), kind="local_path")


def test_entry_points_reject_arguments_without_a_device():
    from edge_proposal_sets_b200 import _lib
    lib = _lib.load()
    d = C.c_void_p(16)                                   # never dereferenced
    ws = lib.eps_local_path_onepass_workspace_bytes(3, 5, 7, 2)
    assert ws >= 512 + 3 * 3 * 4 + 2 * 7 * 4

    def onepass(rowptr=d, col=d, tri=d, n=10, lo=0, hi=5, boff=d, cap=3, mc=7, ctas=2, flags=0, pu=d, pv=d,
                off=d, w=d, wb=ws):
        return lib.eps_local_path_onepass(rowptr, col, tri, n, lo, hi, boff, cap, mc, ctas, flags, pu, pv, d, None,
                                          None, off, w, wb, None)

    for kw, msg in ((dict(rowptr=None), b"null"), (dict(tri=None), b"null"), (dict(boff=None), b"null"),
                    (dict(off=None), b"null"), (dict(hi=11), b"bad owner range"), (dict(lo=5), b"bad owner range"),
                    (dict(lo=-1), b"bad owner range"), (dict(cap=-1), b"bad owner range"),
                    (dict(cap=1 << 31), b"bad owner range"), (dict(mc=-1), b"bad max_count"),
                    (dict(ctas=0), b"bad max_count"), (dict(pu=None), b"missing pair output"),
                    (dict(flags=_lib.EPS_CN_SIGMOID), b"unknown flag bits"), (dict(flags=1 << 8), b"unknown flag bits"),
                    (dict(flags=1 << 11), b"unknown flag bits")):
        assert onepass(**kw) == -1 and msg in lib.eps_last_error(), kw
    assert onepass(wb=ws - 1) == -3 and b"workspace too small" in lib.eps_last_error()
    assert onepass(w=None) == -3

    def pairs(n=10, pu=d, pv=d, M=4, flags=0, score=d, w=d, wb=256):
        return lib.eps_local_path_pairs(d, d, n, pu, pv, M, flags, score, None, None, w, wb, None)

    for kw, msg in ((dict(n=0), b"bad n or M"), (dict(M=-1), b"bad n or M"), (dict(flags=1), b"unknown flag bits"),
                    (dict(flags=1 << 11), b"unknown flag bits"), (dict(pu=None), b"null"),
                    (dict(score=None), b"all NULL")):
        assert pairs(**kw) == -1 and msg in lib.eps_last_error(), kw
    assert pairs(wb=8) == -3 and b"workspace too small" in lib.eps_last_error()
    assert pairs(M=0, pu=None) == 0                      # empty list: nothing to read or write
    # the existing kind field is unchanged: local_path is no score kind
    assert "local_path" not in _lib.SCORE_KINDS and _lib.EPS_VERSION == 203
