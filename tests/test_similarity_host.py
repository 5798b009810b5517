"""Degree-normalised similarity scores on the host: the numpy oracle against exact rational arithmetic and against
networkx, the model names through the CLI and the model table, and the ABI of the kind flags (rejected before any
CUDA call)."""
import argparse
import ctypes as C
import importlib.util
import math
import os
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import graph as og
from similarity_oracle import SIMILARITY_KINDS, similarity_pairs
from util import csr_from_undirected, golden_graph, tiny_graphs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORRECTLY_ROUNDED = ("jaccard", "sorensen", "hub_promoted", "hub_depressed", "preferential_attachment")


def _exact(kind, c, a, b):
    """The score as an exact rational (salton: a float64 reference, it has a square root)."""
    if kind == "preferential_attachment":
        return Fraction(a * b)
    if kind == "salton":
        return 0.0 if a * b == 0 else c / math.sqrt(a * b)
    den = {"jaccard": a + b - c, "sorensen": a + b, "hub_promoted": min(a, b), "hub_depressed": max(a, b),
           "leicht_holme_newman": a * b}[kind]
    num = 2 * c if kind == "sorensen" else c
    return Fraction(0) if den == 0 else Fraction(num, den)


def _f32(x):
    """Correctly rounded fp32 of an exact rational: via float64 the double rounding could differ, so compare the two
    fp32 neighbours of the float64 value with the exact error."""
    if isinstance(x, float):
        return np.float32(x)
    d = np.float32(float(x))
    best = min((np.nextafter(d, np.float32(-np.inf)), d, np.nextafter(d, np.float32(np.inf))),
               key=lambda y: (abs(Fraction(float(y)) - x), int(np.array(y).view(np.uint32)) & 1))
    return np.float32(best)


def _sets(g, u):
    return set(g.col[g.rowptr[u]:g.rowptr[u + 1]].tolist())


def _check_against_fractions(g, edges):
    deg = np.diff(g.rowptr)
    for kind in SIMILARITY_KINDS:
        got = similarity_pairs(g, edges, kind)
        for i, (u, v) in enumerate(edges.T):
            c = len(_sets(g, u) & _sets(g, v))
            x = _exact(kind, c, int(deg[u]), int(deg[v]))
            if kind in CORRECTLY_ROUNDED:
                assert got[i].view(np.uint32) == _f32(x).view(np.uint32), (kind, u, v, got[i], x)
            elif kind == "leicht_holme_newman":
                assert got[i] == np.float32(float(x)), (kind, u, v)     # fp64 quotient rounded once
            else:
                assert abs(float(got[i]) - x) <= 2 ** -23 * abs(x), (kind, u, v)


def _self_loop_graph():
    # self loops on 0 and 3 are stored neighbours (a node is its own common neighbour with itself's neighbours)
    e = np.array([[0, 0], [0, 1], [0, 2], [1, 2], [2, 3], [3, 3], [3, 4]])
    return csr_from_undirected(6, e)                  # 5: isolated


@pytest.mark.parametrize("name", list(tiny_graphs()) + ["selfloop"])
def test_oracle_exact_on_tiny_graphs(name):
    if name == "selfloop":
        g = _self_loop_graph()
    else:
        n, e = tiny_graphs()[name]
        g = csr_from_undirected(n, e)
    uu, vv = np.meshgrid(np.arange(g.n), np.arange(g.n))
    _check_against_fractions(g, np.stack([uu.ravel(), vv.ravel()]))      # every pair, isolated ends included


def test_oracle_hand_values():
    # path 0-1-2-3-4: (0, 2) share node 1; deg 0 = 1, deg 2 = 2
    n, e = tiny_graphs()["path5"]
    g = csr_from_undirected(n, e)
    pair = np.array([[0], [2]])
    want = {"jaccard": 1 / 2, "sorensen": 2 / 3, "salton": 1 / math.sqrt(2), "hub_promoted": 1.0,
            "hub_depressed": 1 / 2, "leicht_holme_newman": 1 / 2, "preferential_attachment": 2.0}
    for kind, w in want.items():
        assert similarity_pairs(g, pair, kind)[0] == np.float32(w), kind
    # star: two leaves share the hub, each of degree 1 -> jaccard 1, pa 1
    n, e = tiny_graphs()["star6"]
    g = csr_from_undirected(n, e)
    assert similarity_pairs(g, np.array([[1], [2]]), "jaccard")[0] == 1.0
    # isolated end: every score 0 (zero denominator / zero product)
    n, e = tiny_graphs()["mixed8"]
    g = csr_from_undirected(n, e)
    for kind in SIMILARITY_KINDS:
        assert similarity_pairs(g, np.array([[6, 6], [7, 0]]), kind).tolist() == [0.0, 0.0], kind


def test_oracle_exact_on_fb_sample():
    z, ei, g = golden_graph("fb")
    rng = np.random.default_rng(5)
    sel = rng.choice(z["sample_edges"].shape[1], 400, replace=False)
    _check_against_fractions(g, z["sample_edges"][:, sel].astype(np.int64))


@pytest.mark.parametrize("gold", ["twitch", "fb"])
def test_jaccard_and_pa_against_networkx(gold):
    nx = pytest.importorskip("networkx")
    z, ei, g = golden_graph(gold)
    G = nx.Graph()
    G.add_nodes_from(range(g.n))
    rows = np.repeat(np.arange(g.n), np.diff(g.rowptr))
    G.add_edges_from(zip(rows.tolist(), g.col.tolist()))
    rng = np.random.default_rng(11)
    sel = rng.choice(z["sample_edges"].shape[1], 2000, replace=False)
    e = z["sample_edges"][:, sel].astype(np.int64)
    e = np.concatenate([e, rng.integers(0, g.n, (2, 500))], 1)          # arbitrary pairs too
    pairs = list(zip(e[0].tolist(), e[1].tolist()))
    jac = np.array([p for _, _, p in nx.jaccard_coefficient(G, pairs)], dtype=np.float64)
    pa = np.array([p for _, _, p in nx.preferential_attachment(G, pairs)], dtype=np.float64)
    # networkx counts |N(u) | N(v)| on sets, which equals a + b - c on a simple graph (these have no self loops)
    assert not bool((rows == g.col).any())
    assert np.array_equal(similarity_pairs(g, e, "jaccard"), jac.astype(np.float32))
    assert np.array_equal(similarity_pairs(g, e, "preferential_attachment"), pa.astype(np.float32))


def _cli(name):
    spec = importlib.util.spec_from_file_location(f"{name}_cli", os.path.join(ROOT, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("kind", SIMILARITY_KINDS)
def test_cli_and_model_table(kind):
    from edge_proposal_sets_b200 import models
    assert kind in models.HEURISTIC_MODELS and kind in models.SUPPORTED_MODELS
    a = _cli("filter").parse_args(["--dataset", "twitch", "--model", kind, "--checkpoint", f"twitch_{kind}||0|0.pt",
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


def test_filter_step_plans_the_fused_path_on_any_graph():
    from edge_proposal_sets_b200 import filter_step
    from edge_proposal_sets_b200.graph import SparseAdj
    rp = torch.tensor([0, 1, 2], dtype=torch.int32)
    col = torch.tensor([1, 0], dtype=torch.int32)
    for val in (None, torch.tensor([2.0, 2.0])):
        adj = SparseAdj(rp, col, val, 2)
        for kind in SIMILARITY_KINDS:
            assert filter_step.heuristic_table(kind, adj) == (adj, None, False, False, kind)
    assert filter_step.heuristic_table("simple", SparseAdj(rp, col, None, 2))[4] is None


def test_kind_flag_bits():
    from edge_proposal_sets_b200 import _lib
    h = open(os.path.join(ROOT, "include", "eps.h")).read()
    assert int(re.search(r"#define EPS_SCORE_KIND_SHIFT (\d+)", h).group(1)) == _lib.EPS_SCORE_KIND_SHIFT
    old = _lib.EPS_CN_SIGMOID | _lib.EPS_CN_GROUPED_BY_V | _lib.EPS_TWOHOP_UPPER
    assert _lib.EPS_SCORE_KIND_MASK & old == 0
    codes = {}
    for m in re.finditer(r"#define EPS_SCORE_(\w+) \((\d) << EPS_SCORE_KIND_SHIFT\)", h):
        if m.group(1) != "KIND_MASK":
            codes[m.group(1)] = int(m.group(2))
    assert sorted(codes.values()) == sorted(_lib.SCORE_KINDS.values()) == list(range(1, 8))
    lib = _lib.load()
    assert lib.eps_score_kinds() == sum(1 << c for c in _lib.SCORE_KINDS.values())


def test_kind_abi_rejects_before_any_cuda_call():
    from edge_proposal_sets_b200 import _lib
    lib = _lib.load()
    d = C.c_void_p(16)                                   # never dereferenced
    jac = _lib.SCORE_KINDS["jaccard"] << _lib.EPS_SCORE_KIND_SHIFT
    unknown = (1 << 11, 1 << 4, 8, 1 << 30)

    def cn_aa(flags, val=None, wt=None):
        return lib.eps_cn_aa(d, d, val, wt, 10, d, d, 5, flags, d, None, d, 256, None)

    def onepass(flags, val=None, wt=None):
        return lib.eps_twohop_onepass(d, d, val, wt, 10, 0, 5, d, 3, flags, d, d, d, None, d, d, 1 << 20, None)

    for fn in (cn_aa, onepass):
        for bad in unknown:
            assert fn(bad) == -1 and b"unknown flag bits" in lib.eps_last_error(), (fn.__name__, bad)
        assert fn(jac | _lib.EPS_CN_SIGMOID) == -1 and b"similarity kind" in lib.eps_last_error()
        assert fn(jac, wt=d) == -1 and b"similarity kind" in lib.eps_last_error()
    assert cn_aa(jac, val=d) == -1 and b"similarity kind" in lib.eps_last_error()
    assert onepass(jac, val=d) == -1 and b"similarity kind" in lib.eps_last_error()


def test_degree_guard_and_unknown_kind():
    from edge_proposal_sets_b200 import _lib, candidates
    from edge_proposal_sets_b200.graph import SparseAdj
    n = (1 << 23) + 1                                        # node 0 adjacent to everyone: 2 * deg = 2^24
    rowptr = torch.cat([torch.tensor([0]), torch.arange(n - 1, 2 * (n - 1) + 1)]).int()
    col = torch.cat([torch.arange(1, n), torch.zeros(n - 1, dtype=torch.int64)]).int()
    hub = SparseAdj(rowptr, col, None, n)
    with pytest.raises(_lib.EpsError, match="2\\^24"):
        candidates.similarity_flags(hub, "jaccard")
    small = SparseAdj(torch.tensor([0, 1, 2], dtype=torch.int32), torch.tensor([1, 0], dtype=torch.int32), None, 2)
    assert candidates.similarity_flags(small, None) == 0
    assert candidates.similarity_flags(small, "salton") == 3 << _lib.EPS_SCORE_KIND_SHIFT
    with pytest.raises(_lib.EpsError, match="unknown similarity kind"):
        candidates.similarity_flags(small, "katz")


def test_wrappers_reject_tables_and_have_no_cpu_fallback():
    from edge_proposal_sets_b200 import _lib, ops
    from edge_proposal_sets_b200.graph import SparseAdj
    adj = SparseAdj(torch.tensor([0, 1, 2], dtype=torch.int32), torch.tensor([1, 0], dtype=torch.int32), None, 2)
    with pytest.raises(_lib.EpsError):
        ops.cn_aa(adj, torch.tensor([[0], [1]]), kind="jaccard")
