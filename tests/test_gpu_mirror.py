"""Mirror mode on the GPU: the upper-triangle K6 / K6+K3 kernel against the full kernel filtered to u > v, and the
filter step with ``mirror=True`` (score every unordered pair once, rebuild the list) against ``mirror=False``, bit for
bit, for every filter model, at boundary values of k and with many slabs; the guards that keep a call on the full
path; two GPUs against one."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import graph as og
from util import golden_graph, spread_linkpred, synth_graph, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEURISTICS = ("simple", "adamic", "adamic_ogb", "resource_allocation")


def _adj_from_pairs(n, pairs):
    """SparseAdj of the symmetric closure of ``pairs`` (self loops kept once)."""
    from edge_proposal_sets_b200.graph import SparseAdj
    p = np.asarray(pairs, np.int64).reshape(-1, 2)
    key = np.unique(np.concatenate([p[:, 0] * n + p[:, 1], p[:, 1] * n + p[:, 0]]))
    row, col = key // n, key % n
    rowptr = np.zeros(n + 1, np.int64)
    rowptr[1:] = np.cumsum(np.bincount(row, minlength=n))
    return SparseAdj(torch.from_numpy(rowptr).int().to(DEV), torch.from_numpy(col).int().to(DEV), None, n)


def _special_graph():
    """A hub, self loops, isolated nodes, a clique, and high ids whose candidates all lie below them."""
    rng = np.random.default_rng(3)
    n = 3000
    pairs = [(0, int(u)) for u in rng.choice(np.arange(1, 2500), 1800, replace=False)]       # hub owner 0
    pairs += [(int(a), int(b)) for a, b in rng.integers(1, 2500, (6000, 2)) if a != b]
    pairs += [(5, 5), (17, 17), (2999, 2999), (2998, 2998)]                                   # self loops
    pairs += [(a, b) for a in range(2600, 2612) for b in range(a + 1, 2612)]                  # a clique
    pairs += [(2990, 10), (2991, 10), (2992, 2990)]         # 2991: candidates 2990 ... only below or equal
    return n, _adj_from_pairs(n, pairs)                     # 2500..2599, 2700..2989: isolated


def _graphs():
    out = {}
    for gold in ("twitch", "fb"):
        z, ei, g = golden_graph(gold)
        out[gold] = to_adj(g, DEV)
    out["special"] = _special_graph()[1]
    return out


@pytest.fixture(scope="module")
def graphs():
    return _graphs()


def _tables(adj):
    from edge_proposal_sets_b200 import filter_step
    out = [("enum", None)]
    for name in HEURISTICS:
        out.append((name, filter_step.heuristic_table(name, adj)))
    return out


@pytest.mark.timeout(600)
@pytest.mark.parametrize("gname", ["twitch", "fb", "special"])
def test_half_kernel_is_the_full_kernel_above_the_diagonal(graphs, gname):
    from edge_proposal_sets_b200 import candidates
    adj = graphs[gname]
    n = adj.n
    ranges = [(0, n), (n // 3, n // 3 + 700), (n - 5, n)]
    for lo, hi in ranges:
        for name, t in _tables(adj):
            if t is None:
                fe, fo = candidates.two_hop(adj, lo, hi, want_offsets=True)
                he, ho = candidates.two_hop(adj, lo, hi, want_offsets=True, upper=True)
                fs = fc = hs = hc = None
            else:
                fe, fs, fc, fo = candidates.two_hop_scored(t[0], t[1], lo, hi, sigmoid=t[2], use_values=t[3],
                                                           want_count=True, want_offsets=True)
                he, hs, hc, ho = candidates.two_hop_scored(t[0], t[1], lo, hi, sigmoid=t[2], use_values=t[3],
                                                           want_count=True, want_offsets=True, upper=True)
            keep = fe[0] > fe[1]
            assert torch.equal(he, fe[:, keep]), (gname, name, lo)
            if fs is not None:
                assert torch.equal(hs.view(torch.int32), fs[keep].view(torch.int32)), (gname, name, lo)
                assert torch.equal(hc, fc[keep]), (gname, name, lo)
            per_owner = torch.bincount(fe[1][keep].long() - lo, minlength=hi - lo)
            assert torch.equal(ho[1:] - ho[:-1], per_owner), (gname, name, lo)
            bound = candidates.owner_bounds(adj, upper=True)[lo:hi]
            assert bool((per_owner <= bound).all())
    if gname == "special":
        e = candidates.two_hop(adj, upper=True)
        assert not bool((e[1] == 2991).any()) and bool((e[1] == 0).any())     # 2991 owns no u > v; the hub does


def _heuristic_model(name):
    from edge_proposal_sets_b200 import models
    if name in ("simple", "adamic"):
        return models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=name)
    return None


def _both(name, model, adj, k, slab, **kw):
    from edge_proposal_sets_b200 import filter_step
    s0, s1 = {}, {}
    full = filter_step.filter_topk(name, model, None, adj, k=k, slab_pairs=slab, stats=s0, mirror=False, **kw)
    half = filter_step.filter_topk(name, model, None, adj, k=k, slab_pairs=slab, stats=s1, mirror=True, **kw)
    return full, half, s0, s1


def _tie_k(scores_sorted):
    """A k inside the longest run of equal scores of a sorted list (its k-th and k+1-th scores are equal)."""
    s = scores_sorted
    eq = np.flatnonzero(s[1:] == s[:-1])
    return int(eq[len(eq) // 2]) + 1 if eq.size else 1


@pytest.mark.timeout(900)
@pytest.mark.parametrize("gname", ["twitch", "fb"])
def test_mirror_equals_full_heuristics(graphs, gname):
    from edge_proposal_sets_b200 import filter_step
    adj = graphs[gname]
    for name in HEURISTICS:
        model = _heuristic_model(name)
        every = filter_step.filter_topk(name, model, None, adj, k=None, mirror=False)
        C = every.shape[0]
        for k, slab in ((1, 1 << 27), (4999, 1 << 27), (_tie_k(every[:, 2].cpu().numpy()), 1 << 27),
                        (C - 1, 1 << 27), (C + 3, 1 << 27), (20001, 1 << 18)):
            full, half, s0, s1 = _both(name, model, adj, k, slab)
            assert s1["mirror"] and not s0["mirror"]
            assert torch.equal(full, half), (gname, name, k, slab)
            assert s1["candidates_scored"] == s0["candidates_scored"] == C
            assert 2 * s1["pairs_evaluated"] == C
            if slab < (1 << 20):
                assert s1["slabs"] > 10
        assert torch.equal(every[:C - 1], filter_step.filter_topk(name, model, None, adj, k=C - 1))


def _gnn(kind, n, H, L):
    import argparse
    from edge_proposal_sets_b200 import models
    from oracle import gnn as ognn
    sd = ognn.random_state_dict(kind, n, 0, H, L, seed=7)
    args = argparse.Namespace(model=kind, dataset="x", num_layers=L, hidden_channels=H, dropout=0.0,
                              use_feature=False, use_learnable_embedding=True)

    class D:
        num_nodes = n
        x = None
    mg = models.build_model(args, D, DEV)
    mg.load_state_dict(sd)
    mg.eval()
    return mg


@pytest.mark.timeout(900)
@pytest.mark.parametrize("kind,prec", [("gcn", "fp32"), ("gcn", "prefilter"), ("sage", "prefilter")])
def test_mirror_equals_full_gnn(graphs, kind, prec):
    adj = graphs["twitch"]
    mg = _gnn(kind, adj.n, 256, 3)
    from edge_proposal_sets_b200 import candidates
    edges = candidates.two_hop(adj)
    pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(edges.shape[1], 200_000, replace=False))).to(DEV)
    spread_linkpred(mg, None, adj, edges[:, pick].contiguous())
    C = edges.shape[1]
    ks = [1, 4999, 100_000] + ([C - 1] if prec == "fp32" else [])
    for k in ks:
        for slab in ((1 << 27, 1 << 20) if k == 4999 else (1 << 27,)):
            full, half, s0, s1 = _both(kind, mg, adj, k, slab, precision=prec)
            assert s1["mirror"] and "prefilter_fallback" not in s1
            assert torch.equal(full, half), (kind, prec, k, slab)
            assert s1["candidates_scored"] == s0["candidates_scored"] == C


@pytest.mark.timeout(600)
def test_guards_keep_the_full_path(graphs):
    from edge_proposal_sets_b200 import filter_step
    from edge_proposal_sets_b200.graph import SparseAdj
    adj = graphs["fb"]
    run = lambda name, a, **kw: filter_step.filter_topk(name, _heuristic_model(name), None, a, stats=kw.pop("st"), **kw)
    # weighted adjacency: weighted AA / CN is not bit-symmetric
    w = SparseAdj(adj.rowptr, adj.col, torch.full((adj.nnz,), 2.0, device=DEV), adj.n)
    for kw in (dict(a=w, k=3000), dict(a=adj, k=3000, owners=(100, 5000)), dict(a=adj, k=3000, per_node=4),
               dict(a=adj, k=None)):
        a = kw.pop("a")
        st0, st1 = {}, {}
        auto = run("adamic_ogb", a, st=st0, **kw)
        full = run("adamic_ogb", a, st=st1, mirror=False, **kw)
        assert st0["mirror"] is False and torch.equal(auto, full), kw
        assert st0["candidates_scored"] == st0["pairs_evaluated"]
    # an adjacency that is not structurally symmetric (one direction of a few edges dropped)
    n = 50
    rowptr = torch.tensor([0] + [3] * n, dtype=torch.int32, device=DEV)
    col = torch.tensor([1, 2, 3], dtype=torch.int32, device=DEV)
    one_way = SparseAdj(rowptr, col, None, n)
    st = {}
    filter_step.filter_topk("simple", _heuristic_model("simple"), None, one_way, k=10, stats=st)
    assert st["mirror"] is False


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from edge_proposal_sets_b200 import filter_step, models
        from util import synth_graph as sg, to_adj as ta
        s, ei, w, g = sg("small")
        adj = ta(g, dev)
        m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="simple")
        ok = True
        for name, model in (("simple", m), ("adamic_ogb", None)):
            st = {}
            single = filter_step.filter_topk(name, model, None, adj, k=4000, mirror=False)
            sharded = filter_step.filter_topk(name, model, None, adj, k=4000, distributed=True, slab_pairs=100000,
                                              stats=st)
            ok = ok and st["mirror"] and torch.equal(single, sharded)
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_gpu_mirror_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=280)
        assert p.exitcode == 0
    assert dict(out) == {0: True, 1: True}
