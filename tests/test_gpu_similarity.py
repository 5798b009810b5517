"""Degree-normalised similarity scores on the GPU: the fused K6+K3 epilogue (full and upper triangle), the two-pass
entry point, K3 grouped and K3 pairs bit for bit against the numpy oracle; the filter step's lists against a stable
sort of the oracle scores, with mirror mode, per-node budgets and weighted graphs; the filter.py -> rank.py flow;
two GPUs against one."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import graph as og, ranking as orank
from per_node_oracle import per_node_topk
from similarity_oracle import SIMILARITY_KINDS, candidates_with_counts, similarity_pairs
from util import golden_graph, synth_graph, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _special_graph():
    """A hub, self loops, isolated nodes and a clique (as in the mirror tests)."""
    rng = np.random.default_rng(3)
    n = 3000
    pairs = [(0, int(u)) for u in rng.choice(np.arange(1, 2500), 1800, replace=False)]
    pairs += [(int(a), int(b)) for a, b in rng.integers(1, 2500, (6000, 2)) if a != b]
    pairs += [(5, 5), (17, 17), (2999, 2999), (2998, 2998)]
    pairs += [(a, b) for a in range(2600, 2612) for b in range(a + 1, 2612)]
    pairs += [(2990, 10), (2991, 10), (2992, 2990)]
    p = np.asarray(pairs, np.int64)
    ei = np.concatenate([p.T, p[:, ::-1].T], 1)
    return og.add_edges("x", ei, np.ones(ei.shape[1], np.float32), np.zeros((2, 0), np.int64), n)


def _weighted_graph():
    """The collab shape in miniature: integer edge weights kept on the graph (the scores must ignore them)."""
    s, ei, w, g = synth_graph("small", dataset="collab")
    m = ei.shape[1] // 2
    wts = np.random.default_rng(4).integers(1, 5, m).astype(np.float32)
    return og.add_edges("collab", ei, np.concatenate([wts, wts]), np.zeros((2, 0), np.int64), s["n"])


@pytest.fixture(scope="module")
def graphs():
    out = {}
    for gold in ("twitch", "fb"):
        out[gold] = golden_graph(gold)[2]
    out["special"] = _special_graph()
    out["weighted"] = _weighted_graph()
    return {k: (g, to_adj(g, DEV)) + candidates_with_counts(g) for k, g in out.items()}


def _bits(t):
    return t.cpu().numpy().view(np.uint32) if torch.is_tensor(t) else np.asarray(t, np.float32).view(np.uint32)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("gname", ["twitch", "fb", "special", "weighted"])
def test_fused_and_k3_bit_exact_against_oracle(graphs, gname):
    from edge_proposal_sets_b200 import candidates, ops
    g, adj, cand, cnt = graphs[gname]
    assert (adj.val is not None) == (gname == "weighted")
    rng = np.random.default_rng(1)
    arb = torch.from_numpy(np.concatenate([rng.integers(0, g.n, (2, 3000)),
                                           np.array([[0, 5, 2700, 2701, 17], [2700, 5, 2701, 2701, 17]]) % g.n], 1)).to(DEV)
    for kind in SIMILARITY_KINDS:
        e, s, c = candidates.two_hop_scored(adj, kind=kind, want_count=True)
        assert np.array_equal(e.cpu().numpy(), cand) and np.array_equal(c.cpu().numpy(), cnt)
        want = similarity_pairs(g, cand, kind, counts=cnt)
        assert np.array_equal(_bits(s), want.view(np.uint32)), (gname, kind)
        # upper triangle = the full kernel above the diagonal
        he, hs = candidates.two_hop_scored(adj, kind=kind, upper=True)
        keep = e[0] > e[1]
        assert torch.equal(he, e[:, keep]) and torch.equal(hs.view(torch.int32), s[keep].view(torch.int32)), kind
        # K3 grouped and K3 pairs on the candidates, K3 pairs on arbitrary pairs (zero denominators included)
        for grouped in (True, False):
            k3 = ops.cn_aa(adj, e, kind=kind, grouped_by_v=grouped)
            assert torch.equal(k3.view(torch.int32), s.view(torch.int32)), (gname, kind, grouped)
        pa = ops.cn_aa(adj, arb, kind=kind)
        assert np.array_equal(_bits(pa), similarity_pairs(g, arb.cpu().numpy().astype(np.int64), kind).view(np.uint32))
    iso = np.flatnonzero(np.diff(g.rowptr) == 0)
    if iso.size:
        z = torch.tensor([[int(iso[0])], [0]], device=DEV)
        assert all(float(ops.cn_aa(adj, z, kind=kind)[0]) == 0.0 for kind in SIMILARITY_KINDS)


def _model(kind):
    from edge_proposal_sets_b200 import models
    return models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=kind)


def _tie_k(s):
    eq = np.flatnonzero(s[1:] == s[:-1])
    return int(eq[len(eq) // 2]) + 1 if eq.size else 1


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("gname", ["fb", "weighted", "special"])
def test_filter_topk_against_stable_sort(graphs, gname):
    from edge_proposal_sets_b200 import candidates, filter_step
    g, adj, cand, cnt = graphs[gname]
    C = cand.shape[1]
    for kind in SIMILARITY_KINDS:
        sc = similarity_pairs(g, cand, kind, counts=cnt)
        order = orank.stable_order_desc(sc)
        ks = [(1, 1 << 27), (4999, 1 << 27), (_tie_k(sc[order]), 1 << 16), (C, 1 << 27), (C + 7, 1 << 18)]
        for k, slab in ks:
            want = orank.sorted_edges(cand, sc, k)
            st0, st1 = {}, {}
            full = filter_step.filter_topk(kind, _model(kind), None, adj, k=k, slab_pairs=slab, stats=st0, mirror=False)
            assert np.array_equal(full.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, kind, k, slab)
            half = filter_step.filter_topk(kind, _model(kind), None, adj, k=k, slab_pairs=slab, stats=st1)
            assert st1["mirror"] and torch.equal(full, half), (gname, kind, k, slab)
        # per-node budgets
        for m in (1, 5):
            got = filter_step.filter_topk(kind, _model(kind), None, adj, k=None, per_node=m, slab_pairs=1 << 16)
            want = per_node_topk(cand, sc, m)
            assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, kind, m)


@pytest.mark.timeout(600)
def test_second_job_takes_k3(graphs):
    """Two heuristic jobs in one call: the first takes the fused kernel, the second K3 on the same candidates."""
    from edge_proposal_sets_b200 import filter_step
    adj = graphs["fb"][1]
    jobs = [("jaccard", _model("jaccard")), ("salton", _model("salton")), ("simple", _model("simple"))]
    out = filter_step.filter_topk_multi(jobs, None, adj, k=3000, slab_pairs=1 << 18)
    for (name, mdl), got in zip(jobs, out):
        assert torch.equal(got, filter_step.filter_topk(name, mdl, None, adj, k=3000)), name


@pytest.mark.timeout(600)
def test_cli_filter_then_rank_jaccard(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    k = 100000
    r = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "filter.py"), "--dataset", "twitch", "--model", "jaccard",
                        "--checkpoint", "twitch_jaccard||0|0.pt", "--topk", str(k)], cwd=tmp_path, env=env,
                       capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-2000:]
    out = tmp_path / "filtered_edges" / "twitch_jaccard__0_0_sorted_edges.pt"
    got = torch.load(out).numpy()
    z, ei, g = golden_graph("twitch")
    cand, cnt = candidates_with_counts(g)
    want = orank.sorted_edges(cand, similarity_pairs(g, cand, "jaccard", counts=cnt), k)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    r2 = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "rank.py"), "--dataset", "twitch", "--model", "jaccard",
                         "--sorted_edge_path", "twitch_jaccard__0_0_sorted_edges.pt", "--num_sorted_edge", str(k),
                         "--runs", "1"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=280)
    assert r2.returncode == 0, r2.stderr[-2000:]
    assert "Hits@50" in r2.stdout and len(list((tmp_path / "curves").glob("*.pt"))) == 1


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
        ok = True
        for name in ("jaccard", "preferential_attachment"):
            m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=name)
            single = filter_step.filter_topk(name, m, None, adj, k=4000, mirror=False)
            for mirror in (False, None):
                sharded = filter_step.filter_topk(name, m, None, adj, k=4000, distributed=True, slab_pairs=100000,
                                                  mirror=mirror)
                ok = ok and torch.equal(single, sharded)
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_gpu_matches_single_gpu():
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
