"""The Local Path index on the GPU: the fused one-pass walk (full and upper triangle, any owner range) and the pair
kernel bit for bit against the numpy / scipy oracle on four graphs; the filter step's lists against a stable sort of
the oracle scores, with mirror mode, per-node budgets and a multi-job call; the filter.py -> rank.py flow; two GPUs
against one."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from local_path_oracle import local_path_pairs, local_path_score, local_path_counts
from oracle import graph as og, ranking as orank
from per_node_oracle import per_node_topk
from similarity_oracle import candidates_with_counts
from util import golden_graph, spread_linkpred, synth_graph, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _special_graph():
    """A hub, self loops, isolated nodes and a clique."""
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
    """The collab shape in miniature: integer edge weights kept on the graph (the score must ignore them)."""
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
    res = {}
    for k, g in out.items():
        cand, cnt = candidates_with_counts(g)
        c2, c3 = local_path_counts(g, cand)
        assert np.array_equal(c2, cnt)
        res[k] = (g, to_adj(g, DEV), cand, cnt, c3, local_path_score(cnt, c3))
    return res


def _bits(t):
    return t.cpu().numpy().view(np.uint32) if torch.is_tensor(t) else np.asarray(t, np.float32).view(np.uint32)


def _model():
    from edge_proposal_sets_b200 import models
    return models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="local_path")


@pytest.mark.timeout(900)
@pytest.mark.parametrize("gname", ["twitch", "fb", "special", "weighted"])
def test_fused_and_pairs_bit_exact_against_oracle(graphs, gname):
    from edge_proposal_sets_b200 import candidates, ops
    g, adj, cand, cnt, c3, sc = graphs[gname]
    assert (adj.val is not None) == (gname == "weighted")
    e, s, c2, k3 = candidates.two_hop_local_path(adj)
    assert np.array_equal(e.cpu().numpy(), cand)
    assert np.array_equal(c2.cpu().numpy(), cnt) and np.array_equal(k3.cpu().numpy(), c3), gname
    assert np.array_equal(_bits(s), sc.view(np.uint32)), gname
    # candidates and c2 equal today's CN call
    ecn, _, ccn = candidates.two_hop_scored(adj, None, want_count=True, use_values=False)
    assert torch.equal(ecn, e) and torch.equal(ccn, c2)
    e2, s2, cc2, off = candidates.two_hop_scored(adj, kind="local_path", want_count=True, want_offsets=True)
    assert torch.equal(e2, e) and torch.equal(s2.view(torch.int32), s.view(torch.int32)) and torch.equal(cc2, c2)
    assert int(off[-1]) == e.shape[1]
    # upper triangle = the full kernel above the diagonal
    he, hs, h2, h3 = candidates.two_hop_local_path(adj, upper=True)
    keep = e[0] > e[1]
    assert torch.equal(he, e[:, keep]) and torch.equal(hs.view(torch.int32), s[keep].view(torch.int32))
    assert torch.equal(h2, c2[keep]) and torch.equal(h3, k3[keep])
    # owner ranges (slabs) concatenate to the full list, in both modes
    cuts = [0, 1, adj.n // 7, adj.n // 2, adj.n - 1, adj.n]
    for upper, (fe, fs) in ((False, (e, s)), (True, (he, hs))):
        parts = [candidates.two_hop_local_path(adj, a, b, upper=upper) for a, b in zip(cuts[:-1], cuts[1:])]
        assert torch.equal(torch.cat([p[0] for p in parts], 1), fe)
        assert torch.equal(torch.cat([p[1] for p in parts]).view(torch.int32), fs.view(torch.int32))
    # the pair kernel on the candidates (shuffled) and on arbitrary pairs: u == v, edges, isolated ends
    rng = np.random.default_rng(1)
    sel = rng.choice(cand.shape[1], min(cand.shape[1], 400_000), replace=False)
    pc = e[:, torch.from_numpy(sel).to(DEV)]
    ps, p2, p3 = ops.local_path(adj, pc, want_counts=True)
    assert torch.equal(ps.view(torch.int32), s[torch.from_numpy(sel).to(DEV)].view(torch.int32))
    assert torch.equal(p2, c2[torch.from_numpy(sel).to(DEV)]) and torch.equal(p3, k3[torch.from_numpy(sel).to(DEV)])
    rows = np.repeat(np.arange(g.n), np.diff(g.rowptr))
    arb = np.concatenate([rng.integers(0, g.n, (2, 3000)), np.stack([rows[:500], g.col[:500]]),
                          np.array([[0, 5, 17, g.n - 1], [0, 5, 17, g.n - 1]])], 1).astype(np.int64)
    ws, w2, w3 = local_path_pairs(g, arb)
    gs, g2, g3 = ops.local_path(adj, torch.from_numpy(arb).to(DEV), want_counts=True)
    assert np.array_equal(g2.cpu().numpy(), w2) and np.array_equal(g3.cpu().numpy(), w3)
    assert np.array_equal(_bits(gs), ws.view(np.uint32))
    assert torch.equal(_model()(None, torch.from_numpy(arb).to(DEV), adj).view(torch.int32), gs.view(torch.int32))


def _tie_k(s):
    eq = np.flatnonzero(s[1:] == s[:-1])
    return int(eq[len(eq) // 2]) + 1 if eq.size else 1


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("gname", ["fb", "special", "weighted"])
def test_filter_topk_against_stable_sort(graphs, gname):
    from edge_proposal_sets_b200 import filter_step
    g, adj, cand, cnt, c3, sc = graphs[gname]
    C = cand.shape[1]
    order = orank.stable_order_desc(sc)
    for k, slab in [(1, 1 << 27), (1, 1 << 14), (_tie_k(sc[order]), 1 << 16), (_tie_k(sc[order]), 1 << 27),
                    (C - 1, 1 << 27), (C - 1, 1 << 16), (C + 7, 1 << 18)]:
        want = orank.sorted_edges(cand, sc, k)
        st0, st1 = {}, {}
        full = filter_step.filter_topk("local_path", _model(), None, adj, k=k, slab_pairs=slab, stats=st0, mirror=False)
        assert np.array_equal(full.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, k, slab)
        half = filter_step.filter_topk("local_path", _model(), None, adj, k=k, slab_pairs=slab, stats=st1)
        assert st1["mirror"] and not st0["mirror"] and torch.equal(full, half), (gname, k, slab)
        assert st0["candidates_scored"] == st1["candidates_scored"] == C
    for m in (1, 5):
        for slab in (1 << 14, 1 << 27):
            got = filter_step.filter_topk("local_path", _model(), None, adj, k=None, per_node=m, slab_pairs=slab)
            want = per_node_topk(cand, sc, m)
            assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, m, slab)


def _gcn(n):
    import argparse
    from edge_proposal_sets_b200 import models
    from oracle import gnn as ognn
    sd = ognn.random_state_dict("gcn", n, 0, 256, 3, seed=7)
    args = argparse.Namespace(model="gcn", dataset="x", num_layers=3, hidden_channels=256, dropout=0.0,
                              use_feature=False, use_learnable_embedding=True)

    class D:
        num_nodes = n
        x = None
    mg = models.build_model(args, D, DEV)
    mg.load_state_dict(sd)
    mg.eval()
    return mg


@pytest.mark.timeout(900)
def test_multi_job_call_equals_single_jobs(graphs):
    """CN + LP + GCN in one call: LP takes the fused walk, CN goes to K3, GCN to K2; each list equals its own call."""
    from edge_proposal_sets_b200 import candidates, filter_step, models
    adj = graphs["fb"][1]
    mg = _gcn(adj.n)
    edges = candidates.two_hop(adj)
    pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(edges.shape[1], 100_000, replace=False))).to(DEV)
    spread_linkpred(mg, None, adj, edges[:, pick].contiguous())
    cn = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="simple")
    for mirror in (False, None):
        jobs = [("simple", cn), ("local_path", _model()), ("gcn", mg)]
        out = filter_step.filter_topk_multi(jobs, None, adj, k=20000, slab_pairs=1 << 19, mirror=mirror)
        for (name, mdl), got in zip(jobs, out):
            assert torch.equal(got, filter_step.filter_topk(name, mdl, None, adj, k=20000, mirror=mirror)), (name, mirror)
    with pytest.raises(ValueError):
        filter_step.filter_topk_multi([("local_path", _model()), ("local_path", _model())], None, adj, k=10)


@pytest.mark.timeout(600)
def test_cli_filter_then_rank_local_path(tmp_path, graphs):
    env = dict(os.environ, PYTHONPATH=ROOT)
    k = 100000
    r = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "filter.py"), "--dataset", "twitch", "--model",
                        "local_path", "--checkpoint", "twitch_local_path||0|0.pt", "--topk", str(k)], cwd=tmp_path,
                       env=env, capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-2000:]
    got = torch.load(tmp_path / "filtered_edges" / "twitch_local_path__0_0_sorted_edges.pt").numpy()
    g, adj, cand, cnt, c3, sc = graphs["twitch"]
    want = orank.sorted_edges(cand, sc, k)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    r2 = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "rank.py"), "--dataset", "twitch", "--model",
                         "local_path", "--sorted_edge_path", "twitch_local_path__0_0_sorted_edges.pt",
                         "--num_sorted_edge", str(k), "--runs", "1"], cwd=tmp_path, env=env, capture_output=True,
                        text=True, timeout=280)
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
        m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="local_path")
        single = filter_step.filter_topk("local_path", m, None, adj, k=4000, mirror=False)
        ok = True
        for mirror in (False, None):
            sharded = filter_step.filter_topk("local_path", m, None, adj, k=4000, distributed=True, slab_pairs=100000,
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
