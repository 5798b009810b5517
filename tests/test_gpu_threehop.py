"""Distance-3 candidates on the GPU: eps_threehop_onepass (full and upper triangle, owner ranges, tiny slabs and a
single owner above the slab size) bit for bit against the scipy oracle on four graphs; the GCN filter lists at hops=3
against a stable sort of the fp32 scores of the oracle candidates, with the prefilter, mirror mode and per-node
budgets; the filter.py --hops 3 -> rank.py flow; two GPUs against one."""
import argparse
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import graph as og, ranking as orank
from per_node_oracle import per_node_topk
from threehop_oracle import three_hop_candidates
from util import golden_graph, spread_linkpred, synth_graph, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _special_graph():
    """A hub, self loops, isolated nodes, a clique and a bipartite component (a 10-cycle with pendant paths)."""
    rng = np.random.default_rng(5)
    n = 3000
    pairs = [(0, int(u)) for u in rng.choice(np.arange(1, 2500), 1500, replace=False)]
    pairs += [(int(a), int(b)) for a, b in rng.integers(1, 2500, (2500, 2)) if a != b]
    pairs += [(5, 5), (17, 17), (2999, 2999), (2998, 2998)]
    pairs += [(a, b) for a in range(2600, 2612) for b in range(a + 1, 2612)]
    cyc = list(range(2700, 2710))
    pairs += [(cyc[i], cyc[(i + 1) % 10]) for i in range(10)] + [(2700, 2750), (2750, 2751), (2705, 2760)]
    p = np.asarray(pairs, np.int64)
    ei = np.concatenate([p.T, p[:, ::-1].T], 1)
    return og.add_edges("x", ei, np.ones(ei.shape[1], np.float32), np.zeros((2, 0), np.int64), n)


@pytest.fixture(scope="module")
def graphs():
    out = {"twitch": golden_graph("twitch")[2], "fb": golden_graph("fb")[2], "special": _special_graph()}
    return {k: (g, to_adj(g, DEV, keep_values=False), three_hop_candidates(g)) for k, g in out.items()}


def _keys(e, n):
    return e[1].long() * n + e[0].long()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("gname", ["twitch", "fb", "special"])
def test_enumeration_bit_exact_against_oracle(graphs, gname):
    from edge_proposal_sets_b200 import candidates, filter_step
    g, adj, cand = graphs[gname]
    e, off = candidates.three_hop(adj, want_offsets=True)
    assert e.dtype == torch.int32 and np.array_equal(e.cpu().numpy(), cand), gname
    assert np.array_equal(off.diff().cpu().numpy(), np.bincount(cand[1], minlength=g.n)) and int(off[0]) == 0
    # the 2-hop set is a subset
    assert bool(torch.isin(_keys(candidates.two_hop(adj), adj.n), _keys(e, adj.n)).all())
    # upper triangle = the full list above the diagonal, with its own offsets
    he, hoff = candidates.three_hop(adj, want_offsets=True, upper=True)
    keep = e[0] > e[1]
    assert torch.equal(he, e[:, keep]) and torch.equal(hoff.diff(), torch.bincount(e[1][keep].long(), minlength=adj.n))
    # owner ranges and slabs (tiny ones, and single owners far above the slab size) concatenate to the full lists
    cuts = [0, 1, adj.n // 7, adj.n // 2, adj.n - 1, adj.n]
    for upper, full in ((False, e), (True, he)):
        parts = [candidates.three_hop(adj, a, b, upper=upper) for a, b in zip(cuts[:-1], cuts[1:])]
        assert torch.equal(torch.cat(parts, 1), full), (gname, upper)
        for slab in (1 << 12, 1 << 20):
            parts = [candidates.three_hop(adj, lo, hi, cap=cap, upper=upper)
                     for lo, hi, cap in filter_step.iter_slabs(adj, 0, adj.n, slab, upper, hops=3)]
            assert torch.equal(torch.cat(parts, 1), full), (gname, upper, slab)
    # the hub owner in a slab of its own, the slab size far below its bound
    b0 = int(candidates.owner_bounds(adj, hops=3)[0])
    slabs = list(filter_step.iter_slabs(adj, 0, 3, max(b0 // 100, 1), hops=3))
    assert slabs[0][:2] == (0, 1) and slabs[0][2] == b0
    assert torch.equal(torch.cat([candidates.three_hop(adj, lo, hi, cap=cap) for lo, hi, cap in slabs], 1),
                       e[:, e[1] < 3])


@pytest.mark.timeout(900)
def test_collab_shape_owner_range():
    from edge_proposal_sets_b200 import candidates, filter_step
    s, ei, w, g = synth_graph("collab")
    adj = to_adj(g, DEV, keep_values=False)
    order = torch.argsort(candidates.owner_bounds(adj, hops=3), descending=True)
    hub = int(order[0])
    for lo, hi in ((hub, hub + 1), (0, 300), (g.n // 2, g.n // 2 + 300)):
        want = three_hop_candidates(g, lo, hi, block=32)
        for upper in (False, True):
            w_ = want[:, want[0] > want[1]] if upper else want
            got = candidates.three_hop(adj, lo, hi, upper=upper)
            assert np.array_equal(got.cpu().numpy(), w_), (lo, hi, upper)
            parts = [candidates.three_hop(adj, a, b, cap=c, upper=upper)
                     for a, b, c in filter_step.iter_slabs(adj, lo, hi, 1 << 14, upper, hops=3)]
            assert torch.equal(torch.cat(parts, 1), got)


def _gcn(n):
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


def _tie_k(s):
    eq = np.flatnonzero(s[1:] == s[:-1])
    return int(eq[len(eq) // 2]) + 1 if eq.size else 1


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("gname", ["fb", "special"])
def test_gcn_lists_against_stable_sort(graphs, gname):
    from edge_proposal_sets_b200 import filter_step
    g, adj, cand = graphs[gname]
    mg = _gcn(adj.n)
    ce = torch.from_numpy(cand).to(DEV)
    pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(cand.shape[1], 100_000, replace=False))).to(DEV)
    spread_linkpred(mg, None, adj, ce[:, pick].contiguous())
    with torch.no_grad():
        s32 = mg.linkpred.score_pairs(mg.embed(None, adj), ce, "fp32").cpu().numpy()
    del ce
    C = cand.shape[1]
    order = orank.stable_order_desc(s32)
    for k, slab in [(1, 1 << 27), (777, 1 << 18), (_tie_k(s32[order]), 1 << 20), (C - 1, 1 << 27), (C + 7, 1 << 22)]:
        want = orank.sorted_edges(cand, s32, k)
        st = {}
        fp32 = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=slab, precision="fp32", mirror=False,
                                       hops=3, stats=st)
        assert np.array_equal(fp32.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, k, slab)
        assert st["hops"] == 3 and not st["mirror"] and st["candidates_scored"] == C
        for prec in ("fp32", "prefilter"):
            st = {}
            half = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=slab, precision=prec, hops=3, stats=st)
            assert st["mirror"] and st["hops"] == 3 and torch.equal(half, fp32), (gname, k, slab, prec)
        if k < C:
            pre = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=slab, precision="prefilter",
                                          mirror=False, hops=3)
            assert torch.equal(pre, fp32), (gname, k, slab)
    for m in (1, 5):
        want = per_node_topk(cand, s32, m)
        for prec, slab in (("fp32", 1 << 16), ("prefilter", 1 << 27)):
            got = filter_step.filter_topk("gcn", mg, None, adj, k=None, per_node=m, slab_pairs=slab, precision=prec,
                                          hops=3)
            assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32)), (gname, m, prec)
    # hops=2 is unchanged by the option
    assert torch.equal(filter_step.filter_topk("gcn", mg, None, adj, k=1000, precision="fp32"),
                       filter_step.filter_topk("gcn", mg, None, adj, k=1000, precision="fp32", hops=2))


@pytest.mark.timeout(900)
def test_cli_filter_hops3_then_rank(tmp_path, graphs):
    from edge_proposal_sets_b200.data import get_data
    from oracle import gnn as ognn
    env = dict(os.environ, PYTHONPATH=ROOT)
    _, _, split_edge, data = get_data(argparse.Namespace(dataset="twitch", use_feature=True), "cpu")
    sd = ognn.random_state_dict("sage", data.num_nodes, data.x.shape[1], 256, 3, seed=4)
    (tmp_path / "models").mkdir()
    for run in range(3):
        torch.save(sd, tmp_path / "models" / f"twitch_sage||0|{run}.pt")
    k = 40000

    def filt(run, *extra):
        r = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "filter.py"), "--dataset", "twitch", "--model",
                            "sage", "--checkpoint", f"twitch_sage||0|{run}.pt", "--topk", str(k), *extra],
                           cwd=tmp_path, env=env, capture_output=True, text=True, timeout=280)
        assert r.returncode == 0, r.stderr[-3000:]
        return r, torch.load(tmp_path / "filtered_edges" / f"twitch_sage__0_{run}_sorted_edges.pt")

    r3, got3 = filt(0, "--hops", "3")
    g, adj, cand = graphs["twitch"]
    assert f"using {cand.shape[1]} edges" in r3.stdout
    assert got3.dtype == torch.float32 and got3.shape == (k, 3) and bool((got3[1:, 2] <= got3[:-1, 2]).all())
    key = got3[:, 1].long().numpy() * g.n + got3[:, 0].long().numpy()
    assert np.isin(key, cand[1].astype(np.int64) * g.n + cand[0]).all()
    two = og.two_hop_candidates(g)
    assert not np.isin(key, two[1].astype(np.int64) * g.n + two[0]).all()      # distance-3 pairs made the list
    _, got_default = filt(1)
    _, got2 = filt(2, "--hops", "2")
    assert torch.equal(got_default, got2) and not torch.equal(got_default, got3)
    r2 = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "rank.py"), "--dataset", "twitch", "--model", "simple",
                         "--sorted_edge_path", "twitch_sage__0_0_sorted_edges.pt", "--num_sorted_edge", str(k),
                         "--runs", "1"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=280)
    assert r2.returncode == 0, r2.stderr[-3000:]
    assert "Hits@50" in r2.stdout


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
        from edge_proposal_sets_b200 import models
        from edge_proposal_sets_b200 import filter_step
        from oracle import gnn as ognn
        from util import synth_graph as sg, to_adj as ta
        s, ei, w, g = sg("small")
        adj = ta(g, dev, keep_values=False)
        args = argparse.Namespace(model="gcn", dataset="x", num_layers=3, hidden_channels=256, dropout=0.0,
                                  use_feature=False, use_learnable_embedding=True)

        class D:
            num_nodes = g.n
            x = None
        mg = models.build_model(args, D, dev)
        mg.load_state_dict(ognn.random_state_dict("gcn", g.n, 0, 256, 3, seed=7))
        mg.eval()
        single = filter_step.filter_topk("gcn", mg, None, adj, k=4000, precision="fp32", mirror=False, hops=3)
        ok = True
        for mirror in (False, None):
            sharded = filter_step.filter_topk("gcn", mg, None, adj, k=4000, distributed=True, slab_pairs=100000,
                                              precision="fp32", mirror=mirror, hops=3)
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
