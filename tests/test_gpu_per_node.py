"""Per-node proposal budgets on the GPU: K4c (segmented top-m select) bit-exact against the oracle, the filter step
in per-node mode on the golden graphs, its invariances, the GNN prefilter, the CLI and the two-GPU merge."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import graph as og
from per_node_oracle import per_node_topk
from util import golden_graph, spread_linkpred, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _np_key(s):
    """K4's order key: ascending key == descending score, -0.0 folded into +0.0."""
    b = (np.asarray(s, np.float32) + np.float32(0.0)).view(np.uint32).astype(np.uint64)
    asc = np.where(b >> 31, b ^ 0xFFFFFFFF, b ^ 0x80000000)
    return (~asc) & 0xFFFFFFFF


def _scores(kind, n, rng):
    if kind == "geometric":
        return rng.geometric(0.45, size=n).astype(np.float32)          # CN-like: long equal runs
    if kind == "all_equal":
        return np.full(n, 0.75, np.float32)
    if kind == "signed_zero":
        return rng.choice(np.array([0.0, -0.0, 1.0, -1.0], np.float32), size=n)
    return rng.choice(np.array([np.inf, -np.inf, 2.0, -0.0, 0.0], np.float32), size=n)


def _layout(m, big):
    sizes = [0, 1, max(m - 1, 0), m, m + 1, 0, 3, 2 * m + 7, 6144, 6145, 20000, 1]
    if big:
        sizes.insert(5, 2_100_000)                                      # larger than shared memory: streamed passes
    return np.array(sizes, np.int64)


def _run(score, sizes, m, margin=None):
    from edge_proposal_sets_b200 import ops
    M = score.size
    off = np.zeros(sizes.size + 1, np.int64)
    off[1:] = np.cumsum(sizes)
    e = np.stack([np.arange(M), np.repeat(np.arange(sizes.size), sizes)]).astype(np.int32)   # u = position, v = segment
    out, sc, kept = ops.segment_topk(torch.from_numpy(score).to(DEV), torch.from_numpy(e).to(DEV),
                                     torch.from_numpy(off).to(DEV), m, margin=margin)
    return e, off, out.cpu().numpy(), sc.cpu().numpy(), kept.cpu().numpy()


@pytest.mark.parametrize("kind", ["geometric", "all_equal", "signed_zero", "inf"])
@pytest.mark.parametrize("m", [1, 3, 100, 5000])
def test_segment_topk_exact_vs_oracle(m, kind):
    rng = np.random.default_rng(m + len(kind))
    sizes = _layout(m, big=kind in ("geometric", "signed_zero"))
    score = _scores(kind, int(sizes.sum()), rng)
    e, off, out, sc, kept = _run(score, sizes, m)
    want = per_node_topk(e, score, m)
    pos = np.sort(want[:, 0].astype(np.int64))                          # the kept set, in position order
    assert np.array_equal(out[0].astype(np.int64), pos) and np.array_equal(out[1], e[1, pos])
    assert np.array_equal(sc.view(np.uint32), score[pos].view(np.uint32))          # score bits, -0.0 kept as is
    assert np.array_equal(np.diff(kept), np.minimum(sizes, m))


@pytest.mark.parametrize("m,margin,kind", [(1, 0.0, "geometric"), (3, 0.5, "geometric"), (100, 1e-3, "sigmoid"),
                                           (5000, 2e-2, "sigmoid"), (100, 0.25, "inf")])
def test_segment_topk_band_is_the_k4b_threshold_per_segment(m, margin, kind):
    rng = np.random.default_rng(m)
    sizes = _layout(m, big=m == 100)
    n = int(sizes.sum())
    score = ((1.0 / (1.0 + np.exp(-rng.standard_normal(n) * 0.5))).astype(np.float32) if kind == "sigmoid"
             else _scores(kind, n, rng))
    e, off, out, sc, kept = _run(score, sizes, m, margin=margin)
    keys = _np_key(score)
    want = []
    for s in range(sizes.size):
        lo, hi = off[s], off[s + 1]
        if hi - lo <= m:
            want.append(np.arange(lo, hi))
            continue
        bound = np.sort(keys[lo:hi])[m - 1]                             # the m-th key of the segment
        last = bound
        if margin > 0:
            sm = np.float32(_key_score(bound))
            kt = int(_np_key(np.array([sm - np.float32(margin)], np.float32))[0])
            last = kt if kt == 0xFFFFFFFF else kt + 1                   # K4b's one ulp of slack
        want.append(lo + np.flatnonzero(keys[lo:hi] <= last))
    want = np.concatenate(want)
    assert np.array_equal(out[0].astype(np.int64), want)
    assert np.array_equal(sc.view(np.uint32), score[want].view(np.uint32))
    assert kept[-1] == want.size


def _key_score(key):
    from edge_proposal_sets_b200 import ops
    return ops.key_to_score(int(key))


def _device_scores(name, adj):
    """Scores of every candidate, in candidate order, from the fused kernel the filter step uses (pinned to the
    oracle by test_gpu_heuristics)."""
    from edge_proposal_sets_b200 import candidates, filter_step
    t = filter_step.heuristic_table(name, adj)
    edges, sc = candidates.two_hop_scored(t[0], t[1], sigmoid=t[2], use_values=t[3])
    return edges.cpu().numpy().astype(np.int64), sc.cpu().numpy()


def _heuristic_model(name):
    from edge_proposal_sets_b200 import models
    if name in ("simple", "adamic"):
        return models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type=name)
    return None


@pytest.mark.timeout(600)
@pytest.mark.parametrize("gold", ["twitch", "fb"])
def test_filter_step_per_node_vs_oracle(gold):
    from edge_proposal_sets_b200 import filter_step
    z, ei, g = golden_graph(gold)
    adj = to_adj(g, DEV)
    cand = og.two_hop_candidates(g)
    slab = 1 << 20
    for name in ("simple", "adamic", "adamic_ogb", "resource_allocation"):
        e, s = _device_scores(name, adj)
        assert np.array_equal(e, cand)
        if name == "simple":
            assert np.array_equal(s, og.two_hop_candidates(g, return_values=True)[1].astype(np.float32))
        model = _heuristic_model(name)
        m = 3
        want = per_node_topk(cand, s, m)
        st = {}
        got = filter_step.filter_topk(name, model, None, adj, k=None, slab_pairs=slab, stats=st, per_node=m)
        assert st["slabs"] > 3 and st["per_node"]["m"] == m and st["per_node"]["survivors"] == [want.shape[0]]
        assert np.array_equal(got.cpu().numpy(), want), name
        got_k = filter_step.filter_topk(name, model, None, adj, k=2000, slab_pairs=slab, per_node=m)
        assert np.array_equal(got_k.cpu().numpy(), want[:2000]), name
        # slab size does not change the result
        one = filter_step.filter_topk(name, model, None, adj, k=2000, slab_pairs=1 << 27, per_node=m)
        assert torch.equal(one, got_k), name


@pytest.mark.timeout(600)
def test_per_node_with_a_budget_above_every_owner_is_the_global_list():
    from edge_proposal_sets_b200 import candidates, filter_step
    z, ei, g = golden_graph("fb")
    adj = to_adj(g, DEV)
    big = int(candidates.owner_counts(adj).max().item())
    for name in ("simple", "adamic_ogb"):
        model = _heuristic_model(name)
        for k in (5000, None):
            glob = filter_step.filter_topk(name, model, None, adj, k=k, slab_pairs=1 << 19)
            per = filter_step.filter_topk(name, model, None, adj, k=k, slab_pairs=1 << 19, per_node=big)
            assert torch.equal(glob, per), (name, k)


def _gcn(n, H, L):
    import argparse
    from edge_proposal_sets_b200 import models
    from oracle import gnn as ognn
    sd = ognn.random_state_dict("gcn", n, 0, H, L, seed=7)
    args = argparse.Namespace(model="gcn", dataset="x", num_layers=L, hidden_channels=H, dropout=0.0,
                              use_feature=False, use_learnable_embedding=True)

    class D:
        num_nodes = n
        x = None
    mg = models.build_model(args, D, DEV)
    mg.load_state_dict(sd)
    mg.eval()
    return mg


@pytest.mark.timeout(600)
def test_gnn_per_node_prefilter_equals_fp32():
    from edge_proposal_sets_b200 import filter_step
    z, ei, g = golden_graph("twitch")
    adj = to_adj(g, DEV)
    mg = _gcn(g.n, 256, 3)
    cand = og.two_hop_candidates(g)
    pick = np.random.default_rng(0).choice(cand.shape[1], 200_000, replace=False)
    spread_linkpred(mg, None, adj, torch.from_numpy(cand[:, np.sort(pick)]).to(DEV))
    m = 10
    for k in (None, 20000):
        f32 = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=1 << 22, precision="fp32", per_node=m)
        st = {}
        pf = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=1 << 22, precision="prefilter",
                                     per_node=m, stats=st)
        assert "prefilter_fallback" not in st and st["prefilter"]["gcn"]["pool"] >= pf.shape[0]
        assert torch.equal(pf, f32), k
        f16 = filter_step.filter_topk("gcn", mg, None, adj, k=k, slab_pairs=1 << 22, precision="f16", per_node=m)
        assert f16.shape == f32.shape
        a = set(map(tuple, f32[:, :2].long().cpu().numpy().tolist()))
        b = set(map(tuple, f16[:, :2].long().cpu().numpy().tolist()))
        assert len(a & b) >= 0.95 * len(a)


@pytest.mark.timeout(280)
def test_filter_cli_per_node_topk_then_rank_prefix(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    k, m = 20000, 3
    r = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "filter.py"), "--dataset", "fb", "--model", "simple",
                        "--checkpoint", "fb_simple||0|0.pt", "--topk", str(k), "--per_node_topk", str(m)],
                       cwd=tmp_path, env=env, capture_output=True, text=True, timeout=250)
    assert r.returncode == 0, r.stderr[-2000:]
    got = torch.load(tmp_path / "filtered_edges" / "fb_simple__0_0_sorted_edges.pt").numpy()
    z, ei, g = golden_graph("fb")
    cand, cn = og.two_hop_candidates(g, return_values=True)
    assert np.array_equal(got, per_node_topk(cand, cn.astype(np.float32), m, k))
    r2 = subprocess.run([sys.executable, "-u", os.path.join(ROOT, "rank.py"), "--dataset", "fb", "--model", "simple",
                         "--sorted_edge_path", "fb_simple__0_0_sorted_edges.pt", "--num_sorted_edge", "5000",
                         "--runs", "1"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=250)
    assert r2.returncode == 0, r2.stderr[-2000:]
    assert "Using 5000 highest scoring edges" in r2.stdout and "Hits@20" in r2.stdout


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
            single = filter_step.filter_topk(name, model, None, adj, k=4000, per_node=5)
            sharded = filter_step.filter_topk(name, model, None, adj, k=4000, distributed=True, slab_pairs=100000,
                                              per_node=5)
            ok = ok and torch.equal(single, sharded)
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_gpu_per_node_matches_single_gpu():
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
