"""K3 (CN / AA / RA) and K6 (candidate enumeration) on the GPU vs the oracle and the golden
vectors produced by the reference itself.  Bit-exact for counts and — because the kernels add the
fp32 terms exactly (64-bit fixed point) and round once, the oracle's order="exact" — for fp32 AA too
when given the oracle's weight table; <=1e-5 relative against the reference's own outputs."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import graph as og, heuristics as oh, ranking as orank
from util import csr_from_undirected, golden_graph, synth_graph, tiny_graphs, to_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t.to(dtype) if dtype else t).to(DEV)


@pytest.fixture(scope="module", params=["twitch", "fb"])
def gold(request):
    z, ei, g = golden_graph(request.param)
    return request.param, z, g, to_adj(g, DEV)


@pytest.mark.parametrize("grouped", [False, True])
def test_sample_vs_reference_golden(gold, grouped):
    from edge_proposal_sets_b200 import ops
    name, z, g, adj = gold
    e = _dev(z["sample_edges"])
    score, cnt = ops.cn_aa(adj, e, None, grouped_by_v=grouped, want_count=True)
    assert np.array_equal(cnt.cpu().numpy(), z["sample_cn"])                       # bit-exact CN
    assert np.array_equal(score.cpu().numpy(), z["sample_cn"].astype(np.float32))
    w = _dev(oh.aa_ogb_weights(g))
    aa = ops.cn_aa(adj, e, w, grouped_by_v=grouped).cpu().numpy()
    # bit-exact against the oracle's exact-sum-rounded-once restatement (the kernels' contract) ...
    assert np.array_equal(aa, oh.aa_ogb_pairs(g, z["sample_edges"].astype(np.int64), order="exact"))
    # ... and within the north_star tolerance of the reference's own output (numpy's reduceat
    # switches to pairwise summation for >= 9 common neighbours, so the last bits can differ)
    ref0 = z["sample_aa"]
    assert np.all(np.abs(aa - ref0) <= 1e-5 * np.abs(ref0))
    few = z["sample_cn"] <= 2       # reduceat computes t0 + (t1 + t2 + ...): same bits up to 2 terms
    assert np.array_equal(aa[few], ref0[few])
    aa_dev = ops.cn_aa(adj, e, adj.aa_ogb_weights(), grouped_by_v=grouped).cpu().numpy()
    ref = z["sample_aa"]
    assert np.all(np.abs(aa_dev - ref) <= 1e-5 * np.abs(ref) + 1e-12)              # north_star tolerance
    ra = ops.cn_aa(adj, e, adj.ra_weights(), grouped_by_v=grouped).cpu().numpy()
    assert np.all(np.abs(ra - z["sample_ra"]) <= 1e-5 * np.abs(z["sample_ra"]) + 1e-12)


def test_models_api_simple_adamic(gold):
    from edge_proposal_sets_b200 import adamic_utils, models
    name, z, g, adj = gold
    e = _dev(z["sample_edges"][:, :5000], torch.int64)                              # reference passes int64 [2,B]
    m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="simple")
    assert np.array_equal(m(None, e, adj).cpu().numpy(), z["sample_cn"][:5000].astype(np.float32))
    m = models.CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="adamic")
    got = m(None, e, adj).cpu().numpy()
    want = oh.adamic_sigmoid_pairs(g, z["sample_edges"][:, :5000].astype(np.int64))
    assert np.max(np.abs(got - want)) <= 1e-6
    pred, edge = adamic_utils.AA(adamic_utils.get_A(adj, adj.n), e)
    assert edge is e and np.allclose(pred.cpu().numpy(), z["sample_aa"][:5000], rtol=1e-5, atol=0)
    ra = adamic_utils.resource_allocation(adj, e.t())
    assert np.allclose(ra.cpu().numpy(), z["sample_ra"][:5000], rtol=1e-5, atol=0)


def test_full_candidate_set_properties(gold):
    """Full size (twitch: 25,556,294 pairs): K6 reproduces the reference's candidate list byte for
    byte, the CN checksum, the AA checksum and the exact CN top-k proposal list."""
    from edge_proposal_sets_b200 import candidates, ops
    name, z, g, adj = gold
    edges = candidates.two_hop(adj)
    N = int(z["num_candidates"])
    assert edges.shape == (2, N)
    assert hashlib.sha256(edges.t().contiguous().t().cpu().numpy().tobytes()).hexdigest() == str(z["cand_sha256"])
    score, cnt = ops.cn_aa(adj, edges, None, grouped_by_v=True, want_count=True)
    assert int(cnt.long().sum()) == int(z["sum_cn"]) and int(cnt.max()) == int(z["max_cn"])
    assert int(cnt.min()) >= 1                                                     # every candidate has a 2-path
    score2 = ops.cn_aa(adj, edges, None, grouped_by_v=False)
    assert torch.equal(score, score2)                                              # both kernels agree
    aa = ops.cn_aa(adj, edges, _dev(oh.aa_ogb_weights(g)), grouped_by_v=True)
    assert abs(float(aa.double().sum()) - float(z["sum_aa"])) <= 1e-7 * float(z["sum_aa"])
    assert torch.equal(aa, ops.cn_aa(adj, edges, _dev(oh.aa_ogb_weights(g)), grouped_by_v=False))
    k = int(z["topk_k"])
    top = ops.topk_edges(edges, score, k)
    uv = top[:, :2].to(torch.int32).cpu().numpy()
    assert hashlib.sha256(np.ascontiguousarray(uv).tobytes()).hexdigest() == str(z["topk_cn_sha256"])
    assert np.array_equal(uv[:64], z["topk_cn_head"]) and np.array_equal(uv[-64:], z["topk_cn_tail"])


def test_weighted_collab_graph():
    from edge_proposal_sets_b200 import ops
    s, ei, w, g = synth_graph("small", dataset="collab")
    wts = np.random.default_rng(3).integers(1, 5, size=ei.shape[1] // 2).astype(np.float32)
    g = og.add_edges("collab", ei, np.concatenate([wts, wts]), np.zeros((2, 0), np.int64), s["n"])
    adj = to_adj(g, DEV)
    assert adj.val is not None
    cand = og.two_hop_candidates(g)
    e = _dev(cand)
    for grouped in (False, True):
        got = ops.cn_aa(adj, e, None, grouped_by_v=grouped).cpu().numpy()
        assert np.array_equal(got, oh.cn_scores_pairs(g, cand))                    # integer weights: exact in any order
        aa = ops.cn_aa(adj, e, _dev(oh.aa_ogb_weights(g)), grouped_by_v=grouped).cpu().numpy()
        assert np.array_equal(aa, oh.aa_ogb_pairs(g, cand, order="exact"))
        assert np.allclose(aa, oh.aa_ogb_pairs(g, cand), rtol=1e-5, atol=0)
    # random (ungrouped, repeated, self) pairs
    rng = np.random.default_rng(4)
    rp = rng.integers(0, s["n"], size=(2, 20000))
    got, cnt = ops.cn_aa(adj, _dev(rp), None, want_count=True)
    assert np.array_equal(cnt.cpu().numpy(), oh.cn_count_pairs(g, rp))
    assert np.array_equal(got.cpu().numpy(), oh.cn_scores_pairs(g, rp))


def test_tiny_graphs_and_edge_cases():
    from edge_proposal_sets_b200 import candidates, ops
    for name, (n, e) in tiny_graphs().items():
        g = csr_from_undirected(n, e)
        adj = to_adj(g, DEV)
        cand = og.two_hop_candidates(g)
        got = candidates.two_hop(adj).cpu().numpy()
        assert np.array_equal(got, cand.astype(np.int32)), name
        if cand.shape[1] == 0:
            assert ops.cn_aa(adj, _dev(cand.astype(np.int32))).numel() == 0        # empty input
            continue
        for grouped in (False, True):
            sc, cnt = ops.cn_aa(adj, _dev(cand), _dev(oh.aa_ogb_weights(g)), grouped_by_v=grouped, want_count=True)
            assert np.array_equal(cnt.cpu().numpy(), oh.cn_count_pairs(g, cand)), name
            assert np.array_equal(sc.cpu().numpy(), oh.aa_ogb_pairs(g, cand, order="exact")), name
    # all pairs incl. isolated nodes and (u,u)
    n, e = tiny_graphs()["mixed8"]
    g = csr_from_undirected(n, e)
    adj = to_adj(g, DEV)
    allp = np.stack(np.meshgrid(np.arange(n), np.arange(n), indexing="ij")).reshape(2, -1)
    for grouped in (False, True):
        cnt = ops.cn_aa(adj, _dev(allp), None, grouped_by_v=grouped, want_count=True)[1].cpu().numpy()
        assert np.array_equal(cnt, oh.cn_count_pairs(g, allp))


@pytest.mark.parametrize("shape", ["tiny", "small"])
def test_candidate_enumeration_vs_oracle(shape):
    from edge_proposal_sets_b200 import candidates
    s, ei, w, g = synth_graph(shape)
    adj = to_adj(g, DEV)
    cand = og.two_hop_candidates(g)
    got = candidates.two_hop(adj)
    assert np.array_equal(got.cpu().numpy(), cand.astype(np.int32))
    # owner-range slabs concatenate to the full list
    mid = s["n"] // 3
    parts = [candidates.two_hop(adj, 0, mid), candidates.two_hop(adj, mid, s["n"])]
    assert torch.equal(torch.cat(parts, 1), got)
    counts = candidates.owner_counts(adj).cpu().numpy()
    assert np.array_equal(counts, np.bincount(cand[1], minlength=s["n"]))


# ---------------------------------------------------------------------------------------------
# K6+K3 fused: candidates and scores from one walk over the 2-paths
# ---------------------------------------------------------------------------------------------

def test_fused_twohop_scored_full_golden(gold):
    """Full candidate set of twitch / fb: same list (sha256), CN / AA / RA bit-identical to K3 on the
    enumerated pairs, checksums and the exact CN top-k list of the golden file."""
    from edge_proposal_sets_b200 import candidates, ops
    name, z, g, adj = gold
    w = _dev(oh.aa_ogb_weights(g))
    edges, aa, cnt = candidates.two_hop_scored(adj, w, want_count=True)
    N = int(z["num_candidates"])
    assert edges.shape == (2, N)
    assert hashlib.sha256(edges.t().contiguous().t().cpu().numpy().tobytes()).hexdigest() == str(z["cand_sha256"])
    assert int(cnt.long().sum()) == int(z["sum_cn"]) and int(cnt.max()) == int(z["max_cn"]) and int(cnt.min()) >= 1
    aa3, cnt3 = ops.cn_aa(adj, edges, w, grouped_by_v=True, want_count=True)
    assert torch.equal(cnt, cnt3) and torch.equal(aa, aa3)                         # fused == per-pair kernel, bit for bit
    assert abs(float(aa.double().sum()) - float(z["sum_aa"])) <= 1e-7 * float(z["sum_aa"])
    e2, cn_score = candidates.two_hop_scored(adj, None)
    assert torch.equal(e2, edges) and torch.equal(cn_score, cnt.float())
    e3, ra = candidates.two_hop_scored(adj, adj.ra_weights())
    assert torch.equal(ra, ops.cn_aa(adj, edges, adj.ra_weights(), grouped_by_v=True))
    e4, sg = candidates.two_hop_scored(adj, w, sigmoid=True)
    assert torch.equal(sg, ops.cn_aa(adj, edges, w, sigmoid=True, grouped_by_v=True))
    k = int(z["topk_k"])
    uv = ops.topk_edges(edges, cn_score, k)[:, :2].to(torch.int32).cpu().numpy()
    assert hashlib.sha256(np.ascontiguousarray(uv).tobytes()).hexdigest() == str(z["topk_cn_sha256"])
    # the sampled pairs of the golden file: the reference's own AA within the north_star tolerance
    pos = _dev(z["sample_index"])
    assert np.array_equal(edges[:, pos].cpu().numpy(), z["sample_edges"])
    got = aa[pos].cpu().numpy()
    assert np.all(np.abs(got - z["sample_aa"]) <= 1e-5 * np.abs(z["sample_aa"]))
    assert np.array_equal(cnt[pos].cpu().numpy(), z["sample_cn"])


@pytest.mark.parametrize("shape", ["tiny", "small"])
def test_fused_twohop_scored_vs_oracle(shape):
    from edge_proposal_sets_b200 import candidates
    s, ei, w, g = synth_graph(shape)
    adj = to_adj(g, DEV)
    cand = og.two_hop_candidates(g)
    wt = oh.aa_ogb_weights(g)
    edges, aa, cnt = candidates.two_hop_scored(adj, _dev(wt), want_count=True)
    assert np.array_equal(edges.cpu().numpy(), cand.astype(np.int32))
    assert np.array_equal(cnt.cpu().numpy(), oh.cn_count_pairs(g, cand))
    assert np.array_equal(aa.cpu().numpy(), oh.aa_ogb_pairs(g, cand, order="exact"))
    assert np.allclose(aa.cpu().numpy(), oh.aa_ogb_pairs(g, cand), rtol=1e-5, atol=0)   # reference (numpy) order
    # owner-range slabs concatenate to the full result
    mid = s["n"] // 3
    a = candidates.two_hop_scored(adj, _dev(wt), 0, mid)
    b = candidates.two_hop_scored(adj, _dev(wt), mid, s["n"])
    assert torch.equal(torch.cat([a[0], b[0]], 1), edges) and torch.equal(torch.cat([a[1], b[1]]), aa)


@pytest.mark.parametrize("shape", ["tiny", "small", "twitch"])
def test_onepass_slots(shape):
    """eps_twohop_onepass (padded per-owner slots sized by a bound, then scan + compaction): the per-owner counts are the
    oracle's, exact bounds give the default-bound results bit for bit (pairs, order, scores, counts, offsets), an owner
    sub-range is the matching slice of the full run, and a bound one too small raises."""
    from edge_proposal_sets_b200 import candidates, ops
    from edge_proposal_sets_b200._lib import EpsError
    if shape == "twitch":
        z, ei, g = golden_graph("twitch")
    else:
        s, ei, w, g = synth_graph(shape)
    adj = to_adj(g, DEV)
    wt = _dev(oh.aa_ogb_weights(g))
    cand = og.two_hop_candidates(g)
    counts = candidates.owner_counts(adj)
    assert np.array_equal(counts.cpu().numpy(), np.bincount(cand[1], minlength=adj.n))
    N = int(counts.sum())
    bound = int(candidates.owner_bounds(adj).sum())
    assert bool((candidates.owner_bounds(adj) >= counts).all()) and bound >= N
    f = candidates.two_hop_scored(adj, wt, want_count=True, want_offsets=True)
    e1 = candidates.two_hop(adj)
    assert e1.shape == (2, N) and torch.equal(e1, f[0])
    c1 = candidates.two_hop_scored(adj, None)
    assert torch.equal(c1[0], e1) and torch.equal(c1[1], f[2].float())
    assert torch.equal(c1[1], ops.cn_aa(adj, e1, None, grouped_by_v=True))
    sg1 = candidates.two_hop_scored(adj, wt, sigmoid=True)
    assert torch.equal(sg1[0], e1) and torch.equal(sg1[1], ops.cn_aa(adj, e1, wt, sigmoid=True, grouped_by_v=True))
    # offsets, a tight capacity, an owner sub-range, and a violated bound
    e, sc, cn, off = candidates._onepass(adj, wt, 0, adj.n, counts, False, True, True)   # exact bounds
    assert torch.equal(off[1:], torch.cumsum(counts, 0)) and int(off[0]) == 0
    for a, b in zip((e, sc, cn, off), f):
        assert torch.equal(a, b)
    lo, hi = adj.n // 3, (2 * adj.n) // 3
    sub = candidates.two_hop_scored(adj, wt, lo, hi, want_count=True)
    a, b = int(off[lo]), int(off[hi])
    for x, y in zip(sub, (e[:, a:b], sc[a:b], cn[a:b])):
        assert torch.equal(x, y)
    short = counts.clone()
    short[int(torch.argmax(counts))] -= 1                       # one owner's bound one too small
    with pytest.raises(EpsError):
        candidates._onepass(adj, wt, 0, adj.n, short, False, True, True)
    # repeated runs are identical (the owners' hand-out order does not reach the outputs)
    for _ in range(3):
        again = candidates.two_hop_scored(adj, wt, want_count=True, want_offsets=True)
        for a, b in zip(again, f):
            assert torch.equal(a, b)


def test_fused_twohop_scored_tiny_graphs():
    from edge_proposal_sets_b200 import candidates
    for name, (n, e) in tiny_graphs().items():
        g = csr_from_undirected(n, e)
        adj = to_adj(g, DEV)
        cand = og.two_hop_candidates(g)
        edges, sc, cnt = candidates.two_hop_scored(adj, _dev(oh.aa_ogb_weights(g)), want_count=True)
        assert np.array_equal(edges.cpu().numpy(), cand.astype(np.int32)), name
        if cand.shape[1]:
            assert np.array_equal(cnt.cpu().numpy(), oh.cn_count_pairs(g, cand)), name
            assert np.array_equal(sc.cpu().numpy(), oh.aa_ogb_pairs(g, cand, order="exact")), name
    # an empty owner range; a weighted graph with ASYMMETRIC values must raise, not fall back
    s, ei, w, g = synth_graph("tiny")
    adj = to_adj(g, DEV)
    e0, s0 = candidates.two_hop_scored(adj, None, 5, 5)
    assert e0.shape == (2, 0) and s0.numel() == 0
    from edge_proposal_sets_b200._lib import EpsError
    g.val = np.random.default_rng(0).random(g.nnz).astype(np.float32) + 0.5
    adjw = to_adj(g, DEV, keep_values=True)
    assert not candidates.values_symmetric(adjw)
    with pytest.raises(EpsError):
        candidates.two_hop_scored(adjw, None)


def test_fused_weighted_collab_equals_pairwise_kernel():
    """collab keeps edge weights: the fused one-pass kernel forms A[u,k]*(A[v,k]*w_k) per 2-path and must
    equal K3 (eps_cn_aa with values) and the oracle bit for bit — CN ('simple'), AA ('adamic_ogb'), and
    the index-only 'adamic' variant; also through filter_topk."""
    from edge_proposal_sets_b200 import candidates, filter_step, ops
    s, ei, w, g = synth_graph("small", dataset="collab")
    wts = np.random.default_rng(3).integers(1, 5, size=ei.shape[1] // 2).astype(np.float32)
    g = og.add_edges("collab", ei, np.concatenate([wts, wts]), np.zeros((2, 0), np.int64), s["n"])
    adj = to_adj(g, DEV)
    assert adj.val is not None and candidates.values_symmetric(adj)
    cand = og.two_hop_candidates(g)
    wt = _dev(oh.aa_ogb_weights(g))
    e, aa, cnt = candidates.two_hop_scored(adj, wt, want_count=True)
    assert np.array_equal(e.cpu().numpy(), cand.astype(np.int32))
    assert np.array_equal(cnt.cpu().numpy(), oh.cn_count_pairs(g, cand))
    assert np.array_equal(aa.cpu().numpy(), oh.aa_ogb_pairs(g, cand, order="exact"))
    assert torch.equal(aa, ops.cn_aa(adj, e, wt, use_values=True, grouped_by_v=True))
    e2, cn = candidates.two_hop_scored(adj, None)                                 # weighted CN
    assert np.array_equal(cn.cpu().numpy(), oh.cn_scores_pairs(g, cand))
    assert torch.equal(cn, ops.cn_aa(adj, e, None, use_values=True, grouped_by_v=True))
    e3, ad = candidates.two_hop_scored(adj, adj.adamic_weights(), sigmoid=True, use_values=False)
    assert torch.equal(ad, ops.cn_aa(adj, e, adj.adamic_weights(), use_values=False, sigmoid=True, grouped_by_v=True))
    # a non-integer but symmetric weighting (products round): still the same fp32 products as K3
    key = np.minimum(np.repeat(np.arange(g.n), np.diff(g.rowptr)), g.col) * g.n + \
        np.maximum(np.repeat(np.arange(g.n), np.diff(g.rowptr)), g.col)
    uk, inv = np.unique(key, return_inverse=True)
    g.val = (np.random.default_rng(9).random(uk.size).astype(np.float32) + 0.25)[inv]
    adj2 = to_adj(g, DEV, keep_values=True)
    assert candidates.values_symmetric(adj2)
    wt2 = _dev(oh.aa_ogb_weights(g))
    e4, aa4 = candidates.two_hop_scored(adj2, wt2)
    assert torch.equal(aa4, ops.cn_aa(adj2, e4, wt2, use_values=True, grouped_by_v=True))
    assert np.array_equal(aa4.cpu().numpy(), oh.aa_ogb_pairs(g, cand, order="exact"))
    # filter_topk takes the fused path for the weighted graph and agrees with the oracle ranking
    for model in ("simple", "adamic_ogb"):
        assert filter_step.heuristic_table(model, adj) is not None
    m = __import__("edge_proposal_sets_b200.models", fromlist=["x"]).CommonNeighborsPredictor(None, 0, None, None, None, None, model_type="adamic_ogb")
    top = filter_step.filter_topk("adamic_ogb", m, None, adj, k=5000, slab_pairs=200000).cpu().numpy()
    # (the device weight table uses CUDA logf: compare with the pairwise kernel on the same table bit for bit,
    # and with the oracle's numpy-logf scores to the north-star 1e-5)
    pair = ops.cn_aa(adj, e, adj.aa_ogb_weights(), use_values=True, grouped_by_v=True)
    assert np.array_equal(top, ops.topk_edges(e, pair, 5000).cpu().numpy())
    g1 = og.add_edges("collab", ei, np.concatenate([wts, wts]), np.zeros((2, 0), np.int64), s["n"])
    want = orank.sorted_edges(cand, oh.aa_ogb_pairs(g1, cand, order="exact"), 5000)
    assert np.allclose(top[:, 2], want[:, 2], rtol=1e-5, atol=0)
