"""K2 tensor-core arm (tcgen05, fp16 operands under a power-of-two scale, fp32 accumulate) vs the fp64 oracle
and the fp32 arm.

Stated tolerance on these (default-init-like) models (DESIGN.md): |sigmoid(score) - fp64 oracle| <= 3e-4 absolute
and the logit within 2e-3 * (1 + |logit|); the ordering statistics below quantify what that does to a top-k.
The filter step does not rely on this number: it calibrates and verifies the deviation per job (filter_step.py)."""
import numpy as np
import pytest
import torch

from oracle import gnn as ognn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _setup(H, L, n, M, seed=0, scale=0.5):
    sd = ognn.random_state_dict("gcn", n, 0, H, L, seed=seed + 1)
    rng = np.random.default_rng(seed)
    h = (rng.standard_normal((n, H)) * scale).astype(np.float32)
    e = rng.integers(0, n, size=(2, M))
    Ws = [sd[f"linkpred.lins.{i}.weight"].to(DEV) for i in range(L)]
    bs = [sd[f"linkpred.lins.{i}.bias"].to(DEV) for i in range(L)]
    return sd, h, e, Ws, bs


@pytest.mark.timeout(120)
@pytest.mark.parametrize("H,L,M", [(256, 2, 128), (256, 2, 70001), (256, 3, 40000), (128, 3, 5000), (64, 2, 999),
                                   (64, 2, 150001), (128, 4, 120000), (256, 3, 9000)])
def test_tc_arm_vs_oracle(H, L, M):
    from edge_proposal_sets_b200 import ops
    sd, h, e, Ws, bs = _setup(H, L, 5000, M)
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    got = ops.linkpred_mlp(hd, ed, Ws, bs, "f16").cpu().numpy()
    want = ognn.linkpred_forward(torch.from_numpy(h), e, sd, L, torch.float64).numpy()
    assert np.isfinite(got).all()
    assert np.max(np.abs(got - want)) <= 3e-4
    logit = ops.linkpred_mlp(hd, ed, Ws, bs, "f16", sigmoid=False).cpu().numpy()
    want_l = ognn.linkpred_forward(torch.from_numpy(h), e, sd, L, torch.float64, return_logit=True).numpy()
    print(f"H={H} L={L}: max |sigmoid dev| {np.max(np.abs(got - want)):.2e}, max logit dev / (1+|logit|) "
          f"{np.max(np.abs(logit - want_l) / (1 + np.abs(want_l))):.2e}")
    assert np.max(np.abs(logit - want_l) / (1 + np.abs(want_l))) <= 2e-3
    # determinism: same inputs -> same bits
    again = ops.linkpred_mlp(hd, ed, Ws, bs, "f16").cpu().numpy()
    assert np.array_equal(got, again)


@pytest.mark.timeout(120)
def test_tc_arm_matches_f16_rounded_oracle_tightly():
    """With the oracle fed the SAME rounded operands — fp16(fp16(h_u s) * fp16(h_v s)) with the arm's
    power-of-two scale s (ops.tc_scale restates the device rule), fp16 weights, fp16 hidden activations
    carried times S = s^2, biases times S — the only difference left is fp32 accumulation order: the kernel
    must agree to ~1e-5, which pins layouts, descriptors and the scale handling exactly."""
    from edge_proposal_sets_b200 import ops
    H, L, M = 256, 3, 20000
    sd, h, e, Ws, bs = _setup(H, L, 3000, M, seed=3)
    hd = torch.from_numpy(h).to(DEV)
    hs, S = ops.tc_scale(hd, Ws, bs)
    assert S == hs * hs and S >= 1.0
    f16 = lambda t: t.to(torch.float16).to(torch.float64)
    ht = torch.from_numpy(h) * hs
    z = f16((f16(ht[e[0]]) * f16(ht[e[1]])).float())
    for i in range(L - 1):
        z = torch.relu(z @ f16(sd[f"linkpred.lins.{i}.weight"]).t() + S * sd[f"linkpred.lins.{i}.bias"].double())
        if i < L - 2:
            z = f16(z.float())
    want = (z @ sd[f"linkpred.lins.{L-1}.weight"].double().t()).reshape(-1) / S + sd[f"linkpred.lins.{L-1}.bias"].double()
    got = ops.linkpred_mlp(hd, torch.from_numpy(e).to(DEV), Ws, bs, "f16", sigmoid=False)
    err = np.abs(got.cpu().numpy() - want.numpy())
    print("f16-rounded oracle: max err", err.max(), "scale", hs)
    assert err.max() <= 5e-5 * (1 + np.abs(want.numpy()).max())


@pytest.mark.timeout(120)
@pytest.mark.parametrize("hmag,wmag", [(1e-3, 1.0), (30.0, 1.0), (0.5, 40.0), (200.0, 0.02)])
def test_tc_arm_scale_keeps_fp16_in_range(hmag, wmag):
    """Tiny and huge embeddings / weights: the device-computed scale keeps every fp16 operand finite and
    inside the normal range, so the arm stays as accurate (relative to the logit's scale) as on benign inputs."""
    from edge_proposal_sets_b200 import ops
    H, L, M = 256, 3, 30000
    sd, h, e, Ws, bs = _setup(H, L, 3000, M, seed=13, scale=hmag)
    Ws = [w * wmag for w in Ws[:-1]] + [Ws[-1]]
    for i in range(L - 1):
        sd[f"linkpred.lins.{i}.weight"] = sd[f"linkpred.lins.{i}.weight"] * wmag
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    got = ops.linkpred_mlp(hd, ed, Ws, bs, "f16", sigmoid=False).cpu().numpy()
    want = ognn.linkpred_forward(torch.from_numpy(h), e, sd, L, torch.float64, return_logit=True).numpy()
    assert np.isfinite(got).all()
    spread = np.abs(want - np.median(want)).max() + 1e-30
    print(f"hmag {hmag} wmag {wmag}: scale {ops.tc_scale(hd, Ws, bs)}, max err / logit spread = {np.abs(got - want).max() / spread:.2e}")
    assert np.abs(got - want).max() <= 4e-3 * spread + 2e-5 * (1 + np.abs(want).max())


@pytest.mark.timeout(120)
def test_tc_arm_ranking_quality():
    from edge_proposal_sets_b200 import ops
    H, L, M, k = 256, 3, 200000, 20000
    sd, h, e, Ws, bs = _setup(H, L, 4000, M, seed=5)
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    tc = ops.linkpred_mlp(hd, ed, Ws, bs, "f16", sigmoid=False)
    fp = ops.linkpred_mlp(hd, ed, Ws, bs, "fp32", sigmoid=False)
    top_tc = set(ops.topk(tc, k)[0].cpu().numpy().tolist())
    top_fp = set(ops.topk(fp, k)[0].cpu().numpy().tolist())
    overlap = len(top_tc & top_fp) / k
    print(f"top-{k} overlap tensor-core-vs-fp32 arm: {overlap:.4f}")
    assert overlap >= 0.995


@pytest.mark.timeout(120)
@pytest.mark.parametrize("H,L", [(256, 3), (256, 2), (128, 3), (64, 2)])
def test_tc_arm_score_is_a_function_of_the_pair_only(H, L):
    """Long pair lists gather from an fp16 copy of h, short ones read the fp32 rows and round them in
    registers; tiles, clusters and ring stages differ too.  Same pair -> same bits, always."""
    from edge_proposal_sets_b200 import ops
    n, M = 3000, 40000                                   # M >= 2n: table path
    sd, h, e, Ws, bs = _setup(H, L, n, M, seed=9)
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    full = ops.linkpred_mlp(hd, ed, Ws, bs, "f16", sigmoid=False)
    for lo, hi in [(0, 5000), (12345, 12345 + 777), (M - 300, M)]:      # M' < 2n: fp32-source path
        part = ops.linkpred_mlp(hd, ed[:, lo:hi].contiguous(), Ws, bs, "f16", sigmoid=False)
        assert torch.equal(part, full[lo:hi])


@pytest.mark.timeout(120)
@pytest.mark.parametrize("H,L,M", [(256, 3, 300001), (128, 2, 77777), (64, 2, 262144)])
def test_tc_arm_owner_major_list_vs_oracle(H, L, M):
    """An owner-major list with ascending u inside an owner, like the candidate slabs: long runs of one staged owner
    row per tile, on the fp16-table path."""
    from edge_proposal_sets_b200 import ops
    n = 6000
    sd, h, e, Ws, bs = _setup(H, L, n, M, seed=7)
    order = np.lexsort((e[0], e[1]))
    e = e[:, order]
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    got = ops.linkpred_mlp(hd, ed, Ws, bs, "f16").cpu().numpy()
    want = ognn.linkpred_forward(torch.from_numpy(h), e, sd, L, torch.float64).numpy()
    assert np.max(np.abs(got - want)) <= 3e-4


@pytest.mark.timeout(120)
def test_tc_context_reuses_table_and_weight_images():
    """ops.LinkpredTC (scale, fp16 table + weight images built once, EPS_MLP_REUSE_WORKSPACE afterwards) returns the
    bits of the one-shot call for every slab of a series — longer, shorter and short-list (M < 2n) ones."""
    from edge_proposal_sets_b200 import ops
    H, L, n = 256, 3, 3000
    sd, h, e, Ws, bs = _setup(H, L, n, 90000, seed=11)
    hd, ed = torch.from_numpy(h).to(DEV), torch.from_numpy(e).to(DEV)
    ctx = ops.LinkpredTC(hd, Ws, bs)
    for lo, hi in [(0, 40000), (40000, 90000), (100, 20100), (5, 1005), (0, 90000)]:
        part = ed[:, lo:hi].contiguous()
        assert torch.equal(ctx.score(part), ops.linkpred_mlp(hd, part, Ws, bs, "f16"))
    assert ctx.prepared
    assert torch.equal(ctx.score(ed, sigmoid=False), ops.linkpred_mlp(hd, ed, Ws, bs, "f16", sigmoid=False))


@pytest.mark.timeout(180)
def test_tc_arm_scores_do_not_depend_on_list_structure():
    """The tensor-core arm's score is a function of (h, weights, u, v) only: where a pair sits in the list (inside a
    long owner run, at a run boundary, in a tile with more owners than the staged-row cache holds) must not change
    its bits."""
    from edge_proposal_sets_b200 import ops
    H, L, n = 256, 3, 6000
    sd, h, _, Ws, bs = _setup(H, L, n, 8, seed=11)
    hd = torch.from_numpy(h).to(DEV)
    rng = np.random.default_rng(5)
    # owner runs of very different lengths: 1 .. 700 pairs, ascending u inside a run (what K6 emits), then a random tail
    lens = rng.integers(1, 700, size=120)
    v = np.repeat(rng.permutation(n)[:120], lens)
    u = np.concatenate([np.sort(rng.integers(0, n, size=l)) for l in lens])
    tail = rng.integers(0, n, size=(2, 3000))
    e = np.concatenate([np.stack([u, v]), tail], axis=1)
    ed = torch.from_numpy(e).to(DEV)
    assert e.shape[1] >= 2 * n                                  # the fp16-table path
    base = ops.linkpred_mlp(hd, ed, Ws, bs, "f16")
    ref = ops.linkpred_mlp(hd, ed, Ws, bs, "fp32")
    assert float((base - ref).abs().max()) <= 3e-4
    # the same pairs in a different order (shuffled: every tile has many owners) score the same
    perm = torch.randperm(ed.shape[1], device=DEV)
    got = ops.linkpred_mlp(hd, ed[:, perm].contiguous(), Ws, bs, "f16")
    assert torch.equal(got, base[perm])
