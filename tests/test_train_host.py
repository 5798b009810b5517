"""Host-side pieces of the training path (SURVEY §8f row 4) on CPU tensors: positive/negative edge
construction (train_and_eval.py:43-56), transposed CSR values for the SpMM backward, the PyG-2.x
checkpoint layout, and the run log against the reference's own logger.py."""
import contextlib
import io
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import refshim
from edge_proposal_sets_b200 import autograd, train_step
from edge_proposal_sets_b200.graph import SparseAdj, add_edges
from edge_proposal_sets_b200.rank_step import RunLog
from util import GOLDEN


def _graph(n=60, m=200, seed=0, dataset="x"):
    g = torch.Generator().manual_seed(seed)
    e = torch.randint(0, n, (2, m), generator=g)
    e = e[:, e[0] != e[1]]
    w = torch.randint(1, 4, (e.shape[1],), generator=g).float()
    return add_edges(dataset, e, w, torch.zeros([2, 0], dtype=torch.long), n)


def test_to_undirected_sorted_unique_both_directions():
    e = torch.tensor([[3, 1, 3, 0], [1, 3, 1, 2]])
    got = train_step.to_undirected(e, 5)
    assert got.tolist() == [[0, 1, 2, 3], [2, 3, 0, 1]]


def test_negative_sampling_returns_distinct_non_edges():
    adj = _graph()
    g = torch.Generator().manual_seed(1)
    neg = train_step.negative_sampling(adj, 500, g)
    assert neg.shape[0] == 2 and 0 < neg.shape[1] <= 500
    dense = torch.zeros(adj.n, adj.n, dtype=torch.bool)
    dense[adj.row(), adj.col.long()] = True
    assert not dense[neg[0], neg[1]].any()
    key = neg[0] * adj.n + neg[1]
    assert torch.unique(key).numel() == key.numel()
    # a nearly complete graph cannot yield more negatives than it has non-edges
    n = 6
    full = torch.tensor([[i, j] for i in range(n) for j in range(n) if i != j]).t()
    k6 = add_edges("x", full, torch.ones(full.shape[1]), torch.zeros([2, 0], dtype=torch.long), n)
    neg = train_step.negative_sampling(k6, 100, g)
    assert neg.shape[1] <= n and bool((neg[0] == neg[1]).all())      # only the self pairs are left


def test_transposed_values_match_dense_transpose():
    adj = _graph(dataset="collab")
    assert adj.val is not None
    rowptr, col, val = adj.gcn_norm()
    vt = autograd.transposed_values(rowptr, col, val, adj.n)
    dense = torch.zeros(adj.n, adj.n)
    row = torch.repeat_interleave(torch.arange(adj.n), (rowptr[1:] - rowptr[:-1]).long())
    dense[row, col.long()] = val
    dense_t = torch.zeros(adj.n, adj.n)
    dense_t[row, col.long()] = vt
    assert torch.equal(dense_t, dense.t())
    assert not torch.equal(vt, val)          # (w*dinv_i)*dinv_j is not bitwise symmetric in general


def test_gcnconv_accepts_pyg2_checkpoint_layout():
    from edge_proposal_sets_b200.models import GCN
    m = GCN(12, 8, 8, 2, 0.0)
    sd = {}
    for k, v in m.state_dict().items():
        sd[k.replace(".weight", ".lin.weight")] = v.t().contiguous().clone() if k.endswith(".weight") else v.clone()
    assert "convs.0.lin.weight" in sd and sd["convs.0.lin.weight"].shape == (8, 12)
    m2 = GCN(12, 8, 8, 2, 0.0)
    m2.load_state_dict(sd)
    for k in m.state_dict():
        assert torch.equal(m.state_dict()[k], m2.state_dict()[k])


def test_link_loss_formula():
    p, q = torch.tensor([0.9, 0.5]), torch.tensor([0.2, 0.4, 0.1])
    want = -(np.log(np.array([0.9, 0.5]) + 1e-8).mean()) - np.log(1 - np.array([0.2, 0.4, 0.1]) + 1e-8).mean()
    assert float(train_step.link_loss(p, q)) == pytest.approx(want, rel=1e-6)


def test_runlog_prints_the_stored_logger_output():
    """RunLog on the results stored in tests/golden/runlog.json prints what the file says and takes the same curve
    point.  The file records its source: written from RunLog itself, because the reference's logger.py was not
    available then, it pins RunLog's output on every checkout; the test below ties it to the reference."""
    gold = json.load(open(os.path.join(GOLDEN, "runlog.json")))
    ours = RunLog(len(gold["results"]))
    for run, rows in enumerate(gold["results"]):
        for r in rows:
            ours.add_result(run, r)

    def cap(*a):
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            ours.print_statistics(*a)
        return buf.getvalue()
    for run in range(len(gold["results"])):
        assert cap(run) == gold["printed"][str(run)]
    assert cap() == gold["printed"]["all"]
    cp = ours.curve_point(1, 77)
    assert [cp[0], float(cp[1]), float(cp[2])] == gold["curve_point_run1"]


@pytest.mark.skipif(not refshim.available(), reason="/root/reference not present")
def test_runlog_prints_what_the_reference_logger_prints():
    sys.path.insert(0, refshim.REFERENCE_ROOT)
    import importlib
    ref_logger = importlib.import_module("logger")
    assert os.path.abspath(ref_logger.__file__).startswith(refshim.REFERENCE_ROOT)
    rng = np.random.default_rng(0)
    ours, ref = RunLog(3), ref_logger.Logger(3)
    for run in range(3):
        for _ in range(5):
            r = tuple(float(v) for v in rng.random(3))
            ours.add_result(run, r)
            ref.add_result(run, r)

    def cap(fn, *a):
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            fn(*a)
        return buf.getvalue()
    for run in range(3):
        assert cap(ours.print_statistics, run) == cap(ref.print_statistics, run)
    assert cap(ours.print_statistics) == cap(ref.print_statistics)
    res = 100 * torch.tensor(ref.results[1])
    am = res[:, 1].argmax().item()
    cp = ours.curve_point(1, 77)
    assert cp[0] == 77 and float(cp[1]) == float(res[am, 1]) and float(cp[2]) == float(res[am, 2])
    from oracle.make_golden_models import runlog_vectors
    want = runlog_vectors(ref_logger.Logger, "")
    gold = json.load(open(os.path.join(GOLDEN, "runlog.json")))
    for key in ("results", "printed", "curve_point_run1"):
        assert gold[key] == want[key], f"tests/golden/runlog.json differs from the reference ({key}): python -m oracle.make_golden_models"
