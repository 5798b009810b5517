"""Shared helpers for the tests: golden fixtures -> oracle CSR and product SparseAdj."""
import os

import numpy as np
import torch

from oracle import graph as og

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    """The arrays of tests/golden/{name}.npz (graph split, whole-set checksums) and {name}_sample.npz (the
    reference's scores on a seeded sample of candidates), in one mapping."""
    z = dict(np.load(os.path.join(GOLDEN, f"{name}.npz")))
    z.update(np.load(os.path.join(GOLDEN, f"{name}_sample.npz")))
    return z


def undirected(train, n):
    """to_undirected as the bundled datasets store edge_index (twitch/data.py:116)."""
    train = np.asarray(train, dtype=np.int64)
    r = np.concatenate([train[:, 0], train[:, 1]])
    c = np.concatenate([train[:, 1], train[:, 0]])
    key = np.unique(r * n + c)
    return np.stack([key // n, key % n])


def golden_graph(name):
    z = load_golden(name)
    n = int(z["n"])
    ei = undirected(z["train_edges"], n)
    g = og.add_edges(name, ei, np.ones(ei.shape[1], np.float32), np.zeros((2, 0), np.int64), n)
    return z, ei, g


def to_adj(g: og.CSR, device, keep_values=None):
    from edge_proposal_sets_b200.graph import SparseAdj
    if keep_values is None:
        keep_values = not bool(np.all(g.val == 1.0))
    val = torch.from_numpy(g.val.astype(np.float32)).to(device) if keep_values else None
    return SparseAdj(torch.from_numpy(g.rowptr.astype(np.int32)).to(device),
                     torch.from_numpy(g.col.astype(np.int32)).to(device), val, g.n)


def synth_graph(name, dataset=None, scale=1.0):
    from edge_proposal_sets_b200 import synth
    s = synth.make_shape(name, scale)
    ei = synth.undirected_edge_index(s["train_edges"])
    w = np.ones(ei.shape[1], np.float32) if s["edge_weight"] is None else np.concatenate([s["edge_weight"]] * 2)
    g = og.add_edges(dataset or name, ei, w, np.zeros((2, 0), np.int64), s["n"])
    return s, ei, w, g


def tiny_graphs():
    """Hand-checkable graphs (SURVEY §8c pin 4): path, star, clique, deg-1 leaves, isolated nodes."""
    out = {}
    out["path5"] = (5, np.array([[0, 1], [1, 2], [2, 3], [3, 4]]))
    out["star6"] = (6, np.array([[0, i] for i in range(1, 6)]))
    out["clique5"] = (5, np.array([[i, j] for i in range(5) for j in range(i + 1, 5)]))
    # two triangles sharing node 2, a pendant leaf 5 on node 4, isolated nodes 6,7
    out["mixed8"] = (8, np.array([[0, 1], [1, 2], [0, 2], [2, 3], [3, 4], [2, 4], [4, 5]]))
    return out


def csr_from_undirected(n, und_edges, dataset="x", weight=None):
    e = np.asarray(und_edges, dtype=np.int64)
    ei = np.concatenate([e.T, e[:, ::-1].T], axis=1)
    w = np.ones(ei.shape[1], np.float32) if weight is None else np.concatenate([weight, weight]).astype(np.float32)
    return og.add_edges(dataset, ei, w, np.zeros((2, 0), np.int64), n)


def spread_linkpred(model, x, adj, sample_edges):
    """Give a seeded random LinkGNN the score spread of a TRAINED filter model (what bench.py does to its synthetic
    model): zero hidden biases and He-uniform hidden weights in the LinkPredictor, output layer rescaled so that the
    fp32 logits of ``sample_edges`` have mean -2 and std 2.  With nn.Linear's default init every candidate scores
    the same to ~1e-4 and a top-k boundary means nothing."""
    from edge_proposal_sets_b200 import ops
    lins = model.linkpred.lins
    with torch.no_grad():
        for lin in lins[:-1]:
            lin.weight.mul_(6.0 ** 0.5)
            lin.bias.zero_()
        lins[-1].bias.zero_()
        h = model.embed(x, adj)
        logit = ops.linkpred_mlp(h, sample_edges, [l.weight for l in lins], [l.bias for l in lins], "fp32", sigmoid=False)
        mean, std = float(logit.double().mean()), float(logit.double().std())
        scale = 2.0 / max(std, 1e-30)
        lins[-1].weight.mul_(scale)
        lins[-1].bias.fill_(-mean * scale - 2.0)
    model._h_key = None
    return model
