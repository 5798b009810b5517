"""Generate tests/golden/linkpred_H{H}_L{L}.npz and tests/golden/model_configs.json by EXECUTING the
reference's own ``models.py`` in the build container.

TEST INFRASTRUCTURE — see ``oracle/__init__.py``.  Run from the repo root:

    python -m oracle.make_golden_models     # needs /root/reference (read-only)

What is pinned:
  * ``LinkPredictor`` (/root/reference/models.py:461-485, plain torch): for three (H, L) shapes the
    reference class is instantiated under ``torch.manual_seed``, put in eval mode and run on seeded
    ``x_i, x_j``; weights, inputs and the fp32 outputs are stored.  The oracle restatement
    (``oracle.gnn.linkpred_forward``) and the K2 kernels are held to these vectors.
  * ``default_model_configs`` (/root/reference/models.py:673-790): the resolved argument namespace
    for every (dataset, model) pair on the scoring path, with nothing set on the command line and
    with every overridable flag set.
  * ``logger.Logger`` (tests/golden/runlog.json): what it prints for three runs of seeded results and
    the curve point rank.py takes from them; ``rank_step.RunLog`` is held to it.
GCNConv / SAGEConv stay unpinned (their arithmetic lives in torch_geometric / torch_sparse, which
are absent here; the import stubs in ``refshim`` carry no arithmetic).
"""
from __future__ import annotations

import argparse
import contextlib
import importlib
import io
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import refshim  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
DATASETS = ["ddi", "collab", "reddit", "twitch", "fb", "email", "ppa"]
MODELS = ["gcn", "sage", "simple", "adamic", "adamic_ogb", "resource_allocation"]
FIELDS = ["num_layers", "hidden_channels", "dropout", "batch_size", "lr", "epochs", "use_feature",
          "use_learnable_embedding"]
SHAPES = [(64, 2, 96), (256, 3, 80), (300, 3, 40)]          # (H, L, B): tiny / ddi-collab-ppa / email


def runlog_vectors(make_logger, source: str) -> dict:
    """Feeds three runs of five seeded (train, valid, test) results to ``make_logger(3)`` and returns them with
    what its ``print_statistics(run)`` / ``print_statistics()`` print and the [index_end, valid, test] point
    rank.py:377-380 takes from run 1 at index_end 77 (the reference Logger has no method for it)."""
    rng = np.random.default_rng(0)
    results = [[[float(v) for v in rng.random(3)] for _ in range(5)] for _ in range(3)]
    log = make_logger(3)
    for run, rows in enumerate(results):
        for r in rows:
            log.add_result(run, tuple(r))

    def printed(*a):
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            log.print_statistics(*a)
        return buf.getvalue()
    res = 100 * torch.tensor(results[1])
    am = res[:, 1].argmax().item()
    return {"source": source, "results": results,
            "printed": {**{str(run): printed(run) for run in range(3)}, "all": printed()},
            "curve_point_run1": [77, float(res[am, 1]), float(res[am, 2])]}


def main():
    assert refshim.available(), "needs /root/reference"
    ref = refshim.reference_models_module()
    for H, L, B in SHAPES:
        blobs = {}
        torch.manual_seed(1000 + H + L)
        lp = ref.LinkPredictor(H, H, 1, L, 0.5)
        lp.eval()
        g = torch.Generator().manual_seed(H * 7 + L)
        x_i, x_j = torch.randn(B, H, generator=g), torch.randn(B, H, generator=g)
        with torch.no_grad():
            y = lp(x_i, x_j)
        tag = f"H{H}_L{L}"
        blobs[f"{tag}/x_i"], blobs[f"{tag}/x_j"], blobs[f"{tag}/y"] = x_i.numpy(), x_j.numpy(), y.numpy()
        for k, v in lp.state_dict().items():
            blobs[f"{tag}/{k}"] = v.numpy()
        np.savez_compressed(os.path.join(OUT, f"linkpred_{tag}.npz"), **blobs)     # one file per shape: < 1 MB each

    table = {}
    for d in DATASETS:
        for m in MODELS:
            a = argparse.Namespace(dataset=d, model=m, **{f: None for f in FIELDS})
            r = ref.default_model_configs(a)
            table[f"{d}/{m}/unset"] = {f: getattr(r, f) for f in FIELDS}
            b = argparse.Namespace(dataset=d, model=m, num_layers=5, hidden_channels=96, dropout=0.25,
                                   batch_size=777, lr=0.5, epochs=3, use_feature=True, use_learnable_embedding=True)
            r = ref.default_model_configs(b)
            table[f"{d}/{m}/set"] = {f: getattr(r, f) for f in FIELDS}
    with open(os.path.join(OUT, "model_configs.json"), "w") as f:
        json.dump(table, f, indent=0, sort_keys=True)
    ref_logger = importlib.import_module("logger")        # REFERENCE_ROOT is on sys.path (reference_models_module)
    assert os.path.abspath(ref_logger.__file__).startswith(os.path.abspath(refshim.REFERENCE_ROOT)), ref_logger.__file__
    with open(os.path.join(OUT, "runlog.json"), "w") as f:
        json.dump(runlog_vectors(ref_logger.Logger, "the reference's logger.py"), f, indent=1)
    print("wrote linkpred_H*_L*.npz, runlog.json,", len(table), "config rows")


if __name__ == "__main__":
    main()
