"""LinkPredictor and default_model_configs against vectors produced by EXECUTING the reference's
own models.py (oracle/make_golden_models.py -> tests/golden/linkpred_H*_L*.npz, model_configs.json)."""
import argparse
import json
import os

import numpy as np
import pytest
import torch

from oracle import gnn as ognn, refshim
from util import GOLDEN

SHAPES = [(64, 2), (256, 3), (300, 3)]
FIELDS = ["num_layers", "hidden_channels", "dropout", "batch_size", "lr", "epochs", "use_feature",
          "use_learnable_embedding"]


def _case(H, L):
    tag = f"H{H}_L{L}"
    z = np.load(os.path.join(GOLDEN, f"linkpred_{tag}.npz"))
    sd = {f"linkpred.lins.{i}.{p}": torch.from_numpy(z[f"{tag}/lins.{i}.{p}"]) for i in range(L) for p in ("weight", "bias")}
    return torch.from_numpy(z[f"{tag}/x_i"]), torch.from_numpy(z[f"{tag}/x_j"]), z[f"{tag}/y"], sd


@pytest.mark.parametrize("H,L", SHAPES)
def test_oracle_linkpred_matches_reference_vectors(H, L):
    """oracle.gnn.linkpred_forward restates models.py:478-485; the reference's own outputs pin it."""
    x_i, x_j, y, sd = _case(H, L)
    B = x_i.shape[0]
    h = torch.cat([x_i, x_j], 0)
    edges = np.stack([np.arange(B), np.arange(B) + B])
    got = ognn.linkpred_forward(h, edges, sd, L, torch.float32).numpy()
    assert y.shape == (B, 1)
    np.testing.assert_allclose(got, y[:, 0], rtol=0, atol=2e-7)
    got64 = ognn.linkpred_forward(h, edges, sd, L, torch.float64).numpy()
    np.testing.assert_allclose(got64, y[:, 0], rtol=0, atol=1e-6)


@pytest.mark.skipif(not refshim.available(), reason="/root/reference not present")
def test_linkpred_fixture_regenerates():
    """The committed vectors are what the reference produces today (same seeds, same torch)."""
    ref = refshim.reference_models_module()
    H, L = 64, 2
    x_i, x_j, y, sd = _case(H, L)
    lp = ref.LinkPredictor(H, H, 1, L, 0.5)
    lp.load_state_dict({k.replace("linkpred.", ""): v for k, v in sd.items()})
    lp.eval()
    with torch.no_grad():
        np.testing.assert_array_equal(lp(x_i, x_j).numpy(), y)


def test_default_model_configs_match_reference_table():
    """models.default_model_configs == /root/reference/models.py:673-790 for every (dataset, model)
    on the scoring path.  'ppa' has no branch in the reference (everything stays None); this build
    fills it with its own documented choice, so only the explicitly-set rows are compared there."""
    from edge_proposal_sets_b200.models import default_model_configs
    table = json.load(open(os.path.join(GOLDEN, "model_configs.json")))
    checked = 0
    for key, want in table.items():
        d, m, mode = key.split("/")
        if mode == "unset":
            if d == "ppa":
                continue
            a = argparse.Namespace(dataset=d, model=m, **{f: None for f in FIELDS})
        else:
            a = argparse.Namespace(dataset=d, model=m, num_layers=5, hidden_channels=96, dropout=0.25, batch_size=777,
                                   lr=0.5, epochs=3, use_feature=True, use_learnable_embedding=True)
        got = default_model_configs(a)
        assert {f: getattr(got, f) for f in FIELDS} == want, key
        checked += 1
    assert checked >= 78


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", SHAPES)
def test_gpu_linkpred_fp32_matches_reference_vectors(H, L):
    """K2 fp32 arm through LinkPredictor.forward(x_i, x_j) — the reference call signature."""
    from edge_proposal_sets_b200.models import LinkPredictor
    x_i, x_j, y, sd = _case(H, L)
    dev = torch.device("cuda:0")
    lp = LinkPredictor(H, H, 1, L, 0.5).to(dev)
    lp.load_state_dict({k.replace("linkpred.", ""): v for k, v in sd.items()})
    lp.eval()
    got = lp(x_i.to(dev), x_j.to(dev)).cpu().numpy()
    assert got.shape == y.shape
    np.testing.assert_allclose(got, y, rtol=0, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(64, 2), (256, 3)])
def test_gpu_linkpred_tcgen05_matches_reference_vectors(H, L):
    """K2 tcgen05 arm (fp16 operands, fp32 accumulate): |sigma - reference| <= 3e-4 (DESIGN §3)."""
    from edge_proposal_sets_b200.models import LinkPredictor
    x_i, x_j, y, sd = _case(H, L)
    dev = torch.device("cuda:0")
    lp = LinkPredictor(H, H, 1, L, 0.5).to(dev)
    lp.load_state_dict({k.replace("linkpred.", ""): v for k, v in sd.items()})
    lp.eval()
    lp.precision = "f16"
    got = lp(x_i.to(dev), x_j.to(dev)).cpu().numpy()
    np.testing.assert_allclose(got, y, rtol=0, atol=3e-4)
