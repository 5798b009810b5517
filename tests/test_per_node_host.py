"""Per-node proposal budgets on the host: the oracle against a brute-force per-owner loop, the filter.py flag,
and the argument checks of the K4c entry points (no device needed)."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import ranking as orank
from per_node_oracle import per_node_topk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _brute_force(e, s, m, k):
    """Every owner's m best by (score desc, candidate index asc), then all kept rows by the same rule."""
    keep = []
    for v in np.unique(e[1]):
        idx = np.flatnonzero(e[1] == v)
        best = sorted(idx.tolist(), key=lambda i: (-float(s[i] + np.float32(0.0)), i))[:m]
        keep.extend(best)
    keep.sort(key=lambda i: (-float(s[i] + np.float32(0.0)), i))
    keep = keep[:k] if k is not None else keep
    return np.array([[e[0, i], e[1, i], s[i]] for i in keep], dtype=np.float32).reshape(-1, 3)


@pytest.mark.parametrize("m", [1, 2, 3, 7, 1000])
@pytest.mark.parametrize("k", [None, 1, 50, 100000])
def test_oracle_per_node_topk_matches_brute_force(m, k):
    rng = np.random.default_rng(m * 7 + (k or 0))
    n_own = 60
    sizes = rng.integers(0, 25, n_own)
    sizes[[3, 17]] = 0                                        # owners without candidates
    v = np.repeat(np.arange(n_own), sizes)
    u = np.concatenate([np.sort(rng.choice(500, size=c, replace=False)) for c in sizes])
    e = np.stack([u, v]).astype(np.int64)
    s = rng.geometric(0.5, size=v.size).astype(np.float32)  # CN-like: heavy ties
    s[rng.integers(0, v.size, 20)] = -0.0
    s[rng.integers(0, v.size, 20)] = 0.0
    got = per_node_topk(e, s, m, k)
    want = _brute_force(e, s, m, k)
    assert got.dtype == np.float32 and np.array_equal(got, want)
    # no owner holds more than m rows; with k=None every owner keeps min(count, m)
    owners, cnt = np.unique(got[:, 1].astype(np.int64), return_counts=True)
    assert np.all(cnt <= m)
    if k is None:
        assert got.shape[0] == int(np.minimum(sizes, m).sum())


def test_oracle_per_node_topk_large_budget_is_the_global_list():
    rng = np.random.default_rng(1)
    v = np.sort(rng.integers(0, 40, 3000))
    e = np.stack([rng.integers(0, 1000, 3000), v])
    s = rng.geometric(0.4, size=3000).astype(np.float32)
    assert np.array_equal(per_node_topk(e, s, 3000, 700), orank.sorted_edges(e, s, 700))
    assert np.array_equal(per_node_topk(e, s, 3000), orank.sorted_edges(e, s))


def _filter_cli():
    spec = importlib.util.spec_from_file_location("filter_cli", os.path.join(ROOT, "filter.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_filter_cli_per_node_topk_flag():
    cli = _filter_cli()
    base = ["--dataset", "fb", "--model", "simple", "--checkpoint", "fb_simple||0|0.pt"]
    assert cli.parse_args(base).per_node_topk is None
    a = cli.parse_args(base + ["--per_node_topk", "10", "--topk", "500"])
    assert a.per_node_topk == 10 and a.topk == 500
    for bad in ("0", "-3", "x"):
        with pytest.raises(SystemExit):
            cli.parse_args(base + ["--per_node_topk", bad])


def test_segment_topk_argument_validation_needs_no_device():
    from edge_proposal_sets_b200 import _lib
    lib = _lib.load()
    ws = lib.eps_segment_topk_workspace_bytes(100)
    assert ws >= 256 and lib.eps_segment_topk_workspace_bytes(0) >= 256
    # null pointers, m < 1 and inconsistent sizes are rejected before any CUDA call
    assert lib.eps_segment_topk_select(None, 10, None, 2, 3, 0.0, 0, None, None, 0, None) == -1
    assert b"null" in lib.eps_last_error()
    buf = (np.zeros(64, np.uint8)).ctypes.data                # any non-null address: never dereferenced here
    assert lib.eps_segment_topk_select(buf, 10, None, 2, 3, 0.0, 0, buf, buf, ws, None) == -1
    assert b"null" in lib.eps_last_error()
    assert lib.eps_segment_topk_select(buf, 10, buf, 2, 0, 0.0, 0, buf, buf, ws, None) == -1
    assert b"m out of range" in lib.eps_last_error()
    assert lib.eps_segment_topk_select(buf, 10, buf, 0, 3, 0.0, 0, buf, buf, ws, None) == -1
    assert b"inconsistent" in lib.eps_last_error()
    assert lib.eps_segment_topk_select(buf, 10, buf, -1, 3, 0.0, 0, buf, buf, ws, None) == -1
    assert lib.eps_segment_topk_select(buf, 10, buf, 2, 3, -1.0, 1, buf, buf, ws, None) == -1
    assert b"margin" in lib.eps_last_error()
    assert lib.eps_segment_topk_write(None, None, None, 10, None, 2, None, None, None, None, None, 0, None) == -1
    assert b"null" in lib.eps_last_error()
    assert lib.eps_segment_topk_write(buf, buf, buf, 10, buf, 2, buf, None, None, None, buf, ws, None) == -1
    assert b"null" in lib.eps_last_error()


def test_segment_topk_wrapper_has_no_cpu_fallback():
    import torch
    from edge_proposal_sets_b200 import _lib, ops
    with pytest.raises(_lib.EpsError):
        ops.segment_topk(torch.zeros(4), torch.zeros((2, 4), dtype=torch.int32), torch.tensor([0, 4]), 2)
