"""The C-ABI library loads on a GPU-less host and exports every symbol include/eps.h declares."""
import ctypes as C
import os
import re

import pytest

from edge_proposal_sets_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "eps.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(eps_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree():
    assert header_functions() == sorted(_lib.SIGNATURES)


def test_library_exports_every_declared_symbol():
    if not os.path.exists(_lib.LIB_PATH):
        from edge_proposal_sets_b200 import build
        build.build()
    lib = C.CDLL(_lib.LIB_PATH)
    for name in header_functions():
        assert hasattr(lib, name), f"{name} declared in include/eps.h but not exported"
    assert _lib.load().eps_version() == _lib.EPS_VERSION


def test_argument_validation_needs_no_device():
    lib = _lib.load()
    # null pointers / bad sizes are rejected before any CUDA call
    assert lib.eps_cn_aa(None, None, None, None, 10, None, None, 5, 0, None, None, None, 0, None) == -1
    assert b"null" in lib.eps_last_error()
    assert lib.eps_topk_f32(None, 10, 3, None, None, None, 0, None) == -1
    assert lib.eps_spmm_csr_f32(None, None, None, None, None, 4, 8, 0, None, 0, None, 0, None) == -1
    assert lib.eps_topk_workspace_bytes(1 << 20, 1000) > 0
    assert lib.eps_linkpred_workspace_bytes(1000, 256, 3, 5000, 0) >= 256
    assert lib.eps_linkpred_workspace_bytes(1000, 256, 3, 5000, 1) >= 256 + 2 * 256 * 256 * 2 + 1000 * 256 * 2
    # on the fp16-table path (M >= 2n) the size does not depend on M: ops.LinkpredTC sizes one buffer for a whole series
    assert len({lib.eps_linkpred_workspace_bytes(1000, 256, 3, M, 1) for M in (2000, 5000, 1 << 20, 1 << 33)}) == 1


def test_no_cpu_fallback():
    import torch
    from edge_proposal_sets_b200 import ops
    from edge_proposal_sets_b200.graph import SparseAdj
    adj = SparseAdj(torch.tensor([0, 1, 2], dtype=torch.int32), torch.tensor([1, 0], dtype=torch.int32), None, 2)
    with pytest.raises(_lib.EpsError):
        ops.cn_aa(adj, torch.tensor([[0], [1]]))
    with pytest.raises(_lib.EpsError):
        ops.topk(torch.zeros(4), 2)
