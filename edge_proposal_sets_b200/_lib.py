"""ctypes binding of libeps_b200.so (the C ABI declared in include/eps.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present every
compute call raises.  ``load()`` only builds the library when asked to (``EPS_AUTO_BUILD=1`` or
``build=True``); on the GPU box the prebuilt in-tree ``.so`` is what is loaded.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libeps_b200.so")

EPS_OK = 0
EPS_VERSION = 203          # must equal EPS_VERSION in include/eps.h (checked by load())
EPS_REDUCE_SUM, EPS_REDUCE_MEAN = 0, 1
EPS_CN_SIGMOID, EPS_CN_GROUPED_BY_V = 1, 2
EPS_TWOHOP_UPPER = 4       # eps_twohop_onepass: only the candidates u > v of every owner v
# degree-normalised similarity scores: a 3-bit kind field at bit 8 of the eps_cn_aa / eps_twohop_onepass flags
EPS_SCORE_KIND_SHIFT = 8
EPS_SCORE_KIND_MASK = 7 << EPS_SCORE_KIND_SHIFT
SCORE_KINDS = {"jaccard": 1, "sorensen": 2, "salton": 3, "hub_promoted": 4, "hub_depressed": 5,
               "leicht_holme_newman": 6, "preferential_attachment": 7}
EPS_MLP_FP32, EPS_MLP_TC_F16 = 0, 1
EPS_MLP_TC_BF16 = EPS_MLP_TC_F16       # round-1 name
EPS_MLP_REUSE_WORKSPACE = 0x100
EPS_CAND_SCORE_CN, EPS_CAND_SCORE_WSUM = 0, 1

_vp, _i32, _i64, _sz, _int = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t, C.c_int

# name -> (restype, argtypes); mirrors include/eps.h one to one
SIGNATURES = {
    "eps_version": (_int, []),
    "eps_last_error": (C.c_char_p, []),
    "eps_spmm_csr_f32": (_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _int, _vp, _int, _vp, _sz, _vp]),
    "eps_spmm_workspace_bytes": (_sz, []),
    "eps_gcn_norm_count": (_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "eps_gcn_norm_fill": (_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "eps_cn_aa": (_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _int, _vp, _vp, _vp, _sz, _vp]),
    "eps_cn_aa_workspace_bytes": (_sz, []),
    "eps_score_kinds": (_int, []),
    "eps_linkpred_mlp": (_int, [_vp, _i32, _i32, _vp, _vp, _i64, C.POINTER(_vp), C.POINTER(_vp), _i32,
                                _int, _int, _vp, _vp, _sz, _vp]),
    "eps_linkpred_workspace_bytes": (_sz, [_i32, _i32, _i32, _i64, _int]),
    "eps_pair_hadamard_f32": (_int, [_vp, _i32, _i32, _vp, _vp, _i64, _vp, _vp]),
    "eps_pair_hadamard_bwd_f32": (_int, [_vp, _i32, _i32, _vp, _vp, _i64, _vp, _vp, _vp]),
    "eps_topk_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "eps_topk_workspace_bytes": (_sz, [_i64, _i64]),
    "eps_pack_edges": (_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "eps_topk_select2_f32": (_int, [_vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "eps_threshold_tiles": (_i64, [_i64]),
    "eps_threshold_workspace_bytes": (_sz, [_i64]),
    "eps_threshold_count": (_int, [_vp, _i64, _vp, C.c_float, _int, _vp, _vp, _sz, _vp]),
    "eps_threshold_write": (_int, [_vp, _vp, _vp, _i64, _vp, C.c_float, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eps_segment_topk_workspace_bytes": (_sz, [_i64]),
    "eps_segment_topk_select": (_int, [_vp, _i64, _vp, _i64, _i64, C.c_float, _int, _vp, _vp, _sz, _vp]),
    "eps_segment_topk_write": (_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "eps_gather_pairs2": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "eps_twohop_onepass": (_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "eps_twohop_onepass_workspace_bytes": (_sz, [_i64, _i32]),
    "eps_local_path_onepass": (_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _i64, _i64, _i32, _int, _vp, _vp, _vp, _vp,
                                      _vp, _vp, _vp, _sz, _vp]),
    "eps_local_path_onepass_workspace_bytes": (_sz, [_i64, _i32, _i64, _i32]),
    "eps_local_path_pairs": (_int, [_vp, _vp, _i32, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "eps_local_path_pairs_workspace_bytes": (_sz, []),
    "eps_threehop_onepass": (_int, [_vp, _vp, _i32, _i32, _i32, _vp, _i64, _i64, _i32, _int, _vp, _vp, _vp, _vp, _sz,
                                    _vp]),
    "eps_threehop_onepass_workspace_bytes": (_sz, [_i64, _i32, _i64, _i32]),
    "eps_comm_unique_id": (_int, [_vp]),
    "eps_comm_init": (_int, [_vp, _int, _int, C.POINTER(_vp)]),
    "eps_comm_destroy": (_int, [_vp]),
    "eps_topk_merge_allgather": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "eps_topk_merge_workspace_bytes": (_sz, [_int, _i64, _i64]),
}

_lib = None


class EpsError(RuntimeError):
    pass


def load(build: bool | None = None) -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if build is None:
        build = os.environ.get("EPS_AUTO_BUILD", "0") == "1"
    if build or not os.path.exists(LIB_PATH):
        if not build and not os.path.exists(LIB_PATH):
            raise EpsError(
                f"{LIB_PATH} is missing: build it with `python -m edge_proposal_sets_b200.build` "
                "(there is no CPU fallback)")
        from . import build as _b
        _b.build()
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise EpsError(f"{LIB_PATH} does not export {name} (built from an older eps.h): "
                           "rebuild it with `python -m edge_proposal_sets_b200.build --force`") from None
        fn.restype = res
        fn.argtypes = args
    got = lib.eps_version()
    if got != EPS_VERSION:
        raise EpsError(f"{LIB_PATH} was built from another eps.h (library version {got}, binding {EPS_VERSION}): "
                       "rebuild it with `python -m edge_proposal_sets_b200.build --force`")
    from . import build as _b
    if _b.is_stale():
        import warnings
        warnings.warn(f"{LIB_PATH} is older than its sources; rebuild with `python -m edge_proposal_sets_b200.build`")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != EPS_OK:
        msg = load().eps_last_error().decode("utf-8", "replace")
        raise EpsError(f"{what} failed with eps_status {status}: {msg}")
