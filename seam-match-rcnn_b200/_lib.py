"""ctypes binding of libseam_b200.so (the C ABI declared in include/seam_b200.h).

There is no CPU implementation behind these calls: if the library is missing, or no B200 is
present, the entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import List, Optional

from . import _build

_HEADER = os.path.join(os.path.dirname(_build.HERE), "include", "seam_b200.h")

SEAM_OK = 0
STATUS_NAMES = {0: "OK", 1: "BAD_ARG", 2: "UNSUPPORTED", 3: "CUDA", 4: "STATE"}
KERNELS = {"aggregate": 0, "nlb_gemm": 1, "prep_queries": 2, "score": 3, "rescore": 4, "exact": 5,
           "prep_gallery": 6, "merge": 7, "tower": 8}
SEAM_MAX_T = 64
SEAM_MAX_K = 32
SEAM_MAX_WORLD = 8


class SeamError(RuntimeError):
    """A C-ABI call returned a non-zero seam_status."""

    def __init__(self, status: int, message: str):
        self.status = status
        super().__init__(f"seam_b200 [{STATUS_NAMES.get(status, status)}]: {message}")


class SeamWeights(C.Structure):
    """struct seam_weights: 13 device pointers in the reference's state_dict order."""
    FIELDS = ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "W_w", "W_b", "concat_w",
              "att_w", "att_b", "last_w", "last_b")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class SeamExchange(C.Structure):
    """struct seam_exchange (include/seam_b200.h): the peer-mapped buffers of the gallery-sharded search."""
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("Q", C.c_int32), ("k", C.c_int32), ("own_max", C.c_int32),
                ("q_lo", C.c_int32 * (SEAM_MAX_WORLD + 1)),
                ("q_all", C.c_void_p * SEAM_MAX_WORLD),
                ("list_margin", C.c_void_p * SEAM_MAX_WORLD), ("list_idx", C.c_void_p * SEAM_MAX_WORLD),
                ("final_score", C.c_void_p * SEAM_MAX_WORLD), ("final_margin", C.c_void_p * SEAM_MAX_WORLD),
                ("final_idx", C.c_void_p * SEAM_MAX_WORLD),
                ("flags", C.c_void_p * SEAM_MAX_WORLD),
                ("step", C.c_void_p), ("done", C.c_void_p), ("q_all_mc", C.c_void_p),
                ("final_score_mc", C.c_void_p), ("final_margin_mc", C.c_void_p), ("final_idx_mc", C.c_void_p)]


class SeamWeightGrads(C.Structure):
    """struct seam_weight_grads: gradient buffers of the 11 aggregator parameters (state_dict order)."""
    FIELDS = ("theta_w", "theta_b", "phi_w", "phi_b", "g_w", "g_b", "W_w", "W_b", "concat_w", "att_w", "att_b")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


# field of seam_weights -> key in TemporalAggregationNLB.state_dict()
WEIGHT_KEYS = {
    "theta_w": "newnlb.theta.weight", "theta_b": "newnlb.theta.bias",
    "phi_w": "newnlb.phi.weight", "phi_b": "newnlb.phi.bias",
    "g_w": "newnlb.g.weight", "g_b": "newnlb.g.bias",
    "W_w": "newnlb.W.weight", "W_b": "newnlb.W.bias",
    "concat_w": "newnlb.concat_project.0.weight",
    "att_w": "attention_scorer.weight", "att_b": "attention_scorer.bias",
    "last_w": "last.weight", "last_b": "last.bias",
}


def declared_symbols() -> List[str]:
    """Every function name declared in include/seam_b200.h."""
    with open(_HEADER) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(seam_[a-z_0-9]+)\s*\(", text)))


_lib: Optional[C.CDLL] = None


def _declare(lib: C.CDLL) -> None:
    vp, i32, i64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
    lib.seam_abi_version.restype = i32
    lib.seam_abi_version.argtypes = []
    lib.seam_exchange_sizeof.restype = sz
    lib.seam_exchange_sizeof.argtypes = []
    lib.seam_create.restype = i32
    lib.seam_create.argtypes = [C.POINTER(vp), i32]
    lib.seam_destroy.restype = None
    lib.seam_destroy.argtypes = [vp]
    lib.seam_last_error.restype = C.c_char_p
    lib.seam_last_error.argtypes = [vp]
    lib.seam_launch_count.restype = C.c_uint64
    lib.seam_launch_count.argtypes = [vp]
    lib.seam_device_stamp.restype = i32
    lib.seam_device_stamp.argtypes = [vp, vp, vp]
    lib.seam_watchdog_read.restype = i32
    lib.seam_watchdog_read.argtypes = [vp, C.POINTER(C.c_uint32), i32]
    lib.seam_profile_enable.restype = i32
    lib.seam_profile_enable.argtypes = [vp, i32]
    lib.seam_profile_read.restype = i32
    lib.seam_profile_read.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(i32)]
    lib.seam_load_weights.restype = i32
    lib.seam_load_weights.argtypes = [vp, C.POINTER(SeamWeights), vp]
    lib.seam_load_scorer.restype = i32
    lib.seam_load_scorer.argtypes = [vp, vp, vp, vp]
    lib.seam_aggregate_workspace_bytes.restype = sz
    lib.seam_aggregate_workspace_bytes.argtypes = [i32]
    lib.seam_aggregate.restype = i32
    lib.seam_aggregate.argtypes = [vp, vp, vp, vp, i32, i32, i64, i64, vp, vp, vp, sz, vp]
    lib.seam_aggregate_f16.restype = i32
    lib.seam_aggregate_f16.argtypes = lib.seam_aggregate.argtypes
    lib.seam_nlb_workspace_bytes.restype = sz
    lib.seam_nlb_workspace_bytes.argtypes = [i32, i32]
    lib.seam_nlb_forward.restype = i32
    lib.seam_nlb_forward.argtypes = [vp, vp, i32, i32, vp, vp, sz, vp]
    lib.seam_prepare_gallery.restype = i32
    lib.seam_prepare_gallery.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    lib.seam_prepare_gallery_f16.restype = i32
    lib.seam_prepare_gallery_f16.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.seam_score_workspace_bytes.restype = sz
    lib.seam_score_workspace_bytes.argtypes = [vp, i32, i32, i32]
    lib.seam_score_partition.restype = i32
    lib.seam_score_partition.argtypes = [i32, i32, i32, i32, C.POINTER(C.c_int32), i32, C.POINTER(C.c_int32)]
    lib.seam_score_plan.restype = i32
    lib.seam_score_plan.argtypes = [vp, i32, i32, C.POINTER(C.c_int64)]
    lib.seam_score_topk.restype = i32
    lib.seam_score_topk.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_score_topk_g16.restype = i32
    lib.seam_score_topk_g16.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_search.restype = i32
    lib.seam_search.argtypes = [vp, vp, vp, vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_search_f16.restype = i32
    lib.seam_search_f16.argtypes = lib.seam_search.argtypes
    lib.seam_search_g16.restype = i32
    lib.seam_search_g16.argtypes = [vp, vp, vp, vp, i32, i32, i64, i64, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_search_f16_g16.restype = i32
    lib.seam_search_f16_g16.argtypes = lib.seam_search_g16.argtypes
    lib.seam_score_dense.restype = i32
    lib.seam_score_dense.argtypes = [vp, vp, i32, vp, i32, vp, vp]
    lib.seam_score_prob.restype = i32
    lib.seam_score_prob.argtypes = [vp, vp, i32, vp, i32, vp, vp]
    lib.seam_rank_fused_distances.restype = i32
    lib.seam_rank_fused_distances.argtypes = [vp, vp, vp, i32, vp, i32, vp, vp, vp, vp]
    lib.seam_rank_of_target.restype = i32
    lib.seam_rank_of_target.argtypes = [vp, vp, i32, vp, i32, vp, vp, vp, vp]
    lib.seam_rank_workspace_bytes.restype = sz
    lib.seam_rank_workspace_bytes.argtypes = [vp, i32, i32]
    lib.seam_rank_of_target_prepared.restype = i32
    lib.seam_rank_of_target_prepared.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_rank_of_target_prepared_g16.restype = i32
    lib.seam_rank_of_target_prepared_g16.argtypes = [vp, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_shard_target_margin.restype = i32
    lib.seam_shard_target_margin.argtypes = [vp, vp, i32, vp, i32, i32, vp, vp, vp]
    lib.seam_shard_target_margin_g16.restype = i32
    lib.seam_shard_target_margin_g16.argtypes = lib.seam_shard_target_margin.argtypes
    lib.seam_shard_rank_count_prepared.restype = i32
    lib.seam_shard_rank_count_prepared.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    lib.seam_shard_rank_count_prepared_g16.restype = i32
    lib.seam_shard_rank_count_prepared_g16.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    xp = C.POINTER(SeamExchange)
    lib.seam_sharded_aggregate.restype = i32
    lib.seam_sharded_aggregate.argtypes = [vp, xp, vp, vp, vp, i32, i32, i64, i64, i32, i32, vp, vp]
    lib.seam_sharded_aggregate_f16.restype = i32
    lib.seam_sharded_aggregate_f16.argtypes = lib.seam_sharded_aggregate.argtypes
    lib.seam_sharded_score_topk.restype = i32
    lib.seam_sharded_score_topk.argtypes = [vp, xp, vp, vp, vp, vp, i32, i32, vp, vp, sz, vp]
    lib.seam_sharded_score_topk_g16.restype = i32
    lib.seam_sharded_score_topk_g16.argtypes = [vp, xp, vp, vp, vp, i32, i32, vp, vp, sz, vp]
    lib.seam_sharded_merge.restype = i32
    lib.seam_sharded_merge.argtypes = [vp, xp, vp, vp, vp, vp]
    lib.seam_aggregate_backward.restype = i32
    lib.seam_aggregate_backward.argtypes = [vp, C.POINTER(SeamWeights), vp, vp, vp, i32, i32, i64, i64, vp, vp,
                                            C.POINTER(SeamWeightGrads), vp]
    lib.seam_score_dense_backward.restype = i32
    lib.seam_score_dense_backward.argtypes = [vp, vp, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.seam_tower_load_weights.restype = i32
    lib.seam_tower_load_weights.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), vp, vp, vp, vp, vp, vp, C.c_float, vp]
    lib.seam_tower_workspace_bytes.restype = sz
    lib.seam_tower_workspace_bytes.argtypes = [i32]
    lib.seam_tower_forward.restype = i32
    lib.seam_tower_forward.argtypes = [vp, vp, i32, vp, vp, vp, sz, vp]
    lib.seam_upload_tracks.restype = i32
    lib.seam_upload_tracks.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp]
    lib.seam_upload_tracks_f16.restype = i32
    lib.seam_upload_tracks_f16.argtypes = lib.seam_upload_tracks.argtypes
    lib.seam_merge_topk.restype = i32
    lib.seam_merge_topk.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen the in-tree library (building it first when nvcc is present and it is stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if build_if_missing:
        try:
            _build.build()
        except RuntimeError:
            if not os.path.exists(path):
                raise
    if not os.path.exists(path):
        raise SeamError(3, f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    _declare(lib)
    _lib = lib
    return lib
