"""seam-match-rcnn_b200: B200-native retrieval hot path of SEAM Match-RCNN.

Temporal aggregation (non-local block + frame-attention pooling), the (q-g)^2 -> linear ->
softmax pair scorer and per-query top-k, as hand-written sm_100a CUDA kernels behind a C ABI
(include/seam_b200.h), with the reference's module surface on top.

The directory name contains a hyphen; import it as ``seam_match_rcnn_b200`` (the alias module
at the repository root registers this directory under that name).
"""
from ._lib import SeamError, declared_symbols, load as load_library          # noqa: F401
from ._build import build as build_library, LIB_PATH                          # noqa: F401
from .engine import SeamEngine, PreparedGallery, get_engine                   # noqa: F401
from .modules import NONLocalBlock1D, MatchPredictor, TemporalAggregationNLB  # noqa: F401
from .retrieval import (ShardedRetriever, RetrievalReport, ProductReport, evaluate_aggregated,   # noqa: F401
                        evaluate_products, evaluate_distance_fusions, product_means, self_distances, search, PeerExchange,
                        search_host, HostTrackStream, bind_to_gpu_numa_node, shard_bounds, all_gather_rows, exchange_layout, K_THRESHOLDS)

__all__ = [
    "SeamError", "SeamEngine", "PreparedGallery", "get_engine", "NONLocalBlock1D", "MatchPredictor",
    "TemporalAggregationNLB", "ShardedRetriever", "RetrievalReport", "evaluate_aggregated", "search",
    "search_host", "HostTrackStream", "ProductReport", "evaluate_products", "evaluate_distance_fusions", "product_means", "self_distances", "PeerExchange",
    "shard_bounds", "all_gather_rows", "exchange_layout", "bind_to_gpu_numa_node", "build_library", "load_library", "declared_symbols", "K_THRESHOLDS",
]
