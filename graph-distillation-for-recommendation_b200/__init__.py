"""gdr — B200-native data-parallel distillation core of ClustGDD.

Four stages behind the reference's own call signatures (see SURVEY.md §8):
  1. adjacency build        graph.py        (deep_robust_utils.py, distill_recsys.py:110-117)
  2. K-hop propagation      propagation.py  (clustgdd_agent_transduct.py:55-65)
  3. k-means / WCSS         kmeans.py       (sklearn KMeans call sites)
  4. coarsened graph        coarsen.py      (graph_compress, build_condensed_bipartite)
  +  edge scoring / top-k   sparsify.py     (ER_estimator, attaw_ER_estimator, graph_sparse; SURVEY §8f item 1)
  +  top-K evaluation       recsys.py       (recommend_topk, ranking_metrics: recall_at_k, distill_recsys.py:446-497)
  +  condensed-model training recsys.py     (LightGCNPropagate: gradients w.r.t. embeddings and edge weights, :684-733;
                                            BPRSampler, bpr_loss: triplet sampling and the BPR loss + gradient)
All arithmetic runs in libgdr_b200.so (hand-written sm_100a CUDA, C ABI in include/gdr.h).
Importing this package loads that library and fails if it has not been built.
"""
from . import _lib

_lib.load()  # no CPU fallback: fail at import time when the CUDA library is missing

from ._lib import GdrError, LIB_PATH  # noqa: E402
from ._dev import launch_count  # noqa: E402
from .graph import (  # noqa: E402
    CSR, coo_to_csr, sym_normalize, is_sparse_tensor, sparse_mx_to_torch_sparse_tensor, to_tensor,
    to_scipy, normalize_adj_tensor, normalize_adj, build_interaction_matrix,
)
from .propagation import propagate, spmm  # noqa: E402
from .kmeans import (  # noqa: E402
    KMeans, MiniBatchKMeans, kmeans_cluster, cluster_means, segment_mean_pool, segment_sum, assign_labels, standard_scale,
)
from .coarsen import (  # noqa: E402
    graph_compress, build_condensed_bipartite, condensed_csr_to_edge_index, coarsen_edges, label_counts,
)
from .sparsify import (  # noqa: E402
    ER_estimator, attaw_ER_estimator, graph_sparse, er_lower, cosine_reweight, softmax_rows, class_edge_weight,
    topk_filter, row_degree,
)
from .recsys import (  # noqa: E402
    BipartiteGraph, lightgcn_propagate, BipartitePropagate, LightGCNPropagate, RankformerGCNGraph,
    rankformer_gcn_forward, recommend_topk, ranking_metrics, BPRSampler, BPRLoss, bpr_loss,
)
from .io import (  # noqa: E402
    induced_subgraph, load_graphsaint, load_rankformer_dataset, read_ui_txt, save_condensed, load_condensed,
    RecDataset, GraphSaintData,
)
from .svd import compute_svd_embeddings, truncated_svd  # noqa: E402
from . import parallel  # noqa: E402

__all__ = [
    "GdrError", "LIB_PATH", "launch_count", "CSR", "coo_to_csr", "sym_normalize", "is_sparse_tensor",
    "sparse_mx_to_torch_sparse_tensor", "to_tensor", "to_scipy", "normalize_adj_tensor", "normalize_adj",
    "build_interaction_matrix", "propagate", "spmm", "KMeans", "MiniBatchKMeans", "kmeans_cluster", "cluster_means",
    "segment_mean_pool", "segment_sum", "assign_labels", "standard_scale", "graph_compress",
    "build_condensed_bipartite", "condensed_csr_to_edge_index", "coarsen_edges", "label_counts",
    "ER_estimator", "attaw_ER_estimator", "graph_sparse", "er_lower", "cosine_reweight", "softmax_rows",
    "class_edge_weight", "topk_filter", "row_degree", "BipartiteGraph", "lightgcn_propagate", "BipartitePropagate", "LightGCNPropagate",
    "RankformerGCNGraph",
    "rankformer_gcn_forward", "recommend_topk", "ranking_metrics", "BPRSampler", "BPRLoss", "bpr_loss",
    "induced_subgraph", "load_graphsaint", "load_rankformer_dataset", "read_ui_txt",
    "save_condensed", "load_condensed", "RecDataset", "GraphSaintData", "compute_svd_embeddings", "truncated_svd",
    "parallel",
]
