"""B200-native tracklet-graph message passing (drop-in for models/mpn.py + the post-processing of inference.py).

Public surface (same names as the reference where one exists):
    MOTMPNet                     models/mpn.py:144
    edge_features                inference.py:453-456
    post_processing              inference.py:70
    post_processing_batched      post_processing for every graph of a batch in one call (new; see INTEGRATION.md)
    pruning, splitting, remove_edges_single_direction, compute_SCC_and_Clusters      utils.py
    ShardedMPN                   row-block sharded forward across the GPUs of one box (new; see DESIGN.md)
    GraphStream                  a stream of host-resident graphs: PCIe copies of neighbouring graphs overlap the kernels (new)
    sharded_post_processing      post_processing for row-block shards: active lists merged across ranks (new; see DESIGN.md)
    compute_P_R_F                inference.py:20-66
    evaluation.{adjusted_rand_score, adjusted_mutual_info_score, homogeneity_score, completeness_score, v_measure_score}
                                 the sklearn.metrics calls of inference.py:509-519
    tracking_table, save_mtmc    inference.py:540-551, main.py:114
    normalize_columns, edge_labels    inference.py:403-404, 446-450
    pack_reid_features, load_packed_features    one packed file + one H->D copy for libs/dataset.py:298-307 / inference.py:399
"""
from . import _lib
from . import evaluation
from .evaluation import compute_P_R_F, clustering_scores
from .tracking_output import relabel_detections, save_mtmc, tracking_table
from .graph_inputs import (edge_labels, load_packed_features, normalize_columns, pack_reid_features,
                           pack_reid_features_from_pickles, read_packed_features)
from .edge_features import edge_features
from .graph import TrackletGraph, graph_for
from .mpn import MOTMPNet
from .pipeline import GraphStream, ShardedGraphStream, unpack_decisions
from .sharded import (CudaPhases, CudaPostOps, ShardedMPN, partition_rows, shard_edges, sharded_forward,
                      sharded_post_processing)
from .postprocess import (compute_SCC_and_Clusters, post_processing, post_processing_batched, pruning,
                          remove_edges_single_direction, split_stats, splitting)

__all__ = ["MOTMPNet", "edge_features", "post_processing", "post_processing_batched", "pruning", "splitting", "remove_edges_single_direction",
           "compute_SCC_and_Clusters", "split_stats", "TrackletGraph", "graph_for", "ShardedMPN", "CudaPhases", "sharded_forward", "partition_rows",
           "shard_edges", "GraphStream", "ShardedGraphStream", "unpack_decisions", "sharded_post_processing", "CudaPostOps", "_lib", "evaluation", "compute_P_R_F", "clustering_scores", "relabel_detections", "tracking_table",
           "save_mtmc", "edge_labels", "normalize_columns", "pack_reid_features", "pack_reid_features_from_pickles",
           "read_packed_features", "load_packed_features"]
