"""ctypes binding of the C ABI in include/mpn_b200.h (libmpn_b200.so, built in-tree by csrc/build.sh).

The product path fails loudly when the library is missing or the device is not sm_100: there is no CPU
or PyTorch fallback for the hot path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmpn_b200.so")

MPN_OK, MPN_ERR_INVALID, MPN_ERR_CUDA, MPN_ERR_UNSORTED, MPN_ERR_WORKSPACE, MPN_ERR_NO_DEVICE = range(6)
MPN_DE, MPN_DH, MPN_MAX_NODE_LAYERS = 4, 32, 8
MPN_SUMS_DOUBLES = 96
ABI_VERSION = 6             # MPN_B200_ABI_VERSION of include/mpn_b200.h (bumped when a struct or a signature changes)
STAGE_ENC0, STAGE_ENC1, STAGE_EDGE, STAGE_NODE, STAGE_APPLY = range(5)
POST_CUT, POST_PRUNE, POST_SPLIT = 1, 2, 4
MPN_X_F32, MPN_X_F16, MPN_X_BF16 = 0, 1, 2      # element kind of the node features x (the *_x entry points)

# offsets inside mpn_weights.small (floats) — keep in sync with include/mpn_b200.h
W_ENC1_W, W_ENC1_B, W_ENC1_G, W_ENC1_BETA = 0, 8, 12, 16
W_ENC2_W, W_ENC2_B, W_ENC2_G, W_ENC2_BETA = 20, 36, 40, 44
W_EDGE_W, W_EDGE_B, W_EDGE_G, W_EDGE_BETA = 48, 320, 324, 328
W_NODE_W, W_NODE_B, W_NODE_G, W_NODE_BETA = 332, 1484, 1516, 1548
W_CLS_W, W_CLS_B = 1580, 1588
W_EDGE_W0, W_NODE_W0, W_SMALL_FLOATS = 1592, 1864, 2888


class MpnGraph(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("n_cols", C.c_int32), ("row_offset", C.c_int32), ("chunk", C.c_int32),
                ("n_edges", C.c_int64), ("max_tasks", C.c_int32), ("layout_hint", C.c_int32),
                ("rowptr", C.c_void_p), ("col", C.c_void_p), ("taskptr", C.c_void_p), ("task_row", C.c_void_p),
                ("n_tasks", C.c_void_p), ("n_graphs", C.c_int32), ("max_graph_nodes", C.c_int32),
                ("node_gid", C.c_void_p), ("graph_nptr", C.c_void_p)]


class MpnWeights(C.Structure):
    _fields_ = [("n_node_layers", C.c_int32), ("node_dims", C.c_int32 * (MPN_MAX_NODE_LAYERS + 1)),
                ("node_w", C.c_void_p * MPN_MAX_NODE_LAYERS), ("node_b", C.c_void_p * MPN_MAX_NODE_LAYERS),
                ("node_gamma", C.c_void_p * MPN_MAX_NODE_LAYERS), ("node_beta", C.c_void_p * MPN_MAX_NODE_LAYERS),
                ("small", C.c_void_p),
                ("node_w_hi", C.c_void_p * MPN_MAX_NODE_LAYERS), ("node_w_lo", C.c_void_p * MPN_MAX_NODE_LAYERS),
                ("node_w_hi16", C.c_void_p * MPN_MAX_NODE_LAYERS), ("node_w_lo16", C.c_void_p * MPN_MAX_NODE_LAYERS),
                ("node_w_scale16", C.c_float * MPN_MAX_NODE_LAYERS), ("node_bn_gmax", C.c_float * MPN_MAX_NODE_LAYERS),
                ("node_bn_bmax", C.c_float * MPN_MAX_NODE_LAYERS),
                ("node_agg", C.c_int32), ("reattach_nodes", C.c_int32), ("reattach_edges", C.c_int32), ("reserved", C.c_int32)]


AGG_SUM, AGG_MEAN, AGG_MAX = 0, 1, 2


MPN_MAX_PEERS = 16


class MpnPeerCtx(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("sums", C.c_void_p * MPN_MAX_PEERS),
                ("flags", C.c_void_p * MPN_MAX_PEERS), ("h", C.c_void_p * MPN_MAX_PEERS),
                ("cstats", C.c_void_p * MPN_MAX_PEERS),
                ("seq_moments", C.c_uint64), ("seq_h", C.c_uint64), ("seq_c", C.c_uint64),
                ("shard_node_encoder", C.c_int32), ("reserved", C.c_int32),
                ("edge_attr", C.c_void_p * MPN_MAX_PEERS), ("node_tables", C.c_void_p * MPN_MAX_PEERS),
                ("block_start", C.c_int32 * (MPN_MAX_PEERS + 1)), ("reserved2", C.c_int32), ("seq_t", C.c_uint64)]
MPN_PEER_CSTAT_COLS = 1024


class MpnError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libmpn_b200 error %d: %s" % (code, message))
        self.code = code


class UnsortedEdgeIndex(MpnError):
    pass


_lib = None

_PROTOS = {
    # name: (restype, argtypes)
    "mpn_abi_version": (C.c_int, []),
    "mpn_last_error": (C.c_char_p, []),
    "mpn_kernel_launches": (C.c_uint64, []),
    "mpn_check_device": (C.c_int, [C.c_int]),
    "mpn_set_pdl": (C.c_int, [C.c_int]),
    "mpn_graph_build": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p]),
    "mpn_graph_build_i32": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_graph_build_deferred": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_cross_camera_edges": (C.c_int64, [C.c_void_p, C.c_int32]),
    "mpn_cross_camera_block_edges": (C.c_int64, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "mpn_graph_build_cross_camera": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "mpn_cross_camera_batched_layout": (C.c_int64, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "mpn_graph_build_cross_camera_batched": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_void_p]),
    "mpn_profile_gram": (C.c_int, [C.c_int]),
    "mpn_profile_gram_ms": (C.c_float, []),
    "mpn_shared_gram_mode": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_shared_gram_row_range": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "mpn_pack_decisions": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "mpn_profile_timeline": (C.c_int, [C.c_int]),
    "mpn_profile_timeline_read": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "mpn_edge_features_workspace_bytes": (C.c_size_t, [C.POINTER(MpnGraph), C.c_int32]),
    "mpn_edge_features": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_int32, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_workspace_bytes": (C.c_size_t, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_int32]),
    "mpn_forward": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_with_edge_features": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                                 C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_plan_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_int32, C.c_int32,
                                  C.c_int64, C.c_int, C.c_void_p, C.c_size_t]),
    "mpn_plan_destroy": (None, [C.c_void_p]),
    "mpn_plan_node_encoder": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_plan_node_tables": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "mpn_plan_sweep": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_plan_sums": (C.c_void_p, [C.c_void_p]),
    "mpn_plan_reduce": (C.c_int, [C.c_void_p, C.c_int32, C.c_int, C.c_void_p]),
    "mpn_plan_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "mpn_plan_node_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "mpn_plan_h_full": (C.c_void_p, [C.c_void_p]),
    "mpn_split_tf32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_split_f16": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_void_p]),
    "mpn_forward_sharded": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(MpnPeerCtx),
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_sharded_with_edge_features": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_void_p, C.c_int32,
                                                         C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                         C.POINTER(MpnPeerCtx), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_decide": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_post_workspace_bytes": (C.c_size_t, [C.POINTER(MpnGraph)]),
    "mpn_cut": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_prune": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                            C.POINTER(C.c_int32), C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_split": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                            C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_split_last_stats": (None, [C.c_void_p]),
    "mpn_scc_labels": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_post_processing": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_post_processing_batched": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_active_edges": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_compact_workspace_bytes": (C.c_size_t, [C.POINTER(MpnGraph)]),
    "mpn_count_active": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_compact_active": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_clear_inactive": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mpn_labels_reference": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
    "mpn_labels_reference_batched": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                              C.c_void_p]),
    "mpn_labels_reference_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.POINTER(C.c_int32)]),
    "mpn_split_exact_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_void_p]),
    "mpn_edge_confusion": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "mpn_contingency_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "mpn_contingency": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(C.c_int64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_expected_mutual_information_host": (C.c_double, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]),
    "mpn_relabel_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "mpn_relabel_detections": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_write_mtmc_txt_host": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
    "mpn_edge_labels": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpn_normalize_columns_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "mpn_normalize_columns": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_normalize_columns_batched": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                                C.c_size_t, C.c_void_p]),
    "mpn_gemm_nt_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "mpn_gram_nt": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                              C.c_void_p]),
    "mpn_gemm_nt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int,
                              C.c_void_p, C.c_size_t, C.c_void_p]),
    # the entry points that read x, with (x, x_kind) in place of an fp32 x
    "mpn_edge_features_x": (C.c_int, [C.POINTER(MpnGraph), C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    "mpn_forward_x": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_with_edge_features_x": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_int32, C.c_void_p,
                                                   C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                   C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_sharded_x": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                        C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.POINTER(MpnPeerCtx), C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_forward_sharded_with_edge_features_x": (C.c_int, [C.POINTER(MpnGraph), C.POINTER(MpnWeights), C.c_void_p, C.c_int32,
                                                           C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                                           C.c_void_p, C.c_void_p, C.c_int, C.POINTER(MpnPeerCtx), C.c_void_p,
                                                           C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpn_plan_node_encoder_x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "mpn_normalize_columns_x": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.c_void_p]),
    "mpn_normalize_columns_batched_x": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                                  C.c_void_p, C.c_size_t, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS.keys())


def lib():
    """Load libmpn_b200.so once.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError("libmpn_b200.so not built: run %s (or __graft_entry__.build()); "
                              "the MPN hot path has no CPU fallback" % os.path.join(_HERE, "csrc", "build.sh"))
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.mpn_abi_version() != ABI_VERSION:
            raise ImportError("libmpn_b200.so ABI version mismatch")
        _lib = l
    return _lib


def check(code):
    if code != MPN_OK:
        msg = lib().mpn_last_error().decode("utf-8", "replace")
        if code == MPN_ERR_UNSORTED:
            raise UnsortedEdgeIndex(code, msg)
        raise MpnError(code, msg)


_DEVICE_OK = set()


def require_device(index: int):
    """Raises unless CUDA device `index` is an sm_100 part.  Cached: cudaGetDeviceProperties costs milliseconds."""
    index = int(index)
    if index not in _DEVICE_OK:
        check(lib().mpn_check_device(index))
        _DEVICE_OK.add(index)
