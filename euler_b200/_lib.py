"""ctypes binding of the C ABI declared in include/euler_b200.h.

The shared library is built in-tree (euler_b200/lib/libeuler_b200.so) by euler_b200/build.py.  There
is no Python/CPU fallback: if the library is missing or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "lib", "libeuler_b200.so")

EU_RNG_MINSTD = 0
EU_RNG_PHILOX = 1


class EulerError(RuntimeError):
    pass


class GraphDesc(C.Structure):
    """eu_graph_desc"""
    _fields_ = [
        ("n_nodes", C.c_int64), ("n_edge_types", C.c_int32), ("n_node_types", C.c_int32),
        ("ids", C.c_void_p), ("node_type", C.c_void_p), ("node_w", C.c_void_p),
        ("grp_ptr", C.c_void_p), ("nbr", C.c_void_p), ("cum_w", C.c_void_p), ("grp_cum", C.c_void_p),
        ("w", C.c_void_p), ("feat_dim", C.c_int32), ("feat", C.c_void_p),
        ("sampler_order", C.c_void_p), ("n_feat_slots", C.c_int32), ("feat_slot_dims", C.c_void_p),
        ("n_u64_slots", C.c_int32), ("u64_ptr", C.c_void_p), ("u64_val", C.c_void_p),
        ("n_bin_slots", C.c_int32), ("bin_ptr", C.c_void_p), ("bin_val", C.c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/euler_b200.h declares
_P, _I64, _I32, _U64, _F = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_float
SIGNATURES = {
    "eu_last_error": (C.c_char_p, []),
    "eu_version": (C.c_char_p, []),
    "eu_launch_count": (_U64, []),
    "eu_graph_create": (C.c_int, [C.POINTER(GraphDesc), C.c_int, C.POINTER(_P)]),
    "eu_graph_create_rmat": (C.c_int, [_I64, _I64, C.c_double, C.c_double, C.c_double, _U64, _I32, _U64,
                                       C.c_int, C.POINTER(_P)]),
    "eu_graph_create_rmat_shard": (C.c_int, [_I64, _I64, C.c_double, C.c_double, C.c_double, _U64, _I32, _U64,
                                             C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "eu_graph_create_rmat_hetero": (C.c_int, [_I64, _I64, _I32, _I32, C.c_double, C.c_double, C.c_double, _U64, _I32, _U64,
                                              C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "eu_graph_load": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "eu_graph_load_ex": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "eu_graph_set_edges": (C.c_int, [_P, _P]),
    "eu_graph_num_edge_records": (_I64, [_P]),
    "eu_graph_edge_dense_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_edge_sparse_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_edge_binary_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_sample_edge": (C.c_int, [_P, _I32, _P, _I32, _P]),
    "eu_get_edge_dense_feature": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_get_edge_sparse_feature": (C.c_int, [_P, _P, _I64, _I32, _I64, _I64, _P, _P]),
    "eu_get_edge_binary_feature": (C.c_int, [_P, _P, _I64, _I32, _I64, _P, _P]),
    "eu_graph_destroy": (C.c_int, [_P]),
    "eu_graph_num_nodes": (_I64, [_P]),
    "eu_graph_num_edges": (_I64, [_P]),
    "eu_graph_num_edge_types": (_I32, [_P]),
    "eu_graph_num_node_types": (_I32, [_P]),
    "eu_graph_feat_dim": (_I32, [_P]),
    "eu_graph_hbm_bytes": (_I64, [_P]),
    "eu_graph_export": (C.c_int, [_P] * 9),
    "eu_graph_edge_type_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_node_type_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_dense_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_dense_feature_dim": (_I32, [_P, _I32]),
    "eu_graph_sparse_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_binary_feature_id": (_I32, [_P, C.c_char_p]),
    "eu_graph_sparse_feature_max_len": (_I64, [_P, _I32]),
    "eu_get_sparse_feature": (C.c_int, [_P, _P, _I64, _I32, _I64, _I64, _P, _P]),
    "eu_get_sparse_feature_host": (C.c_int, [_P, _P, _I64, _I32, _I64, _I64, _P, _P, _P]),
    "eu_get_binary_feature": (C.c_int, [_P, _P, _I64, _I32, _I64, _P, _P]),
    "eu_get_binary_feature_host": (C.c_int, [_P, _P, _I64, _I32, _I64, _P, _P, _P]),
    "eu_ctx_create": (C.c_int, [_P, C.c_int, _U64, _P, C.POINTER(_P)]),
    "eu_ctx_destroy": (C.c_int, [_P]),
    "eu_ctx_set_stream": (C.c_int, [_P, _P]),
    "eu_ctx_seed": (C.c_int, [_P, _U64]),
    "eu_ctx_set_engines": (C.c_int, [_P, _I32, _P]),
    "eu_ctx_reserve": (C.c_int, [_P, _I64]),
    "eu_ctx_sync": (C.c_int, [_P]),
    "eu_ctx_draws": (C.c_int, [_P, C.POINTER(_U64)]),
    "eu_ctx_profile": (C.c_int, [_P, C.c_int]),
    "eu_ctx_profile_read": (C.c_int, [_P, C.c_char_p, _I64]),
    "eu_sample_neighbor": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _I64, _P, _P, _P]),
    "eu_sample_neighbor_host": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _I64, _P, _P, _P]),
    "eu_sample_neighbor_raw": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _P, _P, _P]),
    "eu_sample_neighbor_raw_host": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _P, _P, _P]),
    "eu_get_sorted_full_neighbor": (C.c_int, [_P, _P, _I64, _P, _I32, _I64, _P, _P, _P, _P]),
    "eu_get_top_k_neighbor": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _I64, _P, _P, _P]),
    "eu_sample_neighbor_layerwise": (C.c_int, [_P, _P, _I64, _I32, _P, _I32, _I32, _I64, _I32, _P, _P]),
    "eu_sparse_get_adj": (C.c_int, [_P, _P, _P, _I64, _I32, _I32, _P, _I32, _P]),
    "eu_gen_pair_count": (_I64, [_I32, _I32, _I32]),
    "eu_gen_pair": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P]),
    "eu_sample_fanout": (C.c_int, [_P, _P, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P]),
    "eu_sample_fanout_batched": (C.c_int, [_P, _P, _I32, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P]),
    "eu_sample_fanout_host": (C.c_int, [_P, _P, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P]),
    "eu_sample_fanout_batched_host": (C.c_int, [_P, _P, _I32, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P]),
    "eu_sample_fanout_with_feature": (C.c_int, [_P, _P, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P, _I32, _P, _P, _P, _I32, _P,
                                                _P, _P, _P]),
    "eu_sample_fanout_with_feature_host": (C.c_int, [_P, _P, _I64, _P, _I32, _P, _I32, _I64, _P, _P, _P, _I32, _P, _P, _P, _I32,
                                                     _P, _P, _P, _P]),
    "eu_sage_mean_aggregate_host": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_sample_node": (C.c_int, [_P, _I32, _P, _I32, _P]),
    "eu_sample_node_host": (C.c_int, [_P, _I32, _P, _I32, _P]),
    "eu_build_alias_table": (C.c_int, [_P, _I64, _P, _P, _P]),
    "eu_graph_load_inspect": (C.c_int, [C.c_char_p, C.c_int, C.c_int, _P, _P, _P, _P, _I64, _P, _P]),
    "eu_random_walk": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _F, _F, _I64, _P]),
    "eu_random_walk_host": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _F, _F, _I64, _P]),
    "eu_get_dense_feature": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_get_dense_feature_host": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_get_full_neighbor": (C.c_int, [_P, _P, _I64, _P, _I32, _I64, _P, _P, _P, _P]),
    "eu_unique": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "eu_get_node_type": (C.c_int, [_P, _P, _I64, _P]),
    "eu_get_node_type_host": (C.c_int, [_P, _P, _I64, _P]),
    "eu_get_node_weight_host": (C.c_int, [_P, _P, _I64, _P]),
    "eu_get_full_neighbor_host": (C.c_int, [_P, _P, _I64, _P, _I32, _I64, _P, _P, _P, _P, _P]),
    "eu_gather": (C.c_int, [_P, _P, _I64, _I64, _P, _I64, _P]),
    "eu_scatter_add": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "eu_scatter_max": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "eu_scatter_mean": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "eu_sage_mean_aggregate": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_sage_add_aggregate": (C.c_int, [_P, _P, _I64, _I32, _I32, _P]),
    "eu_gather_host": (C.c_int, [_P, _P, _I64, _I64, _P, _I64, _P]),
    "eu_scatter_add_host": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "eu_scatter_max_host": (C.c_int, [_P, _P, _I64, _P, _I64, _I64, _P]),
    "eu_shard_bucket": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P]),
    "eu_shard_pack_sample": (C.c_int, [_P, _P, _P, _P, _I64, _P]),
    "eu_shard_merge_sample": (C.c_int, [_P, _P, _P, _I64, _I32, _I64, _P, _P, _P, _P]),
    "eu_shard_merge_rows": (C.c_int, [_P, _P, _P, _I64, _I64, _P]),
    "eu_sym_create": (C.c_int, [_P, _I32, _I32, _I64, _I32, _I64, _I32, C.POINTER(_P), _P]),
    "eu_sym_connect": (C.c_int, [_P, _P]),
    "eu_sym_destroy": (C.c_int, [_P]),
    "eu_sym_outputs": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "eu_sym_error": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "eu_sym_sample_hop": (C.c_int, [_P, _P, _I64, _P, _I32, _I32, _I64, _I32, _I32]),
    "eu_sym_sample_hop_batched": (C.c_int, [_P, _P, _I32, _I64, _P, _I32, _I32, _I64, _I32, _I32]),
    "eu_sym_get_dense_feature": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32]),
    "eu_sym_sage_mean": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P]),
    "InitQueryProxy": (C.c_bool, [C.c_char_p]),
    "eu_default_graph": (_P, []),
    "eu_default_ctx": (_P, []),
    "eu_set_default_graph": (C.c_int, [_P, C.c_int, _U64]),
}

_lib = None


def load():
    """Load libeuler_b200.so (raises if it has not been built -- no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise EulerError(
                "%s not found: run `python -m euler_b200.build` (or __graft_entry__.build()). "
                "euler_b200 has no CPU / PyTorch fallback." % SO_PATH)
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI drifted from the header
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise EulerError("euler_b200 error %d: %s" % (rc, load().eu_last_error().decode()))
