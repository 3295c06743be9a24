"""euler_b200 -- B200-native (sm_100a) minibatch-construction path of alibaba/euler.

`import euler_b200 as tf_euler` exposes the reference's op names for this path (sample_neighbor,
sample_fanout, sample_node, random_walk, get_dense_feature, gather / scatter_*), backed by
hand-written CUDA kernels in euler_b200/lib/libeuler_b200.so behind the C ABI of
include/euler_b200.h.  See DESIGN.md / INTEGRATION.md.
"""
from ._lib import EU_RNG_MINSTD, EU_RNG_PHILOX, EulerError  # noqa: F401
from .graph import Context, Graph  # noqa: F401
from .ops import (context, gather, gen_pair, get_edge_binary_feature, get_edge_dense_feature, get_edge_sparse_feature, get_dense_feature, get_edge_type_id, get_full_neighbor, get_graph,  # noqa: F401
                  get_binary_feature, get_node_type_id, get_sorted_full_neighbor, get_sparse_feature, get_top_k_neighbor, initialize_embedded_graph,
                  initialize_graph, random_walk, sage_mean_aggregate, sample_fanout, sample_fanout_batched, sample_fanout_with_feature,
                  sample_edge, sample_neighbor, sample_neighbor_api, sample_neighbor_layerwise, sample_node, scatter_, scatter_add, scatter_max, scatter_mean,
                  scatter_softmax, seed, set_graph, sparse_get_adj, unique)
