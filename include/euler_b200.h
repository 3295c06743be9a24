/* euler_b200 -- C ABI of the B200-native minibatch-construction path of alibaba/euler.
 *
 * This is the drop-in boundary (SURVEY.md section 8b, seam B2).  The reference exports exactly one
 * C symbol, `bool InitQueryProxy(const char*)` (tf_euler/utils/init_query_proxy.cc:19-36); every
 * other entry point of the hot path is a TensorFlow op registered in C++.  Since TF's registry is
 * not part of this build, each TF op of the path is exported here as a flat function with the
 * op's own argument meaning; the reference-side binding a maintainer would add is shown in
 * INTEGRATION.md.  Plain pointers and sizes only -- no torch / TF types.
 *
 * Conventions
 *   - every function returns 0 (EU_OK) or a nonzero eu_status; nothing throws across the ABI;
 *   - `eu_ctx` = one execution lane: a CUDA stream + one RNG engine + scratch.  It plays the role of
 *     one thread of the reference's client pool (euler/client/query_proxy.cc:205-210: 8 threads,
 *     each with its own thread_local engine, euler/common/random.cc:22).  Calls on one ctx are
 *     stream-ordered; different ctxs may run concurrently; the graph is immutable after creation;
 *   - functions without a `_host` suffix take DEVICE pointers and only enqueue work on the ctx
 *     stream (no host synchronisation, capturable in a CUDA graph);
 *   - `_host` variants take HOST pointers and return after the results have landed (this is what a
 *     CPU-tensor framework binds): pageable buffers are staged through pinned memory owned by the ctx,
 *     buffers that are already page-locked (cudaHostAlloc / cudaHostRegister) are DMA'd in place;
 *   - edge-type / count lists are HOST arrays (they are op attributes / tiny tensors upstream).
 */
#ifndef EULER_B200_H_
#define EULER_B200_H_

#include <stdbool.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  EU_OK = 0,
  EU_ERR_INVALID = 1,      /* bad argument */
  EU_ERR_CUDA = 2,         /* a CUDA call failed; see eu_last_error() */
  EU_ERR_NO_GPU = 3,       /* no CUDA device: this library has no CPU fallback */
  EU_ERR_UNSUPPORTED = 4,  /* valid in the reference but outside this path (e.g. `condition`) */
  EU_ERR_IO = 5,
  EU_ERR_STATE = 6         /* e.g. op called before a graph was initialised */
} eu_status;

/* RNG engines.  EU_RNG_MINSTD reproduces the reference's engine and draw order bit-exactly
 * (std::default_random_engine + uniform_real_distribution<double>, euler/common/random.cc:22-28);
 * EU_RNG_PHILOX is a counter-based engine keyed on (node id, draw) for throughput runs: same
 * algorithm, same distribution, different stream. */
typedef enum { EU_RNG_MINSTD = 0, EU_RNG_PHILOX = 1 } eu_rng_kind;

typedef struct eu_graph eu_graph;
typedef struct eu_ctx eu_ctx;

const char* eu_last_error(void);
const char* eu_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t eu_launch_count(void);

/* ------------------------------------------------------------------ graph -------------------- */
/* CSR description, HOST arrays.  Mirrors what a reference Node holds (euler/core/graph/node.h:49-57,
 * node.cc:37-96): for row r and edge type t the adjacency group is
 *   [grp_ptr[r*T+t], grp_ptr[r*T+t+1])  -- neighbor_groups_idx, made global;
 * cum_w is the NODE-GLOBAL cumulative f32 weight exactly as stored (node.cc:59-65); grp_cum[r*T+t] is
 * edge_group_collection.sum_weights_[t].  If cum_w == NULL, `w` (raw weights) must be given and the
 * prefix sums are accumulated the way Node::Init does (sequential f32, eu_graph builds them). */
typedef struct {
  int64_t n_nodes;
  int32_t n_edge_types;    /* T */
  int32_t n_node_types;
  const uint64_t* ids;     /* [n] node id of each row; id 0 is unusable (DEFAULT_UINT64) */
  const int32_t* node_type;/* [n] or NULL (all 0) */
  const float* node_w;     /* [n] or NULL (all 1.0) */
  const int64_t* grp_ptr;  /* [n*T+1] */
  const uint64_t* nbr;     /* [E] */
  const float* cum_w;      /* [E] or NULL */
  const float* grp_cum;    /* [n*T] or NULL (required iff cum_w given and T > 1) */
  const float* w;          /* [E] raw weights, used iff cum_w == NULL */
  int32_t feat_dim;        /* dense f32 feature slot 0: row length, 0 = none */
  const float* feat;       /* [n*feat_dim] or NULL */
  const int64_t* sampler_order; /* [n] rows in the order the global node sampler enumerates them
                                   (graph.cc:349-354 uses unordered_map order); NULL = row order */
  /* optional: several dense f32 feature slots (Node::float_features_idx_, node.h); when
   * n_feat_slots > 0, feat is [n, sum(feat_slot_dims)] and feat_dim must equal that sum */
  int32_t n_feat_slots;
  const int32_t* feat_slot_dims;
  /* optional ragged features (Node::uint64_features_ / binary_features_, euler/core/graph/node.h): slot s of row r is
   * [ptr[r*S+s], ptr[r*S+s+1]) of the value array; S = 0 / NULL = none */
  int32_t n_u64_slots;
  const int64_t* u64_ptr;   /* [n*S+1] */
  const uint64_t* u64_val;
  int32_t n_bin_slots;
  const int64_t* bin_ptr;   /* [n*S+1] */
  const uint8_t* bin_val;
} eu_graph_desc;

int eu_graph_create(const eu_graph_desc* desc, int device, eu_graph** out);
/* Synthetic R-MAT graph generated, sorted and prefix-summed on the device (SURVEY.md section 8d "G-RMAT"):
 * ids 1..n, one node/edge type, n_edges directed edges with (a,b,c,d), adjacency sorted by dst,
 * weight = 1 + (hash(src,dst) % 100) / 10, feat ~ U(-1,1).  feat_dim may be 0. */
int eu_graph_create_rmat(int64_t n_nodes, int64_t n_edges, double a, double b, double c,
                         uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                         eu_graph** out);
/* The rows of that same graph that shard `shard_index` of `shard_number` owns: owner(id) = id % shard_number
 * (the reference's routing (id % partitions) % shards with partitions a multiple of shards,
 * euler/core/kernels/id_split_op.cc:46-49).  The union of the shards is exactly eu_graph_create_rmat's graph. */
int eu_graph_create_rmat_shard(int64_t n_nodes, int64_t n_edges, double a, double b, double c,
                               uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                               int shard_index, int shard_number, eu_graph** out);
/* Heterogeneous variant (BASELINE configs[4]): edge type = hash(edge) % n_edge_types (adjacency grouped by
 * (row, type), one node-global cumulative weight array as node.cc:59-65), node type = id % n_node_types. */
int eu_graph_create_rmat_hetero(int64_t n_nodes, int64_t n_edges, int32_t n_edge_types, int32_t n_node_types, double a,
                                double b, double c, uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                                int shard_index, int shard_number, eu_graph** out);
/* Euler 2.0 on-disk format (euler.meta + the Node and Edge partition files; SURVEY.md Appendix B), shard `shard_index` of
 * `shard_number` with the reference's file filter (graph.cc:90-98).  = Graph::Init, graph.h:53-56. */
int eu_graph_load(const char* data_path, int shard_index, int shard_number, int device,
                  eu_graph** out);
/* load_edges = 0: node data only (Graph::Init's load_data_type "node"); eu_graph_load = load_edges 1 ("all"): the Edge
 * files, when the directory has them, feed eu_sample_edge and the edge feature ops. */
int eu_graph_load_ex(const char* data_path, int shard_index, int shard_number, int device, int load_edges,
                     eu_graph** out);
/* Edge records (Edge files of the Euler format; euler/core/graph/edge.h): needed only by sample_edge and the edge feature ops.
 * HOST arrays; features use the node layout (dense slots concatenated per edge, ragged uint64 / binary slots).
 * sampler_order: edge rows in the order the reference's edge_map_ iterates (graph.cc:372-399); NULL = row order. */
typedef struct {
  int64_t n_edges;
  const uint64_t* src;      /* [nE] */
  const uint64_t* dst;      /* [nE] */
  const int32_t* type;      /* [nE] */
  const float* w;           /* [nE] or NULL (all 1.0) */
  int32_t feat_dim;         /* total dense width, 0 = none */
  const float* feat;        /* [nE * feat_dim] */
  int32_t n_feat_slots;     /* 0 = one slot of feat_dim */
  const int32_t* feat_slot_dims;
  int32_t n_u64_slots; const int64_t* u64_ptr; const uint64_t* u64_val;
  int32_t n_bin_slots; const int64_t* bin_ptr; const uint8_t* bin_val;
  const int64_t* sampler_order;
} eu_edge_desc;
int eu_graph_set_edges(eu_graph* g, const eu_edge_desc* desc);
int64_t eu_graph_num_edge_records(const eu_graph* g);
int32_t eu_graph_edge_dense_feature_id(const eu_graph* g, const char* name);
int32_t eu_graph_edge_sparse_feature_id(const eu_graph* g, const char* name);
int32_t eu_graph_edge_binary_feature_id(const eu_graph* g, const char* name);
int eu_graph_destroy(eu_graph* g);
int64_t eu_graph_num_nodes(const eu_graph* g);
int64_t eu_graph_num_edges(const eu_graph* g);
int32_t eu_graph_num_edge_types(const eu_graph* g);
/* Host-only (no GPU needed): parse an Euler 2.0 data directory exactly as eu_graph_load does -- same file filter, same record
 * decoding, same replay of the reference's node_map_ iteration order (euler/core/graph/graph.cc:349-354) -- and report what would
 * be uploaded: counts and, for the first `cap` entries, node ids and types in GLOBAL SAMPLER ORDER.  Any out pointer may be NULL. */
int eu_graph_load_inspect(const char* data_path, int shard_index, int shard_number, int64_t* n_nodes, int64_t* n_edges,
                          int32_t* n_edge_types, int32_t* n_node_types, int64_t cap, int64_t* order_ids, int32_t* order_types);
/* Host-only helper (no GPU needed): the sampler tables eu_graph_create / eu_graph_load build for the global node and edge samplers --
 * FastWeightedCollection::Init + AliasMethod::Init (euler/common/fast_weighted_collection.h:54-74, alias_method.cc:23-63):
 * weights f32[n] -> prob f32[n], alias i32[n], *sum = the f32 weight sum.  Exposed so the tables can be checked bit for bit
 * against the reference's without a device. */
int eu_build_alias_table(const float* weights, int64_t n, float* prob, int32_t* alias, float* sum);
int32_t eu_graph_num_node_types(const eu_graph* g);
int32_t eu_graph_feat_dim(const eu_graph* g);
int64_t eu_graph_hbm_bytes(const eu_graph* g);
/* Copy the device CSR back to caller-allocated HOST arrays (any pointer may be NULL). */
int eu_graph_export(const eu_graph* g, uint64_t* ids, int32_t* node_type, float* node_w,
                    int64_t* grp_ptr, uint64_t* nbr, float* cum_w, float* grp_cum, float* feat);
/* type-name lookup from euler.meta (tf_euler/python/euler_ops/type_ops.py:31-64); -1 if unknown */
int32_t eu_graph_edge_type_id(const eu_graph* g, const char* name);
int32_t eu_graph_node_type_id(const eu_graph* g, const char* name);
/* dense feature slot of feature `name` (looked up as "dense_"+name like get_dense_feature_op.cc:83);
 * -1 if unknown.  eu_graph_dense_feature_dim: stored width of a slot. */
int32_t eu_graph_dense_feature_id(const eu_graph* g, const char* name);
int32_t eu_graph_dense_feature_dim(const eu_graph* g, int32_t fid);
/* slots of the uint64 ("sparse_"+name, get_sparse_feature_op.cc:75) and binary ("binary_"+name) features; -1 if unknown */
int32_t eu_graph_sparse_feature_id(const eu_graph* g, const char* name);
int32_t eu_graph_binary_feature_id(const eu_graph* g, const char* name);
/* the most uint64 values any node holds in slot `fid` (computed at upload); 0 for an unknown slot.  Sizes the value buffers
 * of eu_sample_fanout_with_feature without a lengths-first call. */
int64_t eu_graph_sparse_feature_max_len(const eu_graph* g, int32_t fid);

/* ------------------------------------------------------------------ contexts ----------------- */
/* stream: a cudaStream_t (NULL = legacy default stream). */
int eu_ctx_create(eu_graph* g, eu_rng_kind rng, uint64_t seed, void* stream, eu_ctx** out);
int eu_ctx_destroy(eu_ctx* c);
int eu_ctx_set_stream(eu_ctx* c, void* stream);
int eu_ctx_seed(eu_ctx* c, uint64_t seed);           /* engine e <- seed + e; stream-ordered */
/* A ctx may carry several engines: batch b of a *_batched call runs on engine b (its own draw stream and
 * its own dedup scope), i.e. each batch is exactly one reference op call on one client thread; batching only
 * shares kernel launches.  seeds == NULL: engine e <- seed + e.  Plain ops use engine 0. */
int eu_ctx_set_engines(eu_ctx* c, int32_t n, const uint64_t* seeds);
/* pre-size scratch (required before graph capture) for hops of up to max_rows rows; it also covers the level scratch of an
 * eu_sample_fanout_with_feature whose levels 1..L hold at most 2 * max_rows ids in all (every count >= 2) */
int eu_ctx_reserve(eu_ctx* c, int64_t max_rows);
int eu_ctx_sync(eu_ctx* c);
/* number of uniforms the MINSTD engine has produced since the last seed (synchronises) */
int eu_ctx_draws(eu_ctx* c, uint64_t* draws);
/* Per-kernel timing: while enabled, every kernel this ctx launches is bracketed by CUDA events on the
 * ctx stream.  eu_ctx_profile_read synchronises and returns "name,rows,launches,total_ms" lines. */
int eu_ctx_profile(eu_ctx* c, int enable);
int eu_ctx_profile_read(eu_ctx* c, char* buf, int64_t cap);

/* ------------------------------------------------------------------ sampling ops ------------- */
/* tf_euler.sample_neighbor -- TF op SampleNeighbor (tf_euler/ops/neighbor_ops.cc:138-163, kernel
 * tf_euler/kernels/sample_neighbor_op.cc:54-129).  nodes i64[B]; etypes i32[K] (host);
 * outputs [B,count]: ids i64 (default_node fill), w f32 (0 fill), t i32 (-1 fill). */
int eu_sample_neighbor(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                       int32_t count, int64_t default_node, int64_t* out_ids, float* out_w,
                       int32_t* out_t);
int eu_sample_neighbor_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                            int32_t K, int32_t count, int64_t default_node, int64_t* out_ids,
                            float* out_w, int32_t* out_t);
/* euler::SampleNeighbor of the C++ api (euler/core/api/api.cc:223-236): one Node::SampleNeighbor per element of `nodes`,
 * in order, WITHOUT the engine's unique/gather rule -- a repeated id draws again.  Engine-form outputs [B,count]: rows
 * without a result (absent node / no edge of the requested types) are (0, 0.0, -1).  Exact-RNG contexts only. */
int eu_sample_neighbor_raw(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                           int32_t count, int64_t* out_ids, float* out_w, int32_t* out_t);
int eu_sample_neighbor_raw_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                int32_t count, int64_t* out_ids, float* out_w, int32_t* out_t);
/* tf_euler.sample_fanout -- TF op SampleFanout (tf_euler/ops/neighbor_ops.cc:228-280, kernel
 * tf_euler/kernels/sample_fanout_op.cc:60-145).  etypes i32[L,K] (host), counts i32[L] (host);
 * out_*[l] point to B*prod(counts[0..l]) elements.  The frontier never leaves the device. */
int eu_sample_fanout(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                     const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                     float* const* out_w, int32_t* const* out_t);
/* nb independent batches of B seeds in one set of launches (nodes / outputs batch-major). */
int eu_sample_fanout_batched(eu_ctx* c, const int64_t* nodes, int32_t nb, int64_t B, const int32_t* etypes, int32_t K,
                             const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                             float* const* out_w, int32_t* const* out_t);
int eu_sample_fanout_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                          int32_t K, const int32_t* counts, int32_t L, int64_t default_node,
                          int64_t* const* out_ids, float* const* out_w, int32_t* const* out_t);
int eu_sample_fanout_batched_host(eu_ctx* c, const int64_t* nodes, int32_t nb, int64_t B, const int32_t* etypes,
                                  int32_t K, const int32_t* counts, int32_t L, int64_t default_node,
                                  int64_t* const* out_ids, float* const* out_w, int32_t* const* out_t);
/* tf_euler.sample_fanout_with_feature -- TF op SampleFanoutWithFeature (tf_euler/python/euler_ops/neighbor_ops.py:49-69, kernel
 * tf_euler/kernels/sample_fanout_with_feature_op.cc:95-274): eu_sample_fanout (same draws, ids, weights and types bit for bit,
 * L <= 16) plus the dense and uint64 features of every level.  Level 0 is `nodes` as given; level l >= 1 is hop l's ENGINE ids
 * (v_select(nb_l), :65-68), so a default-filled slot gets zeros and the sparse default whatever default_node is.  Rows of level
 * i: rows_0 = B, rows_i = rows_{i-1} * counts[i-1]; a hop with count 0 ends the chain (later levels have 0 rows).
 *   dense_fids / dense_dims i32[ND] (host; slot ids as eu_get_dense_feature, -1 = unknown = zeros);
 *   out_dense[i*ND + j] -> f32[rows_i, dense_dims[j]], zero fill; a stored width above dense_dims[j] is clipped to it
 *   (:220-237 copies the whole stored row, past the row's end).
 *   sparse_fids i32[NS], sparse_defaults i64[NS] (host; slot ids as eu_get_sparse_feature);
 *   out_sp_ptr[i*NS + j] -> i64[rows_i + 1] and out_sp_val[i*NS + j] -> i64[rows_i * max(1, eu_graph_sparse_feature_max_len(fid_j))]:
 *   eu_get_sparse_feature's CSR form, a row without values owns one entry = the default (:238-257).
 * (L+1)*ND and (L+1)*NS are at most 64 each (EU_ERR_UNSUPPORTED beyond).  One dense launch and three sparse launches serve all
 * levels and features; no host synchronisation. */
int eu_sample_fanout_with_feature(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                  const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                                  float* const* out_w, int32_t* const* out_t, int32_t ND, const int32_t* dense_fids,
                                  const int32_t* dense_dims, float* const* out_dense, int32_t NS, const int32_t* sparse_fids,
                                  const int64_t* sparse_defaults, int64_t* const* out_sp_ptr, int64_t* const* out_sp_val);
/* host buffers, same sizing; out_sp_val[k] receives out_sp_ptr[k][rows] values */
int eu_sample_fanout_with_feature_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                       const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                                       float* const* out_w, int32_t* const* out_t, int32_t ND, const int32_t* dense_fids,
                                       const int32_t* dense_dims, float* const* out_dense, int32_t NS, const int32_t* sparse_fids,
                                       const int64_t* sparse_defaults, int64_t* const* out_sp_ptr, int64_t* const* out_sp_val);
/* tf_euler.sample_node -- TF op SampleNode (tf_euler/ops/sample_ops.cc:22-37, kernel
 * tf_euler/kernels/sample_node_op.cc:39-96; euler::SampleNode api.cc:32-37).  types i32[n_types]
 * (host); a single -1 means all types.  out i64[count]. */
int eu_sample_node(eu_ctx* c, int32_t count, const int32_t* types, int32_t n_types, int64_t* out);
int eu_sample_node_host(eu_ctx* c, int32_t count, const int32_t* types, int32_t n_types,
                        int64_t* out);
/* tf_euler.random_walk -- TF op RandomWalk (tf_euler/ops/walk_ops.cc:77-107, kernel
 * tf_euler/kernels/random_walk_op.cc:83-289).  etypes i32[L,K] (host); out i64[B,L+1].
 * EU_RNG_MINSTD: the reference's walks bit for bit (serial engine stream, sequential f32 prefix of the biased weights).
 * EU_RNG_PHILOX with one edge type per step on sorted adjacency: node2vec steps by rejection sampling (propose from the
 * stored CDF, accept with bias / max bias) -- the same transition distribution at O(log deg) per step. */
int eu_random_walk(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                   int32_t L, float p, float q, int64_t default_node, int64_t* out);
int eu_random_walk_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                        int32_t K, int32_t L, float p, float q, int64_t default_node, int64_t* out);
/* tf_euler.get_dense_feature, one feature -- TF op GetDenseFeature (tf_euler/ops/feature_ops.cc:94-140,
 * kernel tf_euler/kernels/get_dense_feature_op.cc:63-121).  out f32[M,dim], zero fill. */
int eu_get_dense_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int32_t dim,
                         float* out);
int eu_get_dense_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int32_t dim,
                              float* out);
/* tf_euler.get_sparse_feature, one feature (tf_euler/kernels/get_sparse_feature_op.cc:52-130 over Node::GetUint64Feature
 * node.cc:366-379): the uint64 values of slot `fid` for every node, CSR-style: node i owns out_values[out_ptr[i], out_ptr[i+1]).
 * A node without values (absent node, unknown slot, empty slot) owns exactly ONE entry = default_value (the kernel's
 * SparseTensor gets {i, 0} -> default, :96-99).  cap = 0: lengths only (out_values may be NULL); only the first `cap`
 * entries are written.  The SparseTensor of the reference is indices (i, k - out_ptr[i]), dense_shape [M, max row length]. */
int eu_get_sparse_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap,
                          int64_t* out_ptr, int64_t* out_values);
int eu_get_sparse_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap,
                               int64_t* out_ptr, int64_t* out_values, int64_t* total);
/* tf_euler.get_binary_feature, one feature (tf_euler/kernels/get_binary_feature_op.cc over Node::GetBinaryFeature
 * node.cc:396-409): the bytes of slot `fid` for every node, CSR-style (absent node / unknown slot: empty string). */
int eu_get_binary_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t cap, int64_t* out_ptr, uint8_t* out_bytes);
int eu_get_binary_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t cap, int64_t* out_ptr,
                               uint8_t* out_bytes, int64_t* total);

/* tf_euler.sample_edge -- TF op SampleEdge (tf_euler/kernels/sample_edge_op.cc; Graph::SampleEdge graph.cc:277-301): `count`
 * edges of ONE type drawn by the alias method over the edge weights, out i64[count,3] = (src, dst, type).  Several types or
 * -1 return EU_ERR_STATE: the reference's edge_type_collection_ is never initialised and it returns nothing for them. */
int eu_sample_edge(eu_ctx* c, int32_t count, const int32_t* types, int32_t n_types, int64_t* out);
/* tf_euler.get_edge_dense_feature / _sparse_ / _binary_ (tf_euler/kernels/get_edge_*_feature_op.cc over
 * euler::GetEdge*Feature api.cc:148-205): edges i64[E,3] = (src, dst, type); unknown edges give zeros / the default entry /
 * the empty string.  Device pointers; the ragged variants follow eu_get_sparse_feature's two-call convention. */
int eu_get_edge_dense_feature(eu_ctx* c, const int64_t* edges, int64_t E, int32_t fid, int32_t dim, float* out);
int eu_get_edge_sparse_feature(eu_ctx* c, const int64_t* edges, int64_t E, int32_t fid, int64_t default_value, int64_t cap,
                               int64_t* out_ptr, int64_t* out_values);
int eu_get_edge_binary_feature(eu_ctx* c, const int64_t* edges, int64_t E, int32_t fid, int64_t cap, int64_t* out_ptr, uint8_t* out_bytes);

/* tf_euler.get_full_neighbor core (euler::GetFullNeighbor api.cc:208-221 over Node::GetFullNeighbor node.cc:176-198):
 * for every node the edges of each requested type, in the order the types are given, as (id, weight, type); a missing
 * node has an empty list.  CSR-style output: out_ptr i64[B+1] (device) -- entries of node i are
 * [out_ptr[i], out_ptr[i+1]); only the first `cap` entries are written (cap = 0: lengths only; out_* may be NULL).
 * The _host variant takes host buffers and also returns *total = out_ptr[B]: call it with cap = 0 to size the
 * outputs, then again with cap >= *total (the reference's kernel sizes its SparseTensor the same way,
 * tf_euler/kernels/get_full_neighbor_op.cc). */
int eu_get_full_neighbor(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                         int64_t cap, int64_t* out_ptr, int64_t* out_ids, float* out_w,
                         int32_t* out_t);
int eu_get_full_neighbor_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                              int64_t cap, int64_t* out_ptr, int64_t* out_ids, float* out_w, int32_t* out_t,
                              int64_t* total);

/* tf_euler.get_sorted_full_neighbor (neighbor_ops.py:100-119; Node::GetSortedFullNeighbor node.cc:210-262; engine
 * "order_by id asc", euler/core/kernels/get_neighbor_op.cc:128-141): eu_get_full_neighbor with every node's entries ordered
 * by neighbor id ascending (ties keep the listing order).  Same convention (cap = 0: lengths only; cap must cover the listing). */
int eu_get_sorted_full_neighbor(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                int64_t cap, int64_t* out_ptr, int64_t* out_ids, float* out_w, int32_t* out_t);
/* tf_euler.get_top_k_neighbor (neighbor_ops.py:44-46; tf_euler/kernels/get_top_k_neighbor_op.cc:54-121; engine "order_by
 * weight desc, limit k"): dense [B,k] outputs, heaviest edge first, default_node / 0.0 / -1 fill.  Device pointers; synchronises
 * the stream once (scratch is sized from the listing length). */
int eu_get_top_k_neighbor(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K, int32_t k,
                          int64_t default_node, int64_t* out_ids, float* out_w, int32_t* out_t);
/* tf_euler.sample_neighbor_layerwise (neighbor_ops.py:72-77; tf_euler/kernels/sample_neighbor_layerwise_with_adj_op.cc:54-150 over
 * API_LOCAL_SAMPLE_L, euler/core/kernels/local_sample_layer_op.cc:41-140): nodes i64[batch, n]; per batch row `count` neighbors
 * drawn from the union of the rows' neighbor lists, candidates unique by (dst, type) with summed weights (weight_func 1 = sqrt),
 * out_nb i64[batch, count] (default_node when the union is empty); out_adj (may be NULL) f32[batch, n, count] = 1.0 where
 * out_nb[b, k] is a neighbor of nodes[b, j] -- the dense view of the op's SparseTensor.  Same candidate set, weights and
 * distribution as the reference; the candidate ORDER (an unordered_map<string> artefact upstream) is (dst, type) here.
 * Device pointers; synchronises (scratch is sized from the listing). */
int eu_sample_neighbor_layerwise(eu_ctx* c, const int64_t* nodes, int64_t batch, int32_t n, const int32_t* etypes, int32_t K,
                                 int32_t count, int64_t default_node, int32_t weight_func, int64_t* out_nb, float* out_adj);
/* tf_euler.sparse_get_adj (neighbor_ops.py:33-36; euler/core/kernels/sparse_get_adj_op.cc:34-90): nodes i64[batch, N],
 * nb_nodes i64[batch, M] -> out_adj f32[batch, N, M] = 1.0 where an edge nodes[b, j] -> nb_nodes[b, k] of a listed type exists
 * (dense view of the SparseTensor). */
int eu_sparse_get_adj(eu_ctx* c, const int64_t* nodes, const int64_t* nb_nodes, int64_t batch, int32_t N, int32_t M,
                      const int32_t* etypes, int32_t K, float* out_adj);
/* tf_euler.gen_pair (tf_euler/kernels/gen_pair_op.cc:41-100): skip-gram pairs of walks.  paths i64[B,path_len] ->
 * out i64[B, eu_gen_pair_count(path_len, lw, rw), 2] (device pointers). */
int64_t eu_gen_pair_count(int32_t path_len, int32_t left_win_size, int32_t right_win_size);
int eu_gen_pair(eu_ctx* c, const int64_t* paths, int64_t B, int32_t path_len, int32_t left_win_size, int32_t right_win_size,
                int64_t* out);

/* euler::GetNodeType (euler/core/api/api.cc:50-61; tf_euler get_node_type): type of every node, INT32_MIN
 * (DEFAULT_INT32, euler/common/data_types.cc:23) for ids that are not in the graph. */
int eu_get_node_type(eu_ctx* c, const int64_t* nodes, int64_t B, int32_t* out);
int eu_get_node_type_host(eu_ctx* c, const int64_t* nodes, int64_t B, int32_t* out);
/* Node::GetWeight (euler/core/graph/node.h:78) of every node, 0.0 for ids that are not in the graph (host buffers). */
int eu_get_node_weight_host(eu_ctx* c, const int64_t* nodes, int64_t B, float* out);

/* tf.unique on the device (UniqueDataFlow / SageDataFlow, tf_euler/python/dataflow/neighbor_dataflow.py:84-109): the
 * distinct values of ids in order of FIRST occurrence and, per input, the index of its value in that list.
 * uniq: device i64[n] (first *n_unique valid), inverse: device i32[n], n_unique: device i64[1] (may be NULL). */
int eu_unique(eu_ctx* c, const int64_t* ids, int64_t n, int64_t* uniq, int32_t* inverse, int64_t* n_unique);

/* ------------------------------------------------------------------ message-passing ops ------ */
/* MPGather / MPScatterAdd / MPScatterMax (tf_euler/ops/mp_ops.cc:22-81; kernels
 * tf_euler/kernels/gather_op.cc:31-52, scatter_op.cc:32-92).  f32 data, i32 indices, as registered. */
int eu_gather(eu_ctx* c, const float* params, int64_t N, int64_t D, const int32_t* idx, int64_t E,
              float* out);
int eu_scatter_add(eu_ctx* c, const float* updates, int64_t D, const int32_t* idx, int64_t E,
                   int64_t size, float* out);
int eu_scatter_max(eu_ctx* c, const float* updates, int64_t D, const int32_t* idx, int64_t E,
                   int64_t size, float* out);
/* scatter_mean (tf_euler/python/euler_ops/mp_ops.py:65-69): add / (add(ones) + 1e-7) */
int eu_scatter_mean(eu_ctx* c, const float* updates, int64_t D, const int32_t* idx, int64_t E,
                    int64_t size, float* out);
/* Fused SAGE aggregation for fixed-fanout blocks (sage_dataflow.py:43-46 edge_src = repeat(range(B),count)):
 * out[r,:] = mean_{j<count} feat[row(nbr_ids[r*count+j]),:] with scatter_mean's (count + 1e-7)
 * divisor; ids not in the graph (default fill) contribute zeros, as get_dense_feature would. */
int eu_sage_mean_aggregate(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count,
                           int32_t dim, float* out);
int eu_sage_mean_aggregate_host(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count,
                                int32_t dim, float* out);
/* the same block with aggr = 'add' (scatter_add, tf_euler/kernels/scatter_op.cc:44-55): out[r,:] = sum_j feat[row(nbr_ids[r*count+j]),:] */
int eu_sage_add_aggregate(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, float* out);
int eu_gather_host(eu_ctx* c, const float* params, int64_t N, int64_t D, const int32_t* idx,
                   int64_t E, float* out);
int eu_scatter_add_host(eu_ctx* c, const float* updates, int64_t D, const int32_t* idx, int64_t E,
                        int64_t size, float* out);
int eu_scatter_max_host(eu_ctx* c, const float* updates, int64_t D, const int32_t* idx, int64_t E,
                        int64_t size, float* out);

/* ------------------------------------------------------------------ sharding (multi-GPU) ----- */
/* Replace ID_SPLIT / IDX_MERGE / DATA_MERGE (euler/core/kernels/id_split_op.cc:46-99, idx_merge_op.cc:32-78)
 * either side of an all-to-all.  eu_shard_bucket: stable counting sort of ids by owner
 * (id % num_partitions) % shard_num; sorted_ids[k] came from ids[src_index[k]]; counts[o] / offsets[o]
 * (device, i64[shard_num] / [shard_num+1]) delimit owner o's segment.  eu_shard_merge_sample: replies in
 * sorted order -> original row order + TF packing + engine-id frontier.  eu_shard_merge_rows: the same for
 * fixed-width f32 rows (features). */
int eu_shard_bucket(eu_ctx* c, const int64_t* ids, int64_t rows, int32_t num_partitions, int32_t shard_num,
                    int32_t self_shard, int64_t* sorted_ids, int32_t* src_index, int64_t* counts, int64_t* offsets);
/* ids 0 and 2^64-1 (placeholder / default fill) exist nowhere and are routed to self_shard.
 * eu_shard_pack_sample: (ids, w, t)[n] -> n 16-byte records {id, w | t << 32} so one all-to-all carries a reply;
 * eu_shard_merge_sample consumes records in sorted order. */
int eu_shard_pack_sample(eu_ctx* c, const int64_t* ids, const float* w, const int32_t* t, int64_t n, int64_t* packed);
int eu_shard_merge_sample(eu_ctx* c, const int64_t* packed, const int32_t* src_index, int64_t rows, int32_t count,
                          int64_t default_node, int64_t* eng_ids, int64_t* out_ids, float* out_w, int32_t* out_t);
int eu_shard_merge_rows(eu_ctx* c, const float* rows_in, const int32_t* src_index, int64_t rows, int64_t D,
                        float* out);

/* Peer-memory exchange (csrc/p2p.cu): the all-to-all of a hop / feature fetch done by the kernels themselves over
 * NVLink peer mappings -- no NCCL call, no host sync, CUDA-graph capturable.  One eu_sym per (ctx, rank): a symmetric
 * region exported with cudaIpc; all_gather the 64-byte handles (any out-of-band channel) and eu_sym_connect.
 * Results land in the rank's own symmetric output arrays (eu_sym_outputs), already in request order. */
typedef struct eu_sym eu_sym;
int eu_sym_create(eu_ctx* c, int32_t rank, int32_t world, int64_t max_rows, int32_t max_count, int64_t max_feat_rows,
                  int32_t max_dim, eu_sym** out, void* handle_out /* 64 bytes */);
int eu_sym_connect(eu_sym* s, const void* handles /* world x 64 bytes, rank order */);
int eu_sym_destroy(eu_sym* s);
int eu_sym_outputs(eu_sym* s, int64_t** eng, int64_t** ids, float** w, int32_t** t, float** rows);
int eu_sym_error(eu_sym* s, int* err);   /* 1 if a bounded wait timed out (synchronises) */
int eu_sym_sample_hop(eu_sym* s, const int64_t* seeds, int64_t rows, const int32_t* etypes, int32_t K, int32_t count,
                      int64_t default_node, int32_t num_partitions, int32_t want_packed);
/* nb independent batches per exchange: seeds i64[nb][rows], outputs [nb][rows][count]; batch g is sampled by every
 * shard's engine g (eu_ctx_set_engines) over the requests of rank 0..N-1 for that batch, its own dedup scope. */
int eu_sym_sample_hop_batched(eu_sym* s, const int64_t* seeds, int32_t nb, int64_t rows, const int32_t* etypes, int32_t K,
                              int32_t count, int64_t default_node, int32_t num_partitions, int32_t want_packed);
int eu_sym_get_dense_feature(eu_sym* s, const int64_t* ids, int64_t rows, int32_t fid, int32_t dim, int32_t num_partitions);
/* Sharded eu_sage_mean_aggregate: REMOTE get_dense_feature (euler/core/kernels/remote_op.cc:60-146) fused with the
 * scatter_mean that follows it (tf_euler/python/euler_ops/mp_ops.py:65-69 over sage_dataflow.py:43-46's edge_src).
 * Each owner sums the rows of ITS ids per destination (j ascending) and stores one partial row per destination in the
 * requester's region; the requester adds the partials in rank order and divides by (count + 1e-7).  rows*count ids must
 * fit the inbox (max(max_rows, max_feat_rows)) and world*rows*dim floats the feature region.  out: device f32[rows*dim]. */
int eu_sym_sage_mean(eu_sym* s, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, int32_t num_partitions,
                     float* out);

/* ------------------------------------------------------------------ reference entry point ---- */
/* bool InitQueryProxy(const char* conf) -- tf_euler/utils/init_query_proxy.cc:19-36.  "k=v;k=v";
 * keys of euler/client/query_proxy.cc:41-160 that apply here: mode (local only), data_path,
 * sampler_type, data_type, shard_num(=1); new keys: device, seed, rng (minstd|philox).
 * Returns false only for an empty / malformed list (as the reference does, :22-33); load errors are
 * logged.  Creates the process-wide default graph + ctx used by the *_default accessors. */
bool InitQueryProxy(const char* conf);
eu_graph* eu_default_graph(void);
eu_ctx* eu_default_ctx(void);
int eu_set_default_graph(eu_graph* g, eu_rng_kind rng, uint64_t seed);

#ifdef __cplusplus
}
#endif
#endif /* EULER_B200_H_ */
