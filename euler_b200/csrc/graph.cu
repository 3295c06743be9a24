// HBM-resident graph store: CSR + cumulative weights + id->row table + dense features.
// Replaces euler/core/graph/{graph,node}.cc's unordered_map<NodeID,Node*> of per-node vectors
// (node.h:49-57, graph.h:187-199) with flat arrays laid out for coalesced 128-byte access.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <mutex>

#include "internal.h"

namespace eu {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ------------------------------------------------------------------------------------- kernels
__global__ void k_hash_clear(HashSlot* tab, unsigned long long cap) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  if (i < cap) { tab[i].key = 0; tab[i].row = kEmptyRow; }
}

// Open addressing, linear probing.  A later row with a duplicate id overwrites the earlier one,
// like node_map_[id] = n (graph.cc:162-166): resolved with atomicMax on the row.
__global__ void k_hash_insert(HashSlot* tab, unsigned long long mask, const unsigned long long* ids,
                              int64_t n) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  unsigned long long id = ids[r];
  unsigned long long h = mix64(id) & mask;
  while (true) {
    // claim on the row field: kEmptyRow -> r.  Key is written by the claimer; readers at build
    // time spin on the key of a claimed slot.
    unsigned long long prev = atomicCAS(&tab[h].row, kEmptyRow, (unsigned long long)r);
    if (prev == kEmptyRow) {
      atomicExch(&tab[h].key, id + 1);  // +1: 0 means "key not yet published"
      return;
    }
    unsigned long long k;
    do { k = atomicAdd(&tab[h].key, 0ull); } while (k == 0);
    if (k == id + 1) {
      atomicMax(&tab[h].row, (unsigned long long)r);  // kEmptyRow is never the max of valid rows
      return;
    }
    h = (h + 1) & mask;
  }
}

__global__ void k_hash_finalize(HashSlot* tab, unsigned long long cap) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  if (i < cap && tab[i].row != kEmptyRow) tab[i].key -= 1;
}

// Node::Init accumulation (node.cc:46-70): ONE running f32 sum per node across all its groups,
// per-group f32 sums, and the edge-group CWC's running f32 sum (compact_weighted_collection.h:82-97).
// Sequential per row on purpose: a parallel scan would round differently.
__global__ void k_build_cum(int64_t n, int32_t T, const int64_t* grp_ptr, const float* w,
                            float* cum_w, float* grp_cum) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  float sum_weight = 0.f, cwc = 0.f;
  for (int32_t t = 0; t < T; ++t) {
    float type_weight = 0.f;
    for (int64_t j = grp_ptr[r * T + t]; j < grp_ptr[r * T + t + 1]; ++j) {
      float x = w[j];
      sum_weight = __fadd_rn(sum_weight, x);
      type_weight = __fadd_rn(type_weight, x);
      cum_w[j] = sum_weight;
    }
    cwc = __fadd_rn(cwc, type_weight);
    if (grp_cum) grp_cum[r * T + t] = cwc;
  }
}

// ---- synthetic R-MAT (SURVEY.md section 8d)
__device__ __forceinline__ unsigned long long splitmix(unsigned long long& s) {
  unsigned long long z = (s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// keys == nullptr: only count the edges this shard owns.  Otherwise append key = local_row * n + dst
// (cursor order is irrelevant: the keys are radix-sorted afterwards and equal keys are indistinguishable).
__global__ void k_rmat_edges(unsigned long long* keys, unsigned long long* cursor, int64_t n_edges, int64_t n_nodes,
                             int scale, double a, double b, double c, unsigned long long seed, int N, int shard, int T) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  unsigned long long s = mix64(seed ^ (unsigned long long)e * 0xD6E8FEB86659FD93ull);
  unsigned long long src = 0, dst = 0;
  for (int l = 0; l < scale; ++l) {
    double u = (double)(splitmix(s) >> 11) * (1.0 / 9007199254740992.0);
    int q = u < a ? 0 : (u < a + b ? 1 : (u < a + b + c ? 2 : 3));
    src = (src << 1) | (unsigned long long)(q >> 1);
    dst = (dst << 1) | (unsigned long long)(q & 1);
  }
  // scramble so the heavy corner is not the low ids, then fold into [0, n)
  src = mix64(src + 0x51ED27) % (unsigned long long)n_nodes;
  dst = mix64(dst + 0x51ED27) % (unsigned long long)n_nodes;
  const unsigned long long src_id = src + 1;
  if (N > 1 && (int)(src_id % (unsigned long long)N) != shard) return;
  if (!keys) { atomicAdd(cursor, 1ull); return; }
  const unsigned long long base_id = shard == 0 ? (unsigned long long)N : (unsigned long long)shard;
  const unsigned long long row = N > 1 ? (src_id - base_id) / (unsigned long long)N : src;
  const unsigned long long pos = N > 1 ? atomicAdd(cursor, 1ull) : (unsigned long long)e;
  // heterogeneous graphs: edge type = hash(edge index) % T; adjacency groups are (row, type)
  const unsigned long long et = T > 1 ? mix64(seed * 0x2545F4914F6CDD1Dull + (unsigned long long)e) % (unsigned long long)T : 0ull;
  keys[pos] = (row * (unsigned long long)T + et) * (unsigned long long)n_nodes + dst;
}

__global__ void k_count_src(const unsigned long long* keys, int64_t n_edges, int64_t n_nodes,
                            int64_t* deg) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  atomicAdd((unsigned long long*)&deg[keys[e] / (unsigned long long)n_nodes], 1ull);
}

__global__ void k_rmat_fill(const unsigned long long* keys, int64_t n_edges, int64_t n_nodes,
                            unsigned long long* nbr, float* w, unsigned long long base_id, unsigned long long stride, int T) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  unsigned long long k = keys[e];
  unsigned long long row = k / (unsigned long long)n_nodes / (unsigned long long)T, dst = k % (unsigned long long)n_nodes;
  unsigned long long src = base_id + row * stride - 1;  // global 0-based source index
  nbr[e] = dst + 1;  // ids are 1..n
  unsigned long long h = mix64(src * 0x9E3779B97F4A7C15ull ^ dst);
  w[e] = 1.0f + (float)(h % 100ull) / 10.0f;
}

__global__ void k_iota_ids(unsigned long long* ids, int32_t* ntype, float* nw, int64_t n, unsigned long long base_id,
                           unsigned long long stride, int NT) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  ids[r] = base_id + (unsigned long long)r * stride;
  ntype[r] = (int32_t)(ids[r] % (unsigned long long)NT);  // node type = id % NT
  nw[r] = 1.0f;
}

// feat[row, d] = U(-1,1) from a hash of (global node index, d): identical on every shard layout
__global__ void k_fill_feat(float* feat, int64_t n_local, int32_t dim, unsigned long long seed, unsigned long long base_id,
                            unsigned long long stride) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t total = n_local * (int64_t)dim;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (; i < total; i += step) {
    const unsigned long long row = (unsigned long long)(i / dim), col = (unsigned long long)(i % dim);
    const unsigned long long gi = (base_id + row * stride - 1) * (unsigned long long)dim + col;
    unsigned long long h = mix64(seed ^ (gi * 0x9E3779B97F4A7C15ull));
    feat[i] = (float)((double)(h >> 11) * (2.0 / 9007199254740992.0) - 1.0);
  }
}

// adj_sorted: lets the node2vec step classify neighbors by merging sorted lists in parallel
// (the reference's two-pointer merge, tf_euler/kernels/random_walk_op.cc:140-168, assumes sorted lists too).
__global__ void k_check_adj_sorted(int64_t n_groups, const int64_t* grp_ptr, const unsigned long long* nbr, int* unsorted) {
  int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n_groups) return;
  for (int64_t j = grp_ptr[k] + 1; j < grp_ptr[k + 1]; ++j)
    if ((long long)nbr[j - 1] > (long long)nbr[j]) { *unsorted = 1; return; }
}

static int build_hash(eu_graph* g) {
  DevGraph& d = g->d;
  const int tb = 256;
  if (!d.dense_ids) {   // ids in arithmetic progression resolve by arithmetic (lookup_row): no table (4.3 GB at 100M nodes)
    unsigned long long cap = 64;
    while (cap < (unsigned long long)d.n * 2) cap <<= 1;
    HashSlot* tab = nullptr;
    int rc = g->alloc(&tab, (int64_t)cap);
    if (rc) return rc;
    k_hash_clear<<<(unsigned)ceil_div(cap, tb), tb>>>(tab, cap);
    EU_LAUNCHED();
    if (d.n > 0) {
      k_hash_insert<<<(unsigned)ceil_div(d.n, tb), tb>>>(tab, cap - 1, d.ids, d.n);
      EU_LAUNCHED();
    }
    k_hash_finalize<<<(unsigned)ceil_div(cap, tb), tb>>>(tab, cap);
    EU_LAUNCHED();
    EU_CUDA(cudaDeviceSynchronize());
    d.htab = tab;
    d.hmask = cap - 1;
  }
  {
    int* flag = nullptr;
    EU_CUDA(cudaMalloc(&flag, sizeof(int)));
    EU_CUDA(cudaMemset(flag, 0, sizeof(int)));
    if (d.n * d.T > 0) {
      k_check_adj_sorted<<<(unsigned)ceil_div(d.n * d.T, tb), tb>>>(d.n * d.T, d.grp_ptr, d.nbr, flag);
      EU_LAUNCHED();
    }
    int h = 0;
    EU_CUDA(cudaMemcpy(&h, flag, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(flag);
    d.adj_sorted = h ? 0 : 1;
  }
  return EU_OK;
}

template <typename T>
static int upload(eu_graph* g, const T** dst, const T* src, int64_t count) {
  T* p = nullptr;
  int rc = g->alloc(&p, count);
  if (rc) return rc;
  if (count > 0) EU_CUDA(cudaMemcpy(p, src, sizeof(T) * (size_t)count, cudaMemcpyHostToDevice));
  *dst = p;
  return EU_OK;
}

// Walker alias tables.  RESTATEMENT of AliasMethod::Init (euler/common/alias_method.cc:23-63): the tables must be bit-identical to
// the reference's (the global sampler's draws index them), so the pairing order (two LIFO stacks, light entry first) and every
// f32 / f64 operation -- p = w * n in f32, the donor's remainder (w_heavy + w_light) in f32 then minus the f64 mean, rounded back
// to f32, the > comparison against the f64 mean -- are the reference's; nothing else of that file is used.
static void alias_build(const std::vector<float>& weights, std::vector<float>* prob,
                        std::vector<int32_t>* alias) {
  const size_t n = weights.size();
  prob->assign(n, 0.f);
  alias->assign(n, 0);
  std::vector<float> rem(weights);                 // what is left of each entry's normalised weight
  const double mean = 1 / static_cast<double>(n);
  std::vector<int64_t> light, heavy;               // LIFO: the reference pops the most recently pushed index
  for (size_t i = 0; i < n; i++) (rem[i] > mean ? heavy : light).push_back((int64_t)i);
  while (!heavy.empty() && !light.empty()) {
    const int64_t lo = light.back(); light.pop_back();
    const int64_t hi = heavy.back(); heavy.pop_back();
    (*prob)[lo] = rem[lo] * (float)n;
    (*alias)[lo] = (int32_t)hi;
    const float both = rem[hi] + rem[lo];
    rem[hi] = (float)((double)both - mean);
    (rem[hi] > mean ? heavy : light).push_back(hi);
  }
  for (int64_t i : light) (*prob)[i] = 1.0f;       // leftovers of either stack keep their own slot
  for (int64_t i : heavy) (*prob)[i] = 1.0f;
}

// FastWeightedCollection::Init (fast_weighted_collection.h:54-74): f32 sum, f32 divide, alias.
static float fwc_build(const std::vector<float>& w, std::vector<float>* prob,
                       std::vector<int32_t>* alias) {
  float s = 0.0f;
  for (float x : w) s += x;
  std::vector<float> norm(w);
  for (auto& x : norm) x /= s;
  alias_build(norm, prob, alias);
  return s;
}

void fwc_build_public(const std::vector<float>& w, std::vector<float>* prob, std::vector<int32_t>* alias, float* sum) {
  *sum = fwc_build(w, prob, alias);
}

}  // namespace eu
extern "C" int eu_build_alias_table(const float* weights, int64_t n, float* prob, int32_t* alias, float* sum) {
  if (n < 0 || (n > 0 && (!weights || !prob || !alias))) { eu::set_error("eu_build_alias_table: bad argument"); return EU_ERR_INVALID; }
  std::vector<float> w(weights, weights + n), p;
  std::vector<int32_t> a;
  float s = 0.f;
  eu::fwc_build_public(w, &p, &a, &s);
  for (int64_t i = 0; i < n; ++i) { prob[i] = p[i]; alias[i] = a[i]; }
  if (sum) *sum = s;
  return EU_OK;
}
namespace eu {

// Graph::BuildGlobalSampler, euler/core/graph/graph.cc:333-370.
int graph_build_sampler(eu_graph* g) {
  if (g->sampler_built) return EU_OK;
  DevGraph& d = g->d;
  EU_CUDA(cudaSetDevice(g->device));
  if (d.n >= (int64_t)1 << 31) { set_error("node sampler: > 2^31 nodes unsupported"); return EU_ERR_UNSUPPORTED; }
  int32_t NT = d.n_node_types;
  std::vector<unsigned long long> ids(d.n);
  std::vector<int32_t> nt(d.n);
  std::vector<float> nw(d.n);
  if (d.n > 0) {
    EU_CUDA(cudaMemcpy(ids.data(), d.ids, sizeof(unsigned long long) * d.n, cudaMemcpyDeviceToHost));
    EU_CUDA(cudaMemcpy(nt.data(), d.node_type, sizeof(int32_t) * d.n, cudaMemcpyDeviceToHost));
    EU_CUDA(cudaMemcpy(nw.data(), d.node_w, sizeof(float) * d.n, cudaMemcpyDeviceToHost));
  }
  std::vector<std::vector<unsigned long long>> t_ids(NT);
  std::vector<std::vector<float>> t_w(NT);
  g->type_sums.assign(NT, 0.f);
  for (int64_t i = 0; i < d.n; ++i) {
    int64_t r = g->sampler_order.empty() ? i : g->sampler_order[i];
    int32_t t = nt[r];
    if (t < 0 || t >= NT) { set_error("node type %d out of range", t); return EU_ERR_INVALID; }
    t_ids[t].push_back(ids[r]);
    t_w[t].push_back(nw[r]);
    g->type_sums[t] += nw[r];
  }
  g->samplers.resize(NT);
  for (int32_t t = 0; t < NT; ++t) {
    for (auto& x : t_w[t]) x /= g->type_sums[t];
    std::vector<float> prob;
    std::vector<int32_t> alias;
    TypeSampler& s = g->samplers[t];
    s.n = (int64_t)t_ids[t].size();
    s.fwc_sum = fwc_build(t_w[t], &prob, &alias);
    int rc;
    if ((rc = g->alloc(&s.ids, s.n))) return rc;
    if ((rc = g->alloc(&s.prob, s.n))) return rc;
    if ((rc = g->alloc(&s.alias, s.n))) return rc;
    if (s.n > 0) {
      EU_CUDA(cudaMemcpy(s.ids, t_ids[t].data(), sizeof(unsigned long long) * s.n, cudaMemcpyHostToDevice));
      EU_CUDA(cudaMemcpy(s.prob, prob.data(), sizeof(float) * s.n, cudaMemcpyHostToDevice));
      EU_CUDA(cudaMemcpy(s.alias, alias.data(), sizeof(int32_t) * s.n, cudaMemcpyHostToDevice));
    }
  }
  g->type_fwc_sum = fwc_build(g->type_sums, &g->type_prob, &g->type_alias);
  int rc;
  if ((rc = g->alloc(&g->d_type_prob, NT))) return rc;
  if ((rc = g->alloc(&g->d_type_alias, NT))) return rc;
  if (NT > 0) {
    EU_CUDA(cudaMemcpy(g->d_type_prob, g->type_prob.data(), sizeof(float) * NT, cudaMemcpyHostToDevice));
    EU_CUDA(cudaMemcpy(g->d_type_alias, g->type_alias.data(), sizeof(int32_t) * NT, cudaMemcpyHostToDevice));
  }
  g->sampler_built = true;
  return EU_OK;
}

static int check_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_error("no CUDA device (%s); euler_b200 has no CPU fallback",
              e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    return EU_ERR_NO_GPU;
  }
  if (device < 0 || device >= n) { set_error("device %d out of range (%d)", device, n); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(device));
  return EU_OK;
}

}  // namespace eu

using namespace eu;

extern "C" {

const char* eu_last_error(void) { return eu::g_err; }
const char* eu_version(void) { return "euler_b200 0.1 (sm_100a)"; }
uint64_t eu_launch_count(void) { return eu::g_launches.load(); }

int eu_graph_create(const eu_graph_desc* desc, int device, eu_graph** out) {
  if (!desc || !out) { set_error("null argument"); return EU_ERR_INVALID; }
  if (desc->n_nodes < 0 || desc->n_edge_types < 1 || desc->n_edge_types > EU_MAX_ETYPES ||
      !desc->ids || !desc->grp_ptr || (!desc->cum_w && !desc->w && desc->grp_ptr[desc->n_nodes * desc->n_edge_types] > 0) ||
      (desc->cum_w && desc->n_edge_types > 1 && !desc->grp_cum)) {
    set_error("eu_graph_create: invalid descriptor");
    return EU_ERR_INVALID;
  }
  // id 2^64-1 cannot be a node: the id -> row table stores id + 1 with 0 = "slot not published yet" (and the reference's own
  // id 0 is unusable the same way, DEFAULT_UINT64)
  for (int64_t r = 0; r < desc->n_nodes; ++r)
    if (desc->ids[r] == ~0ull) { set_error("eu_graph_create: node id 2^64-1 is not supported"); return EU_ERR_UNSUPPORTED; }
  int rc = check_device(device);
  if (rc) return rc;
  eu_graph* g = new eu_graph();
  g->device = device;
  DevGraph& d = g->d;
  d.n = desc->n_nodes;
  d.T = desc->n_edge_types;
  d.n_node_types = desc->n_node_types > 0 ? desc->n_node_types : 1;
  d.E = desc->grp_ptr[d.n * d.T];
  const int64_t n = d.n, T = d.T, E = d.E;
#define TRY(x) do { rc = (x); if (rc) { eu_graph_destroy(g); return rc; } } while (0)
  TRY(upload(g, (const uint64_t**)&d.ids, desc->ids, n));
  {
    std::vector<int32_t> nt(n, 0);
    std::vector<float> nw(n, 1.0f);
    TRY(upload(g, &d.node_type, desc->node_type ? desc->node_type : nt.data(), n));
    TRY(upload(g, &d.node_w, desc->node_w ? desc->node_w : nw.data(), n));
  }
  TRY(upload(g, &d.grp_ptr, desc->grp_ptr, n * T + 1));
  TRY(upload(g, (const uint64_t**)&d.nbr, desc->nbr, E));
  if (desc->cum_w) {
    TRY(upload(g, &d.cum_w, desc->cum_w, E));
    if (T > 1) TRY(upload(g, &d.grp_cum, desc->grp_cum, n * T));
  } else {
    float *w = nullptr, *cum = nullptr, *gc = nullptr;
    TRY(g->alloc(&cum, E));
    if (T > 1) TRY(g->alloc(&gc, n * T));
    if (cudaMalloc(&w, sizeof(float) * (size_t)(E > 0 ? E : 1)) != cudaSuccess) { set_error("cudaMalloc w"); eu_graph_destroy(g); return EU_ERR_CUDA; }
    if (E > 0) cudaMemcpy(w, desc->w, sizeof(float) * (size_t)E, cudaMemcpyHostToDevice);
    if (n > 0) {
      k_build_cum<<<(unsigned)ceil_div(n, 128), 128>>>(n, (int32_t)T, d.grp_ptr, w, cum, gc);
      g_launches++;
    }
    cudaError_t e = cudaDeviceSynchronize();
    cudaFree(w);
    if (e != cudaSuccess) { set_error("k_build_cum: %s", cudaGetErrorString(e)); eu_graph_destroy(g); return EU_ERR_CUDA; }
    d.cum_w = cum;
    d.grp_cum = gc;
  }
  d.feat_dim = desc->feat ? desc->feat_dim : 0;
  if (d.feat_dim > 0) TRY(upload(g, &d.feat, desc->feat, n * (int64_t)d.feat_dim));
  if (d.feat_dim > 0) {
    if (desc->n_feat_slots > 0) {
      if (desc->n_feat_slots > EU_MAX_FEAT_SLOTS || !desc->feat_slot_dims) { set_error("bad feature slots"); eu_graph_destroy(g); return EU_ERR_INVALID; }
      int32_t off = 0;
      d.n_slots = desc->n_feat_slots;
      for (int s = 0; s < d.n_slots; ++s) { d.slot_off[s] = off; d.slot_dim[s] = desc->feat_slot_dims[s]; off += desc->feat_slot_dims[s]; }
      if (off != d.feat_dim) { set_error("feat_dim != sum(feat_slot_dims)"); eu_graph_destroy(g); return EU_ERR_INVALID; }
    } else {
      d.n_slots = 1; d.slot_off[0] = 0; d.slot_dim[0] = d.feat_dim;
    }
    for (int s = 0; s < d.n_slots; ++s) g->dense_feature_names.push_back("feat" + std::to_string(s));
  }
  if (desc->n_u64_slots > 0 && desc->u64_ptr) {
    const int64_t S = desc->n_u64_slots;
    d.n_u64_slots = (int32_t)S;
    TRY(upload(g, &d.u64_ptr, desc->u64_ptr, n * S + 1));
    TRY(upload(g, (const uint64_t**)&d.u64_val, desc->u64_val, desc->u64_ptr[n * S]));
    for (int64_t k = 0; k < S; ++k) g->sparse_feature_names.push_back("u64_" + std::to_string(k));
    g->u64_max_len.assign(S, 0);
    for (int64_t r = 0; r < n; ++r)
      for (int64_t k = 0; k < S; ++k)
        g->u64_max_len[k] = std::max(g->u64_max_len[k], desc->u64_ptr[r * S + k + 1] - desc->u64_ptr[r * S + k]);
  }
  if (desc->n_bin_slots > 0 && desc->bin_ptr) {
    const int64_t S = desc->n_bin_slots;
    d.n_bin_slots = (int32_t)S;
    TRY(upload(g, &d.bin_ptr, desc->bin_ptr, n * S + 1));
    TRY(upload(g, (const uint8_t**)&d.bin_val, desc->bin_val, desc->bin_ptr[n * S]));
    for (int64_t k = 0; k < S; ++k) g->binary_feature_names.push_back("bin_" + std::to_string(k));
  }
  // dense id range?
  bool dense = n > 0;
  for (int64_t r = 0; r < n && dense; ++r) dense = desc->ids[r] == desc->ids[0] + (uint64_t)r;
  d.dense_ids = dense ? 1 : 0;
  d.id_base = n > 0 ? desc->ids[0] : 0;
  d.id_stride = 1;
  TRY(build_hash(g));
  if (desc->sampler_order) g->sampler_order.assign(desc->sampler_order, desc->sampler_order + n);
  for (int t = 0; t < T; ++t) g->edge_type_names.push_back(std::to_string(t));
  for (int t = 0; t < d.n_node_types; ++t) g->node_type_names.push_back(std::to_string(t));
#undef TRY
  *out = g;
  return EU_OK;
}

// R-MAT generation, optionally restricted to the rows one shard owns (owner(id) = id % shard_number,
// the reference's (id % partitions) % shards with partitions a multiple of shards, id_split_op.cc:46-49).
// Every shard derives edges, weights and features from the same per-edge / per-node hashes, so the union
// of the shards is exactly the unsharded graph.
static int rmat_create(int64_t n_nodes, int64_t n_edges, double a, double b, double c, uint64_t seed,
                       int32_t feat_dim, uint64_t feat_seed, int device, int shard_index, int shard_number,
                       int T, int NT, eu_graph** out) {
  if (!out || n_nodes <= 0 || n_edges < 0 || shard_number < 1 || shard_index < 0 || shard_index >= shard_number ||
      T < 1 || T > EU_MAX_ETYPES || NT < 1 || NT > EU_MAX_ETYPES || (double)n_nodes * (double)n_nodes * T >= 9.2e18) {
    set_error("eu_graph_create_rmat: bad sizes"); return EU_ERR_INVALID;
  }
  if ((double)n_nodes * (double)n_nodes >= 9.2e18) { set_error("n_nodes too large for 64-bit sort keys"); return EU_ERR_INVALID; }
  int rc = check_device(device);
  if (rc) return rc;
  const int64_t N = shard_number;
  const int64_t base_id = shard_index == 0 ? N : shard_index;           // first owned id (ids are 1..n; 0 is unusable)
  const int64_t n_local = n_nodes >= base_id ? (n_nodes - base_id) / N + 1 : 0;
  eu_graph* g = new eu_graph();
  g->device = device;
  DevGraph& d = g->d;
  d.n = n_local; d.T = T; d.n_node_types = NT;
  const int tb = 256;
#define TRY(x) do { rc = (x); if (rc) { eu_graph_destroy(g); return rc; } } while (0)
#define TRYC(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { set_error("%s -> %s", #x, cudaGetErrorString(_e)); eu_graph_destroy(g); return EU_ERR_CUDA; } } while (0)
  int scale = 1;
  while (((int64_t)1 << scale) < n_nodes) ++scale;
  // pass 1: how many edges does this shard own
  unsigned long long* d_cnt = nullptr;
  TRYC(cudaMalloc(&d_cnt, sizeof(unsigned long long)));
  TRYC(cudaMemset(d_cnt, 0, sizeof(unsigned long long)));
  int64_t E = n_edges;
  if (N > 1 && n_edges > 0) {
    k_rmat_edges<<<(unsigned)ceil_div(n_edges, tb), tb>>>(nullptr, d_cnt, n_edges, n_nodes, scale, a, b, c, seed, (int)N, shard_index, T);
    g_launches++;
    unsigned long long h = 0;
    TRYC(cudaMemcpy(&h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost));
    E = (int64_t)h;
    TRYC(cudaMemset(d_cnt, 0, sizeof(unsigned long long)));
  }
  d.E = E;
  unsigned long long *ids = nullptr, *nbr = nullptr;
  int32_t* ntype = nullptr;
  float *nw = nullptr, *cum = nullptr;
  int64_t* ptr = nullptr;
  TRY(g->alloc(&ids, n_local));
  TRY(g->alloc(&ntype, n_local));
  TRY(g->alloc(&nw, n_local));
  const int64_t n_grp = n_local * T;   // adjacency groups
  float* gcum = nullptr;
  TRY(g->alloc(&ptr, n_grp + 1));
  if (T > 1) TRY(g->alloc(&gcum, n_grp));
  TRY(g->alloc(&nbr, E));
  TRY(g->alloc(&cum, E));
  if (n_local > 0) {
    k_iota_ids<<<(unsigned)ceil_div(n_local, tb), tb>>>(ids, ntype, nw, n_local, (unsigned long long)base_id, (unsigned long long)N, NT);
    g_launches++;
  }
  unsigned long long *k0 = nullptr, *k1 = nullptr;
  float* w = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0, tmp2 = 0;
  TRYC(cudaMalloc(&k0, sizeof(unsigned long long) * (size_t)(E > 0 ? E : 1)));
  TRYC(cudaMalloc(&k1, sizeof(unsigned long long) * (size_t)(E > 0 ? E : 1)));
  if (n_edges > 0) {
    k_rmat_edges<<<(unsigned)ceil_div(n_edges, tb), tb>>>(k0, d_cnt, n_edges, n_nodes, scale, a, b, c, seed, (int)N, shard_index, T);
    g_launches++;
  }
  int end_bit = 1;
  while (end_bit < 64 && ((double)(n_grp > 0 ? n_grp : 1) * (double)n_nodes) >= ldexp(1.0, end_bit)) ++end_bit;
  cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, k0, k1, (int64_t)E, 0, end_bit);
  cub::DeviceScan::ExclusiveSum(nullptr, tmp2, ptr, ptr, (int64_t)(n_grp + 1));
  if (tmp2 > tmp_bytes) tmp_bytes = tmp2;
  TRYC(cudaMalloc(&tmp, tmp_bytes > 0 ? tmp_bytes : 1));
  TRYC(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, k0, k1, (int64_t)E, 0, end_bit));
  TRYC(cudaMemset(ptr, 0, sizeof(int64_t) * (size_t)(n_grp + 1)));
  if (E > 0) {
    k_count_src<<<(unsigned)ceil_div(E, tb), tb>>>(k1, E, n_nodes, ptr);
    g_launches++;
  }
  TRYC(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, ptr, ptr, (int64_t)(n_grp + 1)));
  TRYC(cudaFree(k0)); k0 = nullptr;
  TRYC(cudaMalloc(&w, sizeof(float) * (size_t)(E > 0 ? E : 1)));
  if (E > 0) {
    k_rmat_fill<<<(unsigned)ceil_div(E, tb), tb>>>(k1, E, n_nodes, nbr, w, (unsigned long long)base_id, (unsigned long long)N, T);
    g_launches++;
  }
  if (n_local > 0) {
    k_build_cum<<<(unsigned)ceil_div(n_local, 128), 128>>>(n_local, T, ptr, w, cum, gcum);
    g_launches++;
  }
  TRYC(cudaDeviceSynchronize());
  cudaFree(k1); cudaFree(w); cudaFree(tmp); cudaFree(d_cnt);
  d.ids = ids; d.node_type = ntype; d.node_w = nw; d.grp_ptr = ptr; d.nbr = nbr; d.cum_w = cum;
  d.grp_cum = gcum;
  d.dense_ids = 1; d.id_base = (unsigned long long)base_id; d.id_stride = (unsigned long long)N;
  d.feat_dim = feat_dim;
  if (feat_dim > 0) {
    float* feat = nullptr;
    TRY(g->alloc(&feat, n_local * (int64_t)feat_dim));
    k_fill_feat<<<148 * 8, 256>>>(feat, n_local, feat_dim, feat_seed, (unsigned long long)base_id, (unsigned long long)N);
    g_launches++;
    d.feat = feat;
    d.n_slots = 1; d.slot_off[0] = 0; d.slot_dim[0] = feat_dim;
    g->dense_feature_names.push_back("feat0");
  }
  TRY(build_hash(g));
  for (int t = 0; t < T; ++t) g->edge_type_names.push_back(std::to_string(t));
  for (int t = 0; t < NT; ++t) g->node_type_names.push_back(std::to_string(t));
#undef TRY
#undef TRYC
  *out = g;
  return EU_OK;
}

int eu_graph_create_rmat(int64_t n_nodes, int64_t n_edges, double a, double b, double c,
                         uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                         eu_graph** out) {
  return rmat_create(n_nodes, n_edges, a, b, c, seed, feat_dim, feat_seed, device, 0, 1, 1, 1, out);
}

int eu_graph_create_rmat_hetero(int64_t n_nodes, int64_t n_edges, int32_t n_edge_types, int32_t n_node_types, double a,
                                double b, double c, uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                                int shard_index, int shard_number, eu_graph** out) {
  return rmat_create(n_nodes, n_edges, a, b, c, seed, feat_dim, feat_seed, device, shard_index, shard_number, n_edge_types,
                     n_node_types, out);
}

int eu_graph_create_rmat_shard(int64_t n_nodes, int64_t n_edges, double a, double b, double c,
                               uint64_t seed, int32_t feat_dim, uint64_t feat_seed, int device,
                               int shard_index, int shard_number, eu_graph** out) {
  return rmat_create(n_nodes, n_edges, a, b, c, seed, feat_dim, feat_seed, device, shard_index, shard_number, 1, 1, out);
}

int eu_graph_destroy(eu_graph* g) {
  if (!g) return EU_OK;
  cudaSetDevice(g->device);
  for (void* p : g->allocs) cudaFree(p);
  delete g;
  return EU_OK;
}

int64_t eu_graph_num_nodes(const eu_graph* g) { return g ? g->d.n : -1; }
int64_t eu_graph_num_edges(const eu_graph* g) { return g ? g->d.E : -1; }
int32_t eu_graph_num_edge_types(const eu_graph* g) { return g ? g->d.T : -1; }
int32_t eu_graph_num_node_types(const eu_graph* g) { return g ? g->d.n_node_types : -1; }
int32_t eu_graph_feat_dim(const eu_graph* g) { return g ? g->d.feat_dim : -1; }
int64_t eu_graph_hbm_bytes(const eu_graph* g) { return g ? g->hbm_bytes : -1; }

int eu_graph_export(const eu_graph* g, uint64_t* ids, int32_t* node_type, float* node_w,
                    int64_t* grp_ptr, uint64_t* nbr, float* cum_w, float* grp_cum, float* feat) {
  if (!g) { set_error("null graph"); return EU_ERR_INVALID; }
  const DevGraph& d = g->d;
  EU_CUDA(cudaSetDevice(g->device));
  EU_CUDA(cudaDeviceSynchronize());
#define DL(dst, src, cnt) if ((dst) && (src) && (cnt) > 0) EU_CUDA(cudaMemcpy(dst, src, sizeof(*(dst)) * (size_t)(cnt), cudaMemcpyDeviceToHost))
  DL(ids, d.ids, d.n);
  DL(node_type, d.node_type, d.n);
  DL(node_w, d.node_w, d.n);
  DL(grp_ptr, d.grp_ptr, d.n * d.T + 1);
  DL(nbr, d.nbr, d.E);
  DL(cum_w, d.cum_w, d.E);
  DL(grp_cum, d.grp_cum, d.n * d.T);
  DL(feat, d.feat, d.n * (int64_t)d.feat_dim);
#undef DL
  return EU_OK;
}

int32_t eu_graph_edge_type_id(const eu_graph* g, const char* name) {
  if (!g || !name) return -1;
  for (size_t i = 0; i < g->edge_type_names.size(); ++i)
    if (g->edge_type_names[i] == name) return (int32_t)i;
  return -1;
}
int32_t eu_graph_dense_feature_id(const eu_graph* g, const char* name) {
  if (!g || !name) return -1;
  for (size_t i = 0; i < g->dense_feature_names.size(); ++i)
    if (g->dense_feature_names[i] == name) return (int32_t)i;
  return -1;
}
int32_t eu_graph_sparse_feature_id(const eu_graph* g, const char* name) {
  if (!g || !name) return -1;
  for (size_t i = 0; i < g->sparse_feature_names.size(); ++i)
    if (g->sparse_feature_names[i] == name) return (int32_t)i;
  return -1;
}
int32_t eu_graph_binary_feature_id(const eu_graph* g, const char* name) {
  if (!g || !name) return -1;
  for (size_t i = 0; i < g->binary_feature_names.size(); ++i)
    if (g->binary_feature_names[i] == name) return (int32_t)i;
  return -1;
}
int32_t eu_graph_dense_feature_dim(const eu_graph* g, int32_t fid) {
  if (!g || fid < 0 || fid >= g->d.n_slots) return -1;
  return g->d.slot_dim[fid];
}
int64_t eu_graph_sparse_feature_max_len(const eu_graph* g, int32_t fid) {
  if (!g || fid < 0 || fid >= (int32_t)g->u64_max_len.size()) return 0;
  return g->u64_max_len[fid];
}
int32_t eu_graph_node_type_id(const eu_graph* g, const char* name) {
  if (!g || !name) return -1;
  for (size_t i = 0; i < g->node_type_names.size(); ++i)
    if (g->node_type_names[i] == name) return (int32_t)i;
  return -1;
}

}  // extern "C"
