// Host-side internals shared by the translation units of libeuler_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/euler_b200.h"
#include "common.cuh"

namespace eu {

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define EU_CUDA(call)                                                                    \
  do {                                                                                   \
    cudaError_t _e = (call);                                                             \
    if (_e != cudaSuccess) {                                                             \
      ::eu::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
      return EU_ERR_CUDA;                                                                \
    }                                                                                    \
  } while (0)

#define EU_LAUNCHED()                                                              \
  do {                                                                             \
    ::eu::g_launches.fetch_add(1, std::memory_order_relaxed);                      \
    cudaError_t _e = cudaPeekAtLastError();                                        \
    if (_e != cudaSuccess) {                                                       \
      ::eu::set_error("%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return EU_ERR_CUDA;                                                          \
    }                                                                              \
  } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

struct TypeSampler {      // FastWeightedCollection of one node type (fast_weighted_collection.h:27-100)
  int64_t n = 0;
  unsigned long long* ids = nullptr;  // device, sampler order
  float* prob = nullptr;              // device
  int32_t* alias = nullptr;           // device
  float fwc_sum = 0.f;                // FWC::sum_weight_
};

}  // namespace eu

struct eu_graph {
  int device = 0;
  eu::DevGraph d{};
  std::vector<void*> allocs;
  int64_t hbm_bytes = 0;
  // global node sampler (Graph::BuildGlobalSampler, graph.cc:333-370); built lazily
  bool sampler_built = false;
  std::vector<eu::TypeSampler> samplers;
  std::vector<float> type_sums;        // node_weight_sums_
  std::vector<float> type_prob;        // node_type_collection_ alias tables (host; tiny)
  std::vector<int32_t> type_alias;
  float type_fwc_sum = 0.f;
  float* d_type_prob = nullptr;
  int32_t* d_type_alias = nullptr;
  std::vector<int64_t> sampler_order;  // optional explicit order (rows)
  std::vector<std::string> edge_type_names, node_type_names;
  std::vector<std::string> dense_feature_names;  // per slot, without the "dense_" prefix
  std::vector<std::string> sparse_feature_names, binary_feature_names;   // per slot, without the "sparse_" / "binary_" prefix
  std::vector<int64_t> u64_max_len;    // per uint64 slot: the most values any node holds in it
  // edges (eu_graph_set_edges): device store, per-type alias samplers in edge_map_ order, feature names
  eu::DevEdges e{};
  bool edges_set = false;
  struct EdgeSampler { int64_t n = 0; const int64_t* order = nullptr; const float* prob = nullptr; const int32_t* alias = nullptr; float fwc_sum = 0.f; };
  std::vector<EdgeSampler> edge_samplers;
  std::vector<std::string> edge_dense_names, edge_sparse_names, edge_binary_names;

  template <typename T>
  int alloc(T** p, int64_t count) {
    size_t bytes = (size_t)(count > 0 ? count : 1) * sizeof(T);
    bytes = (bytes + 255) & ~(size_t)255;
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) {
      eu::set_error("cudaMalloc(%zu) -> %s", bytes, cudaGetErrorString(e));
      return EU_ERR_CUDA;
    }
    allocs.push_back(q);
    hbm_bytes += (int64_t)bytes;
    *p = (T*)q;
    return EU_OK;
  }
};

// Device-resident engine state of one ctx.
struct EuRngState {
  uint32_t x;                 // minstd engine state
  uint32_t x_prev;             // engine state before the hop in flight (rows derive theirs from it)
  unsigned long long draws;   // uniforms produced since seed
  unsigned long long calls;   // philox: hop counter (salt)
  unsigned int blocks_done;   // last-block-done ticket
  unsigned int pad2;
  unsigned long long key;     // philox: per-engine key
};

struct eu_ctx {
  eu_graph* g = nullptr;
  eu_rng_kind rng = EU_RNG_MINSTD;
  uint64_t seed = 0;
  cudaStream_t stream = nullptr;
  EuRngState* d_rng = nullptr;       // [n_eng] engines; batch b of a batched call uses engine b, plain ops engine 0
  int n_eng = 1;
  // scratch (device), sized for `cap_rows` (padded) rows of the widest hop
  int64_t cap_rows = 0;
  eu::HashSlot* d_dedup = nullptr;   // two table sets of tab_set_slots slots each
  int64_t tab_set_slots = 0;
  int32_t* d_first = nullptr;        // [rows] first occurrence index of each seed
  int64_t* d_rowof = nullptr;        // [rows] graph row (valid where first==i), -1 if absent
  uint8_t* d_elig = nullptr;         // [rows]
  uint32_t* d_state = nullptr;       // [rows] engine state before the row's first draw (walks)
  uint32_t* d_emask = nullptr;       // [rows/32] eligible-first-occurrence ballots
  uint32_t* d_woff = nullptr;        // [rows/32] F^(count in earlier warps of the block)
  uint32_t* d_blkpre = nullptr;      // [rows/256] count in earlier blocks
  uint32_t* d_blkmul = nullptr;      // [rows/256] F^that count
  int32_t* d_live = nullptr;         // [rows] rows that sample, compacted by k_prepare
  unsigned int* d_nlive = nullptr;   // their number
  unsigned long long* d_front[2] = {nullptr, nullptr};  // engine-id frontier ping-pong [rows]
  unsigned long long* d_levels = nullptr;  // engine ids of every hop of one fanout, back to back (eu_sample_fanout_with_feature)
  int64_t levels_cap = 0;
  // extra scratch for walks / scatter
  void* d_misc = nullptr;
  int64_t misc_bytes = 0;
  float* d_walkv = nullptr;          // node2vec: biased weights of the big rows of one step (walk.cu)
  long long walkv_cap = 0;
  // node2vec: the three prefix kernels of a step (huge / big / small rows) are independent -> forked onto two auxiliary
  // streams and joined back (event fork/join: capturable in a CUDA graph)
  cudaStream_t aux[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
  // pinned staging for *_host calls
  void* h_pin = nullptr;
  int64_t pin_bytes = 0;
  void* d_stage = nullptr;
  int64_t stage_bytes = 0;
  // optional per-kernel timing (eu_ctx_profile): CUDA events on the ctx stream around each kernel
  bool prof = false;
  struct ProfRec { const char* name; int64_t rows; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof_recs;
};

// RAII-free helper: EU_PROF(c, "name", rows) { launch; }  records events around the launch when profiling
struct EuProfScope {
  eu_ctx* c; size_t idx;
  EuProfScope(eu_ctx* c_, const char* name, int64_t rows) : c(c_), idx((size_t)-1) {
    if (!c->prof) return;
    eu_ctx::ProfRec r{name, rows, nullptr, nullptr};
    cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
    cudaEventRecord(r.e0, c->stream);
    c->prof_recs.push_back(r);
    idx = c->prof_recs.size() - 1;
  }
  ~EuProfScope() { if (idx != (size_t)-1) cudaEventRecord(c->prof_recs[idx].e1, c->stream); }
};

namespace eu {
int ctx_reserve(eu_ctx* c, int64_t rows, int64_t table_slots);
int64_t hop_scratch_rows(int nb, int64_t rows_b);
int64_t hop_table_slots(int nb, int64_t rows_b);
int64_t hop_table_cap(int64_t rows_b);   // dedup slots per batch (region stride = cap + 1)
int ctx_misc(eu_ctx* c, int64_t bytes);
int ctx_levels(eu_ctx* c, int64_t ids);   // d_levels holds at least `ids` engine ids
int refuse_growth_in_capture(eu_ctx* c, const char* what);   // EU_ERR_STATE if the ctx stream is being captured
int ctx_stage(eu_ctx* c, int64_t host_bytes, int64_t dev_bytes);
int graph_build_sampler(eu_graph* g);
int launch_state_scan(eu_ctx* c, int64_t rows, unsigned long long uniforms_per_row);
// one sampleNB hop (sample.cu): seeds u64[rows] -> engine ids u64[rows*count] (0 placeholders, may be
// null) and TF-packed outputs (may be null)
int hop(eu_ctx* c, const unsigned long long* seeds, int64_t rows, const int32_t* etypes, int32_t K,
        int32_t count, int64_t default_node, unsigned long long* eng_ids, int64_t* out_ids,
        float* out_w, int32_t* out_t, int hop_index, bool pre_inserted, bool insert_next, int nb,
        const int32_t* rows_act = nullptr, bool raw = false);

// Multi-segment feature fetches: one launch set serves several (ids, output) pairs, e.g. every (level, feature) of a fanout.
// Segment s covers rows [start_s, start_s + rows_s) of the launch; seg_of finds the segment of a row.
constexpr int kMaxFeatSegs = 64;
template <class Seg, int N>
struct SegTable {
  int32_t n;      // segments in use (<= N)
  int64_t rows;   // total rows
  Seg s[N];
};
template <class Seg, int N>
__device__ __forceinline__ int seg_of(const SegTable<Seg, N>& t, int64_t i) {
  if (N == 1) return 0;
  int lo = 0, hi = t.n - 1;   // last segment with start <= i (an empty segment shares its start with the next one)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (t.s[mid].start <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}
struct DenseSeg { const unsigned long long* ids; int64_t rows; int32_t fid; int32_t dim; float* out; };
// one k_feature launch for all segments (mp_ops.cu)
int dense_feature_segments(eu_ctx* c, const DenseSeg* segs, int n);
struct SparseSeg { const unsigned long long* ids; int64_t rows; int32_t fid; int64_t default_value; int64_t cap; int64_t* out_ptr;
                   int64_t* out_values; };
// three launches (lengths, one scan, fill) for all segments, no host sync (features.cu)
int sparse_feature_segments(eu_ctx* c, const SparseSeg* segs, int n);
}  // namespace eu
