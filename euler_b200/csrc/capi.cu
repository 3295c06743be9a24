// Contexts, host-buffer entry points and the reference's InitQueryProxy entry.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <initializer_list>
#include <string>
#include <vector>

#include "internal.h"

namespace eu {

// engine e is seeded with seeds[e] (or seed0 + e when seeds == nullptr)
__global__ void k_seed(EuRngState* rs, int n, unsigned long long seed0, const unsigned long long* seeds) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const unsigned long long seed = seeds ? seeds[e] : seed0 + (unsigned long long)e;
  EuRngState* r = rs + e;
  // std::minstd_rand0::seed(s): x = s mod m, 1 if that is 0 (SURVEY.md Appendix A-13)
  unsigned long long x = seed % 2147483647ull;
  r->x = x == 0 ? 1u : (uint32_t)x;
  r->x_prev = r->x;
  r->draws = 0;
  r->calls = 0;
  r->blocks_done = 0;
  r->key = seed * 0x9E3779B97F4A7C15ull;
}

template <typename T>
static int regrow(T** p, int64_t count) {
  if (*p) cudaFree(*p);
  *p = nullptr;
  void* q = nullptr;
  size_t bytes = (size_t)(count > 0 ? count : 1) * sizeof(T);
  cudaError_t e = cudaMalloc(&q, bytes);
  if (e != cudaSuccess) { set_error("cudaMalloc(%zu) -> %s", bytes, cudaGetErrorString(e)); return EU_ERR_CUDA; }
  *p = (T*)q;
  return EU_OK;
}

// growing scratch frees and re-allocates under a stream synchronise: impossible while the stream is being captured into
// a CUDA graph -- fail loudly and say what to do instead of invalidating the capture
int refuse_growth_in_capture(eu_ctx* c, const char* what) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(c->stream, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone) {
    set_error("%s must grow while the ctx stream is being captured: run the op once (or call eu_ctx_reserve) before the capture", what);
    return EU_ERR_STATE;
  }
  cudaGetLastError();
  return EU_OK;
}

int ctx_reserve(eu_ctx* c, int64_t rows, int64_t table_slots) {
  int rc;
  if ((table_slots > c->tab_set_slots || rows > c->cap_rows) && (rc = refuse_growth_in_capture(c, "the sampling scratch"))) return rc;
  if (table_slots > c->tab_set_slots) {
    EU_CUDA(cudaStreamSynchronize(c->stream));  // growing while the stream still uses the old buffers would be a race
    const int64_t slots = table_slots + 64;
    if ((rc = regrow(&c->d_dedup, 2 * slots))) return rc;  // two table sets: hop l uses set l & 1
    c->tab_set_slots = slots;
    // all-free tables: key 0, row = kEmptyRow (see hop() invariant)
    for (int64_t off = 0; off < 2 * slots; off += (int64_t)1 << 20) {
      int64_t n = std::min<int64_t>((int64_t)1 << 20, 2 * slots - off);
      EU_CUDA(cudaMemset2DAsync(&c->d_dedup[off].key, sizeof(HashSlot), 0x00, 8, (size_t)n, c->stream));
      EU_CUDA(cudaMemset2DAsync(&c->d_dedup[off].row, sizeof(HashSlot), 0xFF, 8, (size_t)n, c->stream));
    }
  }
  if (rows <= c->cap_rows) return EU_OK;
  EU_CUDA(cudaStreamSynchronize(c->stream));
  if ((rc = regrow(&c->d_first, rows))) return rc;
  if ((rc = regrow(&c->d_rowof, rows))) return rc;
  if ((rc = regrow(&c->d_elig, rows))) return rc;
  if ((rc = regrow(&c->d_state, rows))) return rc;
  if ((rc = regrow(&c->d_emask, rows / 32 + 2))) return rc;
  if ((rc = regrow(&c->d_woff, rows / 32 + 2))) return rc;
  if ((rc = regrow(&c->d_blkpre, rows / 256 + 66))) return rc;
  if ((rc = regrow(&c->d_blkmul, rows / 256 + 66))) return rc;
  if ((rc = regrow(&c->d_live, rows))) return rc;
  if (!c->d_nlive && (rc = regrow(&c->d_nlive, 4))) return rc;
  if ((rc = regrow(&c->d_front[0], rows))) return rc;
  if ((rc = regrow(&c->d_front[1], rows))) return rc;
  c->cap_rows = rows;
  return EU_OK;
}

int ctx_misc(eu_ctx* c, int64_t bytes) {
  if (bytes <= c->misc_bytes) return EU_OK;
  if (int rc0 = refuse_growth_in_capture(c, "the op scratch")) return rc0;
  EU_CUDA(cudaStreamSynchronize(c->stream));
  char* p = (char*)c->d_misc;
  int rc = regrow(&p, bytes);
  c->d_misc = p;
  if (rc) { c->misc_bytes = 0; return rc; }
  c->misc_bytes = bytes;
  return EU_OK;
}

int ctx_levels(eu_ctx* c, int64_t ids) {
  if (ids <= c->levels_cap) return EU_OK;
  if (int rc0 = refuse_growth_in_capture(c, "the fanout level scratch")) return rc0;
  EU_CUDA(cudaStreamSynchronize(c->stream));
  int rc = regrow(&c->d_levels, ids);
  c->levels_cap = rc ? 0 : ids;
  return rc;
}

int ctx_stage(eu_ctx* c, int64_t host_bytes, int64_t dev_bytes) {
  if (host_bytes > c->pin_bytes) {
    if (c->h_pin) cudaFreeHost(c->h_pin);
    c->h_pin = nullptr; c->pin_bytes = 0;
    EU_CUDA(cudaHostAlloc(&c->h_pin, (size_t)host_bytes, cudaHostAllocDefault));
    c->pin_bytes = host_bytes;
  }
  if (dev_bytes > c->stage_bytes) {
    EU_CUDA(cudaStreamSynchronize(c->stream));
    char* p = (char*)c->d_stage;
    int rc = regrow(&p, dev_bytes);
    c->d_stage = p;
    if (rc) { c->stage_bytes = 0; return rc; }
    c->stage_bytes = dev_bytes;
  }
  return EU_OK;
}

static inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }

// Bump allocator over the ctx staging buffers: the same offsets are used on the pinned host
// side and on the device side.
struct Stage {
  int64_t off = 0;
  int64_t take(int64_t bytes) { int64_t o = off; off += align256(bytes); return o; }
};

// A caller's host buffer that is already page-locked (cudaHostAlloc / cudaHostRegister -- e.g. a framework's pinned
// tensor) is DMA'd directly; only pageable memory goes through the ctx's pinned staging buffer (a pageable
// cudaMemcpyAsync would serialise against the host, and the extra memcpy costs more than PCIe for wide feature rows).
static bool host_is_pinned(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

static std::mutex g_default_mu;
static eu_graph* g_default_graph = nullptr;
static eu_ctx* g_default_ctx = nullptr;

}  // namespace eu

using namespace eu;

extern "C" {

int eu_ctx_create(eu_graph* g, eu_rng_kind rng, uint64_t seed, void* stream, eu_ctx** out) {
  if (!g || !out || (rng != EU_RNG_MINSTD && rng != EU_RNG_PHILOX)) { set_error("eu_ctx_create: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(g->device));
  eu_ctx* c = new eu_ctx();
  c->g = g; c->rng = rng; c->seed = seed; c->stream = (cudaStream_t)stream;
  cudaError_t e = cudaMalloc(&c->d_rng, sizeof(EuRngState));
  if (e != cudaSuccess) { set_error("cudaMalloc rng -> %s", cudaGetErrorString(e)); delete c; return EU_ERR_CUDA; }
  k_seed<<<1, 64, 0, c->stream>>>(c->d_rng, 1, seed, nullptr);
  g_launches++;
  *out = c;
  return EU_OK;
}

int eu_ctx_destroy(eu_ctx* c) {
  if (!c) return EU_OK;
  cudaSetDevice(c->g->device);
  cudaStreamSynchronize(c->stream);
  cudaFree(c->d_rng); cudaFree(c->d_dedup); cudaFree(c->d_first); cudaFree(c->d_rowof);
  cudaFree(c->d_elig); cudaFree(c->d_state); cudaFree(c->d_emask); cudaFree(c->d_woff); cudaFree(c->d_blkpre); cudaFree(c->d_blkmul); cudaFree(c->d_live); cudaFree(c->d_nlive); cudaFree(c->d_front[0]); cudaFree(c->d_front[1]); cudaFree(c->d_levels);
  cudaFree(c->d_misc); cudaFree(c->d_stage); cudaFree(c->d_walkv);
  for (int i = 0; i < 2; ++i) { if (c->aux[i]) cudaStreamDestroy(c->aux[i]); if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]); }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->h_pin) cudaFreeHost(c->h_pin);
  delete c;
  return EU_OK;
}

int eu_ctx_set_stream(eu_ctx* c, void* stream) {
  if (!c) { set_error("null ctx"); return EU_ERR_INVALID; }
  c->stream = (cudaStream_t)stream;
  return EU_OK;
}

int eu_ctx_seed(eu_ctx* c, uint64_t seed) {
  if (!c) { set_error("null ctx"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  c->seed = seed;
  k_seed<<<1, 64, 0, c->stream>>>(c->d_rng, c->n_eng, seed, nullptr);
  EU_LAUNCHED();
  return EU_OK;
}

// n engines, engine e seeded with seeds[e] (seeds == NULL: seed + e).  Batch b of a *_batched call uses engine b.
int eu_ctx_set_engines(eu_ctx* c, int32_t n, const uint64_t* seeds) {
  if (!c || n < 1 || n > 64) { set_error("eu_ctx_set_engines: 1..64 engines"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  EuRngState* r = nullptr;
  EU_CUDA(cudaMalloc(&r, sizeof(EuRngState) * n));
  unsigned long long* d_seeds = nullptr;
  if (seeds) {
    EU_CUDA(cudaMalloc(&d_seeds, sizeof(unsigned long long) * n));
    EU_CUDA(cudaMemcpy(d_seeds, seeds, sizeof(unsigned long long) * n, cudaMemcpyHostToDevice));
    c->seed = seeds[0];
  }
  cudaFree(c->d_rng);
  c->d_rng = r;
  c->n_eng = n;
  k_seed<<<1, 64, 0, c->stream>>>(c->d_rng, n, c->seed, d_seeds);
  EU_LAUNCHED();
  EU_CUDA(cudaStreamSynchronize(c->stream));
  if (d_seeds) cudaFree(d_seeds);
  return EU_OK;
}

int eu_ctx_reserve(eu_ctx* c, int64_t max_rows) {
  if (!c || max_rows < 0) { set_error("eu_ctx_reserve: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  const int nb = c->n_eng;
  int rc = ctx_reserve(c, max_rows + 256 * nb, 4 * max_rows + 65 * nb);
  if (rc) return rc;
  // eu_sample_fanout_with_feature keeps every level's engine ids: at most 2 * max_rows when every count is >= 2
  if ((rc = ctx_levels(c, 2 * max_rows))) return rc;
  return ctx_misc(c, 256 + 4 * max_rows);
}

int eu_ctx_sync(eu_ctx* c) {
  if (!c) { set_error("null ctx"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  return EU_OK;
}

int eu_ctx_draws(eu_ctx* c, uint64_t* draws) {
  if (!c || !draws) { set_error("eu_ctx_draws: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  EuRngState h;
  EU_CUDA(cudaMemcpyAsync(&h, c->d_rng, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  *draws = h.draws;
  return EU_OK;
}

int eu_ctx_profile(eu_ctx* c, int enable) {
  if (!c) { set_error("null ctx"); return EU_ERR_INVALID; }
  c->prof = enable != 0;
  return EU_OK;
}

// Synchronises, then writes "name,rows,launches,total_ms\n" lines (aggregated) into buf and clears the log.
int eu_ctx_profile_read(eu_ctx* c, char* buf, int64_t cap) {
  if (!c || !buf || cap <= 0) { set_error("eu_ctx_profile_read: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  std::map<std::pair<std::string, int64_t>, std::pair<int64_t, double>> agg;
  for (auto& r : c->prof_recs) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    auto& a = agg[std::make_pair(std::string(r.name), r.rows)];
    a.first += 1; a.second += ms;
    cudaEventDestroy(r.e0); cudaEventDestroy(r.e1);
  }
  c->prof_recs.clear();
  std::string out;
  char line[256];
  for (auto& kv : agg) {
    snprintf(line, sizeof(line), "%s,%lld,%lld,%.6f\n", kv.first.first.c_str(), (long long)kv.first.second,
             (long long)kv.second.first, kv.second.second);
    out += line;
  }
  if ((int64_t)out.size() + 1 > cap) { set_error("profile buffer too small"); return EU_ERR_INVALID; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return EU_OK;
}

// ------------------------------------------------------------------------------ host variants
// Pattern: copy inputs into pinned memory, H2D on the ctx stream, run the device op, D2H into
// pinned memory, synchronise, copy out.  The pinned hop keeps the copies asynchronous-capable
// (pageable cudaMemcpyAsync would serialise against the host).

// Host-buffer staging of one call: inputs go H2D, outputs come D2H, all on the ctx stream.  Pinned caller buffers are
// DMA'd in place; pageable ones pass through the ctx's pinned stage (copied out after the final synchronise).
struct HostIO {
  eu_ctx* c;
  Stage st;
  struct Out { void* user; int64_t off; int64_t bytes; };
  std::vector<Out> outs;
  int64_t take(int64_t bytes) { return st.take(bytes); }
  // size the stage: the device side always, the pinned host side only if some caller buffer is pageable
  int begin(std::initializer_list<const void*> user_bufs) {
    bool all = true;
    for (const void* p : user_bufs) all = all && (!p || host_is_pinned(p));
    return ctx_stage(c, all ? 0 : st.off, st.off);
  }
  // device address of stage offset `off`
  char* dev(int64_t off) const { return (char*)c->d_stage + off; }
  int in(int64_t off, const void* user, int64_t bytes) {
    if (bytes <= 0) return EU_OK;
    const void* src = user;
    if (!host_is_pinned(user)) { memcpy((char*)c->h_pin + off, user, (size_t)bytes); src = (char*)c->h_pin + off; }
    EU_CUDA(cudaMemcpyAsync(dev(off), src, (size_t)bytes, cudaMemcpyHostToDevice, c->stream));
    return EU_OK;
  }
  int out(int64_t off, void* user, int64_t bytes) {
    if (bytes <= 0 || !user) return EU_OK;
    if (host_is_pinned(user)) {
      EU_CUDA(cudaMemcpyAsync(user, dev(off), (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    } else {
      EU_CUDA(cudaMemcpyAsync((char*)c->h_pin + off, dev(off), (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
      outs.push_back({user, off, bytes});
    }
    return EU_OK;
  }
  int finish() {
    EU_CUDA(cudaStreamSynchronize(c->stream));
    for (auto& o : outs) memcpy(o.user, (char*)c->h_pin + o.off, (size_t)o.bytes);
    return EU_OK;
  }
};

int eu_sample_fanout_batched_host(eu_ctx* c, const int64_t* nodes, int32_t nb, int64_t B, const int32_t* etypes,
                                  int32_t K, const int32_t* counts, int32_t L, int64_t default_node,
                                  int64_t* const* out_ids, float* const* out_w, int32_t* const* out_t) {
  if (!c || nb < 1 || B < 0 || L < 0 || L > 16 || !counts || (B > 0 && !nodes)) { set_error("eu_sample_fanout_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  HostIO io{c};
  const int64_t o_nodes = io.take(8 * B * nb);
  int64_t o_ids[16], o_w[16], o_t[16], n_l[16];
  int64_t rows = B * nb;
  for (int l = 0; l < L; ++l) {
    if (counts[l] < 0) { set_error("negative count"); return EU_ERR_INVALID; }
    rows *= counts[l];
    n_l[l] = rows;
    o_ids[l] = io.take(8 * rows); o_w[l] = io.take(4 * rows); o_t[l] = io.take(4 * rows);
  }
  int rc;
  {
    bool all = host_is_pinned(nodes);
    for (int l = 0; l < L && all; ++l)
      all = (!out_ids || !out_ids[l] || host_is_pinned(out_ids[l])) && (!out_w || !out_w[l] || host_is_pinned(out_w[l])) &&
            (!out_t || !out_t[l] || host_is_pinned(out_t[l]));
    rc = ctx_stage(c, all ? 0 : io.st.off, io.st.off);
  }
  if (rc) return rc;
  if ((rc = io.in(o_nodes, nodes, 8 * B * nb))) return rc;
  int64_t* d_ids[16]; float* d_w[16]; int32_t* d_t[16];
  for (int l = 0; l < L; ++l) { d_ids[l] = (int64_t*)io.dev(o_ids[l]); d_w[l] = (float*)io.dev(o_w[l]); d_t[l] = (int32_t*)io.dev(o_t[l]); }
  rc = eu_sample_fanout_batched(c, (const int64_t*)io.dev(o_nodes), nb, B, etypes, K, counts, L, default_node, d_ids, d_w, d_t);
  if (rc) return rc;
  for (int l = 0; l < L; ++l) {
    if (out_ids && (rc = io.out(o_ids[l], out_ids[l], 8 * n_l[l]))) return rc;
    if (out_w && (rc = io.out(o_w[l], out_w[l], 4 * n_l[l]))) return rc;
    if (out_t && (rc = io.out(o_t[l], out_t[l], 4 * n_l[l]))) return rc;
  }
  return io.finish();
}

int eu_sample_fanout_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                          int32_t K, const int32_t* counts, int32_t L, int64_t default_node,
                          int64_t* const* out_ids, float* const* out_w, int32_t* const* out_t) {
  return eu_sample_fanout_batched_host(c, nodes, 1, B, etypes, K, counts, L, default_node, out_ids, out_w, out_t);
}

// Host buffers for eu_sample_fanout_with_feature, sized as for the device entry point (out_sp_val[i*NS+j] holds
// rows_i * max(1, eu_graph_sparse_feature_max_len(fid_j)) values).  Only the value prefix each out_sp_ptr covers is copied back.
int eu_sample_fanout_with_feature_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                       const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                                       float* const* out_w, int32_t* const* out_t, int32_t ND, const int32_t* dense_fids,
                                       const int32_t* dense_dims, float* const* out_dense, int32_t NS, const int32_t* sparse_fids,
                                       const int64_t* sparse_defaults, int64_t* const* out_sp_ptr, int64_t* const* out_sp_val) {
  if (!c || B < 0 || L < 0 || L > 16 || ND < 0 || NS < 0 || (L > 0 && !counts) || (B > 0 && !nodes) ||
      (int64_t)(L + 1) * ND > kMaxFeatSegs || (int64_t)(L + 1) * NS > kMaxFeatSegs || (ND > 0 && (!dense_dims || !out_dense)) ||
      (NS > 0 && (!sparse_fids || !out_sp_ptr || !out_sp_val))) {
    set_error("eu_sample_fanout_with_feature_host: bad argument");
    return EU_ERR_INVALID;
  }
  EU_CUDA(cudaSetDevice(c->g->device));
  HostIO io{c};
  int64_t rows[17];
  rows[0] = B;
  for (int l = 0; l < L; ++l) {
    if (counts[l] < 0) { set_error("negative count"); return EU_ERR_INVALID; }
    rows[l + 1] = rows[l] * counts[l];
  }
  const int64_t o_nodes = io.take(8 * B);
  int64_t o_ids[16], o_w[16], o_t[16];
  for (int l = 0; l < L; ++l) { o_ids[l] = io.take(8 * rows[l + 1]); o_w[l] = io.take(4 * rows[l + 1]); o_t[l] = io.take(4 * rows[l + 1]); }
  std::vector<int64_t> o_dense((L + 1) * ND), o_ptr((L + 1) * NS), o_val((L + 1) * NS), ptr_last((L + 1) * NS);
  std::vector<float*> d_dense((L + 1) * ND);
  std::vector<int64_t*> d_ptr((L + 1) * NS), d_val((L + 1) * NS);
  for (int i = 0; i <= L; ++i) {
    for (int j = 0; j < ND; ++j) o_dense[i * ND + j] = io.take(4 * rows[i] * (dense_dims[j] > 0 ? dense_dims[j] : 0));
    for (int j = 0; j < NS; ++j) {
      o_ptr[i * NS + j] = io.take(8 * (rows[i] + 1));
      o_val[i * NS + j] = io.take(8 * rows[i] * std::max<int64_t>(1, eu_graph_sparse_feature_max_len(c->g, sparse_fids[j])));
    }
  }
  int rc = ctx_stage(c, io.st.off, io.st.off);   // always through the pinned stage: the value prefix is known only at the end
  if (rc) return rc;
  if ((rc = io.in(o_nodes, nodes, 8 * B))) return rc;
  int64_t* d_ids[16]; float* d_w[16]; int32_t* d_t[16];
  for (int l = 0; l < L; ++l) { d_ids[l] = (int64_t*)io.dev(o_ids[l]); d_w[l] = (float*)io.dev(o_w[l]); d_t[l] = (int32_t*)io.dev(o_t[l]); }
  for (size_t k = 0; k < d_dense.size(); ++k) d_dense[k] = (float*)io.dev(o_dense[k]);
  for (size_t k = 0; k < d_ptr.size(); ++k) { d_ptr[k] = (int64_t*)io.dev(o_ptr[k]); d_val[k] = (int64_t*)io.dev(o_val[k]); }
  rc = eu_sample_fanout_with_feature(c, (const int64_t*)io.dev(o_nodes), B, etypes, K, counts, L, default_node, d_ids, d_w, d_t, ND,
                                     dense_fids, dense_dims, d_dense.data(), NS, sparse_fids, sparse_defaults, d_ptr.data(), d_val.data());
  if (rc) return rc;
  for (int l = 0; l < L; ++l) {
    if (out_ids && (rc = io.out(o_ids[l], out_ids[l], 8 * rows[l + 1]))) return rc;
    if (out_w && (rc = io.out(o_w[l], out_w[l], 4 * rows[l + 1]))) return rc;
    if (out_t && (rc = io.out(o_t[l], out_t[l], 4 * rows[l + 1]))) return rc;
  }
  for (int i = 0; i <= L; ++i)
    for (int j = 0; j < ND; ++j)
      if ((rc = io.out(o_dense[i * ND + j], out_dense[i * ND + j], 4 * rows[i] * (dense_dims[j] > 0 ? dense_dims[j] : 0)))) return rc;
  // the pointer arrays first: they say how many values to bring back
  for (size_t k = 0; k < o_ptr.size(); ++k) EU_CUDA(cudaMemcpyAsync((char*)c->h_pin + o_ptr[k], io.dev(o_ptr[k]), 8 * (size_t)(rows[k / NS] + 1), cudaMemcpyDeviceToHost, c->stream));
  if ((rc = io.finish())) return rc;
  for (size_t k = 0; k < o_ptr.size(); ++k) {
    const int64_t n = rows[k / NS];
    const int64_t* hp = (const int64_t*)((char*)c->h_pin + o_ptr[k]);
    memcpy(out_sp_ptr[k], hp, 8 * (size_t)(n + 1));
    ptr_last[k] = hp[n];
    EU_CUDA(cudaMemcpyAsync((char*)c->h_pin + o_val[k], io.dev(o_val[k]), 8 * (size_t)ptr_last[k], cudaMemcpyDeviceToHost, c->stream));
  }
  EU_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t k = 0; k < o_val.size(); ++k) memcpy(out_sp_val[k], (char*)c->h_pin + o_val[k], 8 * (size_t)ptr_last[k]);
  return EU_OK;
}

int eu_sample_neighbor_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                            int32_t K, int32_t count, int64_t default_node, int64_t* out_ids,
                            float* out_w, int32_t* out_t) {
  return eu_sample_fanout_host(c, nodes, B, etypes, K, &count, 1, default_node, &out_ids, &out_w, &out_t);
}

int eu_sample_neighbor_raw_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K, int32_t count,
                                int64_t* out_ids, float* out_w, int32_t* out_t) {
  if (!c || B < 0 || count < 0 || (B > 0 && (!nodes || (count > 0 && (!out_ids || !out_w || !out_t))))) { set_error("eu_sample_neighbor_raw_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  HostIO io{c};
  const int64_t n = B * count;
  const int64_t o_nodes = io.take(8 * B), o_ids = io.take(8 * n), o_w = io.take(4 * n), o_t = io.take(4 * n);
  int rc = io.begin({nodes, out_ids, out_w, out_t});
  if (rc) return rc;
  if ((rc = io.in(o_nodes, nodes, 8 * B))) return rc;
  rc = eu_sample_neighbor_raw(c, (const int64_t*)io.dev(o_nodes), B, etypes, K, count, (int64_t*)io.dev(o_ids), (float*)io.dev(o_w), (int32_t*)io.dev(o_t));
  if (rc) return rc;
  if ((rc = io.out(o_ids, out_ids, 8 * n)) || (rc = io.out(o_w, out_w, 4 * n)) || (rc = io.out(o_t, out_t, 4 * n))) return rc;
  return io.finish();
}

int eu_sample_node_host(eu_ctx* c, int32_t count, const int32_t* types, int32_t n_types, int64_t* out) {
  if (!c || count < 0 || (count > 0 && !out)) { set_error("eu_sample_node_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  int rc = ctx_stage(c, 8 * (int64_t)count + 256, 8 * (int64_t)count + 256);
  if (rc) return rc;
  rc = eu_sample_node(c, count, types, n_types, (int64_t*)c->d_stage);
  if (rc) return rc;
  EU_CUDA(cudaMemcpyAsync(c->h_pin, c->d_stage, 8 * (size_t)count, cudaMemcpyDeviceToHost, c->stream));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  memcpy(out, c->h_pin, 8 * (size_t)count);
  return EU_OK;
}

int eu_random_walk_host(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes,
                        int32_t K, int32_t L, float p, float q, int64_t default_node, int64_t* out) {
  if (!c || B < 0 || L < 0 || (B > 0 && (!nodes || !out))) { set_error("eu_random_walk_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  Stage st;
  const int64_t o_nodes = st.take(8 * B), o_out = st.take(8 * B * (L + 1));
  int rc = ctx_stage(c, st.off, st.off);
  if (rc) return rc;
  char* hp = (char*)c->h_pin; char* dp = (char*)c->d_stage;
  memcpy(hp + o_nodes, nodes, 8 * (size_t)B);
  EU_CUDA(cudaMemcpyAsync(dp + o_nodes, hp + o_nodes, 8 * (size_t)B, cudaMemcpyHostToDevice, c->stream));
  rc = eu_random_walk(c, (const int64_t*)(dp + o_nodes), B, etypes, K, L, p, q, default_node, (int64_t*)(dp + o_out));
  if (rc) return rc;
  EU_CUDA(cudaMemcpyAsync(hp + o_out, dp + o_out, 8 * (size_t)(B * (L + 1)), cudaMemcpyDeviceToHost, c->stream));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  memcpy(out, hp + o_out, 8 * (size_t)(B * (L + 1)));
  return EU_OK;
}

int eu_get_dense_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int32_t dim, float* out) {
  if (!c || M < 0 || dim < 0 || (M > 0 && (!nodes || !out))) { set_error("eu_get_dense_feature_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  HostIO io{c};
  const int64_t o_nodes = io.take(8 * M), o_out = io.take(4 * M * dim);
  int rc = io.begin({nodes, out});
  if (rc) return rc;
  if ((rc = io.in(o_nodes, nodes, 8 * M))) return rc;
  rc = eu_get_dense_feature(c, (const int64_t*)io.dev(o_nodes), M, fid, dim, (float*)io.dev(o_out));
  if (rc) return rc;
  if ((rc = io.out(o_out, out, 4 * M * dim))) return rc;
  return io.finish();
}

// eu_sage_mean_aggregate with host buffers: only the neighbor ids go up and only the [rows, dim] means come down -- the
// rows*count feature rows the unfused composition (get_dense_feature_host + scatter_mean) would move never leave HBM.
int eu_sage_mean_aggregate_host(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, float* out) {
  if (!c || rows < 0 || count < 0 || dim <= 0 || (rows > 0 && (!nbr_ids || !out))) { set_error("eu_sage_mean_aggregate_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  HostIO io{c};
  const int64_t o_ids = io.take(8 * rows * count), o_out = io.take(4 * rows * dim);
  int rc = io.begin({nbr_ids, out});
  if (rc) return rc;
  if ((rc = io.in(o_ids, nbr_ids, 8 * rows * count))) return rc;
  rc = eu_sage_mean_aggregate(c, (const int64_t*)io.dev(o_ids), rows, count, dim, (float*)io.dev(o_out));
  if (rc) return rc;
  if ((rc = io.out(o_out, out, 4 * rows * dim))) return rc;
  return io.finish();
}

int eu_gather_host(eu_ctx* c, const float* params, int64_t N, int64_t D, const int32_t* idx, int64_t E, float* out) {
  if (!c || N < 0 || D <= 0 || E < 0) { set_error("eu_gather_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  Stage st;
  const int64_t o_p = st.take(4 * N * D), o_i = st.take(4 * E), o_o = st.take(4 * E * D);
  int rc = ctx_stage(c, st.off, st.off);
  if (rc) return rc;
  char* hp = (char*)c->h_pin; char* dp = (char*)c->d_stage;
  memcpy(hp + o_p, params, 4 * (size_t)(N * D));
  memcpy(hp + o_i, idx, 4 * (size_t)E);
  EU_CUDA(cudaMemcpyAsync(dp + o_p, hp + o_p, (size_t)(o_o - o_p), cudaMemcpyHostToDevice, c->stream));
  rc = eu_gather(c, (const float*)(dp + o_p), N, D, (const int32_t*)(dp + o_i), E, (float*)(dp + o_o));
  if (rc) return rc;
  EU_CUDA(cudaMemcpyAsync(hp + o_o, dp + o_o, 4 * (size_t)(E * D), cudaMemcpyDeviceToHost, c->stream));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  memcpy(out, hp + o_o, 4 * (size_t)(E * D));
  return EU_OK;
}

static int scatter_host(int op, eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) {
  if (!c || D <= 0 || E < 0 || size < 0) { set_error("scatter_host: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  Stage st;
  const int64_t o_u = st.take(4 * E * D), o_i = st.take(4 * E), o_o = st.take(4 * size * D);
  int rc = ctx_stage(c, st.off, st.off);
  if (rc) return rc;
  char* hp = (char*)c->h_pin; char* dp = (char*)c->d_stage;
  memcpy(hp + o_u, u, 4 * (size_t)(E * D));
  memcpy(hp + o_i, idx, 4 * (size_t)E);
  EU_CUDA(cudaMemcpyAsync(dp + o_u, hp + o_u, (size_t)(o_o - o_u), cudaMemcpyHostToDevice, c->stream));
  const float* du = (const float*)(dp + o_u); const int32_t* di = (const int32_t*)(dp + o_i); float* dout = (float*)(dp + o_o);
  rc = op == 0 ? eu_scatter_add(c, du, D, di, E, size, dout) : eu_scatter_max(c, du, D, di, E, size, dout);
  if (rc) return rc;
  EU_CUDA(cudaMemcpyAsync(hp + o_o, dp + o_o, 4 * (size_t)(size * D), cudaMemcpyDeviceToHost, c->stream));
  EU_CUDA(cudaStreamSynchronize(c->stream));
  memcpy(out, hp + o_o, 4 * (size_t)(size * D));
  return EU_OK;
}
int eu_scatter_add_host(eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) { return scatter_host(0, c, u, D, idx, E, size, out); }
int eu_scatter_max_host(eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) { return scatter_host(1, c, u, D, idx, E, size, out); }

// ------------------------------------------------------------------------------ InitQueryProxy
eu_graph* eu_default_graph(void) { std::lock_guard<std::mutex> l(g_default_mu); return g_default_graph; }
eu_ctx* eu_default_ctx(void) { std::lock_guard<std::mutex> l(g_default_mu); return g_default_ctx; }

int eu_set_default_graph(eu_graph* g, eu_rng_kind rng, uint64_t seed) {
  std::lock_guard<std::mutex> l(g_default_mu);
  if (g_default_ctx) { eu_ctx_destroy(g_default_ctx); g_default_ctx = nullptr; }
  g_default_graph = g;
  if (!g) return EU_OK;
  return eu_ctx_create(g, rng, seed, nullptr, &g_default_ctx);
}

// tf_euler/utils/init_query_proxy.cc:19-36: split on ';' then '=', false only when the list is
// empty or an item is not exactly k=v; the graph-load status is NOT propagated (:34).
bool InitQueryProxy(const char* conf) {
  if (!conf) return false;
  std::map<std::string, std::string> kv;
  std::string s(conf);
  size_t pos = 0;
  int items = 0;
  while (pos <= s.size()) {
    size_t end = s.find(';', pos);
    if (end == std::string::npos) end = s.size();
    std::string item = s.substr(pos, end - pos);
    pos = end + 1;
    if (item.empty()) continue;
    size_t eq = item.find('=');
    if (eq == std::string::npos || item.find('=', eq + 1) != std::string::npos) return false;
    kv[item.substr(0, eq)] = item.substr(eq + 1);
    ++items;
  }
  if (items == 0) return false;
  std::string mode = kv.count("mode") ? kv["mode"] : "local";
  if (mode != "local") {
    fprintf(stderr, "[euler_b200] ERROR InitQueryProxy: mode=%s is not on this path (only mode=local; sharding is eu_* over NCCL)\n", mode.c_str());
    return true;
  }
  int device = kv.count("device") ? atoi(kv["device"].c_str()) : 0;
  uint64_t seed = kv.count("seed") ? strtoull(kv["seed"].c_str(), nullptr, 10) : 1;
  eu_rng_kind rng = (kv.count("rng") && kv["rng"] == "philox") ? EU_RNG_PHILOX : EU_RNG_MINSTD;
  eu_graph* g = nullptr;
  int rc = eu_graph_load(kv["data_path"].c_str(), 0, 1, device, &g);
  if (rc != EU_OK) {
    fprintf(stderr, "[euler_b200] ERROR InitQueryProxy: graph load failed: %s\n", eu_last_error());
    return true;
  }
  rc = eu_set_default_graph(g, rng, seed);
  if (rc != EU_OK) fprintf(stderr, "[euler_b200] ERROR InitQueryProxy: %s\n", eu_last_error());
  return true;
}

}  // extern "C"
