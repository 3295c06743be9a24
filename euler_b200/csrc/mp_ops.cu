// Dense feature fetch and message-passing gather / scatter aggregation (f32 data, i32 indices).
//
// Reference semantics (file:line relative to /root/reference):
//   GetDenseFeature   tf_euler/kernels/get_dense_feature_op.cc:63-121 over euler/core/api/api.cc:63-78
//   MPGather          tf_euler/kernels/gather_op.cc:42-51
//   MPScatterAdd      tf_euler/kernels/scatter_op.cc:44-55   (zero init, serial adds in index order)
//   MPScatterMax      tf_euler/kernels/scatter_op.cc:77-91   (init -1e9, strict >)
//   scatter_mean      tf_euler/python/euler_ops/mp_ops.py:65-69
//
// All are HBM-bound row moves: one (sub-)warp per row, 128-bit loads/stores, no shared memory
// (no reuse).  scatter_* has two paths chosen on the device (no host sync):
//   sorted indices (what SageDataFlow / fixed-fanout blocks produce, sage_dataflow.py:43-46):
//     warp per OUTPUT row, its edges found by binary search, accumulated left to right -> the
//     reference's summation order, bit-exact, no atomics;
//   unsorted indices: vector atomics (red.global.add.v4.f32), order-free, within 1e-5 relative.
#include <stdlib.h>

#include <algorithm>

#include "internal.h"

namespace eu {

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// lanes per row for a row of D floats moved as float4 (D % 4 == 0): smallest power of two >= D/4, <= 32
static inline int lanes_per_row(int64_t D) {
  int64_t v = D / 4;
  int g = 1;
  while (g < 32 && g < v) g <<= 1;
  return g;
}

// ---------------------------------------------------------------------------- feature fetch
// Per segment: out[r, 0:dim] = feat[row(ids[r]), soff : soff + min(sdim, dim)], zeros elsewhere / for unknown ids.  A stored
// width wider than dim is clipped to dim.
struct FeatSeg {
  const unsigned long long* ids;
  float* out;
  int64_t start;          // first row of the segment in the launch
  int32_t dim, soff, sdim;
};
template <bool VEC, int N>
__global__ void __launch_bounds__(256) k_feature(DevGraph g, SegTable<FeatSeg, N> t, int G) {
  const int sh = 31 - __clz(G);   // G is a power of two
  const int sub = (int)(threadIdx.x & (G - 1));
  const int64_t stride = ((int64_t)gridDim.x * blockDim.x) >> sh;
  // grid-stride over the rows: the launcher may cap the grid (EU_FEATURE_CTAS CTAs per SM) so that this HBM-bound copy leaves
  // SM residency to the issue-bound sampling kernels of the other lanes
  for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> sh; i < t.rows; i += stride) {
    const FeatSeg& q = t.s[seg_of(t, i)];
    const int32_t dim = q.dim, soff = q.soff, sdim = q.sdim;
    const int64_t r = i - q.start;
    const int64_t row = sdim > 0 ? lookup_row(g, __ldg(q.ids + r)) : -1;
    const int32_t fd = sdim;  // stored width of this slot
    float* o = q.out + r * (int64_t)dim;
    const float* f = row >= 0 ? g.feat + row * (int64_t)g.feat_dim + soff : nullptr;
    if (VEC) {
      for (int32_t d = sub * 4; d < dim; d += G * 4) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (f && d < fd) v = ldg4(f + d);  // VEC requires fd % 4 == 0 so a float4 never straddles fd
        st4(o + d, v);
      }
    } else {
      for (int32_t d = sub; d < dim; d += G) o[d] = (f && d < fd) ? __ldg(f + d) : 0.f;
    }
  }
}

// ---------------------------------------------------------------------------- gather
template <bool VEC>
__global__ void __launch_bounds__(256) k_gather(const float* __restrict__ params, int64_t D,
                                                const int32_t* __restrict__ idx, int64_t E, int G,
                                                float* __restrict__ out) {
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t i = tid >> (31 - __clz(G));   // G is a power of two
  const int sub = (int)(tid & (G - 1));
  if (i >= E) return;
  const float* src = params + (int64_t)__ldg(idx + i) * D;  // no bounds check, as gather_op.cc:47-51
  float* o = out + i * D;
  if (VEC) {
    for (int64_t d = sub * 4; d < D; d += G * 4) st4(o + d, ldg4(src + d));
  } else {
    for (int64_t d = sub; d < D; d += G) o[d] = __ldg(src + d);
  }
}

// ---------------------------------------------------------------------------- scatter
__global__ void k_check_sorted(const int32_t* __restrict__ idx, int64_t E, int* unsorted) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e + 1 < E && __ldg(idx + e) > __ldg(idx + e + 1)) *unsorted = 1;
}

__device__ __forceinline__ int64_t lower_bound_i32(const int32_t* __restrict__ a, int64_t n, int64_t key) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

enum { OP_ADD = 0, OP_MAX = 1, OP_MEAN = 2 };

// sorted path: G lanes per OUTPUT row r; edges [lb(r), lb(r+1)) reduced in index order.
template <int OP, bool VEC>
__global__ void __launch_bounds__(256) k_scatter_sorted(const float* __restrict__ upd, int64_t D,
                                                        const int32_t* __restrict__ idx, int64_t E,
                                                        int64_t size, int G, const int* unsorted,
                                                        float* __restrict__ out) {
  if (*unsorted) return;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t r = tid >> (31 - __clz(G));   // G is a power of two
  const int sub = (int)(tid & (G - 1));
  if (r >= size) return;
  const int64_t b = lower_bound_i32(idx, E, r), e = lower_bound_i32(idx, E, r + 1);
  const float init = OP == OP_MAX ? -1e9f : 0.f;
  const float denom = __fadd_rn((float)(e - b), 1e-7f);
  float* o = out + r * D;
  if (VEC) {
    for (int64_t d = sub * 4; d < D; d += G * 4) {
      float4 acc = make_float4(init, init, init, init);
      for (int64_t k = b; k < e; ++k) {
        float4 v = ldg4(upd + k * D + d);
        if (OP == OP_MAX) {
          acc.x = v.x > acc.x ? v.x : acc.x; acc.y = v.y > acc.y ? v.y : acc.y;
          acc.z = v.z > acc.z ? v.z : acc.z; acc.w = v.w > acc.w ? v.w : acc.w;
        } else {
          acc.x = __fadd_rn(acc.x, v.x); acc.y = __fadd_rn(acc.y, v.y);
          acc.z = __fadd_rn(acc.z, v.z); acc.w = __fadd_rn(acc.w, v.w);
        }
      }
      if (OP == OP_MEAN) {
        acc.x = __fdiv_rn(acc.x, denom); acc.y = __fdiv_rn(acc.y, denom);
        acc.z = __fdiv_rn(acc.z, denom); acc.w = __fdiv_rn(acc.w, denom);
      }
      st4(o + d, acc);
    }
  } else {
    for (int64_t d = sub; d < D; d += G) {
      float acc = init;
      for (int64_t k = b; k < e; ++k) {
        float v = __ldg(upd + k * D + d);
        if (OP == OP_MAX) acc = v > acc ? v : acc; else acc = __fadd_rn(acc, v);
      }
      if (OP == OP_MEAN) acc = __fdiv_rn(acc, denom);
      o[d] = acc;
    }
  }
}

// unsorted path ------------------------------------------------------------------------------
__global__ void k_fill_if(float* __restrict__ out, int64_t n, float v, const int* unsorted) {
  if (!*unsorted) return;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[i] = v;
}

__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  // total order trick: non-negative floats compare like signed ints, negative like reversed unsigned
  if (v != v) return;  // NaN never wins `upd > out`
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

template <int OP, bool VEC>
__global__ void __launch_bounds__(256) k_scatter_atomic(const float* __restrict__ upd, int64_t D,
                                                        const int32_t* __restrict__ idx, int64_t E, int G,
                                                        const int* unsorted, float* __restrict__ out,
                                                        float* __restrict__ cnt) {
  if (!*unsorted) return;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t i = tid >> (31 - __clz(G));   // G is a power of two
  const int sub = (int)(tid & (G - 1));
  if (i >= E) return;
  const int64_t r = __ldg(idx + i);
  float* o = out + r * D;
  const float* u = upd + i * D;
  if (OP == OP_MEAN && sub == 0) atomicAdd(cnt + r, 1.0f);
  if (VEC && OP != OP_MAX) {
    for (int64_t d = sub * 4; d < D; d += G * 4) atomicAdd(reinterpret_cast<float4*>(o + d), ldg4(u + d));
  } else {
    const int step = VEC ? 4 : 1;
    for (int64_t d = sub * step; d < D; d += G * step)
      for (int q = 0; q < step; ++q) {
        if (OP == OP_MAX) atomic_max_f32(o + d + q, __ldg(u + d + q));
        else atomicAdd(o + d + q, __ldg(u + d + q));
      }
  }
}

__global__ void k_mean_div(float* __restrict__ out, int64_t D, int64_t size, const float* __restrict__ cnt,
                           const int* unsorted) {
  if (!*unsorted) return;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < size * D) out[i] = __fdiv_rn(out[i], __fadd_rn(cnt[i / D], 1e-7f));
}

// ---------------------------------------------------------------------------- fused SAGE mean
// out[r,:] = (sum_j feat[row(ids[r*count+j]),:]) / (count + 1e-7), j ascending (== get_dense_feature
// followed by scatter_mean over edge_src = repeat(range(rows), count)).  One warp per output row;
// the `count` id->row lookups run in parallel across lanes, then NV float4 per lane are accumulated.
// NV float4 per lane: rows of up to NV * 128 floats.  FULL: the width is exactly NV * 128 (128 / 256: no column guards, the
// width is a compile-time constant); otherwise any multiple of 4 up to NV * 128 (e.g. 64 of configs[4]) with guarded columns.
template <int NV, bool FULL>
__global__ void __launch_bounds__(256) k_sage_mean(DevGraph g, const unsigned long long* __restrict__ ids,
                                                   int64_t rows, int32_t count, bool mean, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int32_t fd = FULL ? NV * 128 : g.feat_dim;    // == dim, a multiple of 4, <= NV * 128 (checked by the launcher)
  const float* __restrict__ feat = g.feat + lane * 4;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // grid-stride, one warp per output row (the launcher may cap the grid: EU_SAGE_CTAS CTAs per SM)
  for (int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; r < rows; r += nwarps) {
  float4 acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int32_t j0 = 0; j0 < count; j0 += 32) {
    // the id -> row lookups of up to 32 neighbors run in parallel across the lanes (rows < 2^31: launcher)
    int32_t my = -1;
    if (j0 + lane < count) my = (int32_t)lookup_row(g, __ldg(ids + r * count + j0 + lane));
    // Only neighbors that exist are visited, in ascending j.  Skipping an absent one is exact: it would add a
    // row of +0.0 and the accumulator can never be -0.0 (it starts at +0.0 and x + (-0.0) keeps +0.0's sign).
    unsigned valid = __ballot_sync(0xffffffffu, my >= 0);
    while (valid) {  // warp-uniform
      float4 v[4][NV];
      int n = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {  // 4 independent row reads in flight
        if (valid) {
          const int j = __ffs(valid) - 1;
          valid &= valid - 1;
          const int32_t row = __shfl_sync(0xffffffffu, my, j);
          const float* p = feat + (int64_t)row * fd;
#pragma unroll
          for (int t = 0; t < NV; ++t) v[q][t] = (FULL || lane * 4 + t * 128 < fd) ? ldg4(p + t * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
          n = q + 1;
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q < n) {
#pragma unroll
          for (int t = 0; t < NV; ++t) {
            acc[t].x = __fadd_rn(acc[t].x, v[q][t].x); acc[t].y = __fadd_rn(acc[t].y, v[q][t].y);
            acc[t].z = __fadd_rn(acc[t].z, v[q][t].z); acc[t].w = __fadd_rn(acc[t].w, v[q][t].w);
          }
        }
      }
    }
  }
  const float denom = __fadd_rn((float)count, 1e-7f);
  float* o = out + r * (int64_t)fd + lane * 4;
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    float4 a = acc[t];
    if (mean) { a.x = __fdiv_rn(a.x, denom); a.y = __fdiv_rn(a.y, denom); a.z = __fdiv_rn(a.z, denom); a.w = __fdiv_rn(a.w, denom); }
    if (FULL || lane * 4 + t * 128 < fd) st4(o + t * 128, a);
  }
  }
}

// generic width fallback: G lanes... one warp per row, scalar columns
__global__ void __launch_bounds__(256) k_sage_mean_generic(DevGraph g, const unsigned long long* __restrict__ ids,
                                                           int64_t rows, int32_t count, int32_t dim, bool mean,
                                                           float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int32_t fd = g.feat_dim;
  const float denom = __fadd_rn((float)count, 1e-7f);
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; r < rows; r += nwarps)
    for (int32_t d = lane; d < dim; d += 32) {
      float acc = 0.f;
      for (int32_t j = 0; j < count; ++j) {
        const int64_t row = lookup_row(g, __ldg(ids + r * count + j));
        acc = __fadd_rn(acc, (row >= 0 && d < fd) ? __ldg(g.feat + row * (int64_t)fd + d) : 0.f);
      }
      out[r * (int64_t)dim + d] = mean ? __fdiv_rn(acc, denom) : acc;
    }
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// CTAs per SM of the HBM-bound row movers (0 = one CTA per 8 rows / as many as the rows need).  A capped, persistent grid keeps
// the copy at HBM speed (a few warps per SM cover the bandwidth-delay product) while the issue-bound sampling kernels of the
// other lanes stay resident beside it.
static inline unsigned capped_grid(int64_t want_blocks, const char* env, int dflt) {
  static int cached_sage = -1, cached_feat = -1;
  int& cached = env[3] == 'S' ? cached_sage : cached_feat;
  if (cached < 0) { const char* e = getenv(env); cached = e ? std::max(0, atoi(e)) : dflt; }
  const int64_t cap = cached > 0 ? (int64_t)148 * cached : want_blocks;
  return (unsigned)std::max<int64_t>(1, std::min(want_blocks, cap));
}

// One k_feature launch over the segments.  The float4 path is taken for the whole launch when every segment allows it; the lanes
// per row follow the widest segment.  Unknown slot ids (outside [0, n_slots)) give zero rows (Node::GetFloat32Feature skips
// them, node.cc:353-364; api.cc:71-73).
template <int N>
static int launch_feature(eu_ctx* c, const DenseSeg* segs, int n) {
  const DevGraph& d = c->g->d;
  SegTable<FeatSeg, N> t{};
  t.n = n;
  bool vec = d.feat_dim % 4 == 0;
  int32_t wmax = 0;
  for (int k = 0; k < n; ++k) {
    const DenseSeg& a = segs[k];
    const bool have = a.fid >= 0 && a.fid < d.n_slots;
    FeatSeg& q = t.s[k];
    q.ids = a.ids; q.out = a.out; q.start = t.rows; q.dim = a.dim;
    q.soff = have ? d.slot_off[a.fid] : 0;
    q.sdim = have ? d.slot_dim[a.fid] : 0;
    t.rows += a.rows;
    if (a.rows > 0 && a.dim > 0) {
      vec = vec && a.dim % 4 == 0 && q.soff % 4 == 0 && q.sdim % 4 == 0 && aligned16(a.out);
      wmax = std::max(wmax, a.dim);
    }
  }
  if (t.rows == 0 || wmax == 0) return EU_OK;
  const int G = vec ? lanes_per_row(wmax) : (wmax >= 32 ? 32 : 1);
  const unsigned blocks = capped_grid(ceil_div(t.rows * G, 256), "EU_FEATURE_CTAS", 0);
  EuProfScope ps(c, "k_feature", t.rows);
  if (vec) k_feature<true, N><<<blocks, 256, 0, c->stream>>>(d, t, G);
  else k_feature<false, N><<<blocks, 256, 0, c->stream>>>(d, t, G);
  EU_LAUNCHED();
  return EU_OK;
}

int dense_feature_segments(eu_ctx* c, const DenseSeg* segs, int n) {
  if (n < 1 || n > kMaxFeatSegs) { set_error("dense features: %d segments (1..%d)", n, kMaxFeatSegs); return EU_ERR_UNSUPPORTED; }
  for (int k = 0; k < n; ++k)
    if (segs[k].rows < 0 || segs[k].dim < 0 || (segs[k].rows > 0 && segs[k].dim > 0 && (!segs[k].ids || !segs[k].out))) {
      set_error("dense features: bad segment %d", k);
      return EU_ERR_INVALID;
    }
  return n == 1 ? launch_feature<1>(c, segs, n) : launch_feature<kMaxFeatSegs>(c, segs, n);
}

template <int OP>
static int scatter(eu_ctx* c, const float* upd, int64_t D, const int32_t* idx, int64_t E, int64_t size,
                   float* out) {
  if (!c || D <= 0 || E < 0 || size < 0 || (E > 0 && (!upd || !idx)) || (size > 0 && !out)) {
    set_error("scatter: bad argument");
    return EU_ERR_INVALID;
  }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (size == 0) return EU_OK;
  int rc = ctx_misc(c, 256 + (OP == OP_MEAN ? (int64_t)sizeof(float) * size : 0));
  if (rc) return rc;
  int* unsorted = (int*)c->d_misc;
  float* cnt = (float*)((char*)c->d_misc + 256);
  cudaStream_t s = c->stream;
  EU_CUDA(cudaMemsetAsync(unsorted, 0, sizeof(int), s));
  if (OP == OP_MEAN) EU_CUDA(cudaMemsetAsync(cnt, 0, sizeof(float) * size, s));
  const bool vec = (D % 4 == 0) && aligned16(upd) && aligned16(out);
  const int G = vec ? lanes_per_row(D) : (D >= 32 ? 32 : 1);
  const int tb = 256;
  if (E > 1) {
    k_check_sorted<<<(unsigned)ceil_div(E, tb), tb, 0, s>>>(idx, E, unsorted);
    EU_LAUNCHED();
  }
  const unsigned gs = (unsigned)ceil_div(size * G, tb), ge = (unsigned)ceil_div((E > 0 ? E : 1) * G, tb);
  EuProfScope ps(c, "scatter(sorted+fallback)", E);
  if (vec) k_scatter_sorted<OP, true><<<gs, tb, 0, s>>>(upd, D, idx, E, size, G, unsorted, out);
  else k_scatter_sorted<OP, false><<<gs, tb, 0, s>>>(upd, D, idx, E, size, G, unsorted, out);
  EU_LAUNCHED();
  k_fill_if<<<148 * 4, tb, 0, s>>>(out, size * D, OP == OP_MAX ? -1e9f : 0.f, unsorted);
  EU_LAUNCHED();
  if (E > 0) {
    if (vec) k_scatter_atomic<OP, true><<<ge, tb, 0, s>>>(upd, D, idx, E, G, unsorted, out, cnt);
    else k_scatter_atomic<OP, false><<<ge, tb, 0, s>>>(upd, D, idx, E, G, unsorted, out, cnt);
    EU_LAUNCHED();
  }
  if (OP == OP_MEAN) {
    k_mean_div<<<(unsigned)ceil_div(size * D, tb), tb, 0, s>>>(out, D, size, cnt, unsorted);
    EU_LAUNCHED();
  }
  return EU_OK;
}

}  // namespace eu

using namespace eu;

extern "C" {

int eu_get_dense_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int32_t dim, float* out) {
  if (!c || M < 0 || dim < 0 || (M > 0 && (!nodes || (dim > 0 && !out)))) { set_error("eu_get_dense_feature: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (M == 0 || dim == 0) return EU_OK;
  const DenseSeg seg{(const unsigned long long*)nodes, M, fid, dim, out};
  return launch_feature<1>(c, &seg, 1);
}

int eu_gather(eu_ctx* c, const float* params, int64_t N, int64_t D, const int32_t* idx, int64_t E, float* out) {
  (void)N;
  if (!c || D <= 0 || E < 0 || (E > 0 && (!params || !idx || !out))) { set_error("eu_gather: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (E == 0) return EU_OK;
  const bool vec = (D % 4 == 0) && aligned16(params) && aligned16(out);
  const int G = vec ? lanes_per_row(D) : (D >= 32 ? 32 : 1);
  const unsigned blocks = (unsigned)ceil_div(E * G, 256);
  if (vec) k_gather<true><<<blocks, 256, 0, c->stream>>>(params, D, idx, E, G, out);
  else k_gather<false><<<blocks, 256, 0, c->stream>>>(params, D, idx, E, G, out);
  EU_LAUNCHED();
  return EU_OK;
}

int eu_scatter_add(eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) {
  return scatter<OP_ADD>(c, u, D, idx, E, size, out);
}
int eu_scatter_max(eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) {
  return scatter<OP_MAX>(c, u, D, idx, E, size, out);
}
int eu_scatter_mean(eu_ctx* c, const float* u, int64_t D, const int32_t* idx, int64_t E, int64_t size, float* out) {
  return scatter<OP_MEAN>(c, u, D, idx, E, size, out);
}

static int fanout_aggregate(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, bool mean, float* out) {
  if (!c || rows < 0 || count < 0 || dim <= 0 || (rows > 0 && (!nbr_ids || !out))) { set_error("eu_sage_mean_aggregate: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (rows == 0) return EU_OK;
  const DevGraph& d = c->g->d;
  const unsigned blocks = capped_grid(ceil_div(rows * 32, 256), "EU_SAGE_CTAS", 0);
  const unsigned long long* ids = (const unsigned long long*)nbr_ids;
  EuProfScope ps(c, mean ? "k_sage_mean" : "k_sage_add", rows);
  // float4 path: one slot of the full stored width, a multiple of 4 floats up to 1024 (D = 64 of configs[4], 128, 256, ...)
  const bool v4 = d.n < ((int64_t)1 << 31) && d.n_slots == 1 && dim == d.feat_dim && (dim & 3) == 0 && dim <= 1024 && aligned16(out) && aligned16(d.feat);
  if (v4 && dim == 128) k_sage_mean<1, true><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else if (v4 && dim == 256) k_sage_mean<2, true><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else if (v4 && dim <= 128) k_sage_mean<1, false><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else if (v4 && dim <= 256) k_sage_mean<2, false><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else if (v4 && dim <= 512) k_sage_mean<4, false><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else if (v4) k_sage_mean<8, false><<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, mean, out);
  else k_sage_mean_generic<<<blocks, 256, 0, c->stream>>>(d, ids, rows, count, dim, mean, out);
  EU_LAUNCHED();
  return EU_OK;
}


int eu_sage_mean_aggregate(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, float* out) {
  return fanout_aggregate(c, nbr_ids, rows, count, dim, true, out);
}
// the scatter_add variant over the same fixed-fanout blocks (aggr='add': GCN / the per-relation sums of configs[4]):
// get_dense_feature + scatter_add over edge_src = repeat(range(rows), count), fused
int eu_sage_add_aggregate(eu_ctx* c, const int64_t* nbr_ids, int64_t rows, int32_t count, int32_t dim, float* out) {
  return fanout_aggregate(c, nbr_ids, rows, count, dim, false, out);
}

}  // extern "C"
