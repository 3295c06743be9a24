// Ragged node features on the HBM-resident graph: uint64 ("sparse") and binary features (SURVEY.md section 8f, next-2).
// Reference semantics (file:line relative to /root/reference):
//   Node::GetUint64Feature / GetBinaryFeature   euler/core/graph/node.cc:330-409   slot s = [idx[s-1], idx[s]) of the node's array
//   tf_euler GetSparseFeature                   tf_euler/kernels/get_sparse_feature_op.cc:52-130  a node without values gets one
//                                               entry {i, 0} = default_value
//   tf_euler GetBinaryFeature                   tf_euler/kernels/get_binary_feature_op.cc          one string per node
// Same shape as the full-neighbor listing: per-node lengths -> cub inclusive scan -> copy; no host sync in the device entry points.
// The kernels walk a table of segments, so one length launch, one scan and one fill serve every (level, feature) of
// eu_sample_fanout_with_feature; the single-feature entry points are the one-segment case.
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "internal.h"

namespace eu {

// row slice of slot `fid`: [b, e) in the value array, b == e when the node / slot does not exist
__device__ __forceinline__ void ragged_slice(const int64_t* __restrict__ ptr, int32_t S, int64_t row, int32_t fid, int64_t* b, int64_t* e) {
  *b = *e = 0;
  if (row < 0 || fid < 0 || fid >= S || !ptr) return;
  *b = ptr[row * S + fid];
  *e = ptr[row * S + fid + 1];
}

// Segment s of a launch: rows [start, start + rows) fetch slot `fid` of ids[0 .. rows).  lens[1 + i] is the length of launch row
// i (lens[0] = 0); after the inclusive scan, lens[i] is where row i's values begin in the launch, and segment s owns
// out_ptr[r] = lens[start + r] - lens[start].  The one-segment entry points scan straight into their out_ptr (lens == out_ptr).
struct RaggedSeg {
  const unsigned long long* ids;
  long long* out_ptr;          // [rows + 1]; written by k_ragged_fill only when the launch scans into scratch
  long long* out_values;       // SPARSE
  unsigned char* out_bytes;    // binary
  int64_t start, cap;          // cap: entries of the value buffer
  long long default_value;
  int32_t fid;
};

template <bool SPARSE, int N>
__global__ void k_ragged_len(DevGraph g, SegTable<RaggedSeg, N> t, long long* __restrict__ lens) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i == 0) lens[0] = 0;
  if (i >= t.rows) return;
  const RaggedSeg& q = t.s[seg_of(t, i)];
  int64_t b, e;
  const int64_t row = lookup_row(g, q.ids[i - q.start]);
  if (SPARSE) ragged_slice(g.u64_ptr, g.n_u64_slots, row, q.fid, &b, &e);
  else ragged_slice(g.bin_ptr, g.n_bin_slots, row, q.fid, &b, &e);
  long long len = e - b;
  if (SPARSE && len == 0) len = 1;   // one default entry (get_sparse_feature_op.cc:96-99)
  lens[i + 1] = len;
}

template <bool SPARSE, int N>
__global__ void __launch_bounds__(256) k_ragged_fill(DevGraph g, SegTable<RaggedSeg, N> t, const long long* __restrict__ lens,
                                                     bool write_ptr) {
  const int lane = threadIdx.x & 31;
  const int64_t gtid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  if (write_ptr && gtid < t.n) t.s[N == 1 ? 0 : gtid].out_ptr[0] = 0;   // also for segments without rows
  for (int64_t i = gtid >> 5; i < t.rows; i += nwarps) {
    const RaggedSeg& q = t.s[seg_of(t, i)];
    const int64_t r = i - q.start;
    int64_t b, e;
    const int64_t row = lookup_row(g, q.ids[r]);
    if (SPARSE) ragged_slice(g.u64_ptr, g.n_u64_slots, row, q.fid, &b, &e);
    else ragged_slice(g.bin_ptr, g.n_bin_slots, row, q.fid, &b, &e);
    const long long base = lens[q.start];
    const int64_t o = lens[i] - base;
    if (write_ptr && lane == 0) q.out_ptr[r + 1] = lens[i + 1] - base;
    const int64_t cap = q.cap;
    if (SPARSE) {
      if (e == b) { if (lane == 0 && o < cap) q.out_values[o] = q.default_value; continue; }
      for (int64_t k = lane; k < e - b; k += 32) if (o + k < cap) q.out_values[o + k] = (long long)g.u64_val[b + k];
    } else {
      for (int64_t k = lane; k < e - b; k += 32) if (o + k < cap) q.out_bytes[o + k] = g.bin_val[b + k];
    }
  }
}

// length launch, one scan, fill launch.  lens: [rows + 1], the single segment's out_ptr or scratch behind the scan's temporary
// storage in ctx_misc (write_ptr: the fill then writes every segment's out_ptr).
template <bool SPARSE, int N>
static int ragged_launch(eu_ctx* c, const SegTable<RaggedSeg, N>& t, long long* lens, bool write_ptr, bool fill, size_t tmp) {
  const DevGraph& d = c->g->d;
  cudaStream_t s = c->stream;
  k_ragged_len<SPARSE, N><<<(unsigned)ceil_div(std::max<int64_t>(t.rows, 1), 256), 256, 0, s>>>(d, t, lens);
  EU_LAUNCHED();
  EU_CUDA(cub::DeviceScan::InclusiveSum(c->d_misc, tmp, lens, lens, (int)(t.rows + 1), s));
  EU_LAUNCHED();
  if (fill) {
    const unsigned blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(t.rows * 32, 256), 148 * 8));
    k_ragged_fill<SPARSE, N><<<blocks, 256, 0, s>>>(d, t, lens, write_ptr);
    EU_LAUNCHED();
  }
  return EU_OK;
}

template <bool SPARSE>
static int ragged_get(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap, int64_t* out_ptr,
                      int64_t* out_values, uint8_t* out_bytes, const char* what) {
  if (!c || M < 0 || cap < 0 || !out_ptr || (M > 0 && !nodes) || (cap > 0 && !(SPARSE ? (void*)out_values : (void*)out_bytes))) {
    set_error("%s: bad argument", what);
    return EU_ERR_INVALID;
  }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (M >= ((int64_t)1 << 31)) { set_error("%s: more than 2^31 nodes", what); return EU_ERR_UNSUPPORTED; }
  size_t tmp = 0;
  cub::DeviceScan::InclusiveSum((void*)nullptr, tmp, (long long*)nullptr, (long long*)nullptr, (int)(M + 1), c->stream);
  int rc = ctx_misc(c, (int64_t)tmp + 256);
  if (rc) return rc;
  SegTable<RaggedSeg, 1> t{};
  t.n = 1;
  t.rows = M;
  t.s[0] = RaggedSeg{(const unsigned long long*)nodes, (long long*)out_ptr, (long long*)out_values, out_bytes, 0, cap,
                     (long long)default_value, fid};
  return ragged_launch<SPARSE, 1>(c, t, (long long*)out_ptr, false, cap > 0 && M > 0, tmp);
}

int sparse_feature_segments(eu_ctx* c, const SparseSeg* segs, int n) {
  if (n < 1 || n > kMaxFeatSegs) { set_error("sparse features: %d segments (1..%d)", n, kMaxFeatSegs); return EU_ERR_UNSUPPORTED; }
  SegTable<RaggedSeg, kMaxFeatSegs> t{};
  t.n = n;
  for (int k = 0; k < n; ++k) {
    const SparseSeg& a = segs[k];
    if (a.rows < 0 || a.cap < 0 || !a.out_ptr || (a.rows > 0 && !a.ids) || (a.cap > 0 && !a.out_values)) {
      set_error("sparse features: bad segment %d", k);
      return EU_ERR_INVALID;
    }
    t.s[k] = RaggedSeg{a.ids, (long long*)a.out_ptr, (long long*)a.out_values, nullptr, t.rows, a.cap, (long long)a.default_value, a.fid};
    t.rows += a.rows;
  }
  if (t.rows >= ((int64_t)1 << 31)) { set_error("sparse features: more than 2^31 rows in all"); return EU_ERR_UNSUPPORTED; }
  size_t tmp = 0;
  cub::DeviceScan::InclusiveSum((void*)nullptr, tmp, (long long*)nullptr, (long long*)nullptr, (int)(t.rows + 1), c->stream);
  const int64_t lens_off = ((int64_t)tmp + 255) & ~(int64_t)255;
  int rc = ctx_misc(c, lens_off + 8 * (t.rows + 1));
  if (rc) return rc;
  return ragged_launch<true, kMaxFeatSegs>(c, t, (long long*)((char*)c->d_misc + lens_off), true, true, tmp);
}

// host buffers: lengths first (total), then the values when cap allows
template <bool SPARSE>
static int ragged_get_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap, int64_t* out_ptr,
                           void* out_vals, int64_t* total, const char* what) {
  if (!c || M < 0 || cap < 0 || !out_ptr || (M > 0 && !nodes)) { set_error("%s: bad argument", what); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  unsigned long long* d_nodes = nullptr;
  long long* d_ptr = nullptr;
  char* d_vals = nullptr;
  EU_CUDA(cudaMalloc(&d_nodes, 8 * (size_t)std::max<int64_t>(M, 1)));
  EU_CUDA(cudaMalloc(&d_ptr, 8 * (size_t)(M + 1)));
  const size_t esz = SPARSE ? 8 : 1;
  int rc = EU_OK;
  do {
    if (M > 0 && cudaMemcpyAsync(d_nodes, nodes, 8 * (size_t)M, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { rc = EU_ERR_CUDA; break; }
    rc = ragged_get<SPARSE>(c, (const int64_t*)d_nodes, M, fid, default_value, 0, (int64_t*)d_ptr, nullptr, nullptr, what);
    if (rc) break;
    if (cudaMemcpyAsync(out_ptr, d_ptr, 8 * (size_t)(M + 1), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = EU_ERR_CUDA; break; }
    const int64_t tot = out_ptr[M];
    if (total) *total = tot;
    const int64_t n = std::min(cap, tot);
    if (n > 0) {
      if (!out_vals) { set_error("%s: null output", what); rc = EU_ERR_INVALID; break; }
      if (cudaMalloc(&d_vals, esz * (size_t)n) != cudaSuccess) { set_error("%s: cudaMalloc failed", what); rc = EU_ERR_CUDA; break; }
      rc = ragged_get<SPARSE>(c, (const int64_t*)d_nodes, M, fid, default_value, n, (int64_t*)d_ptr, SPARSE ? (int64_t*)d_vals : nullptr,
                              SPARSE ? nullptr : (uint8_t*)d_vals, what);
      if (rc) break;
      if (cudaMemcpyAsync(out_vals, d_vals, esz * (size_t)n, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
          cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = EU_ERR_CUDA; break; }
    }
  } while (false);
  cudaFree(d_nodes); cudaFree(d_ptr); cudaFree(d_vals);
  if (rc == EU_ERR_CUDA) set_error("%s: CUDA error %s", what, cudaGetErrorString(cudaGetLastError()));
  return rc;
}

}  // namespace eu

using namespace eu;

extern "C" {

int eu_get_sparse_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap, int64_t* out_ptr,
                          int64_t* out_values) {
  return ragged_get<true>(c, nodes, M, fid, default_value, cap, out_ptr, out_values, nullptr, "eu_get_sparse_feature");
}
int eu_get_sparse_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t default_value, int64_t cap, int64_t* out_ptr,
                               int64_t* out_values, int64_t* total) {
  return ragged_get_host<true>(c, nodes, M, fid, default_value, cap, out_ptr, out_values, total, "eu_get_sparse_feature_host");
}
int eu_get_binary_feature(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t cap, int64_t* out_ptr, uint8_t* out_bytes) {
  return ragged_get<false>(c, nodes, M, fid, 0, cap, out_ptr, nullptr, out_bytes, "eu_get_binary_feature");
}
int eu_get_binary_feature_host(eu_ctx* c, const int64_t* nodes, int64_t M, int32_t fid, int64_t cap, int64_t* out_ptr, uint8_t* out_bytes,
                               int64_t* total) {
  return ragged_get_host<false>(c, nodes, M, fid, 0, cap, out_ptr, out_bytes, total, "eu_get_binary_feature_host");
}

}  // extern "C"
