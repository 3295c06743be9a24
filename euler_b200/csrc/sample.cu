// Weighted neighbor sampling / multi-hop fanout / global node sampling on the HBM-resident CSR.
//
// Reference semantics reproduced (file:line relative to /root/reference):
//   Node::__SampleNeighbor            euler/core/graph/node.cc:98-161
//   RandomSelect                      euler/common/compact_weighted_collection.h:30-52
//   euler::SampleNeighbor             euler/core/api/api.cc:223-236
//   engine: ID_UNIQUE -> API_SAMPLE_NB -> gather   euler/core/kernels/id_unique_op.cc:41-66,
//       sample_neighbor_op.cc:37-147 (default fill :135-143), idx_gather_op.cc:45-55,
//       data_gather_op.cc:34-46; rule euler/parser/compiler.cc:76-90
//   TF packing                        tf_euler/kernels/sample_neighbor_op.cc:79-81,114-122
//   fanout chaining                   tf_euler/kernels/sample_fanout_op.cc:36-43,116-140
//   Graph::SampleNode / alias         euler/core/graph/graph.cc:221-275, euler/common/alias_method.cc:66-78
//
// B200 design: one warp per seed row, one lane per draw.  The reference's single serial engine
// stream is reproduced by (1) a device hash that resolves each seed's first occurrence
// (ID_UNIQUE order), (2) a multiplicative prefix "scan" that hands every first-occurrence row the
// engine state it would have had in the serial loop, (3) lanes jumping ahead A^(2*k*lane).
// Duplicate seeds re-derive the identical row from the first occurrence's state, so there is no
// gather pass and the frontier (engine ids) stays in HBM between hops.
#include <algorithm>

#include <stdlib.h>

#include "internal.h"

namespace eu {

struct ETypes {
  int32_t K;
  int32_t v[EU_MAX_ETYPES];
};

// A launch covers `nb` independent batches of `rows_b` seeds each (nb = 1 for the plain ops).  Batch b has
// its own engine (EuRngState[b]), its own dedup scope (table region b) and its own serial draw order, i.e.
// it is exactly one reference op call on one client thread; batching only shares the kernel launches.
struct Geom {
  int32_t nb;        // batches
  int32_t nblk_b;    // 256-row blocks per batch
  int64_t rows_b;    // seeds per batch (dense in the seed / output arrays)
  int64_t rows_pad;  // nblk_b * 256: stride of the per-row scratch arrays
  int64_t cap_b;     // dedup slots per batch (power of two) ; region stride = cap_b + 1
  const int32_t* rows_act;  // device, [nb] or null: only the first rows_act[b] (<= rows_b) seeds of batch b exist -- the
                            // sharded owner path sizes a launch for the worst case and learns the real counts on the device
};

// ---------------------------------------------------------------------------- 1. seed dedup
// grid (blocks per batch, nb): a block past the batch's real row count (sharded owner inputs are sized for the worst case)
// leaves at once
__global__ void k_dedup_insert(HashSlot* tabs, Geom gm, const unsigned long long* __restrict__ seeds) {
  const int b = blockIdx.y;
  const int64_t li = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t rows_here = gm.rows_act ? (int64_t)gm.rows_act[b] : gm.rows_b;
  if (li >= rows_here) return;
  const unsigned long long id = seeds[b * gm.rows_b + li];
  // Warp-aggregate: frontiers are full of runs of equal ids (a default row is `count` zeros, hubs repeat)
  // and equal ids hammer one slot.  The lowest lane of each id group carries the group's minimum
  // index, so only it touches the table.
  const unsigned act = __activemask();
  const unsigned peers = __match_any_sync(act, id);
  if ((threadIdx.x & 31) != __ffs(peers) - 1) return;
  dedup_insert_one(tabs + (int64_t)b * (gm.cap_b + 1), (unsigned long long)dedup_cap_eff(gm.cap_b, gm.rows_act, b) - 1, id, li);
}

__device__ __forceinline__ int64_t dedup_first(const HashSlot* tab, unsigned long long mask,
                                               unsigned long long id) {
  unsigned long long tag = id + 1;
  if (tag == 0ull) return (int64_t)tab[mask + 1].row;
  unsigned long long h = mix64(id) & mask;
  while (true) {
    const ulonglong2 s = *reinterpret_cast<const ulonglong2*>(tab + h);
    if (s.x == tag) return (int64_t)s.y;
    h = (h + 1) & mask;
  }
}

// edge_group_collection.sum_weights_[t]; for T == 1 it is not stored: the single group's f32 sum is
// the row's last cumulative weight (node.cc:59-68 accumulates both with the same additions).
__device__ __forceinline__ float grp_cum_at(const DevGraph& g, int64_t row, int32_t t) {
  if (g.grp_cum) return __ldg(g.grp_cum + row * g.T + t);
  const int64_t b = g.grp_ptr[row], e = g.grp_ptr[row + 1];
  return e > b ? __ldg(g.cum_w + e - 1) : 0.f;
}

// Row eligibility = "would Node::SampleNeighbor return `count` entries" (node.cc:106-148), i.e.
// does this row consume uniforms.  mode 0: K==1; 1: strict subset; 2: all groups.
__device__ __forceinline__ bool row_eligible(const DevGraph& g, int64_t row, const ETypes& et, int mode) {
  if (row < 0) return false;
  const int32_t T = g.T;
  if (mode == 0) {
    int32_t t = et.v[0];
    if (t < 0 || t >= T) return false;
    return g.grp_ptr[row * T + t + 1] > g.grp_ptr[row * T + t];
  }
  if (mode == 1) {
    float s = 0.f;
    for (int32_t i = 0; i < et.K; ++i) {
      int32_t t = et.v[i];
      if (t < 0 || t >= T) return false;
      float pre = t > 0 ? grp_cum_at(g, row, t - 1) : 0.f;
      s = __fadd_rn(s, __fsub_rn(grp_cum_at(g, row, t), pre));
    }
    return s != 0.f;
  }
  return grp_cum_at(g, row, T - 1) != 0.f;
}

// outputs k_prepare needs to finish rows that cannot sample, and the list of rows that can
struct PrepOut {
  unsigned long long* eng_ids;
  long long* out_ids;
  float* out_w;
  int32_t* out_t;
  int32_t count;
  long long default_node;
  HashSlot* next_tabs;
  int64_t next_cap_b;
  int32_t* live;           // [nb*rows_b] global indices of rows that sample
  unsigned int* n_live;    // their number (zeroed before the launch)
};

// ---------------------------------------------------------------------------- 2. prepare
// Per row: first occurrence (ID_UNIQUE), graph row and eligibility of first occurrences.  The number
// of ELIGIBLE FIRST-OCCURRENCE rows before row i of its batch -- its position in the reference's serial
// draw order -- is kept as a 3-level count: emask[ii/32] (ballot), woff[ii/32] (count in earlier warps of
// the block), blkpre[b][ii/256] (count in earlier blocks of the batch; exclusive prefix written by the last
// block of the batch to finish, which also advances that batch's engine by total * draws_per_row uniforms).
// grid = (nblk_b, nb); ii = b * rows_pad + li indexes the scratch arrays.
static constexpr int kPrepBlock = 256;

__global__ void __launch_bounds__(kPrepBlock) k_prepare(DevGraph g, const HashSlot* tabs, Geom gm,
                                                        const unsigned long long* __restrict__ seeds,
                                                        ETypes et, int mode, uint32_t F, unsigned long long draws_per_row,
                                                        int32_t* first, int64_t* rowof, uint32_t* emask, uint32_t* wmul,
                                                        uint32_t* blkpre, uint32_t* blkmul, EuRngState* rngs, PrepOut po) {
  __shared__ uint32_t s_w[kPrepBlock / 32];
  __shared__ bool s_last;
  const int b = blockIdx.y;
  const int64_t li = blockIdx.x * (int64_t)kPrepBlock + threadIdx.x;
  const int64_t ii = b * gm.rows_pad + li;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  EuRngState* rng = rngs + b;
  bool e = false;      // eligible FIRST occurrence: takes a slot of the serial draw order
  bool own = false;    // this row samples (its id is eligible, whether or not it is the first occurrence)
  const int64_t rows_here = gm.rows_act ? (int64_t)gm.rows_act[b] : gm.rows_b;
  // blocks past the batch's real rows (worst-case-sized sharded owner inputs) neither scan nor take a ticket: the launch
  // costs its live rows, not its capacity.  Block 0 always stays (it advances the engine of an empty batch).
  const uint32_t nblk_act = (uint32_t)max((int64_t)1, (rows_here + kPrepBlock - 1) / kPrepBlock);
  if (blockIdx.x >= nblk_act) return;
  if (li < rows_here) {
    const int64_t w = b * gm.rows_b + li;
    const unsigned long long id = seeds[w];
    // raw mode (tabs == null): euler::SampleNeighbor draws every occurrence of an id independently (api.cc:223-236)
    const int64_t f = tabs ? dedup_first(tabs + (int64_t)b * (gm.cap_b + 1), (unsigned long long)dedup_cap_eff(gm.cap_b, gm.rows_act, b) - 1, id) : li;
    first[ii] = (int32_t)f;
    // A duplicate has the same id, hence the same graph row and eligibility as its first occurrence: every row
    // resolves its own, so rows that cannot sample are finished right here and never reach k_sample.
    const int64_t row = lookup_row(g, id);
    own = row_eligible(g, row, et, mode);
    e = own && f == li;
    if (own) {
      rowof[ii] = row;
    } else {
      const int64_t ob = w * (int64_t)po.count;
      for (int32_t j = 0; j < po.count; ++j) {
        if (po.eng_ids) po.eng_ids[ob + j] = 0ull;
        if (po.out_ids) { po.out_ids[ob + j] = po.default_node; po.out_w[ob + j] = 0.f; po.out_t[ob + j] = -1; }
      }
      if (po.next_tabs)  // its `count` zeros enter the next hop's dedup table with their minimum index
        dedup_insert_one(po.next_tabs + (int64_t)b * (po.next_cap_b + 1), (unsigned long long)po.next_cap_b - 1, 0ull,
                         li * (int64_t)po.count);
    }
  }
  // compact the rows that do sample (order is irrelevant: a row's engine state depends only on its position)
  {
    const uint32_t om = __ballot_sync(0xffffffffu, own);
    uint32_t basepos = 0;
    if (lane == 0 && om) basepos = atomicAdd(po.n_live, (unsigned int)__popc(om));
    basepos = __shfl_sync(0xffffffffu, basepos, 0);
    if (own) po.live[basepos + __popc(om & ((1u << lane) - 1u))] = (int32_t)(b * gm.rows_b + li);
  }
  const uint32_t m = __ballot_sync(0xffffffffu, e);
  if (lane == 0) s_w[wid] = __popc(m);
  __syncthreads();
  if (lane == 0) {  // rows_pad is a multiple of 256: every group of the block exists in the scratch arrays
    uint32_t off = 0;
    for (int k = 0; k < wid; ++k) off += s_w[k];
    emask[ii >> 5] = m;
    // F^(eligible rows in earlier warps of this block), off < 256: the rows multiply instead of exponentiating
    uint32_t fp = 1, fb = F;
    for (; off; off >>= 1) { if (off & 1) fp = modmul(fp, fb); fb = modmul(fb, fb); }
    wmul[ii >> 5] = fp;
  }
  uint32_t* bp = blkpre + (int64_t)b * gm.nblk_b;
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
    for (int k = 0; k < kPrepBlock / 32; ++k) tot += s_w[k];
    bp[blockIdx.x] = tot;
    __threadfence();
    s_last = atomicAdd(&rng->blocks_done, 1u) == nblk_act - 1;
  }
  __syncthreads();
  if (!s_last) return;
  // last block of this batch: exclusive prefix over the batch's per-block counts, in place
  __threadfence();
  __shared__ uint32_t s_scan[kPrepBlock];
  uint32_t carry = 0;
  for (uint32_t base = 0; base < nblk_act; base += kPrepBlock) {
    const uint32_t k = base + threadIdx.x;
    const uint32_t v = k < nblk_act ? __ldcg(bp + k) : 0u;  // written by other blocks: read at L2
    s_scan[threadIdx.x] = v;
    __syncthreads();
    for (int off = 1; off < kPrepBlock; off <<= 1) {
      uint32_t t = threadIdx.x >= off ? s_scan[threadIdx.x - off] : 0u;
      __syncthreads();
      s_scan[threadIdx.x] += t;
      __syncthreads();
    }
    if (k < nblk_act) {
      uint32_t pre = carry + s_scan[threadIdx.x] - v;   // eligible rows in earlier blocks of the batch
      bp[k] = pre;
      uint32_t fp = 1, fb = F;
      for (; pre; pre >>= 1) { if (pre & 1) fp = modmul(fp, fb); fb = modmul(fb, fb); }
      blkmul[(int64_t)b * gm.nblk_b + k] = fp;          // F^pre
    }
    carry += s_scan[kPrepBlock - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    // engine after this hop = x * F^total; rows read x_prev
    uint32_t fp = 1, base = F;
    for (uint32_t t = carry; t; t >>= 1) { if (t & 1) fp = modmul(fp, base); base = modmul(base, base); }
    rng->x_prev = rng->x;
    rng->x = modmul(rng->x, fp);
    rng->draws += (unsigned long long)carry * draws_per_row;
    rng->blocks_done = 0;
  }
}

// ---------------------------------------------------------------------------- 3. engine-state scan (walks)
// state_before[i] = x * F^(#eligible rows before i), F = A^(uniforms per row * 2).
// One block; thread t owns a contiguous chunk.  Also advances the ctx engine.
__global__ void __launch_bounds__(1024) k_state_scan(const uint8_t* __restrict__ elig, int64_t rows,
                                                     uint32_t F, unsigned long long draws_per_row,
                                                     uint32_t* state, EuRngState* rng) {
  __shared__ uint32_t s_part[1024];
  __shared__ uint32_t s_cnt[1024];
  const int t = threadIdx.x;
  const int64_t chunk = (rows + 1023) / 1024;
  const int64_t b = t * chunk, e = min(rows, b + chunk);
  uint32_t prod = 1, cnt = 0;
  for (int64_t i = b; i < e; ++i)
    if (elig[i]) { prod = modmul(prod, F); ++cnt; }
  s_part[t] = prod;
  s_cnt[t] = cnt;
  __syncthreads();
  // inclusive Hillis-Steele scan of products (modmul is associative and commutative)
  for (int off = 1; off < 1024; off <<= 1) {
    uint32_t v = 1, c = 0;
    if (t >= off) { v = s_part[t - off]; c = s_cnt[t - off]; }
    __syncthreads();
    if (t >= off) { s_part[t] = modmul(s_part[t], v); s_cnt[t] += c; }
    __syncthreads();
  }
  const uint32_t x0 = rng->x;
  uint32_t run = modmul(x0, t > 0 ? s_part[t - 1] : 1u);
  for (int64_t i = b; i < e; ++i) {
    state[i] = run;
    if (elig[i]) run = modmul(run, F);
  }
  __syncthreads();
  if (t == 1023) {
    rng->x = modmul(x0, s_part[1023]);
    rng->draws += (unsigned long long)s_cnt[1023] * draws_per_row;
  }
}

// ---------------------------------------------------------------------------- 4. sample
struct SampleArgs {
  const unsigned long long* seeds;  // [nb*rows_b]
  Geom gm;
  int32_t count;
  long long default_node;
  ETypes et;
  int mode;
  // minstd: serial-stream position of a first-occurrence row f of batch b =
  //   blkpre[b][f/256] + woff[ff/32] + popc(emask[ff/32] & lanes_below(f%32)), ff = b*rows_pad + f;
  //   engine state = rng[b].x_prev * F^pos = x_prev * blkmul[b][f/256] * wmul[ff/32] * F^popc
  const int32_t* live;          // rows that sample (compacted by k_prepare); null => every row (philox)
  const unsigned int* n_live;
  const int32_t* first;
  const int64_t* rowof;
  const uint32_t* emask;
  const uint32_t* wmul;         // F^(eligible rows in earlier warps of the block)
  const uint32_t* blkmul;       // F^(eligible rows in earlier blocks of the batch)
  uint32_t F;                   // A^(2 * uniforms per row) mod M
  uint32_t lanepow[32];         // A^(2 * uniforms per draw * lane): a lane's jump from the row state
  uint32_t stride;              // A^(2 * uniforms per draw * SG)
  int sg_log;                   // log2 of the lanes per row (SG)
  int stage;                    // 1: TMA-stage mid rows in shared memory (EU_SAMPLE_STAGE=0 turns it off for A/B runs)
  HashSlot* clear_tab;          // dedup tables of THIS hop (all batches), cleared here for the next user
  int64_t clear_n;
  HashSlot* next_tabs;          // dedup tables of the NEXT hop: this hop's engine ids are its seeds (or null)
  int64_t next_cap_b;
  // philox
  unsigned long long key;
  const EuRngState* rngs;
  // outputs
  unsigned long long* eng_ids;  // [nb*rows_b*count] engine ids (0 placeholder) = next frontier; may be null
  long long* out_ids;           // [nb*rows_b*count] TF-packed; may be null
  float* out_w;
  int32_t* out_t;
};

// shuffle binary search over the SG lane-resident values c of a lane group (non-decreasing, +inf padded):
// first local index in [lo,hi] with (double)c > r, else hi.
__device__ __forceinline__ int lane_upper_bound(float c, int lo, int hi, float thr, unsigned gmask, int SG) {
#pragma unroll
  for (int it = 0; it < 5; ++it) {
    int mid = (lo + hi) >> 1;
    float v = __shfl_sync(gmask, c, mid, SG);
    bool go = lo < hi;
    bool gt = v >= thr;   // (double)v > r, see gt_threshold
    hi = (go && gt) ? mid : hi;
    lo = (go && !gt) ? mid + 1 : lo;
  }
  return lo;
}

// One lane GROUP (SG lanes, SG = 2^k >= min(count, 32)) per sampling row, one lane per draw; a warp carries 32/SG
// rows, and a persistent grid strides over the live rows: with fanout 10 two rows share a warp (the kernel is
// issue-bound, profiles/r01_*: every instruction a lane group spares is throughput), and the per-block set-up
// (jump tables, table wipe, parameter loads) is paid once per CTA instead of once per 8 rows.
template <bool PHILOX, int CTAS>
__global__ void __launch_bounds__(256, CTAS) k_sample(DevGraph g, SampleArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t gtid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  __shared__ uint32_t s_lanepow[32];  // A^(2k*lane)
  __shared__ uint32_t s_fpow[32];     // F^k, k < 32
  // TMA-staged adjacency tiles: a row longer than the group's lanes but of at most kStageF * SG cumulative weights is copied
  // into the group's slice of shared memory by ONE cp.async.bulk (the elected lane issues it right after the row bounds are
  // known and the whole group goes on to derive its engine states; the draws then wait on the slice's mbarrier), and every
  // inverse-CDF search of that row is a shared-memory binary search instead of an 8-ary descent through L2.
  constexpr int kStageF = 16;
  __shared__ __align__(128) float s_stage[256 * kStageF];
  __shared__ __align__(8) unsigned long long s_bar[32];
  const int SG = 1 << a.sg_log;
  const int sl = lane & (SG - 1);                    // lane inside its group = draw index modulo SG
  const unsigned gmask = SG == 32 ? 0xffffffffu : (((1u << SG) - 1u) << (lane - sl));
  const bool can_stage = a.sg_log >= 3 && a.stage;   // <= 32 groups per CTA, slices of >= 256 B
  unsigned long long* const bar = &s_bar[can_stage ? (threadIdx.x >> a.sg_log) : 0];
  float* const sm = s_stage + (threadIdx.x - sl) * kStageF;   // this group's slice: kStageF * SG floats, 16-byte aligned
  const int64_t capg = (int64_t)SG * kStageF;
  uint32_t phase = 0;                                // parity of the slice's barrier (uniform over the group)
  if (can_stage && sl == 0) mbar_init(bar, 1);
  if (!PHILOX && threadIdx.x < 32) {
    s_lanepow[threadIdx.x] = a.lanepow[threadIdx.x];
    uint32_t fp = 1, fb = a.F;
    for (uint32_t e = threadIdx.x; e; e >>= 1) { if (e & 1) fp = modmul(fp, fb); fb = modmul(fb, fb); }
    s_fpow[threadIdx.x] = fp;
  }
  fence_mbar_init();
  __syncthreads();
  if (!PHILOX) {
    // k_prepare (the only reader of this hop's dedup tables) has finished: wipe them
    if (!a.gm.rows_act) {
      for (int64_t s = gtid; s < a.clear_n; s += (int64_t)gridDim.x * blockDim.x) { a.clear_tab[s].key = 0; a.clear_tab[s].row = kEmptyRow; }
    } else if (a.clear_n) {   // worst-case-sized regions (sharded owner): only the slots the live rows could touch
      for (int b = 0; b < a.gm.nb; ++b) {
        HashSlot* tab = a.clear_tab + (int64_t)b * (a.gm.cap_b + 1);
        const int64_t n = dedup_cap_eff(a.gm.cap_b, a.gm.rows_act, b) + 1;
        for (int64_t s = gtid; s < n; s += (int64_t)gridDim.x * blockDim.x) { tab[s].key = 0; tab[s].row = kEmptyRow; }
      }
    }
  }
  const int32_t count = a.count;
  const int32_t T = g.T;
  const int64_t total = PHILOX ? a.gm.nb * a.gm.rows_b : (int64_t)__ldg(a.n_live);   // empty rows were finished by k_prepare
  const int64_t qstride = (((int64_t)gridDim.x * blockDim.x) >> 5) << (5 - a.sg_log);
  const uint32_t upd = a.mode == 0 ? 1u : 2u;        // uniforms per draw
  const uint32_t stride = a.stride;                  // A^(2 * upd * SG): a lane's jump to its next draw

  for (int64_t q = ((gtid >> 5) << (5 - a.sg_log)) + (lane >> a.sg_log); q < total; q += qstride) {
    const int64_t w = PHILOX ? q : (int64_t)a.live[q];
    const int bidx = (int)(w / a.gm.rows_b);
    const int64_t li = w - bidx * a.gm.rows_b;
    if (PHILOX && a.gm.rows_act && li >= a.gm.rows_act[bidx]) continue;   // rows past the batch's real count do not exist
    const int64_t obase = w * (int64_t)count;
    const EuRngState* rng = a.rngs + bidx;
    HashSlot* ntab = a.next_tabs ? a.next_tabs + (int64_t)bidx * (a.next_cap_b + 1) : nullptr;
    const unsigned long long nmask = (unsigned long long)a.next_cap_b - 1;
    const int64_t nbase = li * (int64_t)count;  // index of this row's first id inside the next hop's batch

    int64_t row;
    bool ok;
    uint32_t st = 0;
    unsigned long long seed_id = 0;
    if (PHILOX) {
      seed_id = a.seeds[w];
      row = lookup_row(g, seed_id);
      ok = row_eligible(g, row, a.et, a.mode);
    } else {
      const int64_t ib = bidx * a.gm.rows_pad;
      const int32_t f = a.first[ib + li];
      const uint32_t m = a.emask[(ib + f) >> 5];
      ok = (m >> (f & 31)) & 1u;
      if (ok) {
        row = a.rowof[ib + li];
        st = modmul(modmul(rng->x_prev, a.blkmul[(int64_t)bidx * a.gm.nblk_b + f / kPrepBlock]),
                    modmul(a.wmul[(ib + f) >> 5], s_fpow[__popc(m & ((1u << (f & 31)) - 1u))]));
      } else {
        row = -1;
      }
    }
    if (!ok) {
      for (int32_t j = sl; j < count; j += SG) {
        if (a.eng_ids) a.eng_ids[obase + j] = 0ull;
        if (a.out_ids) { a.out_ids[obase + j] = a.default_node; a.out_w[obase + j] = 0.f; a.out_t[obase + j] = -1; }
      }
      if (!PHILOX && ntab && sl == 0) dedup_insert_one(ntab, nmask, 0ull, nbase);  // `count` zeros
      continue;
    }

    const int64_t* gp = g.grp_ptr + row * T;
    const int64_t base = gp[0];
    const int64_t rlen = gp[T] - base;  // whole row
    // stage the row's cumulative weights in the group's lanes when it fits
    const bool small_row = rlen <= SG;
    float c = __int_as_float(0x7f800000);  // +inf
    if (small_row && sl < rlen) c = __ldg(g.cum_w + base + sl);
    // mid row: stage [base - mis, base + rlen) rounded to 16 bytes (the copy starts at the 16-byte boundary below the row;
    // arrays are allocated in 256-byte units, so the rounded end stays inside the allocation)
    const int mis = (int)((reinterpret_cast<uintptr_t>(g.cum_w + base) & 15u) >> 2);
    const bool mid_row = can_stage && !small_row && rlen + mis <= capg;   // uniform over the group (one row per group)
    if (mid_row && sl == 0) {
      const uint32_t bytes = (uint32_t)((((rlen + mis) << 2) + 15) & ~15ll);
      fence_proxy_async_smem();        // the group's reads of the previous tile (ordered by its closing __syncwarp) before the TMA write
      mbar_arrive_expect_tx(bar, bytes);
      bulk_copy_g2s(sm, g.cum_w + base - mis, bytes, bar);
    }
    const float* const srow = sm + mis;   // srow[k] = cum_w[base + k]

    // mode 0: fixed group
    int64_t gb = 0, ge = 0;  // group [gb, ge] inclusive, global indices
    float lim_b = 0.f, lim_e = 0.f;
    if (a.mode == 0) {
      const int32_t t = a.et.v[0];
      gb = gp[t];
      ge = gp[t + 1] - 1;
      lim_b = gb == base ? 0.f : __ldg(g.cum_w + gb - 1);
      lim_e = __ldg(g.cum_w + ge);
    }
    // modes 1/2: type-pick table in the group's lanes (SG >= table size, see hop()): tc[k] = prefix over listed
    // types (1) or grp_cum (2)
    float tc = __int_as_float(0x7f800000);
    int ntc = 0;
    if (a.mode == 1) {
      ntc = a.et.K;
      float sum = 0.f, mine = 0.f;
      for (int32_t i = 0; i < ntc; ++i) {
        int32_t t = a.et.v[i];
        float pre = t > 0 ? grp_cum_at(g, row, t - 1) : 0.f;
        sum = __fadd_rn(sum, __fsub_rn(grp_cum_at(g, row, t), pre));
        if (i == sl) mine = sum;
      }
      if (sl < ntc) tc = mine;
    } else if (a.mode == 2) {
      ntc = T;
      if (sl < T) tc = grp_cum_at(g, row, sl);
    }
    const float tc_end = __shfl_sync(gmask, tc, ntc > 0 ? ntc - 1 : 0, SG);

    // engine state before this lane's first draw
    uint32_t x = 0;
    if (!PHILOX) x = modmul(st, s_lanepow[sl]);
    const uint32_t salt = PHILOX ? (uint32_t)rng->calls : 0u;
    const unsigned long long pkey = PHILOX ? a.key ^ rng->key : 0ull;

    if (mid_row) {   // the tile has landed?  (bounded: a copy that never completes is a bug, not something to wait out)
      const long long t0 = clock64();
      while (!mbar_try_wait(bar, phase))
        if (clock64() - t0 > 4000000000LL) __trap();   // ~2 s
      phase ^= 1u;
    }
    bool keep = true;
    bool bad = false;
    for (int32_t j0 = 0; j0 < count; j0 += SG) {
      const int32_t j = j0 + sl;
      const bool active = j < count;
      double u_t = 0.0, u_n = 0.0;
      if (PHILOX) {
        philox_uniform2(seed_id, (uint32_t)j, salt, pkey, u_t, u_n);
      } else {
        uint32_t xs = x;
        if (upd == 2u) u_t = minstd_uniform(xs);
        u_n = minstd_uniform(xs);
        x = modmul(x, stride);
      }
      int32_t etype = a.mode == 0 ? a.et.v[0] : 0;
      int64_t b = gb, e = ge;
      float lb = lim_b, le = lim_e;
      if (a.mode != 0) {
        // type pick: RandomSelect(sum_weights_, 0, n-1)
        const float tt = gt_threshold(pick_r(u_t, 0.f, tc_end));
        int k = lane_upper_bound(tc, 0, ntc - 1, tt, gmask, SG);
        etype = a.mode == 1 ? a.et.v[k] : k;
        b = gp[etype];
        e = gp[etype + 1] - 1;
        if (e < b) {  // zero-weight group reached through the fall-through: UB in the reference (SURVEY A-17)
          bad = bad || active;
          b = base; e = base;  // keep addresses valid
        }
        lb = b == base ? 0.f : __ldg(g.cum_w + b - 1);
        le = __ldg(g.cum_w + e);
      }
      const float thr = gt_threshold(pick_r(u_n, lb, le));
      int64_t m;
      float wgt;
      if (small_row) {
        int li2 = lane_upper_bound(c, (int)(b - base), (int)(e - base), thr, gmask, SG);
        float hi_v = __shfl_sync(gmask, c, li2, SG);
        float lo_v = __shfl_sync(gmask, c, li2 > 0 ? li2 - 1 : 0, SG);
        m = base + li2;
        wgt = __fsub_rn(hi_v, li2 > 0 ? lo_v : 0.f);
      } else if (mid_row) {
        int lo = (int)(b - base), hi = (int)(e - base);   // first index in [lo, hi] with cum >= thr, else hi
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (srow[mid] >= thr) hi = mid; else lo = mid + 1;
        }
        m = base + lo;
        wgt = __fsub_rn(srow[lo], lo > 0 ? srow[lo - 1] : 0.f);
      } else {
        m = b + upper_bound_clamped(g.cum_w + b, 0, (int32_t)(e - b), thr);
        float hi_v = __ldg(g.cum_w + m);
        float lo_v = m > base ? __ldg(g.cum_w + m - 1) : 0.f;
        wgt = __fsub_rn(hi_v, lo_v);
      }
      const unsigned long long nid = active ? __ldg(g.nbr + m) : 0ull;
      if (j0 == 0) {
        // TF packing keeps the row iff its first engine id != DEFAULT_UINT64 (0)
        unsigned long long first_id = __shfl_sync(gmask, nid, 0, SG);
        keep = first_id != 0ull;
      }
      if (active) {
        if (a.eng_ids) a.eng_ids[obase + j] = nid;
        if (a.out_ids) {
          a.out_ids[obase + j] = keep ? (long long)nid : a.default_node;
          a.out_w[obase + j] = keep ? wgt : 0.f;
          a.out_t[obase + j] = keep ? etype : -1;
        }
      }
      if (!PHILOX && ntab && a.mode == 0) {
        // mode 0 cannot hit the `bad` path: the ids are final, enter them into the next hop's dedup table now
        const unsigned act = __ballot_sync(gmask, active);
        if (active) {
          const unsigned peers = __match_any_sync(act, nid);
          if (lane == __ffs(peers) - 1) dedup_insert_one(ntab, nmask, nid, nbase + j);
        }
      }
    }
    if (__any_sync(gmask, bad)) {
      for (int32_t j = sl; j < count; j += SG) {
        if (a.eng_ids) a.eng_ids[obase + j] = 0ull;
        if (a.out_ids) { a.out_ids[obase + j] = a.default_node; a.out_w[obase + j] = 0.f; a.out_t[obase + j] = -1; }
      }
    }
    if (!PHILOX && ntab && a.mode != 0) {
      // the engine ids just written are the next hop's seeds: enter them into its dedup table now
      // (each lane re-reads its own stores), so the next hop needs no insert kernel
      for (int32_t j0 = 0; j0 < count; j0 += SG) {
        const int32_t j = j0 + sl;
        const bool active = j < count;
        const unsigned long long nid = active ? a.eng_ids[obase + j] : 0ull;
        const unsigned act = __ballot_sync(gmask, active);
        if (active) {
          const unsigned peers = __match_any_sync(act, nid);
          if (lane == __ffs(peers) - 1) dedup_insert_one(ntab, nmask, nid, nbase + j);
        }
      }
    }
    if (mid_row) __syncwarp(gmask);   // every lane is done with the tile before the group's next row overwrites it
  }
}

__global__ void k_bump_calls(EuRngState* rngs, int nb) {
  if (threadIdx.x < nb) rngs[threadIdx.x].calls += 1;
}

// ---------------------------------------------------------------------------- global node sampler
struct NodeSamplerDev {
  int32_t n_types;
  const unsigned long long* ids[EU_MAX_ETYPES];
  const float* prob[EU_MAX_ETYPES];
  const int32_t* alias[EU_MAX_ETYPES];
  long long n[EU_MAX_ETYPES];
  const float* type_prob;
  const int32_t* type_alias;
  // mode 0: single type `type0`; 1: all types (alias over types); 2: CWC over listed types
  int mode;
  int32_t type0;
  int32_t n_sub;
  int32_t sub_ids[EU_MAX_ETYPES];
  float sub_cum[EU_MAX_ETYPES];
};

// AliasMethod::Next (alias_method.cc:66-78): column = floor(n*U1); U2 < prob[column] ? column : alias
__device__ __forceinline__ long long alias_next(const float* prob, const int32_t* alias, long long n,
                                                double u1, double u2) {
  long long col = (long long)floor(__dmul_rn((double)n, u1));
  bool coin = u2 < (double)__ldg(prob + col);
  return coin ? col : (long long)__ldg(alias + col);
}

template <bool PHILOX>
__global__ void k_sample_node(NodeSamplerDev s, int32_t count, int32_t upd, unsigned long long key,
                              EuRngState* rng, long long* out) {
  const int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < count) {
    double u[4] = {0, 0, 0, 0};
    if (PHILOX) {
      philox_uniform2(0x5A4D504C45ull, (uint32_t)j, (uint32_t)rng->calls, key, u[0], u[1]);
      philox_uniform2(0x5A4D504C46ull, (uint32_t)j, (uint32_t)rng->calls, key, u[2], u[3]);
      if (s.mode == 0) { u[2] = u[0]; u[3] = u[1]; }  // keep "node pick" in u[2],u[3]
    } else {
      uint32_t x = modmul(rng->x, modpow_a(2ull * upd * (unsigned long long)j));
      if (s.mode == 1) { u[0] = minstd_uniform(x); u[1] = minstd_uniform(x); }
      if (s.mode == 2) { u[0] = minstd_uniform(x); }
      u[2] = minstd_uniform(x);
      u[3] = minstd_uniform(x);
    }
    int32_t t = s.type0;
    if (s.mode == 1) {
      t = (int32_t)alias_next(s.type_prob, s.type_alias, s.n_types, u[0], u[1]);
    } else if (s.mode == 2) {
      double r = pick_r(u[0], 0.f, s.sub_cum[s.n_sub - 1]);
      int k = 0;
      while (k < s.n_sub - 1 && !((double)s.sub_cum[k] > r)) ++k;
      t = s.sub_ids[k];
    }
    long long col = alias_next(s.prob[t], s.alias[t], s.n[t], u[2], u[3]);
    out[j] = (long long)__ldg(s.ids[t] + col);
  }
}

__global__ void k_advance_engine(EuRngState* rng, unsigned long long uniforms) {
  rng->x = modmul(rng->x, modpow_a(2ull * uniforms));
  rng->draws += uniforms;
  rng->calls += 1;
}

// ---------------------------------------------------------------------------- host side
// engine-state scan over c->d_elig[0..rows): c->d_state[i] = state before row i's first draw
int launch_state_scan(eu_ctx* c, int64_t rows, unsigned long long uniforms_per_row) {
  k_state_scan<<<1, 1024, 0, c->stream>>>(c->d_elig, rows, modpow_a(2ull * uniforms_per_row), uniforms_per_row,
                                          c->d_state, c->d_rng);
  EU_LAUNCHED();
  return EU_OK;
}

static int classify(const DevGraph& d, const int32_t* etypes, int32_t K, ETypes* et, int* mode) {
  if (K < 0 || K > EU_MAX_ETYPES) { set_error("edge_types: K=%d unsupported (max %d)", K, EU_MAX_ETYPES); return EU_ERR_UNSUPPORTED; }
  et->K = K;
  for (int i = 0; i < K; ++i) et->v[i] = etypes[i];
  // node.cc:106-148: K==1 -> that group; 1<K<T -> sub collection; K==0 or K>=T -> all groups
  if (K == 1) *mode = 0;
  else if (K > 1 && K < d.T) *mode = 1;
  else *mode = 2;
  return EU_OK;
}

static Geom make_geom(int nb, int64_t rows_b) {
  Geom gm{};
  gm.nb = nb;
  gm.rows_b = rows_b;
  gm.nblk_b = (int32_t)ceil_div(rows_b > 0 ? rows_b : 1, kPrepBlock);
  gm.rows_pad = (int64_t)gm.nblk_b * kPrepBlock;
  gm.cap_b = 64;
  while (gm.cap_b < rows_b * 2) gm.cap_b <<= 1;
  gm.rows_act = nullptr;
  return gm;
}

// scratch needed by a hop over nb batches of rows_b seeds (see ctx_reserve)
int64_t hop_scratch_rows(int nb, int64_t rows_b) { return make_geom(nb, rows_b).rows_pad * nb; }
int64_t hop_table_slots(int nb, int64_t rows_b) { return (make_geom(nb, rows_b).cap_b + 1) * nb; }
int64_t hop_table_cap(int64_t rows_b) { return make_geom(1, rows_b).cap_b; }

// One sampleNB hop over nb batches: seeds (device u64[nb*rows_b]) -> engine ids (device u64[nb*rows_b*count], may
// be null) and TF-packed outputs (may be null).  Batch b uses engine b of the ctx.
int hop(eu_ctx* c, const unsigned long long* seeds, int64_t rows_b, const int32_t* etypes,
        int32_t K, int32_t count, int64_t default_node, unsigned long long* eng_ids,
        int64_t* out_ids, float* out_w, int32_t* out_t, int hop_index, bool pre_inserted, bool insert_next, int nb,
        const int32_t* rows_act, bool raw) {
  const int64_t rows = rows_b * nb;
  if (rows == 0 || count == 0) return EU_OK;
  if (nb < 1 || nb > c->n_eng) { set_error("hop: %d batches but the ctx has %d engines", nb, c->n_eng); return EU_ERR_INVALID; }
  const DevGraph& d = c->g->d;
  SampleArgs a{};
  int rc = classify(d, etypes, K, &a.et, &a.mode);
  if (rc) return rc;
  if (a.mode != 0 && d.T > 32) { set_error("T > 32 unsupported"); return EU_ERR_UNSUPPORTED; }
  cudaStream_t s = c->stream;
  Geom gm = make_geom(nb, rows_b);
  gm.rows_act = rows_act;
  a.seeds = seeds; a.gm = gm; a.count = count; a.default_node = default_node;
  a.eng_ids = eng_ids; a.out_ids = (long long*)out_ids; a.out_w = out_w; a.out_t = out_t;
  a.rngs = c->d_rng;
  // lanes per row: the smallest power of two that holds a row's draws (and the type-pick table of modes 1/2)
  {
    int need = std::min<int>(count, 32);
    if (a.mode == 1) need = std::max<int>(need, std::min<int>(a.et.K, 32));
    if (a.mode == 2) need = std::max<int>(need, std::min<int>(d.T, 32));
    a.sg_log = 0;
    while ((1 << a.sg_log) < need) ++a.sg_log;
  }
  // persistent grid: 8 CTAs per SM stride over the (live) rows.  EU_SAMPLE_CTAS = CTAs per SM (1..8; 6 also relaxes the
  // register cap); read once (C++11 static initialisation is thread-safe: the ABI is re-entrant across ctxs)
  static const int stage_rows = [] { const char* e = getenv("EU_SAMPLE_STAGE"); return e ? (atoi(e) != 0 ? 1 : 0) : 1; }();
  a.stage = stage_rows;
  static const int grid_ctas = [] { const char* e = getenv("EU_SAMPLE_CTAS"); return e ? std::min(8, std::max(1, atoi(e))) : 8; }();
  const int ctas = grid_ctas == 6 ? 6 : 8;
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(ceil_div(rows * 32, (int64_t)(32 >> a.sg_log)), 256), 148 * grid_ctas);
  if (c->rng == EU_RNG_PHILOX) {
    a.key = c->seed;
    { EuProfScope ps(c, "k_sample<philox>", rows); if (ctas == 6) k_sample<true, 6><<<blocks, 256, 0, s>>>(d, a); else k_sample<true, 8><<<blocks, 256, 0, s>>>(d, a); }
    EU_LAUNCHED();
    k_bump_calls<<<1, 64, 0, s>>>(c->d_rng, nb);
    EU_LAUNCHED();
    return EU_OK;
  }
  if (rows >= ((int64_t)1 << 31) || nb > 64) { set_error("rows >= 2^31 or more than 64 batches"); return EU_ERR_UNSUPPORTED; }
  const Geom ng = make_geom(nb, rows_b * count);  // next hop's geometry (its seeds = this hop's engine ids)
  const bool chain = insert_next && eng_ids;
  rc = ctx_reserve(c, std::max(gm.rows_pad, chain ? ng.rows_pad : 0) * nb, (std::max(gm.cap_b, chain ? ng.cap_b : 0) + 1) * nb);
  if (rc) return rc;
  const int tb = kPrepBlock;
  // Two table sets, hop l uses set l & 1; batch b owns region b (stride cap_b + 1) of a set.  Invariant: both
  // sets are all-free when an op starts (cleared at allocation; every k_sample wipes its own hop's regions once
  // k_prepare has consumed them).  The seeds of hop l+1 are entered into the other set by hop l's k_sample
  // (pre_inserted), so only the first hop of a chain needs the insert kernel.
  HashSlot* tabs = c->d_dedup + (hop_index & 1) * c->tab_set_slots;
  HashSlot* ntabs = c->d_dedup + ((hop_index + 1) & 1) * c->tab_set_slots;
  if (raw && (pre_inserted || insert_next)) { set_error("hop: raw mode does not chain"); return EU_ERR_INVALID; }
  if (!pre_inserted && !raw) {
    EuProfScope ps(c, "k_dedup_insert", rows);
    k_dedup_insert<<<dim3((unsigned)ceil_div(gm.rows_b, tb), (unsigned)nb), tb, 0, s>>>(tabs, gm, seeds);
    EU_LAUNCHED();
  }
  const unsigned long long upr = (unsigned long long)count * (a.mode == 0 ? 1 : 2);
  const uint32_t F = modpow_a(2ull * upr);
  { EuProfScope ps(c, "k_prepare", rows);
    PrepOut po{};
    po.eng_ids = eng_ids; po.out_ids = (long long*)out_ids; po.out_w = out_w; po.out_t = out_t;
    po.count = count; po.default_node = default_node;
    if (chain) { po.next_tabs = ntabs; po.next_cap_b = ng.cap_b; }
    po.live = c->d_live; po.n_live = c->d_nlive;
    EU_CUDA(cudaMemsetAsync(c->d_nlive, 0, sizeof(unsigned int), s));
    k_prepare<<<dim3((unsigned)gm.nblk_b, (unsigned)nb), tb, 0, s>>>(d, raw ? nullptr : tabs, gm, seeds, a.et, a.mode, F, upr, c->d_first,
                                                                     c->d_rowof, c->d_emask, c->d_woff, c->d_blkpre, c->d_blkmul,
                                                                     c->d_rng, po); }
  EU_LAUNCHED();
  a.first = c->d_first; a.rowof = c->d_rowof; a.emask = c->d_emask; a.wmul = c->d_woff; a.blkmul = c->d_blkmul;
  a.live = c->d_live; a.n_live = c->d_nlive;
  a.F = F;
  const uint32_t upd = a.mode == 0 ? 1u : 2u;
  for (uint32_t k = 0; k < 32; ++k) a.lanepow[k] = modpow_a(2ull * upd * k);
  a.stride = modpow_a(2ull * upd * (unsigned long long)(1u << a.sg_log));
  a.clear_tab = tabs;
  a.clear_n = raw ? 0 : (gm.cap_b + 1) * nb;   // raw mode never touched the dedup tables
  if (chain) {
    a.next_tabs = ntabs;
    a.next_cap_b = ng.cap_b;
  }
  { EuProfScope ps(c, "k_sample<minstd>", rows); if (ctas == 6) k_sample<false, 6><<<blocks, 256, 0, s>>>(d, a); else k_sample<false, 8><<<blocks, 256, 0, s>>>(d, a); }
  EU_LAUNCHED();
  return EU_OK;
}

// The hop chain of a fanout over nb batches.  levels == null: the engine ids of hops 0..L-2 live in the ping-pong frontier only.
// Otherwise hop l writes its engine ids, the last hop's included, to levels + (rows of hops 0..l-1): the caller keeps every
// level's frontier (d_levels, sized by the caller).
static int fanout_chain(eu_ctx* c, const int64_t* nodes, int32_t nb, int64_t B, const int32_t* etypes, int32_t K,
                        const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids, float* const* out_w,
                        int32_t* const* out_t, unsigned long long* levels) {
  // a hop with count 0 delivers nothing and neither does any hop after it: stop the chain BEFORE it, so that no hop enters
  // ids into a dedup table that nobody would consume and wipe (the tables must be all-free when an op returns)
  for (int l = 0; l < L; ++l)
    if (counts[l] == 0) { L = l; break; }
  if (B == 0) return EU_OK;
  int64_t rows_b = B, max_rows = hop_scratch_rows(nb, B), max_slots = hop_table_slots(nb, B), widest = B * nb;
  for (int l = 0; l < L; ++l) {
    rows_b *= counts[l];
    if (l + 1 < L) { max_rows = std::max(max_rows, hop_scratch_rows(nb, rows_b)); max_slots = std::max(max_slots, hop_table_slots(nb, rows_b)); }
    widest = std::max(widest, rows_b * nb);
  }
  int rc = ctx_reserve(c, std::max(max_rows, widest), max_slots);
  if (rc) return rc;
  const unsigned long long* seeds = (const unsigned long long*)nodes;
  rows_b = B;
  for (int l = 0; l < L; ++l) {
    unsigned long long* eng = levels ? levels : (l + 1 < L) ? c->d_front[l & 1] : nullptr;
    rc = hop(c, seeds, rows_b, etypes + (int64_t)l * K, K, counts[l], default_node, eng,
             out_ids ? out_ids[l] : nullptr, out_w ? out_w[l] : nullptr, out_t ? out_t[l] : nullptr,
             l, /*pre_inserted=*/l > 0 && c->rng == EU_RNG_MINSTD, /*insert_next=*/l + 1 < L, nb);
    if (rc) return rc;
    seeds = eng;
    rows_b *= counts[l];
    if (levels) levels += rows_b * nb;
  }
  return EU_OK;
}

}  // namespace eu

using namespace eu;

extern "C" {

int eu_sample_neighbor(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                       int32_t count, int64_t default_node, int64_t* out_ids, float* out_w,
                       int32_t* out_t) {
  if (!c || B < 0 || count < 0 || (K > 0 && !etypes)) { set_error("eu_sample_neighbor: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  return hop(c, (const unsigned long long*)nodes, B, etypes, K, count, default_node, nullptr, out_ids, out_w, out_t, 0, false, false, 1);
}

// euler::SampleNeighbor (euler/core/api/api.cc:223-236): one Node::SampleNeighbor per element of node_ids, in order --
// NO unique / gather (that is the engine's rule, euler/parser/compiler.cc:76-90, which the op entry points above apply):
// a repeated id draws again and consumes its own uniforms.  Engine-form outputs: a row that has no result (absent node, no
// edge of the requested types) is `count` x (0, 0.0, -1); out_ids is what api.cc callers get as std::get<0>.
int eu_sample_neighbor_raw(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                           int32_t count, int64_t* out_ids, float* out_w, int32_t* out_t) {
  if (!c || B < 0 || count < 0 || (K > 0 && !etypes)) { set_error("eu_sample_neighbor_raw: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (c->rng != EU_RNG_MINSTD) { set_error("eu_sample_neighbor_raw: exact-RNG contexts only (philox rows are keyed on the node id: duplicates would repeat)"); return EU_ERR_UNSUPPORTED; }
  return hop(c, (const unsigned long long*)nodes, B, etypes, K, count, /*default_node=*/0, nullptr, out_ids, out_w, out_t, 0, false, false, 1,
             nullptr, /*raw=*/true);
}

int eu_sample_fanout_batched(eu_ctx* c, const int64_t* nodes, int32_t nb, int64_t B, const int32_t* etypes, int32_t K,
                             const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                             float* const* out_w, int32_t* const* out_t) {
  if (!c || nb < 1 || B < 0 || L < 0 || !counts || (K > 0 && !etypes)) { set_error("eu_sample_fanout: bad argument"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  if (nb > c->n_eng) { set_error("eu_sample_fanout_batched: %d batches but the ctx has %d engines (eu_ctx_set_engines)", nb, c->n_eng); return EU_ERR_INVALID; }
  for (int l = 0; l < L; ++l)
    if (counts[l] < 0) { set_error("negative count"); return EU_ERR_INVALID; }
  return fanout_chain(c, nodes, nb, B, etypes, K, counts, L, default_node, out_ids, out_w, out_t, nullptr);
}

int eu_sample_fanout(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                     const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                     float* const* out_w, int32_t* const* out_t) {
  return eu_sample_fanout_batched(c, nodes, 1, B, etypes, K, counts, L, default_node, out_ids, out_w, out_t);
}

// tf_euler.sample_fanout_with_feature (tf_euler/kernels/sample_fanout_with_feature_op.cc): the sample_fanout chain (:59-64), then
// the features of every level's ENGINE ids (v_select(nb_i), :65-68).  Level 0 is `nodes` as given; a default-filled slot of a
// later level has no node (engine id 0), so it gets zeros and the sparse default whatever default_node is.
int eu_sample_fanout_with_feature(eu_ctx* c, const int64_t* nodes, int64_t B, const int32_t* etypes, int32_t K,
                                  const int32_t* counts, int32_t L, int64_t default_node, int64_t* const* out_ids,
                                  float* const* out_w, int32_t* const* out_t, int32_t ND, const int32_t* dense_fids,
                                  const int32_t* dense_dims, float* const* out_dense, int32_t NS, const int32_t* sparse_fids,
                                  const int64_t* sparse_defaults, int64_t* const* out_sp_ptr, int64_t* const* out_sp_val) {
  if (!c || B < 0 || L < 0 || L > 16 || ND < 0 || NS < 0 || (L > 0 && !counts) || (K > 0 && !etypes) || (B > 0 && !nodes) ||
      (ND > 0 && (!dense_fids || !dense_dims || !out_dense)) ||
      (NS > 0 && (!sparse_fids || !sparse_defaults || !out_sp_ptr || !out_sp_val))) {
    set_error("eu_sample_fanout_with_feature: bad argument");
    return EU_ERR_INVALID;
  }
  if ((int64_t)(L + 1) * ND > kMaxFeatSegs || (int64_t)(L + 1) * NS > kMaxFeatSegs) {
    set_error("eu_sample_fanout_with_feature: (L+1)*ND = %d and (L+1)*NS = %d, at most %d each", (L + 1) * ND, (L + 1) * NS, kMaxFeatSegs);
    return EU_ERR_UNSUPPORTED;
  }
  for (int l = 0; l < L; ++l)
    if (counts[l] < 0) { set_error("negative count"); return EU_ERR_INVALID; }
  for (int j = 0; j < ND; ++j)
    if (dense_dims[j] < 0) { set_error("negative dense dimension"); return EU_ERR_INVALID; }
  EU_CUDA(cudaSetDevice(c->g->device));
  int64_t rows[17];
  rows[0] = B;
  for (int l = 0; l < L; ++l) rows[l + 1] = rows[l] * counts[l];
  int64_t level_ids = 0;
  for (int l = 1; l <= L; ++l) level_ids += rows[l];
  int rc = ctx_levels(c, level_ids);
  if (rc) return rc;
  rc = fanout_chain(c, nodes, 1, B, etypes, K, counts, L, default_node, out_ids, out_w, out_t, c->d_levels);
  if (rc) return rc;
  const unsigned long long* lv[17];
  lv[0] = (const unsigned long long*)nodes;
  for (int l = 1; l <= L; ++l) lv[l] = l == 1 ? c->d_levels : lv[l - 1] + rows[l - 1];
  if (ND > 0) {
    DenseSeg segs[kMaxFeatSegs];
    for (int i = 0; i <= L; ++i)
      for (int j = 0; j < ND; ++j) segs[i * ND + j] = DenseSeg{lv[i], rows[i], dense_fids[j], dense_dims[j], out_dense[i * ND + j]};
    if ((rc = dense_feature_segments(c, segs, (L + 1) * ND))) return rc;
  }
  if (NS > 0) {
    SparseSeg segs[kMaxFeatSegs];
    for (int i = 0; i <= L; ++i)
      for (int j = 0; j < NS; ++j) {
        const int64_t cap = rows[i] * std::max<int64_t>(1, eu_graph_sparse_feature_max_len(c->g, sparse_fids[j]));
        segs[i * NS + j] = SparseSeg{lv[i], rows[i], sparse_fids[j], sparse_defaults[j], cap, out_sp_ptr[i * NS + j], out_sp_val[i * NS + j]};
      }
    if ((rc = sparse_feature_segments(c, segs, (L + 1) * NS))) return rc;
  }
  return EU_OK;
}

int eu_sample_node(eu_ctx* c, int32_t count, const int32_t* types, int32_t n_types, int64_t* out) {
  if (!c || count < 0 || n_types < 1 || !types) { set_error("eu_sample_node: bad argument"); return EU_ERR_INVALID; }
  eu_graph* g = c->g;
  EU_CUDA(cudaSetDevice(g->device));
  int rc = graph_build_sampler(g);
  if (rc) return rc;
  const int32_t NT = g->d.n_node_types;
  if (NT > EU_MAX_ETYPES) { set_error("more than %d node types", EU_MAX_ETYPES); return EU_ERR_UNSUPPORTED; }
  NodeSamplerDev s{};
  s.n_types = NT;
  for (int t = 0; t < NT; ++t) {
    s.ids[t] = g->samplers[t].ids; s.prob[t] = g->samplers[t].prob; s.alias[t] = g->samplers[t].alias;
    s.n[t] = g->samplers[t].n;
  }
  s.type_prob = g->d_type_prob; s.type_alias = g->d_type_alias;
  uint32_t upd;
  // api.cc:32-37 dispatch; Graph::SampleNode graph.cc:221-275.  Empty result == reference returns
  // an empty vector (the TF kernel then aborts with "SampleNode Result Size 0", sample_node_op.cc:83-86).
  if (n_types == 1) {
    int32_t t = types[0];
    if (t == -1) {
      if (g->type_fwc_sum == 0.f) { set_error("sample_node: total node weight is 0"); return EU_ERR_STATE; }
      s.mode = 1; upd = 4;
    } else {
      if (t < 0 || t >= NT) { set_error("sample_node: node type %d out of range", t); return EU_ERR_INVALID; }
      if (g->samplers[t].fwc_sum == 0.f) { set_error("sample_node: node type %d is empty", t); return EU_ERR_STATE; }
      s.mode = 0; s.type0 = t; upd = 2;
    }
  } else {
    s.mode = 2; upd = 3;
    float sum = 0.f;
    for (int t = 0; t < NT; ++t) {
      bool in = false;
      for (int k = 0; k < n_types; ++k) in |= types[k] == t;
      if (in) { sum += g->type_sums[t]; s.sub_ids[s.n_sub] = t; s.sub_cum[s.n_sub] = sum; ++s.n_sub; }
    }
    if (!(sum > 0)) { set_error("sample_node: listed node types are empty"); return EU_ERR_STATE; }
  }
  if (count == 0) return EU_OK;
  const unsigned blocks = (unsigned)ceil_div(count, 256);
  if (c->rng == EU_RNG_PHILOX)
    k_sample_node<true><<<blocks, 256, 0, c->stream>>>(s, count, upd, c->seed, c->d_rng, (long long*)out);
  else
    k_sample_node<false><<<blocks, 256, 0, c->stream>>>(s, count, upd, c->seed, c->d_rng, (long long*)out);
  EU_LAUNCHED();
  k_advance_engine<<<1, 1, 0, c->stream>>>(c->d_rng, (unsigned long long)upd * (unsigned long long)count);
  EU_LAUNCHED();
  return EU_OK;
}

}  // extern "C"
