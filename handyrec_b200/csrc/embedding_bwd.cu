// embedding_bwd.cu -- a13, the embedding backward of a whole feature group as a two-level radix partition whose second
// level is fused with the segmented reduction and the row update (no global sort, no atomics on gradients, deterministic).
//
// Reference arithmetic replaced: TF autodiff of CustomEmbedding / SequencePoolingLayer (layers/tools.py:87-101,
// layers/sequence.py:26-46): dW[r,:] = sum over the positions that looked row r up of the upstream gradient (IndexedSlices,
// de-duplicated inside the Keras optimisers) followed by the optimiser's row update; features/group.py:289 adds 2*l2*W.
//
// Design (B200: 148 SMs, 227 KB shared memory per SM, the id matrix of a batch lives in the 126 MB L2):
//   level 1  every table is cut into power-of-two row ranges ("units", bin = id >> shift) sized so that a uniform batch puts
//            between 45 % and 90 % of UB_CAP = 4096 positions into each.  bwd_prep_kernel transposes the id matrix (invalid /
//            padding ids -> 0xFFFFFFFF), split_count / split_scan / split_scatter are ONE stable counting pass: positions
//            are moved, in (column, sample) order, into one contiguous list per unit -- (row inside the unit, packed
//            position).  Ranks come from __match_any_sync + per-warp shared-memory counters: integer work only.
//   level 2  bwd_unit_kernel: ONE CTA owns a unit, i.e. it is the only writer of those rows.  It loads the unit's list
//            (coalesced), sorts the <= 4096 (row, position) pairs in shared memory (stable block radix sort over `shift` bits
//            only) and walks the sorted list warp by warp with a segmented shuffle scan: the upstream gradient rows are
//            gathered straight from dout (128-bit loads, U*E rows in flight per warp), equal rows are summed in list order
//            (fixed order -> bit-reproducible), and each finished run updates its row once (SGD / lazy Adam / add into the
//            dense gradient buffer of a dense-updated table).
//   skew     (Zipf ids, tiny tables) a list longer than 4096 is split by a 64-bin histogram of its row range; the bins are
//            dealt out by count quantiles to the unit's UB_HELPERS CTAs (helper CTAs of ordinary units exit at once), each of
//            which splits its share again until a pass fits; a single row with more than 4096 positions is reduced by all
//            lanes of a CTA in list order; rows the host already knows to be that hot (tables with fewer rows than units)
//            are split over slices of their list whose partial sums bwd_unit_combine_kernel adds in slice order.
// HBM/L2 traffic per step = ids twice + positions written and read once (16 B per position) + every upstream gradient row
// once + every touched table row once (read-modify-write): the algorithmic bytes of SURVEY 8(d) plus 24 B per position.
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include <stdlib.h>

#include <algorithm>
#include <new>
#include <vector>

#include "plan.cuh"

namespace hrb {

constexpr int UB_THREADS = 256;
constexpr int UB_IPT = 16;
constexpr int UB_CAP = UB_THREADS * UB_IPT;  // positions one pass sorts in shared memory
constexpr int UB_EXPECT_MAX = 3686;          // 0.9 * UB_CAP: expected positions per unit under uniform ids lie in (max/2, max]
constexpr int UB_MAX_COLS = 256;
constexpr int UB_MAX_BINS = 256;             // units per table
constexpr int UB_BINS = 64;
constexpr int UB_STACK = 256;
constexpr int UB_WARPS = UB_THREADS / 32;
constexpr int UB_HELPERS = 4;                // CTAs per unit; all but the first only work when the unit overflows
constexpr int UB_TILE = 4096;                // samples per split tile
constexpr int SPLIT_ROUNDS = UB_TILE / UB_WARPS / 32;  // rounds of 32 samples a warp of the split kernel walks
constexpr uint32_t UB_INVALID = 0xFFFFFFFFu;
constexpr uint32_t UB_NONE = 0xFFFFFFFEu;
constexpr int UB_SLICE_TARGET = 4096;        // positions per slice of a row the host knows to be hot
constexpr int UB_PARTIAL_LD = 32 * 4 + 4;
constexpr int UB_GATHER = 8;                 // warp batches whose gradient rows are in flight together
constexpr int UB_APPLY = 2;                  // row updates a lane group has in flight together

static inline size_t ub_align(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ids[B, ids_ld] -> idsT[pos_cols][ldT] (invalid, padding and out-of-range ids become UB_INVALID; so does the tail b >= batch)
__global__ void __launch_bounds__(256) bwd_prep_kernel(const FieldDev* __restrict__ fields, const int32_t* __restrict__ pos_field,
                                                      int32_t pos_cols, const int32_t* __restrict__ ids, int64_t ids_ld, int64_t batch,
                                                      int64_t ldT, uint32_t* __restrict__ idsT) {
  __shared__ uint32_t tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t b0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int c = c0 + tx;
  int ids_col = 0, pool = 0;
  int64_t rows = 0;
  if (c < pos_cols) {
    const FieldDev& f = fields[pos_field[c]];
    ids_col = f.ids_col + (c - f.pos_col);
    pool = f.pool;
    rows = f.rows;
  }
  for (int r = ty; r < 32; r += 8) {
    const int64_t b = b0 + r;
    uint32_t v = UB_INVALID;
    if (b < batch && c < pos_cols) {
      const int32_t id = ids[b * ids_ld + ids_col];
      const bool valid = (pool == HRB_POOL_NONE || id != 0) && id >= 0 && (int64_t)id < rows;
      if (valid) v = (uint32_t)id;
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int cc = c0 + r;
    const int64_t b = b0 + tx;
    if (cc < pos_cols && b < ldT) idsT[(int64_t)cc * ldT + b] = tile[tx][r];
  }
}

// 1/n_valid per (sample, mean-pooled field), 1 elsewhere (sequence.py:43-46)
__global__ void __launch_bounds__(256) bwd_scale_kernel(const FieldDev* __restrict__ fields, int32_t n_fields,
                                                       const int32_t* __restrict__ ids, int64_t ids_ld, int64_t batch,
                                                       float* __restrict__ scale) {
  const int64_t total = batch * n_fields;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_fields;
    const int fi = (int)(i - b * n_fields);
    const FieldDev& f = fields[fi];
    float s = 1.0f;
    if (f.pool == HRB_POOL_MEAN) {
      const int32_t* idp = ids + b * ids_ld + f.ids_col;
      int cnt = 0;
      for (int l = 0; l < f.seq_len; ++l) {
        const int32_t id = idp[l];
        cnt += (id != 0 && id >= 0 && (int64_t)id < f.rows);
      }
      s = cnt > 0 ? __fdiv_rn(1.0f, (float)cnt) : 0.f;
    }
    scale[i] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// level 1: one stable counting pass that groups the positions of every table by unit (bin = id >> shift)
// ---------------------------------------------------------------------------------------------------------------------
struct SplitArgs {
  const TableSplitDev* splits;
  const TileDev* tiles;
  const uint32_t* idsT;
  int64_t ldT;
  uint32_t* tile_cnt;   // [n_tiles][UB_MAX_BINS]: positions of (tile, bin), then their first slot in the entry arrays
  uint32_t* list_cnt;   // [n_lists]
  uint32_t* list_off;   // [n_lists]
  uint32_t* ent_row;    // row inside the unit
  uint32_t* ent_pos;    // (local column << 24) | sample
};

// warp w of the CTA walks samples [chunk*4096 + w*512, +512) of the tile's column in SPLIT_ROUNDS rounds of 32 (coalesced)
template <bool SCATTER>
__global__ void __launch_bounds__(UB_THREADS) split_kernel(SplitArgs a) {
  __shared__ uint32_t wcnt[UB_WARPS][UB_MAX_BINS];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const TileDev tile = a.tiles[blockIdx.x];
  const TableSplitDev ts = a.splits[tile.table];
  for (int i = tid; i < UB_WARPS * UB_MAX_BINS; i += UB_THREADS) (&wcnt[0][0])[i] = 0;
  __syncthreads();
  const uint32_t* colp = a.idsT + (int64_t)tile.pos_col * a.ldT;
  const int64_t b0 = (int64_t)tile.chunk * UB_TILE + w * (UB_TILE / UB_WARPS);
  uint32_t packed[SPLIT_ROUNDS];  // SCATTER: (bin << 16) | rank inside (warp, bin)
  uint32_t idv[SPLIT_ROUNDS];     // all rounds' ids are fetched up front: one L2 round trip instead of one per round
#pragma unroll
  for (int k = 0; k < SPLIT_ROUNDS; ++k) {
    const int64_t b = b0 + k * 32 + lane;
    idv[k] = b < a.ldT ? __ldg(colp + b) : UB_INVALID;
  }
#pragma unroll
  for (int k = 0; k < SPLIT_ROUNDS; ++k) {
    const uint32_t id = idv[k];
    const uint32_t bin = id == UB_INVALID ? UB_INVALID : id >> ts.shift;
    const uint32_t peers = __match_any_sync(0xffffffffu, bin);
    const int leader = __ffs(peers) - 1;
    uint32_t base = 0;
    if (bin != UB_INVALID && lane == leader) {
      base = wcnt[w][bin];
      wcnt[w][bin] = base + __popc(peers);
    }
    if (SCATTER) {
      base = __shfl_sync(0xffffffffu, base, leader);
      packed[k] = bin == UB_INVALID ? UB_INVALID : (bin << 16) | (base + __popc(peers & ((1u << lane) - 1u)));
    }
    __syncwarp();
  }
  __syncthreads();
  uint32_t* tc = a.tile_cnt + (size_t)blockIdx.x * UB_MAX_BINS;
  if (!SCATTER) {
    for (int u = tid; u < ts.n_bins; u += UB_THREADS) {
      uint32_t t = 0;
#pragma unroll
      for (int ww = 0; ww < UB_WARPS; ++ww) t += wcnt[ww][u];
      tc[u] = t;
    }
    return;
  }
  for (int u = tid; u < ts.n_bins; u += UB_THREADS) {  // first slot of (warp, bin): tile offset + the warps before
    uint32_t run = tc[u];
#pragma unroll
    for (int ww = 0; ww < UB_WARPS; ++ww) {
      const uint32_t t = wcnt[ww][u];
      wcnt[ww][u] = run;
      run += t;
    }
  }
  __syncthreads();
  const uint32_t mask = (1u << ts.shift) - 1u;
#pragma unroll
  for (int k = 0; k < SPLIT_ROUNDS; ++k) {
    if (packed[k] == UB_INVALID) continue;
    const int64_t b = b0 + k * 32 + lane;
    const uint32_t id = idv[k];
    const uint32_t dst = wcnt[w][packed[k] >> 16] + (packed[k] & 0xFFFFu);
    a.ent_row[dst] = id & mask;
    a.ent_pos[dst] = ((uint32_t)tile.col_local << 24) | (uint32_t)b;
  }
}

// one CTA per table: exclusive scan of the tile counts per bin (tiles in (column, chunk) order) and of the bin totals
__global__ void __launch_bounds__(UB_MAX_BINS) split_scan_kernel(SplitArgs a) {
  __shared__ uint32_t tot[UB_MAX_BINS];
  const TableSplitDev ts = a.splits[blockIdx.x];
  const int u = threadIdx.x;
  uint32_t run = 0;
  if (u < ts.n_bins) {
    for (int t = 0; t < ts.n_tiles; ++t) {
      uint32_t* p = a.tile_cnt + (size_t)(ts.first_tile + t) * UB_MAX_BINS + u;
      const uint32_t c = *p;
      *p = run;
      run += c;
    }
  }
  tot[u] = u < ts.n_bins ? run : 0;
  __syncthreads();
  for (int off = 1; off < UB_MAX_BINS; off <<= 1) {  // inclusive Hillis-Steele scan over the bins
    const uint32_t v = u >= off ? tot[u - off] : 0;
    __syncthreads();
    tot[u] += v;
    __syncthreads();
  }
  if (u < ts.n_bins) {
    const uint32_t base = ts.ent_base + tot[u] - run;
    a.list_cnt[ts.first_list + u] = run;
    a.list_off[ts.first_list + u] = base;
    for (int t = 0; t < ts.n_tiles; ++t) a.tile_cnt[(size_t)(ts.first_tile + t) * UB_MAX_BINS + u] += base;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// level 2: the unit kernel
// ---------------------------------------------------------------------------------------------------------------------
struct UnitArgs {
  const UnitDev* units;
  const TableDev* tables;
  const ColDev* cols;
  const int32_t* col_start;
  const uint32_t* list_cnt;
  const uint32_t* list_off;
  const uint32_t* ent_row;
  const uint32_t* ent_pos;
  const float* dout;
  int64_t dout_ld;
  const float* scale;  // nullptr: no mean-pooled field in the plan
  int32_t n_fields;
  int32_t n_units;     // units of this launch (grid = n_units * UB_HELPERS)
  hrb_opt_params opt;
  float lr_t;
  float* partials;     // [n_partials][UB_PARTIAL_LD]: slice sums of host-known hot rows (+ position count)
  int32_t debug;       // -DHRB_DEVTOOLS builds only (HRB_BWD_DEBUG): 1 no sort, 2 no row updates, 4 no gradient gathers
};
#ifdef HRB_DEVTOOLS
#define HRB_UDBG(b) (a.debug & (b))
#else
#define HRB_UDBG(b) 0
#endif

template <int G>
struct UnitSmem {
  typedef cub::BlockRadixSort<uint32_t, UB_THREADS, UB_IPT, uint32_t> Sort;
  uint32_t row[UB_CAP];
  uint32_t pos[UB_CAP];  // (local column << 24) | sample
  union {
    typename Sort::TempStorage sort;
    float4 red[UB_THREADS];
  } u;
  ColDev cols[UB_MAX_COLS];
  int hist[UB_BINS];
  int wcnt[UB_WARPS];
  uint32_t st_lo[UB_STACK], st_hi[UB_STACK];  // bit 31 of st_hi: known to overflow (skip the optimistic pass)
  int sp;
  float4 stage_acc[UB_WARPS][32 * UB_GATHER];  // finished runs of one gather group, waiting for their batched row update
  uint32_t stage_row[UB_WARPS][(32 / G) * UB_GATHER];
  float4 head_acc[UB_WARPS][G], tail_acc[UB_WARPS][G];
  uint32_t head_row[UB_WARPS], tail_row[UB_WARPS];
  int head_valid[UB_WARPS], tail_valid[UB_WARPS], single[UB_WARPS];
};

template <int G>
__device__ __forceinline__ float4 unit_load_grad(const UnitArgs& a, const ColDev* cols, uint32_t packed, int q) {
  const uint32_t b = packed & 0xFFFFFFu;
  const ColDev c = cols[packed >> 24];
  float4 v = ldg_nc_na(reinterpret_cast<const float4*>(a.dout + (int64_t)b * a.dout_ld + c.out_col) + q);
  if (a.scale != nullptr) {
    const float s = __ldg(a.scale + (int64_t)b * a.n_fields + c.field);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
  }
  return v;
}

// Stable compaction of the list entries [i_lo, i_hi) whose row lies in [lo, hi) into s.row / s.pos (list order).  Every warp
// owns one contiguous stripe of the list: pass 1 counts its hits, pass 2 re-reads the rows (L2) and writes the hits at their
// place.  Returns the number found; nothing is written when it exceeds UB_CAP.
template <int G>
__device__ int unit_compact(UnitSmem<G>& s, const uint32_t* __restrict__ lrow, const uint32_t* __restrict__ lpos, int i_lo, int i_hi,
                            uint32_t lo, uint32_t hi) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint32_t span = hi - lo;
  const int stripe = ((i_hi - i_lo + UB_WARPS - 1) / UB_WARPS + 31) / 32 * 32;
  const int w_lo = min(i_hi, i_lo + stripe * w), w_hi = min(i_hi, w_lo + stripe);
  int cnt = 0;
  for (int i0 = w_lo; i0 < w_hi; i0 += 32 * 4) {
    uint32_t v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * 32 + lane;
      v[k] = i < w_hi ? __ldg(lrow + i) : UB_INVALID;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) cnt += (v[k] - lo) < span;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  __syncthreads();
  if (lane == 0) s.wcnt[w] = cnt;
  __syncthreads();
  int base = 0, total = 0;
#pragma unroll
  for (int ww = 0; ww < UB_WARPS; ++ww) {
    const int c = s.wcnt[ww];
    if (ww < w) base += c;
    total += c;
  }
  if (total > UB_CAP || total == 0) return total;
  for (int i0 = w_lo; i0 < w_hi; i0 += 32) {
    const int i = i0 + lane;
    const uint32_t v = i < w_hi ? __ldg(lrow + i) : UB_INVALID;
    const bool hit = (v - lo) < span;
    const uint32_t bal = __ballot_sync(0xffffffffu, hit);
    if (hit) {
      const int o = base + __popc(bal & ((1u << lane) - 1u));
      s.row[o] = v - lo;
      s.pos[o] = __ldg(lpos + i);
    }
    base += __popc(bal);
  }
  return total;
}

// Sort the m <= UB_CAP entries by row (stable) and reduce equal rows in list order; every finished run updates its row.
// Rows in s.row are relative to `row0` (absolute row of the table = row0 + s.row[i]); keys are < key_end.
template <int MODE, int G>
__device__ void unit_sort_reduce(UnitSmem<G>& s, const UnitArgs& a, const TableDev& T, int m, int64_t row0, uint32_t key_end) {
  constexpr int E = 32 / G;  // entries per warp batch
  constexpr int U = UB_GATHER;  // batches whose gradient rows are in flight together
  const int tid = threadIdx.x;
  __syncthreads();
  if (m > 1 && !HRB_UDBG(1)) {
    uint32_t k[UB_IPT], v[UB_IPT];
#pragma unroll
    for (int j = 0; j < UB_IPT; ++j) {
      const int i = tid * UB_IPT + j;
      k[j] = i < m ? s.row[i] : key_end - 1;  // padding: the largest key; the sort is stable, so it stays behind the real entries
      v[j] = i < m ? s.pos[i] : 0u;
    }
    int bits = 1;
    while (bits < 32 && ((key_end - 1) >> bits) != 0) ++bits;
    __syncthreads();
    typename UnitSmem<G>::Sort(s.u.sort).Sort(k, v, 0, bits);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < UB_IPT; ++j) {
      const int i = tid * UB_IPT + j;
      if (i < m) {
        s.row[i] = k[j];
        s.pos[i] = v[j];
      }
    }
  }
  __syncthreads();
  const int lane = tid & 31, w = tid >> 5, e = lane / G, q = lane % G;
  const int per = ((m + UB_WARPS - 1) / UB_WARPS + E - 1) / E * E;
  const int seg_lo = w * per;
  const int seg_hi = min(m, seg_lo + per);
  if (lane == 0) {
    s.head_valid[w] = 0;
    s.tail_valid[w] = 0;
    s.single[w] = 0;
  }
  uint32_t head_row = UB_NONE;
  if (w > 0 && seg_lo < seg_hi && s.row[seg_lo - 1] == s.row[seg_lo]) head_row = s.row[seg_lo];
  uint32_t carry_row = UB_NONE;
  float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
  int stage_n = 0;  // warp-uniform: finished runs staged since the last flush
  // A finished run (lanes q = 0..G-1 of one entry hold its sum; `closing` is uniform over them): it is parked in the warp's
  // staging area -- the row updates are then issued UB_APPLY at a time per lane group (flush) instead of one dependent
  // read-modify-write per batch -- unless it continues the previous warp's last run (head slot, stitched at the end).
  auto close = [&](bool closing, uint32_t r, const float4& v) {  // called by the whole warp
    const bool head = closing && r == head_row;
    if (head) {
      s.head_acc[w][q] = v;
      if (q == 0) {
        s.head_valid[w] = 1;
        s.head_row[w] = r;
      }
    }
    const bool st = closing && !head;
    const uint32_t bal = __ballot_sync(0xffffffffu, st && q == 0);
    if (st) {
      const int slot = stage_n + __popc(bal & ((1u << (lane - q)) - 1u));
      s.stage_acc[w][slot * G + q] = v;
      if (q == 0) s.stage_row[w][slot] = r;
    }
    stage_n += __popc(bal);
  };
  auto flush = [&]() {
    __syncwarp();
    for (int j0 = 0; j0 < stage_n; j0 += E * UB_APPLY) {
      int64_t rr[UB_APPLY];
      float4 vv[UB_APPLY];
      bool ok[UB_APPLY];
#pragma unroll
      for (int u = 0; u < UB_APPLY; ++u) {
        const int j = j0 + u * E + e;
        ok[u] = j < stage_n;
        rr[u] = ok[u] ? row0 + s.stage_row[w][j] : 0;
        vv[u] = ok[u] ? s.stage_acc[w][j * G + q] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (!HRB_UDBG(2)) apply_table_rows<MODE, UB_APPLY>(T, a.opt, a.lr_t, rr, ok, q, vv);
    }
    stage_n = 0;
    __syncwarp();
  };
  // segmented scan over warp batches; finished runs are staged and their rows updated UB_APPLY at a time (flush)
  for (int k0 = seg_lo; k0 < seg_hi; k0 += E * U) {
    uint32_t r[U];
    float4 g[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = k0 + u * E + e;
      r[u] = UB_INVALID;
      g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < seg_hi) {
        r[u] = s.row[i];
        if (!HRB_UDBG(4)) g[u] = unit_load_grad<G>(a, s.cols, s.pos[i], q);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int nvalid = min(E, seg_hi - (k0 + u * E));  // warp-uniform
      if (nvalid <= 0) continue;
      const int e_end = nvalid - 1;
      float4 acc = g[u];
      const uint32_t row = r[u];
#pragma unroll
      for (int off = 1; off < E; off <<= 1) {  // segmented inclusive scan over the batch (keys are sorted)
        const uint32_t orow = __shfl_up_sync(0xffffffffu, row, off * G);
        const float ox = __shfl_up_sync(0xffffffffu, acc.x, off * G), oy = __shfl_up_sync(0xffffffffu, acc.y, off * G);
        const float oz = __shfl_up_sync(0xffffffffu, acc.z, off * G), ow = __shfl_up_sync(0xffffffffu, acc.w, off * G);
        if (e >= off && orow == row) {
          acc.x = ox + acc.x; acc.y = oy + acc.y; acc.z = oz + acc.z; acc.w = ow + acc.w;
        }
      }
      const uint32_t rnext = __shfl_down_sync(0xffffffffu, row, G);
      const uint32_t first_row = __shfl_sync(0xffffffffu, row, q);
      if (carry_row == first_row) {
        if (row == first_row) {
          acc.x = carry.x + acc.x; acc.y = carry.y + acc.y; acc.z = carry.z + acc.z; acc.w = carry.w + acc.w;
        }
      }
      // the run left open by the previous batch ended at the batch boundary
      close(carry_row != first_row && carry_row != UB_NONE && e == 0, carry_row, carry);
      close(e < e_end && rnext != row, row, acc);
      carry_row = __shfl_sync(0xffffffffu, row, e_end * G + q);
      carry.x = __shfl_sync(0xffffffffu, acc.x, e_end * G + q);
      carry.y = __shfl_sync(0xffffffffu, acc.y, e_end * G + q);
      carry.z = __shfl_sync(0xffffffffu, acc.z, e_end * G + q);
      carry.w = __shfl_sync(0xffffffffu, acc.w, e_end * G + q);
    }
    flush();
  }
  if (carry_row != UB_NONE && e == 0) {  // the segment's last run: may continue in the next warp's segment
    if (carry_row == head_row) {         // the whole segment is one run that also continues the previous one
      s.head_acc[w][q] = carry;
      if (q == 0) {
        s.head_valid[w] = 1;
        s.head_row[w] = carry_row;
        s.single[w] = 1;
      }
    } else {
      s.tail_acc[w][q] = carry;
      if (q == 0) {
        s.tail_valid[w] = 1;
        s.tail_row[w] = carry_row;
      }
    }
  }
  __syncthreads();
  if (tid < G) {  // stitch the runs that cross warp segments, in segment order
    bool open = false;
    uint32_t crow = 0;
    float4 cacc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ww = 0; ww < UB_WARPS; ++ww) {
      if (s.head_valid[ww]) {
        const float4 h = s.head_acc[ww][tid];
        cacc.x += h.x; cacc.y += h.y; cacc.z += h.z; cacc.w += h.w;
        if (!s.single[ww]) {
          apply_table_row<MODE>(T, a.opt, a.lr_t, row0 + crow, tid, cacc);
          open = false;
        }
      } else if (open) {
        apply_table_row<MODE>(T, a.opt, a.lr_t, row0 + crow, tid, cacc);
        open = false;
      }
      if (s.tail_valid[ww]) {
        crow = s.tail_row[ww];
        cacc = s.tail_acc[ww][tid];
        open = true;
      }
    }
    if (open) apply_table_row<MODE>(T, a.opt, a.lr_t, row0 + crow, tid, cacc);
  }
  __syncthreads();
}

// One row with more positions than a pass holds (or one slice of such a row): every lane group adds its share of the row's
// positions in list order, the groups are combined by a fixed tree.  `row` == UB_INVALID: every entry of [i_lo, i_hi) belongs
// to the row (single-row units).  Result (lanes tid < G): the gradient sum; returns the position count.
template <int G>
__device__ int unit_single_row(UnitSmem<G>& s, const UnitArgs& a, const uint32_t* __restrict__ lrow, const uint32_t* __restrict__ lpos,
                               int i_lo, int i_hi, uint32_t row, float4& out) {
  constexpr int NG = UB_THREADS / G;
  constexpr int U = 4;
  const int tid = threadIdx.x, g = tid / G, q = tid % G;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int n_total = 0;
  for (int c0 = i_lo; c0 < i_hi; c0 += UB_CAP) {  // chunks of the list in order
    const int c1 = min(i_hi, c0 + UB_CAP);
    int cnt;
    if (row == UB_INVALID) {
      cnt = c1 - c0;
      __syncthreads();
      for (int i = tid; i < cnt; i += UB_THREADS) s.pos[i] = __ldg(lpos + c0 + i);
    } else {
      cnt = unit_compact<G>(s, lrow, lpos, c0, c1, row, row + 1);
    }
    __syncthreads();
    for (int i0 = g; i0 < cnt; i0 += NG * U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * NG;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < cnt) v[u] = unit_load_grad<G>(a, s.cols, s.pos[i], q);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
      }
    }
    n_total += cnt;
    __syncthreads();
  }
  s.u.red[tid] = acc;
  __syncthreads();
  for (int stride = UB_THREADS / 2; stride >= G; stride >>= 1) {
    if (tid < stride) {
      const float4 o = s.u.red[tid + stride];
      float4 mm = s.u.red[tid];
      mm.x += o.x; mm.y += o.y; mm.z += o.z; mm.w += o.w;
      s.u.red[tid] = mm;
    }
    __syncthreads();
  }
  out = s.u.red[tid < G ? tid : 0];
  __syncthreads();
  return n_total;
}

// 64-bin histogram of the rows of list entries [0, cnt) that fall into [lo, hi)
template <int G>
__device__ void unit_histogram(UnitSmem<G>& s, const uint32_t* __restrict__ lrow, int cnt, uint32_t lo, uint32_t hi, uint32_t width) {
  const int tid = threadIdx.x;
  const uint32_t span = hi - lo;
  __syncthreads();
  if (tid < UB_BINS) s.hist[tid] = 0;
  __syncthreads();
  for (int i0 = tid; i0 < cnt; i0 += UB_THREADS * 4) {
    uint32_t v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * UB_THREADS;
      v[k] = i < cnt ? __ldg(lrow + i) : UB_INVALID;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if ((v[k] - lo) < span) atomicAdd(&s.hist[(v[k] - lo) / width], 1);  // integer counts: the order does not matter
  }
  __syncthreads();
}

template <int MODE, int G>
__global__ void __launch_bounds__(UB_THREADS, 2) bwd_unit_kernel(UnitArgs a, int unit_base) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  UnitSmem<G>& s = *reinterpret_cast<UnitSmem<G>*>(smem_raw);
  const int tid = threadIdx.x;
  const int helper = blockIdx.x / a.n_units;  // CTAs [0, n_units) are the owners, the helpers come behind them
  const UnitDev unit = a.units[unit_base + blockIdx.x % a.n_units];
  const int cnt = (int)a.list_cnt[unit.list];
  if (helper > 0 && (cnt <= UB_CAP || unit.n_slices > 1 || unit.row_hi - unit.row_lo == 1)) return;
  if (cnt == 0) {
    // an untouched row; a slice still has to report "no positions" to bwd_unit_combine_kernel (the workspace is not zeroed)
    if (unit.n_slices > 1 && tid == 0) a.partials[(size_t)(unit.partial_idx + unit.slice) * UB_PARTIAL_LD + 32 * 4] = 0.f;
    return;
  }
  const uint32_t* lrow = a.ent_row + a.list_off[unit.list];
  const uint32_t* lpos = a.ent_pos + a.list_off[unit.list];
  const TableDev T = a.tables[unit.table];
  const int c0 = a.col_start[unit.table];
  const int ncol = a.col_start[unit.table + 1] - c0;
  for (int i = tid; i < ncol; i += UB_THREADS) s.cols[i] = a.cols[c0 + i];
  __syncthreads();
  const uint32_t span = unit.row_hi - unit.row_lo;
  if (unit.n_slices > 1) {  // one slice of a row the host knows to be hot: partial sum + position count
    const int i_lo = (int)((int64_t)cnt * unit.slice / unit.n_slices), i_hi = (int)((int64_t)cnt * (unit.slice + 1) / unit.n_slices);
    float4 sum;
    const int n = unit_single_row<G>(s, a, lrow, lpos, i_lo, i_hi, UB_INVALID, sum);
    float* p = a.partials + (size_t)(unit.partial_idx + unit.slice) * UB_PARTIAL_LD;
    if (tid < G) reinterpret_cast<float4*>(p)[tid] = sum;
    if (tid == 0) p[32 * 4] = (float)n;
    return;
  }
  if (span == 1) {  // a single-row unit: no sort, whatever its length
    float4 sum;
    unit_single_row<G>(s, a, lrow, lpos, 0, cnt, UB_INVALID, sum);
    if (tid < G) apply_table_row<MODE>(T, a.opt, a.lr_t, (int64_t)unit.row_lo, tid, sum);
    return;
  }
  if (cnt <= UB_CAP) {  // the ordinary case: the whole list in one pass
    for (int i = tid; i < cnt; i += UB_THREADS) {
      s.row[i] = __ldg(lrow + i);
      s.pos[i] = __ldg(lpos + i);
    }
    if (HRB_UDBG(8)) return;
    unit_sort_reduce<MODE, G>(s, a, T, cnt, (int64_t)unit.row_lo, span);
    return;
  }
  // overflow: the unit's UB_HELPERS CTAs share its row range by count quantiles of a 64-bin histogram (every CTA computes the
  // same histogram, so they agree on the shares without talking to each other)
  {
    const uint32_t width = (span + UB_BINS - 1) / UB_BINS;
    unit_histogram<G>(s, lrow, cnt, 0, span, width);
    if (tid == 0) {
      int64_t before = 0;
      uint32_t my_lo = span, my_hi = 0;
      int mine = 0;
      for (int bin = 0; bin < UB_BINS; ++bin) {
        const uint32_t blo = (uint32_t)bin * width;
        if (blo >= span) break;
        const int c = s.hist[bin];
        if (c > 0 && (int)(before * UB_HELPERS / cnt) == helper) {  // the bin goes to the CTA its first position falls to
          my_lo = min(my_lo, blo);
          my_hi = max(my_hi, min(span, blo + width));
          mine += c;
        }
        before += c;
      }
      s.sp = 0;
      if (mine > 0) {
        s.st_lo[0] = my_lo;
        s.st_hi[0] = my_hi | (mine > UB_CAP ? 0x80000000u : 0u);
        s.sp = 1;
      }
    }
    __syncthreads();
  }
  while (true) {
    const int sp = s.sp;
    if (sp == 0) break;
    const uint32_t lo = s.st_lo[sp - 1];
    const uint32_t hi_raw = s.st_hi[sp - 1];
    const uint32_t hi = hi_raw & 0x7FFFFFFFu;
    __syncthreads();
    if (tid == 0) s.sp = sp - 1;
    if (!(hi_raw & 0x80000000u)) {
      const int m = unit_compact<G>(s, lrow, lpos, 0, cnt, lo, hi);
      if (m <= UB_CAP) {
        if (m > 0) unit_sort_reduce<MODE, G>(s, a, T, m, (int64_t)unit.row_lo + lo, hi - lo);
        __syncthreads();
        continue;
      }
    }
    if (hi - lo == 1) {
      float4 sum;
      const int n = unit_single_row<G>(s, a, lrow, lpos, 0, cnt, lo, sum);
      if (n > 0 && tid < G) apply_table_row<MODE>(T, a.opt, a.lr_t, (int64_t)unit.row_lo + lo, tid, sum);
      __syncthreads();
      continue;
    }
    // split [lo, hi) by a 64-bin histogram into sub-ranges that fit one pass
    const uint32_t sub = hi - lo;
    const uint32_t width = (sub + UB_BINS - 1) / UB_BINS;
    unit_histogram<G>(s, lrow, cnt, lo, hi, width);
    if (tid == 0) {
      int top = s.sp;
      int acc = 0;
      uint32_t start = lo;
      for (int bin = 0; bin < UB_BINS; ++bin) {
        const uint32_t blo = lo + (uint32_t)bin * width;
        if (blo >= hi) break;
        const uint32_t bhi = min(hi, blo + width);
        const int c = s.hist[bin];
        if (c > UB_CAP) {  // this bin alone overflows: its own range, split again (or a single hot row)
          if (acc > 0 && top < UB_STACK) { s.st_lo[top] = start; s.st_hi[top] = blo; ++top; }
          if (top < UB_STACK) { s.st_lo[top] = blo; s.st_hi[top] = bhi | 0x80000000u; ++top; }
          start = bhi;
          acc = 0;
        } else if (acc + c > UB_CAP) {
          if (top < UB_STACK) { s.st_lo[top] = start; s.st_hi[top] = blo; ++top; }
          start = blo;
          acc = c;
        } else {
          acc += c;
        }
      }
      if (acc > 0 && top < UB_STACK) { s.st_lo[top] = start; s.st_hi[top] = hi; ++top; }
      s.sp = top;
    }
    __syncthreads();
  }
}

// hot rows split over list slices: add the slice sums in slice order, update the row once
template <int MODE, int G>
__global__ void __launch_bounds__(256) bwd_unit_combine_kernel(UnitArgs a, const SliceGroupDev* __restrict__ groups, int group_base, int n_groups) {
  const int gi = blockIdx.x * (blockDim.x / G) + threadIdx.x / G, q = threadIdx.x % G;
  if (gi >= n_groups) return;
  const SliceGroupDev sg = groups[group_base + gi];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float n = 0.f;
  for (int sl = 0; sl < sg.n_slices; ++sl) {
    const float* p = a.partials + (size_t)(sg.partial_idx + sl) * UB_PARTIAL_LD;
    const float cnt = p[32 * 4];
    if (cnt > 0.f) {  // an empty slice wrote only its count
      const float4 v = reinterpret_cast<const float4*>(p)[q];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    n += cnt;
  }
  if (n > 0.f) apply_table_row<MODE>(a.tables[sg.table], a.opt, a.lr_t, (int64_t)sg.row, q, acc);
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
struct UnitHost {
  UnitDev d;
  int32_t g;
  int64_t expect;
};

static inline int64_t unit_ldT(int64_t batch) { return (batch + 15) / 16 * 16; }  // 64-byte aligned id columns

// (Re)build the unit decomposition of `plan` for `batch` samples.  Units are ordered by G, then largest first.
static int build_units(const hrb_plan* plan, int64_t batch) {
  UnitSet& us = plan->units;
  if (us.batch == batch) return HRB_OK;
  us.ok = false;
  us.batch = batch;
  std::vector<UnitHost> units;
  std::vector<SliceGroupDev> groups;
  std::vector<int32_t> group_g;
  std::vector<TableSplitDev> splits(plan->n_tables);
  std::vector<TileDev> tiles;
  int32_t n_partials = 0, n_lists = 0;
  const int64_t n_chunks = (unit_ldT(batch) + UB_TILE - 1) / UB_TILE;
  std::vector<int32_t> col_pos;  // position column of every (table-major) column, as hrb_plan_create orders them
  for (int t = 0; t < plan->n_tables; ++t)
    for (int f = 0; f < plan->n_fields; ++f) {
      if (plan->fields[f].table != t) continue;
      for (int l = 0; l < plan->fields[f].seq_len; ++l) col_pos.push_back(plan->fdev_host[f].pos_col + l);
    }
  for (int t = 0; t < plan->n_tables; ++t) {
    const TableDev& td = plan->tdev_host[t];
    const int64_t ncol = plan->col_start_host[t + 1] - plan->col_start_host[t];
    TableSplitDev& sp = splits[t];
    sp = TableSplitDev{n_lists, 0, 0, (int32_t)tiles.size(), 0, (uint32_t)(batch * plan->col_start_host[t])};
    if (ncol == 0) continue;
    const int64_t n_t = batch * ncol;
    // the largest power-of-two row range whose expected share of the table's positions (uniform ids) is <= UB_EXPECT_MAX
    int shift = 0;
    while (shift < 31 && (int64_t)(2ll << shift) * n_t <= (int64_t)UB_EXPECT_MAX * td.rows) ++shift;
    const int64_t range = 1ll << shift;
    const int64_t n_bins = (td.rows + range - 1) / range;
    if (n_bins > UB_MAX_BINS) return HRB_OK;  // us.ok stays false: the caller takes the sorted path
    sp.n_bins = (int32_t)n_bins;
    sp.shift = shift;
    sp.n_tiles = (int32_t)(ncol * n_chunks);
    for (int64_t cl = 0; cl < ncol; ++cl)
      for (int64_t ch = 0; ch < n_chunks; ++ch)
        tiles.push_back(TileDev{t, (int32_t)cl, col_pos[plan->col_start_host[t] + cl], (int32_t)ch});
    const int32_t g = td.dim / 4;
    for (int64_t bin = 0; bin < n_bins; ++bin) {
      const int64_t lo = bin * range, hi = std::min<int64_t>(td.rows, lo + range);
      const int64_t expect = n_t * (hi - lo) / td.rows;
      UnitHost u{};
      u.d.table = t;
      u.d.row_lo = (uint32_t)lo;
      u.d.row_hi = (uint32_t)hi;
      u.d.n_slices = 1;
      u.d.list = n_lists + (int32_t)bin;
      u.g = g;
      u.expect = expect;
      if (hi - lo == 1 && expect > 2 * UB_SLICE_TARGET) {  // a row of a tiny table: split over slices of its list
        int64_t ns = (expect + UB_SLICE_TARGET - 1) / UB_SLICE_TARGET;
        if (ns > 64) ns = 64;
        groups.push_back(SliceGroupDev{t, (uint32_t)lo, n_partials, (int32_t)ns});
        group_g.push_back(g);
        for (int64_t sl = 0; sl < ns; ++sl) {
          UnitHost v = u;
          v.d.slice = (int32_t)sl;
          v.d.n_slices = (int32_t)ns;
          v.d.partial_idx = n_partials;
          v.expect = expect / ns;
          units.push_back(v);
        }
        n_partials += (int32_t)ns;
      } else {
        units.push_back(u);
      }
    }
    n_lists += (int32_t)n_bins;
  }
  std::stable_sort(units.begin(), units.end(), [](const UnitHost& x, const UnitHost& y) {
    if (x.g != y.g) return x.g < y.g;
    return x.expect > y.expect;
  });
  std::vector<size_t> gorder(groups.size());
  for (size_t i = 0; i < gorder.size(); ++i) gorder[i] = i;
  std::stable_sort(gorder.begin(), gorder.end(), [&](size_t x, size_t y) { return group_g[x] < group_g[y]; });
  std::vector<UnitDev> ud(units.size());
  std::vector<SliceGroupDev> gd(groups.size());
  us.n_g = 0;
  for (size_t i = 0; i < units.size(); ++i) {
    ud[i] = units[i].d;
    if (us.n_g == 0 || us.g_values[us.n_g - 1] != units[i].g) {
      if (us.n_g >= 8) return fail(HRB_UNSUPPORTED, "embedding backward: more than 8 distinct embedding dims in one plan");
      us.g_values[us.n_g] = units[i].g;
      us.g_unit_off[us.n_g] = (int32_t)i;
      ++us.n_g;
    }
  }
  us.g_unit_off[us.n_g] = (int32_t)units.size();
  for (size_t i = 0; i < gorder.size(); ++i) gd[i] = groups[gorder[i]];
  us.g_group_off[0] = 0;  // groups are sorted by G like the units: prefix sums of the per-G counts
  for (int gi = 0; gi < us.n_g; ++gi) {
    int32_t cnt = 0;
    for (size_t i = 0; i < group_g.size(); ++i) cnt += group_g[i] == us.g_values[gi];
    us.g_group_off[gi + 1] = us.g_group_off[gi] + cnt;
  }
  if (us.d_blob) cudaFree(us.d_blob);
  us.d_blob = nullptr;
  const size_t sz_u = ub_align(sizeof(UnitDev) * (ud.size() + 1)), sz_g = ub_align(sizeof(SliceGroupDev) * (gd.size() + 1));
  const size_t sz_s = ub_align(sizeof(TableSplitDev) * (splits.size() + 1)), sz_t = ub_align(sizeof(TileDev) * (tiles.size() + 1));
  HRB_CUDA(cudaMalloc(&us.d_blob, sz_u + sz_g + sz_s + sz_t));
  char* d = (char*)us.d_blob;
  if (!ud.empty()) HRB_CUDA(cudaMemcpy(d, ud.data(), sizeof(UnitDev) * ud.size(), cudaMemcpyHostToDevice));
  if (!gd.empty()) HRB_CUDA(cudaMemcpy(d + sz_u, gd.data(), sizeof(SliceGroupDev) * gd.size(), cudaMemcpyHostToDevice));
  HRB_CUDA(cudaMemcpy(d + sz_u + sz_g, splits.data(), sizeof(TableSplitDev) * splits.size(), cudaMemcpyHostToDevice));
  if (!tiles.empty()) HRB_CUDA(cudaMemcpy(d + sz_u + sz_g + sz_s, tiles.data(), sizeof(TileDev) * tiles.size(), cudaMemcpyHostToDevice));
  us.d_units = (UnitDev*)d;
  us.d_groups = (SliceGroupDev*)(d + sz_u);
  us.d_splits = (TableSplitDev*)(d + sz_u + sz_g);
  us.d_tiles = (TileDev*)(d + sz_u + sz_g + sz_s);
  us.n_units = (int32_t)ud.size();
  us.n_groups = (int32_t)gd.size();
  us.n_partials = n_partials;
  us.n_lists = n_lists;
  us.n_tiles = (int32_t)tiles.size();
  us.ok = true;
  return HRB_OK;
}

bool unit_path_supported(const hrb_plan* plan, int64_t batch) {
  if (!(plan->unit_path_ok && !plan->has_max && batch < (1ll << 24) && batch > 0)) return false;
  std::lock_guard<std::mutex> lock(plan->unit_mu);
  return build_units(plan, batch) == HRB_OK && plan->units.ok;
}

struct UnitWs {
  size_t idsT, scale, partials, ent_row, ent_pos, tile_cnt, list_cnt, list_off, total;
};
static UnitWs carve_unit_ws(const hrb_plan* plan, int64_t batch) {
  const UnitSet& us = plan->units;
  UnitWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += ub_align(bytes);
    return o;
  };
  const size_t n = (size_t)batch * plan->pos_cols;
  w.idsT = take((size_t)plan->pos_cols * unit_ldT(batch) * 4);
  w.scale = take((size_t)batch * plan->n_fields * 4 + 4);
  w.partials = take((size_t)(us.n_partials + 1) * UB_PARTIAL_LD * 4);
  w.ent_row = take(n * 4 + 4);
  w.ent_pos = take(n * 4 + 4);
  w.tile_cnt = take((size_t)(us.n_tiles + 1) * UB_MAX_BINS * 4);
  w.list_cnt = take((size_t)(us.n_lists + 1) * 4);
  w.list_off = take((size_t)(us.n_lists + 1) * 4);
  w.total = off;
  return w;
}

size_t unit_workspace_bytes(const hrb_plan* plan, int64_t batch) {  // call after unit_path_supported(plan, batch)
  std::lock_guard<std::mutex> lock(plan->unit_mu);
  return carve_unit_ws(plan, batch).total;
}

template <int MODE, int G>
static int launch_units(UnitArgs a, const UnitSet& us, int gi, cudaStream_t st) {
  static bool attr = false;
  const size_t smem = sizeof(UnitSmem<G>);
  if (!attr) {
    HRB_CUDA(cudaFuncSetAttribute(bwd_unit_kernel<MODE, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  const int n = us.g_unit_off[gi + 1] - us.g_unit_off[gi];
  if (n > 0) {
    a.n_units = n;
    bwd_unit_kernel<MODE, G><<<n * (HRB_UDBG(32) ? 1 : UB_HELPERS), UB_THREADS, smem, st>>>(a, us.g_unit_off[gi]);
    HRB_LAUNCH_CHECK();
  }
  const int ng = us.g_group_off[gi + 1] - us.g_group_off[gi];
  if (ng > 0) {
    const int gpb = 256 / G;
    bwd_unit_combine_kernel<MODE, G><<<(ng + gpb - 1) / gpb, 256, 0, st>>>(a, us.d_groups, us.g_group_off[gi], ng);
    HRB_LAUNCH_CHECK();
  }
  return HRB_OK;
}

int run_unit_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const float* dout, int64_t dout_ld,
                    const hrb_opt_params& opt, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  std::lock_guard<std::mutex> lock(plan->unit_mu);
  int rc = build_units(plan, batch);
  if (rc != HRB_OK) return rc;
  const UnitSet& us = plan->units;
  if (!us.ok) return fail(HRB_UNSUPPORTED, "embedding backward: unit path not available for this plan / batch");
  const UnitWs ws = carve_unit_ws(plan, batch);
  if (ws.total > workspace_bytes) return fail(HRB_WORKSPACE, "hrb_lookup_bwd_update: workspace %zu < required %zu bytes", workspace_bytes, ws.total);
  char* base = (char*)workspace;
  const int64_t ldT = unit_ldT(batch);
  uint32_t* idsT = (uint32_t*)(base + ws.idsT);
  float* scale = (float*)(base + ws.scale);
  dim3 pg((unsigned)((ldT + 31) / 32), (unsigned)((plan->pos_cols + 31) / 32));
  bwd_prep_kernel<<<pg, 256, 0, st>>>(plan->d_fields, plan->d_pos_field, plan->pos_cols, ids, ids_ld, batch, ldT, idsT);
  HRB_LAUNCH_CHECK();
  if (plan->has_mean) {
    int64_t blocks = (batch * plan->n_fields + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    bwd_scale_kernel<<<(unsigned)blocks, 256, 0, st>>>(plan->d_fields, plan->n_fields, ids, ids_ld, batch, scale);
    HRB_LAUNCH_CHECK();
  }
  SplitArgs sa{us.d_splits, us.d_tiles, idsT, ldT, (uint32_t*)(base + ws.tile_cnt), (uint32_t*)(base + ws.list_cnt),
               (uint32_t*)(base + ws.list_off), (uint32_t*)(base + ws.ent_row), (uint32_t*)(base + ws.ent_pos)};
  if (us.n_tiles > 0) {
    split_kernel<false><<<us.n_tiles, UB_THREADS, 0, st>>>(sa);
    HRB_LAUNCH_CHECK();
    split_scan_kernel<<<plan->n_tables, UB_MAX_BINS, 0, st>>>(sa);
    HRB_LAUNCH_CHECK();
    split_kernel<true><<<us.n_tiles, UB_THREADS, 0, st>>>(sa);
    HRB_LAUNCH_CHECK();
  }
  UnitArgs a{};
  a.units = us.d_units;
  a.tables = plan->d_tables;
  a.cols = plan->d_cols;
  a.col_start = plan->d_col_start;
  a.list_cnt = sa.list_cnt;
  a.list_off = sa.list_off;
  a.ent_row = sa.ent_row;
  a.ent_pos = sa.ent_pos;
  a.dout = dout;
  a.dout_ld = dout_ld;
  a.scale = plan->has_mean ? scale : nullptr;
  a.n_fields = plan->n_fields;
  a.opt = opt;
  a.lr_t = opt.opt == HRB_OPT_ADAM_LAZY ? opt.lr * sqrtf(opt.bias_corr2) / opt.bias_corr1 : 0.f;
  a.partials = (float*)(base + ws.partials);
#ifdef HRB_DEVTOOLS
  {
    static int dbg = -1;
    if (dbg < 0) {
      const char* e = getenv("HRB_BWD_DEBUG");
      dbg = e ? atoi(e) : 0;
    }
    a.debug = dbg;
  }
#endif
  const int mode = upd_mode(opt.opt);
  for (int gi = 0; gi < us.n_g; ++gi) {
#define HRB_UNITS(GG)                                                                      \
  rc = mode == UPD_ADAM      ? launch_units<UPD_ADAM, GG>(a, us, gi, st)                   \
       : mode == UPD_ADAGRAD ? launch_units<UPD_ADAGRAD, GG>(a, us, gi, st)                \
       : mode == UPD_FTRL    ? launch_units<UPD_FTRL, GG>(a, us, gi, st)                   \
                             : launch_units<UPD_SGD, GG>(a, us, gi, st);                   \
  break;
    switch (us.g_values[gi]) {
      case 1: HRB_UNITS(1)
      case 2: HRB_UNITS(2)
      case 4: HRB_UNITS(4)
      case 8: HRB_UNITS(8)
      case 16: HRB_UNITS(16)
      case 32: HRB_UNITS(32)
      default: rc = fail(HRB_UNSUPPORTED, "embedding backward: dim %d", us.g_values[gi] * 4);
    }
#undef HRB_UNITS
    if (rc != HRB_OK) return rc;
  }
  return HRB_OK;
}

}  // namespace hrb
