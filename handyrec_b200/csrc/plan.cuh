// plan.cuh -- the lookup plan (hrb_plan) and its device-side field / table descriptors, shared by lookup.cu and
// embedding_bwd.cu.
#pragma once
#include <cstddef>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace hrb {

struct FieldDev {
  const float* table;
  int64_t rows;
  uint32_t key_base;  // first key of this field's table in the global (table,row) key space
  int32_t dim;
  int32_t seq_len;
  int32_t pool;
  int32_t ids_col;
  int32_t out_col;
  int32_t pos_col;  // first column in the dense position space (prefix sum of seq_len)
  int32_t table_idx;
};

struct TableDev {
  float* w;
  float* m;     // optimiser state: Adam first moment / Adagrad or Ftrl accumulator
  float* v;     // Adam second moment / Ftrl linear
  int64_t rows;
  uint32_t key_base;
  int32_t dim;
  float* grad;  // non-null: a13 adds the row's gradient sum here instead of updating the row (hrb_plan_set_dense_grads)
};

// Row-update modes of apply_table_row(s) and of every kernel that dispatches on them.  UPD_DENSE_ADD is lookup.cu's
// dense-gradient face (hrb_embedding_bwd_dense), which never reaches apply_table_row(s).
enum UpdMode : int { UPD_SGD = 0, UPD_ADAM = 1, UPD_DENSE_ADD = 2, UPD_ADAGRAD = 3, UPD_FTRL = 4 };

// hrb_opt -> UpdMode of the row update
inline int upd_mode(int32_t opt) {
  return opt == HRB_OPT_ADAM_LAZY ? UPD_ADAM : opt == HRB_OPT_ADAGRAD ? UPD_ADAGRAD : opt == HRB_OPT_FTRL ? UPD_FTRL : UPD_SGD;
}

// The caller's hrb_opt_params: the Ftrl fields at its end are read only when opt == HRB_OPT_FTRL (a caller built against the
// shorter struct of the other optimisers passes fewer bytes), zero otherwise.
inline hrb_opt_params load_opt(const hrb_opt_params* p) {
  hrb_opt_params o{};
  memcpy(&o, p, offsetof(hrb_opt_params, l1));
  if (o.opt == HRB_OPT_FTRL) {
    o.l1 = p->l1;
    o.l2 = p->l2;
    o.lr_power = p->lr_power;
    o.l2_shrinkage = p->l2_shrinkage;
  }
  return o;
}

// Keras Ftrl on the four floats of a row chunk (ftrl_elem, common.cuh); a: accumulator, l: linear
__device__ __forceinline__ void ftrl_row4(float4& w, float4& a, float4& l, const float4& g, const hrb_opt_params& o) {
  w.x = ftrl_elem(w.x, a.x, l.x, g.x, o.lr, o.l1, o.l2, o.lr_power, o.l2_shrinkage);
  w.y = ftrl_elem(w.y, a.y, l.y, g.y, o.lr, o.l1, o.l2, o.lr_power, o.l2_shrinkage);
  w.z = ftrl_elem(w.z, a.z, l.z, g.z, o.lr, o.l1, o.l2, o.lr_power, o.l2_shrinkage);
  w.w = ftrl_elem(w.w, a.w, l.w, g.w, o.lr, o.l1, o.l2, o.lr_power, o.l2_shrinkage);
}

// Keras Adagrad (ResourceSparseApplyAdagradV2, eps outside the square root) on one float of a row; acc is the table's
// accumulator (TableDev::m)
__device__ __forceinline__ void adagrad_elem(float& w, float& acc, float g, float lr, float eps) {
  acc = fmaf(g, g, acc);
  w -= lr * g / (sqrtf(acc) + eps);
}

// One touched row of one table takes its update (a13).  MODE: UpdMode (SGD, lazy Adam, Adagrad, Ftrl).  A table with a dense-gradient
// buffer (hrb_plan_set_dense_grads) receives the gradient sum instead and is stepped by the caller's dense optimiser.
template <int MODE>
__device__ __forceinline__ void apply_table_row(const TableDev& t, const hrb_opt_params& opt, float lr_t, int64_t row, int q, float4 g) {
  if (q * 4 >= t.dim) return;
  const int64_t off = row * (t.dim >> 2) + q;
  if (t.grad != nullptr) {
    float4* gp = reinterpret_cast<float4*>(t.grad) + off;
    float4 o = *gp;
    o.x += g.x; o.y += g.y; o.z += g.z; o.w += g.w;
    *gp = o;
    return;
  }
  float4* wp = reinterpret_cast<float4*>(t.w) + off;
  float4 w = *wp;
  if (MODE == UPD_FTRL) {  // issue the accumulator and linear loads with the weight's
    float4* ap = reinterpret_cast<float4*>(t.m) + off;
    float4* lp = reinterpret_cast<float4*>(t.v) + off;
    float4 a = *ap, l = *lp;
    const float l2 = opt.l2_scale;
    g.x = fmaf(l2, w.x, g.x); g.y = fmaf(l2, w.y, g.y); g.z = fmaf(l2, w.z, g.z); g.w = fmaf(l2, w.w, g.w);
    ftrl_row4(w, a, l, g, opt);
    *ap = a;
    *lp = l;
    *wp = w;
    return;
  }
  const float l2 = opt.l2_scale;
  g.x = fmaf(l2, w.x, g.x); g.y = fmaf(l2, w.y, g.y); g.z = fmaf(l2, w.z, g.z); g.w = fmaf(l2, w.w, g.w);
  if (MODE == UPD_SGD) {
    const float lr = opt.lr;
    w.x -= lr * g.x; w.y -= lr * g.y; w.z -= lr * g.z; w.w -= lr * g.w;
  } else if (MODE == UPD_ADAGRAD) {
    float4* ap = reinterpret_cast<float4*>(t.m) + off;
    float4 a = *ap;
    const float lr = opt.lr, e = opt.eps;
    adagrad_elem(w.x, a.x, g.x, lr, e); adagrad_elem(w.y, a.y, g.y, lr, e);
    adagrad_elem(w.z, a.z, g.z, lr, e); adagrad_elem(w.w, a.w, g.w, lr, e);
    *ap = a;
  } else {
    float4* mp = reinterpret_cast<float4*>(t.m) + off;
    float4* vp = reinterpret_cast<float4*>(t.v) + off;
    float4 m = *mp, v = *vp;
    const float b1 = opt.beta1, b2 = opt.beta2, e = opt.eps, lr = lr_t;
    m.x = b1 * m.x + (1.f - b1) * g.x; m.y = b1 * m.y + (1.f - b1) * g.y;
    m.z = b1 * m.z + (1.f - b1) * g.z; m.w = b1 * m.w + (1.f - b1) * g.w;
    v.x = b2 * v.x + (1.f - b2) * g.x * g.x; v.y = b2 * v.y + (1.f - b2) * g.y * g.y;
    v.z = b2 * v.z + (1.f - b2) * g.z * g.z; v.w = b2 * v.w + (1.f - b2) * g.w * g.w;
    w.x -= lr * m.x / (sqrtf(v.x) + e); w.y -= lr * m.y / (sqrtf(v.y) + e);
    w.z -= lr * m.z / (sqrtf(v.z) + e); w.w -= lr * m.w / (sqrtf(v.w) + e);
    *mp = m;
    *vp = v;
  }
  *wp = w;
}

// The same update for N rows of one table at once: every load is issued before the first dependent instruction, so a lane
// group has N read-modify-writes in flight instead of one (the embedding backward is latency-bound otherwise).
template <int MODE, int N>
__device__ __forceinline__ void apply_table_rows(const TableDev& t, const hrb_opt_params& opt, float lr_t, const int64_t (&row)[N],
                                                 const bool (&ok_in)[N], int q, float4 (&g)[N]) {
  const bool in_dim = q * 4 < t.dim;
  bool ok[N];
  int64_t off[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    ok[i] = ok_in[i] && in_dim;
    off[i] = row[i] * (t.dim >> 2) + q;
  }
  if (t.grad != nullptr) {
    float4 o[N];
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (ok[i]) o[i] = reinterpret_cast<float4*>(t.grad)[off[i]];
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (ok[i]) {
        o[i].x += g[i].x; o[i].y += g[i].y; o[i].z += g[i].z; o[i].w += g[i].w;
        reinterpret_cast<float4*>(t.grad)[off[i]] = o[i];
      }
    return;
  }
  float4 w[N], m[N], v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if (ok[i]) {
      w[i] = reinterpret_cast<float4*>(t.w)[off[i]];
      if (MODE != UPD_SGD) m[i] = reinterpret_cast<float4*>(t.m)[off[i]];
      if (MODE == UPD_ADAM || MODE == UPD_FTRL) v[i] = reinterpret_cast<float4*>(t.v)[off[i]];
    }
  }
  const float l2 = opt.l2_scale;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if (!ok[i]) continue;
    float4 gi = g[i], wi = w[i];
    gi.x = fmaf(l2, wi.x, gi.x); gi.y = fmaf(l2, wi.y, gi.y); gi.z = fmaf(l2, wi.z, gi.z); gi.w = fmaf(l2, wi.w, gi.w);
    if (MODE == UPD_SGD) {
      const float lr = opt.lr;
      wi.x -= lr * gi.x; wi.y -= lr * gi.y; wi.z -= lr * gi.z; wi.w -= lr * gi.w;
    } else if (MODE == UPD_ADAGRAD) {
      float4 ai = m[i];
      const float lr = opt.lr, e = opt.eps;
      adagrad_elem(wi.x, ai.x, gi.x, lr, e); adagrad_elem(wi.y, ai.y, gi.y, lr, e);
      adagrad_elem(wi.z, ai.z, gi.z, lr, e); adagrad_elem(wi.w, ai.w, gi.w, lr, e);
      reinterpret_cast<float4*>(t.m)[off[i]] = ai;
    } else if (MODE == UPD_FTRL) {
      float4 ai = m[i], li = v[i];
      ftrl_row4(wi, ai, li, gi, opt);
      reinterpret_cast<float4*>(t.m)[off[i]] = ai;
      reinterpret_cast<float4*>(t.v)[off[i]] = li;
    } else {
      float4 mi = m[i], vi = v[i];
      const float b1 = opt.beta1, b2 = opt.beta2, e = opt.eps, lr = lr_t;
      mi.x = b1 * mi.x + (1.f - b1) * gi.x; mi.y = b1 * mi.y + (1.f - b1) * gi.y;
      mi.z = b1 * mi.z + (1.f - b1) * gi.z; mi.w = b1 * mi.w + (1.f - b1) * gi.w;
      vi.x = b2 * vi.x + (1.f - b2) * gi.x * gi.x; vi.y = b2 * vi.y + (1.f - b2) * gi.y * gi.y;
      vi.z = b2 * vi.z + (1.f - b2) * gi.z * gi.z; vi.w = b2 * vi.w + (1.f - b2) * gi.w * gi.w;
      wi.x -= lr * mi.x / (sqrtf(vi.x) + e); wi.y -= lr * mi.y / (sqrtf(vi.y) + e);
      wi.z -= lr * mi.z / (sqrtf(vi.z) + e); wi.w -= lr * mi.w / (sqrtf(vi.w) + e);
      reinterpret_cast<float4*>(t.m)[off[i]] = mi;
      reinterpret_cast<float4*>(t.v)[off[i]] = vi;
    }
    reinterpret_cast<float4*>(t.w)[off[i]] = wi;
  }
}

// ---- row-range units of the embedding backward (embedding_bwd.cu) -----------------------------------------------------
struct UnitDev {        // one CTA's share of one table: rows [row_lo, row_hi), whose positions form list `list`
  int32_t table;
  uint32_t row_lo, row_hi;
  int32_t slice, n_slices;  // n_slices > 1: ONE very hot row split over slices of its list (partials summed in slice order)
  int32_t partial_idx;      // first partial slot of the slice group
  int32_t list;             // index of the unit's position list (list_cnt / list_off)
  int32_t pad_;
};
struct ColDev {         // one position column of a table (a plain feature has one, a sequence feature seq_len)
  int32_t pos_col;      // row of the transposed id matrix
  int32_t out_col;      // first gradient column in dout
  int32_t field;        // field index (for the mean-pooling scale)
  int32_t pad_;
};
struct SliceGroupDev {  // a hot row whose slices are combined by bwd_unit_combine_kernel
  int32_t table;
  uint32_t row;
  int32_t partial_idx, n_slices;
};
struct TableSplitDev {  // how the positions of one table are split into unit lists: bin = id >> shift
  int32_t first_list, n_bins, shift;
  int32_t first_tile, n_tiles;
  uint32_t ent_base;    // first slot of this table's lists in the entry arrays
};
struct TileDev {        // 4096 samples of one position column
  int32_t table, col_local, pos_col, chunk;
};
struct UnitSet {        // units of one (plan, batch), grouped by G = dim/4
  int64_t batch = -1;
  void* d_blob = nullptr;
  UnitDev* d_units = nullptr;
  SliceGroupDev* d_groups = nullptr;
  TableSplitDev* d_splits = nullptr;
  TileDev* d_tiles = nullptr;
  int32_t n_units = 0, n_groups = 0, n_partials = 0, n_lists = 0, n_tiles = 0;
  int32_t g_values[8] = {0};                   // distinct G values
  int32_t g_unit_off[9] = {0};                 // units of g_values[i] are [g_unit_off[i], g_unit_off[i+1])
  int32_t g_group_off[9] = {0};
  int32_t n_g = 0;
  bool ok = false;                             // false: this (plan, batch) needs the sorted fallback (too many bins per table)
};

}  // namespace hrb

struct hrb_plan {
  int32_t n_tables = 0, n_fields = 0;
  std::vector<hrb_table_desc> tables;
  std::vector<hrb_field_desc> fields;
  std::vector<hrb::FieldDev> fdev_host;
  std::vector<hrb::TableDev> tdev_host;
  uint64_t total_rows = 0;
  int key_bits = 1;
  int32_t pos_cols = 0;    // sum of seq_len
  int32_t out_chunks = 0;  // sum of dim/4
  int32_t max_dim = 0;
  bool uniform_dim = true;
  bool contiguous_out = true;  // out_col_f == out_col_0 + f*D (needs uniform_dim)
  bool all_len1 = true;
  bool has_max = false;
  // device copies (one allocation)
  void* dev_blob = nullptr;
  hrb::FieldDev* d_fields = nullptr;
  hrb::TableDev* d_tables = nullptr;
  int32_t* d_chunk_field = nullptr;  // out chunk -> field
  int32_t* d_chunk_q = nullptr;      // out chunk -> 4-column group inside the field
  int32_t* d_pos_field = nullptr;    // position column -> field
  uint32_t* d_hot_keys = nullptr;    // keys of every row of the tiny ("hot") tables (see bwd_hot_kernel)
  int32_t n_hot_keys = 0;
  std::vector<uint32_t> hot_lo, hot_len;
  // row-sharded tables read over NVLink peer mappings (hrb_plan_set_peers): owner = id % n_ranks, local row = id / n_ranks
  int32_t n_ranks = 1;
  const float** d_peer_tab = nullptr;  // [n_ranks][n_tables] device pointers (peer-mapped for the other ranks)
  int64_t* d_full_rows = nullptr;      // [n_tables] full vocabulary sizes
  // sort-free backward (embedding_bwd.cu): per-table column lists + the unit decomposition of the last batch size seen
  hrb::ColDev* d_cols = nullptr;       // position columns grouped by table
  int32_t* d_col_start = nullptr;      // [n_tables + 1]
  std::vector<int32_t> col_start_host;
  bool unit_path_ok = false;           // every table: dim/4 a power of two <= 32, at most 256 position columns
  bool has_mean = false;
  int32_t bwd_algo = 0;                // hrb_bwd_algo (hrb_plan_set_bwd_algo)
  mutable std::mutex unit_mu;
  mutable hrb::UnitSet units;
};


namespace hrb {
// embedding_bwd.cu: the sort-free backward of a whole group (row-range units, in-shared-memory sort + segmented reduction)
bool unit_path_supported(const hrb_plan* plan, int64_t batch);
size_t unit_workspace_bytes(const hrb_plan* plan, int64_t batch);
int run_unit_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const float* dout, int64_t dout_ld,
                    const hrb_opt_params& opt, void* workspace, size_t workspace_bytes, cudaStream_t st);
}  // namespace hrb
