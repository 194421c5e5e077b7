// clip.cu -- Keras gradient clipping (OptimizerV2 clipvalue / clipnorm / global_clipnorm) on the device.
//
// Reference: keras/optimizer_v2/optimizer_v2.py `_transform_gradients` (clipvalue, then clipnorm, then global_clipnorm),
// tf.clip_by_value, tf.clip_by_norm and tf.clip_by_global_norm.  The passes run in place between "every gradient is known" and
// the first parameter update; the optimiser kernels themselves are unchanged.
//
// Squared norms are reduced in float64 with a fixed order: every CTA writes its partial to the workspace and the last CTA to
// finish sums the partials in CTA order (and re-zeroes its entry's completion counter), so two runs give the same bits and
// sumsq[var] is within a few float32 roundings of the exact sum.  Workspace layout: one counter per entry point in the first
// 16 bytes (the two entries may share a workspace; neither one's partials cover a counter), then the float64 partials.
#include <math.h>

#include <algorithm>

#include "plan.cuh"

namespace hrb {

constexpr int kClipThreads = 256;
constexpr int kClipSegBlocks = 128;  // CTAs per segment of hrb_clip_prepare_multi at most
constexpr int kClipPlanBlocks = 512;  // CTAs of hrb_plan_clip_grads at most
constexpr int kClipPrepPartials = HRB_MULTI_MAX * kClipSegBlocks;

// clip_by_value without turning a NaN into a bound: comparisons with NaN are false, so it passes through (v = +inf: no clamp)
__device__ __forceinline__ float clamp_v(float x, float v) { return x > v ? v : (x < -v ? -v : x); }

__device__ __forceinline__ double block_sum(double s) {
  __shared__ double red[kClipThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __syncthreads();  // red may still be read by a previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
#pragma unroll
    for (int k = 0; k < kClipThreads / 32; ++k) t += red[k];
  return t;  // valid in thread 0
}

struct ClipPrepArgs {
  float* g[HRB_MULTI_MAX];
  const float* w[HRB_MULTI_MAX];
  int64_t n[HRB_MULTI_MAX];
  float l2[HRB_MULTI_MAX];
  int32_t var[HRB_MULTI_MAX];
  int32_t first_block[HRB_MULTI_MAX + 1];
  int32_t count;
};

// g <- clamp(fmaf(l2, w, g), -v, v) (the fmaf of every optimiser kernel, so that the optimiser may then run with l2 = 0);
// sumsq[var] += sum g'^2 when sumsq != nullptr
__global__ void __launch_bounds__(kClipThreads) clip_prepare_kernel(const ClipPrepArgs a, float v, float* __restrict__ sumsq,
                                                                      double* __restrict__ partial, unsigned int* __restrict__ counter) {
  int t = 0;
  while (t + 1 < a.count && (int)blockIdx.x >= a.first_block[t + 1]) ++t;
  const int64_t nb = a.first_block[t + 1] - a.first_block[t];
  const int64_t b = blockIdx.x - a.first_block[t];
  float* __restrict__ g = a.g[t];
  const float* __restrict__ w = a.w[t];
  const float l2 = a.l2[t];
  double s = 0.0;
  for (int64_t i = b * kClipThreads + threadIdx.x; i < a.n[t]; i += nb * kClipThreads) {
    float x = g[i];
    if (w != nullptr) x = fmaf(l2, w[i], x);
    x = clamp_v(x, v);
    g[i] = x;
    s = __fma_rn((double)x, (double)x, s);
  }
  if (sumsq == nullptr) return;
  s = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
  if (!last_block(counter)) return;
  __shared__ double seg[HRB_MULTI_MAX];
  if (threadIdx.x < a.count) {
    double u = 0.0;
    for (int k = a.first_block[threadIdx.x]; k < a.first_block[threadIdx.x + 1]; ++k) u += __ldcg(partial + k);
    seg[threadIdx.x] = u;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < a.count; ++k) sumsq[a.var[k]] = (float)((double)sumsq[a.var[k]] + seg[k]);
    *counter = 0u;
  }
}

// g *= scale[var]
__global__ void __launch_bounds__(kClipThreads) clip_apply_kernel(const ClipPrepArgs a, const float* __restrict__ scale) {
  int t = 0;
  while (t + 1 < a.count && (int)blockIdx.x >= a.first_block[t + 1]) ++t;
  const int64_t nb = a.first_block[t + 1] - a.first_block[t];
  const int64_t b = blockIdx.x - a.first_block[t];
  float* __restrict__ g = a.g[t];
  const float s = scale[a.var[t]];
  for (int64_t i = b * kClipThreads + threadIdx.x; i < a.n[t]; i += nb * kClipThreads) g[i] *= s;
}

// valid positions of field f in one sample, as the backward counts them (bwd_keys_kernel): in-range ids, and for pooled fields
// ids != 0
__device__ __forceinline__ int field_valid(const FieldDev& f, const int32_t* __restrict__ ids_row) {
  int cnt = 0;
  for (int l = 0; l < f.seq_len; ++l) {
    const int32_t id = __ldg(ids_row + f.ids_col + l);
    cnt += (f.pool == HRB_POOL_NONE || id != 0) && id >= 0 && (int64_t)id < f.rows;
  }
  return cnt;
}

// One (dnn, fm) part of a position value: p = part * inv, clamped to [-v, v]; the value the backward reads back for it is the
// part itself unless the clamp binds, then +-v * n (so that * inv gives the clamped value).  Returns that value, c = clamp(p).
__device__ __forceinline__ float clip_part(float part, float inv, float n_scale, float v, float& c) {
  const float p = part * inv;
  c = clamp_v(p, v);
  return (p > v || p < -v) ? c * n_scale : part;
}

// Per (sample, field, 4 floats): the DNN part in dx and the FM part in fm are clamped separately per position and dx receives
// their sum; per table, sum over valid positions of (p_dnn'^2 + p_fm'^2).  Fields in an outer loop: a CTA's sums of one field
// are reduced before the next field starts, in field order.
__global__ void __launch_bounds__(kClipThreads) plan_clip_grads_kernel(const FieldDev* __restrict__ fields, int32_t n_fields,
                                                                         int32_t n_tables, int32_t G, const int32_t* __restrict__ ids,
                                                                         int64_t ids_ld, int64_t batch, float* __restrict__ dx,
                                                                         int64_t dx_ld, const float* __restrict__ fm, int64_t fm_ld,
                                                                         int32_t out0, float v, float* __restrict__ sumsq,
                                                                         double* __restrict__ partial, unsigned int* __restrict__ counter) {
  extern __shared__ double tab_sum[];  // n_tables
  for (int t = threadIdx.x; t < n_tables; t += kClipThreads) tab_sum[t] = 0.0;
  const int64_t total = batch * G;
  for (int fi = 0; fi < n_fields; ++fi) {
    const FieldDev f = fields[fi];
    double s = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)kClipThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kClipThreads) {
      const int64_t b = i / G;
      const int q = (int)(i - b * G);
      const int n = field_valid(f, ids + b * ids_ld);
      const float inv = f.pool == HRB_POOL_MEAN ? (n > 0 ? __fdiv_rn(1.0f, (float)n) : 0.f) : 1.0f;
      const float n_scale = f.pool == HRB_POOL_MEAN ? (float)n : 1.0f;
      float4* dp = reinterpret_cast<float4*>(dx + b * dx_ld + f.out_col) + q;
      float4 d = *dp;
      float4 m = fm != nullptr ? __ldg(reinterpret_cast<const float4*>(fm + b * fm_ld + (f.out_col - out0)) + q)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
      float cd, cf;
      double e = 0.0;
      d.x = clip_part(d.x, inv, n_scale, v, cd) + clip_part(m.x, inv, n_scale, v, cf); e = __fma_rn((double)cd, (double)cd, __fma_rn((double)cf, (double)cf, e));
      d.y = clip_part(d.y, inv, n_scale, v, cd) + clip_part(m.y, inv, n_scale, v, cf); e = __fma_rn((double)cd, (double)cd, __fma_rn((double)cf, (double)cf, e));
      d.z = clip_part(d.z, inv, n_scale, v, cd) + clip_part(m.z, inv, n_scale, v, cf); e = __fma_rn((double)cd, (double)cd, __fma_rn((double)cf, (double)cf, e));
      d.w = clip_part(d.w, inv, n_scale, v, cd) + clip_part(m.w, inv, n_scale, v, cf); e = __fma_rn((double)cd, (double)cd, __fma_rn((double)cf, (double)cf, e));
      *dp = d;
      s = __fma_rn((double)n, e, s);
    }
    if (sumsq == nullptr) continue;
    s = block_sum(s);
    if (threadIdx.x == 0) tab_sum[f.table_idx] += s;
  }
  if (sumsq == nullptr) return;
  __syncthreads();
  for (int t = threadIdx.x; t < n_tables; t += kClipThreads) partial[(int64_t)blockIdx.x * n_tables + t] = tab_sum[t];
  if (!last_block(counter)) return;
  for (int t = threadIdx.x; t < n_tables; t += kClipThreads) {
    double u = 0.0;
    for (int k = 0; k < (int)gridDim.x; ++k) u += __ldcg(partial + (int64_t)k * n_tables + t);
    sumsq[t] = (float)((double)sumsq[t] + u);
  }
  __syncthreads();
  if (threadIdx.x == 0) *counter = 0u;
}

// dx[b, field f] *= scale[table of f]
__global__ void __launch_bounds__(kClipThreads) plan_clip_apply_kernel(const FieldDev* __restrict__ fields, int32_t n_fields, int32_t G,
                                                                         int64_t batch, float* __restrict__ dx, int64_t dx_ld,
                                                                         const float* __restrict__ scale) {
  const int64_t total = batch * n_fields * G;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / (n_fields * G);
    const int r = (int)(i - b * n_fields * G);
    const int fi = r / G, q = r - fi * G;
    const float s = scale[fields[fi].table_idx];
    float4* dp = reinterpret_cast<float4*>(dx + b * dx_ld + fields[fi].out_col) + q;
    float4 d = *dp;
    d.x *= s; d.y *= s; d.z *= s; d.w *= s;
    *dp = d;
  }
}

// s = c / max(norm, c) per variable, or one s from the global norm (NaN when it is not finite).  max() propagates a NaN norm.
__global__ void clip_scales_kernel(const float* __restrict__ sumsq, int32_t n_vars, float c, int32_t global, float* __restrict__ scale) {
  if (global) {
    __shared__ float s_all;
    if (threadIdx.x == 0) {
      double tot = 0.0;
      for (int k = 0; k < n_vars; ++k) tot += (double)sumsq[k];
      const float norm = (float)sqrt(tot);
      s_all = isfinite(norm) ? __fdiv_rn(c, norm <= c ? c : norm) : NAN;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < n_vars; k += blockDim.x) scale[k] = s_all;
    return;
  }
  for (int k = threadIdx.x; k < n_vars; k += blockDim.x) {
    const float norm = sqrtf(sumsq[k]);
    scale[k] = __fdiv_rn(c, norm <= c ? c : norm);
  }
}

constexpr size_t kClipCounterBytes = 16;  // [0]: hrb_clip_prepare_multi's counter, [1]: hrb_plan_clip_grads's
enum ClipCounter { kPrepCounter = 0, kPlanCounter = 1 };

static size_t clip_ws_bytes(int32_t n_tables) {
  const size_t parts = std::max<size_t>(kClipPrepPartials, (size_t)kClipPlanBlocks * (size_t)std::max(n_tables, 1));
  return kClipCounterBytes + parts * sizeof(double);
}
static unsigned int* ws_counter(void* ws, ClipCounter c) { return (unsigned int*)ws + c; }
static double* ws_partials(void* ws) { return (double*)((char*)ws + kClipCounterBytes); }

static void fill_segments(ClipPrepArgs& a, int32_t c0, int32_t count, float* const* g, const float* const* w, const int64_t* n,
                          const float* l2, const int32_t* var) {
  a = ClipPrepArgs{};
  int blocks = 0;
  for (int32_t i = c0; i < count && i < c0 + HRB_MULTI_MAX; ++i) {
    if (n[i] == 0) continue;
    const int k = a.count++;
    a.g[k] = g[i];
    a.w[k] = w != nullptr ? w[i] : nullptr;
    a.n[k] = n[i];
    a.l2[k] = l2 != nullptr ? l2[i] : 0.f;
    a.var[k] = var[i];
    a.first_block[k] = blocks;
    blocks += (int)std::min<int64_t>(kClipSegBlocks, (n[i] + 2047) / 2048);
  }
  a.first_block[a.count] = blocks;
}

static int check_segments(const char* fn, int32_t count, float* const* g, const int64_t* n, const int32_t* var, int32_t n_vars) {
  HRB_REQUIRE(count >= 0 && (count == 0 || (g && n && var)), "%s: bad argument", fn);
  for (int32_t i = 0; i < count; ++i) {
    HRB_REQUIRE(n[i] >= 0 && (n[i] == 0 || g[i]), "%s: null or negative segment %d", fn, i);
    HRB_REQUIRE(var[i] >= 0 && (n_vars < 0 || var[i] < n_vars), "%s: segment %d has variable index %d", fn, i, var[i]);
  }
  return HRB_OK;
}

static int plan_fields_ok(const hrb_plan* plan, const char* fn) {
  HRB_REQUIRE(plan->uniform_dim && plan->max_dim % 4 == 0, "%s: the plan's fields need one embedding dim, a multiple of 4", fn);
  if (plan->has_max) return fail(HRB_UNSUPPORTED, "%s: max-pooled fields are not supported", fn);
  return HRB_OK;
}

}  // namespace hrb

using namespace hrb;

HRB_API int hrb_clip_workspace_bytes(int32_t n_tables, size_t* bytes) {
  HRB_REQUIRE(bytes && n_tables >= 0, "hrb_clip_workspace_bytes: bad argument");
  *bytes = clip_ws_bytes(n_tables);
  return HRB_OK;
}

HRB_API int hrb_clip_prepare_multi(int32_t count, float* const* g_host, const float* const* w_host, const int64_t* n_host,
                                   const float* l2_scale_host, const int32_t* var_host, float clipvalue, float* sumsq, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (int rc = check_segments("hrb_clip_prepare_multi", count, g_host, n_host, var_host, -1)) return rc;
  HRB_REQUIRE(!(clipvalue < 0.f), "hrb_clip_prepare_multi: clipvalue %g < 0", (double)clipvalue);
  HRB_REQUIRE(sumsq == nullptr || (workspace && workspace_bytes >= clip_ws_bytes(0)), "hrb_clip_prepare_multi: workspace too small");
  for (int32_t i = 0; w_host && i < count; ++i)
    HRB_REQUIRE(w_host[i] != nullptr || l2_scale_host == nullptr || l2_scale_host[i] == 0.f,
                "hrb_clip_prepare_multi: segment %d has l2 but no weights", i);
  double* partial = sumsq != nullptr ? ws_partials(workspace) : nullptr;
  unsigned int* counter = sumsq != nullptr ? ws_counter(workspace, kPrepCounter) : nullptr;
  for (int32_t c0 = 0; c0 < count; c0 += HRB_MULTI_MAX) {
    ClipPrepArgs a;
    fill_segments(a, c0, count, g_host, w_host, n_host, l2_scale_host, var_host);
    if (a.count == 0) continue;
    clip_prepare_kernel<<<a.first_block[a.count], kClipThreads, 0, (cudaStream_t)stream>>>(a, clipvalue, sumsq, partial, counter);
    HRB_LAUNCH_CHECK();
  }
  return HRB_OK;
}

HRB_API int hrb_clip_scales(const float* sumsq, int32_t n_vars, float clipnorm, int32_t global, float* scale, void* stream) {
  HRB_REQUIRE(sumsq && scale && n_vars >= 0 && clipnorm >= 0.f, "hrb_clip_scales: bad argument");
  if (n_vars == 0) return HRB_OK;
  clip_scales_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(sumsq, n_vars, clipnorm, global, scale);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_clip_apply_multi(int32_t count, float* const* g_host, const int64_t* n_host, const int32_t* var_host, const float* scale,
                                 void* stream) {
  if (int rc = check_segments("hrb_clip_apply_multi", count, g_host, n_host, var_host, -1)) return rc;
  HRB_REQUIRE(count == 0 || scale, "hrb_clip_apply_multi: null scale");
  for (int32_t c0 = 0; c0 < count; c0 += HRB_MULTI_MAX) {
    ClipPrepArgs a;
    fill_segments(a, c0, count, g_host, nullptr, n_host, nullptr, var_host);
    if (a.count == 0) continue;
    clip_apply_kernel<<<a.first_block[a.count], kClipThreads, 0, (cudaStream_t)stream>>>(a, scale);
    HRB_LAUNCH_CHECK();
  }
  return HRB_OK;
}

HRB_API int hrb_plan_clip_grads(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* dx, int64_t dx_ld,
                                const float* fm, int64_t fm_ld, float clipvalue, float* sumsq, void* workspace, size_t workspace_bytes,
                                void* stream) {
  HRB_REQUIRE(plan && batch >= 0, "hrb_plan_clip_grads: bad argument");
  if (int rc = plan_fields_ok(plan, "hrb_plan_clip_grads")) return rc;
  HRB_REQUIRE(!(clipvalue < 0.f), "hrb_plan_clip_grads: clipvalue %g < 0", (double)clipvalue);
  HRB_REQUIRE(fm == nullptr || plan->contiguous_out, "hrb_plan_clip_grads: an FM part needs contiguous field columns");
  HRB_REQUIRE(sumsq == nullptr || (workspace && workspace_bytes >= clip_ws_bytes(plan->n_tables)), "hrb_plan_clip_grads: workspace too small");
  if (batch == 0 || plan->n_fields == 0) return HRB_OK;
  HRB_REQUIRE(ids && dx && ids_ld >= plan->pos_cols && aligned16(dx) && dx_ld % 4 == 0 && (fm == nullptr || (aligned16(fm) && fm_ld % 4 == 0)),
              "hrb_plan_clip_grads: null or misaligned buffer");
  const int32_t G = plan->max_dim / 4;
  const int64_t blocks = std::min<int64_t>(kClipPlanBlocks, (batch * G + kClipThreads - 1) / kClipThreads);
  const size_t smem = sizeof(double) * std::max(plan->n_tables, 1);
  HRB_REQUIRE(smem <= 48 * 1024, "hrb_plan_clip_grads: too many tables (%d)", plan->n_tables);
  double* partial = sumsq != nullptr ? ws_partials(workspace) : nullptr;
  unsigned int* counter = sumsq != nullptr ? ws_counter(workspace, kPlanCounter) : nullptr;
  plan_clip_grads_kernel<<<(unsigned)blocks, kClipThreads, smem, (cudaStream_t)stream>>>(
      plan->d_fields, plan->n_fields, plan->n_tables, G, ids, ids_ld, batch, dx, dx_ld, fm, fm_ld, plan->fields[0].out_col, clipvalue,
      sumsq, partial, counter);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_plan_clip_apply(const hrb_plan* plan, float* dx, int64_t dx_ld, int64_t batch, const float* scale, void* stream) {
  HRB_REQUIRE(plan && batch >= 0, "hrb_plan_clip_apply: bad argument");
  if (int rc = plan_fields_ok(plan, "hrb_plan_clip_apply")) return rc;
  if (batch == 0 || plan->n_fields == 0) return HRB_OK;
  HRB_REQUIRE(dx && scale && aligned16(dx) && dx_ld % 4 == 0, "hrb_plan_clip_apply: null or misaligned buffer");
  const int32_t G = plan->max_dim / 4;
  const int64_t total = batch * plan->n_fields * G;
  const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 8);
  plan_clip_apply_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(plan->d_fields, plan->n_fields, G, batch, dx, dx_ld, scale);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
