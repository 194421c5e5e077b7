// misc.cu -- DeepFM head + loss, Dice activation, dense-parameter optimisers.
//
// Reference: models/ranking/context_aware/DeepFM.py:86-88 (dnn + fm -> sigmoid), Keras
// binary_crossentropy on a sigmoid output (= sigmoid cross-entropy with logits),
// layers/activation.py:27-42 (Dice), Keras Adam / SGD / Adagrad / Ftrl update formulas.
#include "common.cuh"

namespace hrb {

// WEIGHTED: Keras' sample weights enter at the loss, loss_sum += w*l and dlogit = (p-y)*w*grad_scale; w = 1 leaves every bit of
// prob and dlogit as the unweighted instantiation computes them
template <bool WEIGHTED>
__global__ void __launch_bounds__(256) sigmoid_bce_kernel(const float* __restrict__ dnn, const float* __restrict__ fmv,
                                                         const float* __restrict__ label, const float* __restrict__ weight,
                                                         int64_t batch, float grad_scale, float* __restrict__ prob,
                                                         float* __restrict__ dlogit, float* __restrict__ loss_sum) {
  __shared__ float red[8];
  float local = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < batch; i += (int64_t)gridDim.x * blockDim.x) {
    const float z = dnn[i] + (fmv != nullptr ? fmv[i] : 0.f);
    const float p = sigmoidf_(z);
    const float y = label[i];
    // max(z,0) - z*y + log1p(exp(-|z|))  (tf.nn.sigmoid_cross_entropy_with_logits)
    const float l = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
    if (prob != nullptr) prob[i] = p;
    if constexpr (WEIGHTED) {
      const float w = weight[i];
      local += w * l;
      if (dlogit != nullptr) dlogit[i] = (p - y) * w * grad_scale;
    } else {
      local += l;
      if (dlogit != nullptr) dlogit[i] = (p - y) * grad_scale;
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0 && loss_sum != nullptr) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k];
    atomicAdd(loss_sum, t);
  }
}

// Keras binary_crossentropy on PROBABILITIES (no cached logits): p is clipped to [eps, 1-eps]; the gradient of the clip is 0 outside
template <bool WEIGHTED>
__global__ void __launch_bounds__(256) clipped_bce_kernel(const float* __restrict__ prob, const float* __restrict__ label,
                                                         const float* __restrict__ weight, int64_t n, float eps, float grad_scale,
                                                         float* __restrict__ dprob, float* __restrict__ loss_sum) {
  __shared__ float red[8];
  float local = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float p0 = prob[i], y = label[i];
    const float p = fminf(fmaxf(p0, eps), 1.0f - eps);
    if constexpr (WEIGHTED) {
      const float w = weight[i];
      local -= w * (y * logf(p) + (1.0f - y) * logf(1.0f - p));
      if (dprob != nullptr) dprob[i] = (p0 >= eps && p0 <= 1.0f - eps) ? ((1.0f - y) / (1.0f - p) - y / p) * w * grad_scale : 0.f;
    } else {
      local -= y * logf(p) + (1.0f - y) * logf(1.0f - p);
      if (dprob != nullptr) dprob[i] = (p0 >= eps && p0 <= 1.0f - eps) ? ((1.0f - y) / (1.0f - p) - y / p) * grad_scale : 0.f;
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0 && loss_sum != nullptr) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k];
    atomicAdd(loss_sum, t);
  }
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                  float* __restrict__ v, int64_t n, float lr_t, float b1, float b2,
                                                  float eps, float l2_scale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float w = p[i];
    const float gi = fmaf(l2_scale, w, g[i]);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] = w - lr_t * mi / (sqrtf(vi) + eps);
  }
}

__global__ void __launch_bounds__(256) sgd_kernel(float* __restrict__ p, const float* __restrict__ g, int64_t n, float lr,
                                                 float l2_scale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float w = p[i];
    p[i] = w - lr * fmaf(l2_scale, w, g[i]);
  }
}

// Keras Adagrad (ResourceApplyAdagradV2): eps outside the square root, no step counter
__device__ __forceinline__ float adagrad_update(float w, float& acc, float g, float lr, float eps) {
  acc = fmaf(g, g, acc);
  return w - lr * g / (sqrtf(acc) + eps);
}

__global__ void __launch_bounds__(256) adagrad_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ acc, int64_t n,
                                                     float lr, float eps, float l2_scale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float w = p[i];
    float a = acc[i];
    p[i] = adagrad_update(w, a, fmaf(l2_scale, w, g[i]), lr, eps);
    acc[i] = a;
  }
}

// Keras Ftrl (ResourceApplyFtrl / V2; ftrl_elem, common.cuh).  row_touched != nullptr: elements of rows (dim floats) whose flag is
// 0 are neither read nor written -- the rows an embedding table's IndexedSlices gradient does not list keep their bits.
__global__ void __launch_bounds__(256) ftrl_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ acc,
                                                  float* __restrict__ lin, int64_t n, float lr, float l1, float l2, float lr_power,
                                                  float l2_shrinkage, float l2_scale, const float* __restrict__ row_touched, int32_t dim) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (row_touched != nullptr && row_touched[i / dim] == 0.f) continue;
    const float w = p[i];
    float a = acc[i], l = lin[i];
    p[i] = ftrl_elem(w, a, l, fmaf(l2_scale, w, g[i]), lr, l1, l2, lr_power, l2_shrinkage);
    acc[i] = a;
    lin[i] = l;
  }
}

// Many small parameter tensors in ONE launch (the layer-by-layer models step 12-27 tensors: one launch each was 0.4 ms of
// host time per step).  Block b works on the tensor whose block range contains it; same arithmetic as adam_kernel / sgd_kernel /
// adagrad_kernel / ftrl_kernel.  m holds the Adagrad or Ftrl accumulator, v the Ftrl linear slot.
struct MultiArgs {
  float* p[HRB_MULTI_MAX];
  const float* g[HRB_MULTI_MAX];
  float* m[HRB_MULTI_MAX];
  float* v[HRB_MULTI_MAX];
  int64_t n[HRB_MULTI_MAX];
  float l2[HRB_MULTI_MAX];
  int32_t first_block[HRB_MULTI_MAX + 1];
  int32_t count;
};
enum MultiOpt { MULTI_SGD, MULTI_ADAM, MULTI_ADAGRAD, MULTI_FTRL };
struct FtrlArgs {
  float l1, l2, lr_power, l2_shrinkage;
};
template <int OPT>
__global__ void __launch_bounds__(256) multi_step_kernel(const MultiArgs a, float lr_t, float b1, float b2, float eps, const FtrlArgs f) {
  int t = 0;
  while (t + 1 < a.count && (int)blockIdx.x >= a.first_block[t + 1]) ++t;
  const int64_t nb = a.first_block[t + 1] - a.first_block[t];
  const int64_t b = blockIdx.x - a.first_block[t];
  float* __restrict__ p = a.p[t];
  const float* __restrict__ g = a.g[t];
  const float l2 = a.l2[t];
  for (int64_t i = b * blockDim.x + threadIdx.x; i < a.n[t]; i += nb * blockDim.x) {
    const float w = p[i];
    const float gi = fmaf(l2, w, g[i]);
    if (OPT == MULTI_ADAM) {
      const float mi = b1 * a.m[t][i] + (1.f - b1) * gi;
      const float vi = b2 * a.v[t][i] + (1.f - b2) * gi * gi;
      a.m[t][i] = mi;
      a.v[t][i] = vi;
      p[i] = w - lr_t * mi / (sqrtf(vi) + eps);
    } else if (OPT == MULTI_ADAGRAD) {
      float acc = a.m[t][i];
      p[i] = adagrad_update(w, acc, gi, lr_t, eps);
      a.m[t][i] = acc;
    } else if (OPT == MULTI_FTRL) {
      float acc = a.m[t][i], lin = a.v[t][i];
      p[i] = ftrl_elem(w, acc, lin, gi, lr_t, f.l1, f.l2, f.lr_power, f.l2_shrinkage);
      a.m[t][i] = acc;
      a.v[t][i] = lin;
    } else {
      p[i] = w - lr_t * gi;
    }
  }
}

// ---- Dice ---------------------------------------------------------------------------------
// column sums of f(x) over a row slab; 32 columns x 8 row lanes per CTA, one atomic per column per CTA
template <int MODE>  // 0: sum x   1: sum (x-mean)^2   2: {sum dz, sum dz*zhat} for the BN backward
__global__ void __launch_bounds__(256) dice_colstat_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                          int64_t rows, int32_t units, int64_t rows_per_block,
                                                          const float* __restrict__ alpha, const float* __restrict__ mean,
                                                          const float* __restrict__ var, float eps,
                                                          float* __restrict__ out0, float* __restrict__ out1) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  __shared__ float r0s[8][33], r1s[8][33];
  const int64_t rbeg = (int64_t)blockIdx.y * rows_per_block;
  const int64_t rend = min(rows, rbeg + rows_per_block);
  float s0 = 0.f, s1 = 0.f;
  if (n < units) {
    const float mu = MODE >= 1 ? mean[n] : 0.f;
    const float rstd = MODE == 2 ? rsqrtf(var[n] + eps) : 0.f;
    const float al = MODE == 2 ? alpha[n] : 0.f;
    for (int64_t r = rbeg + ry; r < rend; r += 8) {
      const float v = __ldg(x + r * units + n);
      if (MODE == 0) {
        s0 += v;
      } else if (MODE == 1) {
        const float c = v - mu;
        s0 = fmaf(c, c, s0);
      } else {
        const float zh = (v - mu) * rstd;
        const float p = sigmoidf_(zh);
        const float dz = __ldg(dy + r * units + n) * v * (1.f - al) * p * (1.f - p);
        s0 += dz;
        s1 = fmaf(dz, zh, s1);
      }
    }
  }
  r0s[ry][threadIdx.x & 31] = s0;
  r1s[ry][threadIdx.x & 31] = s1;
  __syncthreads();
  if (ry == 0 && n < units) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      a += r0s[k][threadIdx.x & 31];
      b += r1s[k][threadIdx.x & 31];
    }
    atomicAdd(out0 + n, a);
    if (MODE == 2) atomicAdd(out1 + n, b);
  }
}

__global__ void scale_kernel(float* __restrict__ v, int32_t n, float s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= s;
}

__global__ void __launch_bounds__(256) dice_apply_kernel(const float* __restrict__ x, int64_t total, int32_t units,
                                                        const float* __restrict__ alpha, const float* __restrict__ mean,
                                                        const float* __restrict__ var, float eps, float* __restrict__ y) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i % units);
    const float v = x[i];
    const float p = sigmoidf_((v - mean[n]) * rsqrtf(var[n] + eps));  // activation.py:40-41
    y[i] = p * v + (1.0f - p) * alpha[n] * v;                          // activation.py:42
  }
}

// dx and dalpha.  training: BN backward through the batch statistics (sums in stat = {sum dz, sum dz*zhat}).
__global__ void __launch_bounds__(256) dice_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                      int64_t rows, int32_t units, int64_t rows_per_block,
                                                      const float* __restrict__ alpha, const float* __restrict__ mean,
                                                      const float* __restrict__ var, float eps, int32_t training,
                                                      const float* __restrict__ stat, float* __restrict__ dx,
                                                      float* __restrict__ dalpha) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  __shared__ float red[8][33];
  const int64_t rbeg = (int64_t)blockIdx.y * rows_per_block;
  const int64_t rend = min(rows, rbeg + rows_per_block);
  float da = 0.f;
  if (n < units) {
    const float mu = mean[n], rstd = rsqrtf(var[n] + eps), al = alpha[n];
    const float inv_rows = 1.0f / (float)rows;
    const float m_dz = training ? stat[n] * inv_rows : 0.f;
    const float m_dzz = training ? stat[units + n] * inv_rows : 0.f;
    for (int64_t r = rbeg + ry; r < rend; r += 8) {
      const float v = __ldg(x + r * units + n);
      const float g = __ldg(dy + r * units + n);
      const float zh = (v - mu) * rstd;
      const float p = sigmoidf_(zh);
      const float dz = g * v * (1.f - al) * p * (1.f - p);
      float d = g * (p + (1.f - p) * al);
      d += training ? rstd * (dz - m_dz - zh * m_dzz) : rstd * dz;
      dx[r * units + n] = d;
      da = fmaf(g * (1.f - p), v, da);
    }
  }
  red[ry][threadIdx.x & 31] = da;
  __syncthreads();
  if (ry == 0 && n < units && dalpha != nullptr) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) a += red[k][threadIdx.x & 31];
    atomicAdd(dalpha + n, a);
  }
}

// dense features -> the head columns of the DNN input row (layers/utils.py:28-36 casts ints to fp32)
template <typename T>
__global__ void __launch_bounds__(256) pack_dense_kernel(const T* __restrict__ src, int64_t src_ld, int64_t batch,
                                                        int32_t n, int32_t n_pad, float* __restrict__ dst, int64_t dst_ld) {
  const int64_t total = batch * n_pad;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_pad;
    const int c = (int)(i - b * n_pad);
    dst[b * dst_ld + c] = c < n ? (float)src[b * src_ld + c] : 0.0f;
  }
}

static inline unsigned ew_grid(int64_t n) {
  int64_t b = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

static inline void slab_grid(int64_t rows, int32_t units, dim3& grid, int64_t& rpb) {
  int yb = (int)min((int64_t)sm_count() * 2, (rows + 63) / 64);
  if (yb < 1) yb = 1;
  rpb = (rows + yb - 1) / yb;
  grid = dim3((units + 31) / 32, yb);
}

}  // namespace hrb

using namespace hrb;

HRB_API int hrb_sigmoid_bce(const float* dnn_logit, const float* fm_logit, const float* label, int64_t batch,
                            float grad_scale, float* prob, float* dlogit, float* loss_sum, void* stream) {
  HRB_REQUIRE(dnn_logit && label && batch >= 0, "hrb_sigmoid_bce: null/negative argument");
  if (batch == 0) return HRB_OK;
  sigmoid_bce_kernel<false><<<ew_grid(batch), 256, 0, (cudaStream_t)stream>>>(dnn_logit, fm_logit, label, nullptr, batch, grad_scale,
                                                                             prob, dlogit, loss_sum);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_sigmoid_bce_weighted(const float* dnn_logit, const float* fm_logit, const float* label, const float* weight,
                                     int64_t batch, float grad_scale, float* prob, float* dlogit, float* loss_sum, void* stream) {
  HRB_REQUIRE(dnn_logit && label && weight && batch >= 0, "hrb_sigmoid_bce_weighted: null/negative argument");
  if (batch == 0) return HRB_OK;
  sigmoid_bce_kernel<true><<<ew_grid(batch), 256, 0, (cudaStream_t)stream>>>(dnn_logit, fm_logit, label, weight, batch, grad_scale,
                                                                            prob, dlogit, loss_sum);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_clipped_bce(const float* prob, const float* label, int64_t n, float eps, float grad_scale, float* dprob,
                            float* loss_sum, void* stream) {
  HRB_REQUIRE(prob && label && n >= 0, "hrb_clipped_bce: null/negative argument");
  if (n == 0) return HRB_OK;
  clipped_bce_kernel<false><<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(prob, label, nullptr, n, eps, grad_scale, dprob, loss_sum);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_clipped_bce_weighted(const float* prob, const float* label, const float* weight, int64_t n, float eps, float grad_scale,
                                     float* dprob, float* loss_sum, void* stream) {
  HRB_REQUIRE(prob && label && weight && n >= 0, "hrb_clipped_bce_weighted: null/negative argument");
  if (n == 0) return HRB_OK;
  clipped_bce_kernel<true><<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(prob, label, weight, n, eps, grad_scale, dprob, loss_sum);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_adam_step(float* param, const float* grad, float* m, float* v, int64_t n, float lr, float beta1,
                          float beta2, float eps, float bias_corr1, float bias_corr2, float l2_scale, void* stream) {
  HRB_REQUIRE(param && grad && m && v && n >= 0 && bias_corr1 > 0.f && bias_corr2 > 0.f, "hrb_adam_step: bad argument");
  if (n == 0) return HRB_OK;
  const float lr_t = lr * sqrtf(bias_corr2) / bias_corr1;  // Keras Adam: lr * sqrt(1-b2^t)/(1-b1^t), eps un-corrected
  adam_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(param, grad, m, v, n, lr_t, beta1, beta2, eps, l2_scale);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_adagrad_step(float* param, const float* grad, float* acc, int64_t n, float lr, float eps, float l2_scale, void* stream) {
  HRB_REQUIRE(param && grad && acc && n >= 0, "hrb_adagrad_step: bad argument");
  if (n == 0) return HRB_OK;
  adagrad_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(param, grad, acc, n, lr, eps, l2_scale);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_ftrl_step(float* param, const float* grad, float* acc, float* lin, int64_t n, float lr, float l1, float l2, float lr_power,
                          float l2_shrinkage, float l2_scale, const float* row_touched, int32_t dim, void* stream) {
  HRB_REQUIRE(param && grad && acc && lin && n >= 0 && lr > 0.f, "hrb_ftrl_step: bad argument");
  HRB_REQUIRE(row_touched == nullptr || (dim > 0 && n % dim == 0), "hrb_ftrl_step: n = %lld is not a multiple of dim = %d", (long long)n, dim);
  if (n == 0) return HRB_OK;
  ftrl_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(param, grad, acc, lin, n, lr, l1, l2, lr_power, l2_shrinkage, l2_scale,
                                                            row_touched, dim);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_sgd_step(float* param, const float* grad, int64_t n, float lr, float l2_scale, void* stream) {
  HRB_REQUIRE(param && grad && n >= 0, "hrb_sgd_step: bad argument");
  if (n == 0) return HRB_OK;
  sgd_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(param, grad, n, lr, l2_scale);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

static int multi_step(int opt, int32_t count, float* const* param, const float* const* grad, float* const* m, float* const* v,
                      const int64_t* n, const float* l2_scale, float lr_t, float b1, float b2, float eps, cudaStream_t st,
                      FtrlArgs f = FtrlArgs{}) {
  for (int32_t c0 = 0; c0 < count; c0 += HRB_MULTI_MAX) {
    MultiArgs a{};
    int blocks = 0;
    for (int32_t i = c0; i < count && i < c0 + HRB_MULTI_MAX; ++i) {
      HRB_REQUIRE(n[i] >= 0 && (n[i] == 0 || (param[i] && grad[i] && (opt == MULTI_SGD || m[i]) && ((opt != MULTI_ADAM && opt != MULTI_FTRL) || v[i]))),
                  "multi-tensor step: null tensor %d", i);
      if (n[i] == 0) continue;
      const int k = a.count++;
      a.p[k] = param[i];
      a.g[k] = grad[i];
      a.m[k] = opt != MULTI_SGD ? m[i] : nullptr;
      a.v[k] = (opt == MULTI_ADAM || opt == MULTI_FTRL) ? v[i] : nullptr;
      a.n[k] = n[i];
      a.l2[k] = l2_scale ? l2_scale[i] : 0.f;
      a.first_block[k] = blocks;
      blocks += (int)std::min<int64_t>(sm_count() * 2, (n[i] + 1023) / 1024);  // >= 1 block, 4 elements per thread for large tensors
    }
    if (a.count == 0) continue;
    a.first_block[a.count] = blocks;
    if (opt == MULTI_ADAM) multi_step_kernel<MULTI_ADAM><<<blocks, 256, 0, st>>>(a, lr_t, b1, b2, eps, f);
    else if (opt == MULTI_ADAGRAD) multi_step_kernel<MULTI_ADAGRAD><<<blocks, 256, 0, st>>>(a, lr_t, b1, b2, eps, f);
    else if (opt == MULTI_FTRL) multi_step_kernel<MULTI_FTRL><<<blocks, 256, 0, st>>>(a, lr_t, b1, b2, eps, f);
    else multi_step_kernel<MULTI_SGD><<<blocks, 256, 0, st>>>(a, lr_t, b1, b2, eps, f);
    HRB_LAUNCH_CHECK();
  }
  return HRB_OK;
}

HRB_API int hrb_adam_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* m_host,
                                float* const* v_host, const int64_t* n_host, const float* l2_scale_host, float lr, float beta1,
                                float beta2, float eps, float bias_corr1, float bias_corr2, void* stream) {
  HRB_REQUIRE(count >= 0 && (count == 0 || (param_host && grad_host && m_host && v_host && n_host)) && bias_corr1 > 0.f,
              "hrb_adam_step_multi: bad argument");
  return multi_step(MULTI_ADAM, count, param_host, grad_host, m_host, v_host, n_host, l2_scale_host, lr * sqrtf(bias_corr2) / bias_corr1, beta1, beta2,
                    eps, (cudaStream_t)stream);
}

HRB_API int hrb_sgd_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, const int64_t* n_host,
                               const float* l2_scale_host, float lr, void* stream) {
  HRB_REQUIRE(count >= 0 && (count == 0 || (param_host && grad_host && n_host)), "hrb_sgd_step_multi: bad argument");
  return multi_step(MULTI_SGD, count, param_host, grad_host, nullptr, nullptr, n_host, l2_scale_host, lr, 0.f, 0.f, 0.f, (cudaStream_t)stream);
}

HRB_API int hrb_adagrad_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* acc_host,
                                   const int64_t* n_host, const float* l2_scale_host, float lr, float eps, void* stream) {
  HRB_REQUIRE(count >= 0 && (count == 0 || (param_host && grad_host && acc_host && n_host)), "hrb_adagrad_step_multi: bad argument");
  return multi_step(MULTI_ADAGRAD, count, param_host, grad_host, acc_host, nullptr, n_host, l2_scale_host, lr, 0.f, 0.f, eps,
                    (cudaStream_t)stream);
}

HRB_API int hrb_ftrl_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* acc_host,
                                float* const* lin_host, const int64_t* n_host, const float* l2_scale_host, float lr, float l1, float l2,
                                float lr_power, float l2_shrinkage, void* stream) {
  HRB_REQUIRE(count >= 0 && (count == 0 || (param_host && grad_host && acc_host && lin_host && n_host)) && lr > 0.f,
              "hrb_ftrl_step_multi: bad argument");
  return multi_step(MULTI_FTRL, count, param_host, grad_host, acc_host, lin_host, n_host, l2_scale_host, lr, 0.f, 0.f, 0.f,
                    (cudaStream_t)stream, FtrlArgs{l1, l2, lr_power, l2_shrinkage});
}

HRB_API int hrb_dice_fwd(const float* x, int64_t rows, int32_t units, const float* alpha, float* mean, float* var,
                         float eps, int32_t training, float* y, void* stream) {
  HRB_REQUIRE(x && alpha && mean && var && y && rows >= 0 && units > 0, "hrb_dice_fwd: null/negative argument");
  if (rows == 0) return HRB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (training) {
    dim3 grid;
    int64_t rpb;
    slab_grid(rows, units, grid, rpb);
    HRB_CUDA(cudaMemsetAsync(mean, 0, sizeof(float) * units, st));
    HRB_CUDA(cudaMemsetAsync(var, 0, sizeof(float) * units, st));
    dice_colstat_kernel<0><<<grid, 256, 0, st>>>(x, nullptr, rows, units, rpb, nullptr, nullptr, nullptr, eps, mean, nullptr);
    scale_kernel<<<(units + 255) / 256, 256, 0, st>>>(mean, units, 1.0f / (float)rows);
    dice_colstat_kernel<1><<<grid, 256, 0, st>>>(x, nullptr, rows, units, rpb, nullptr, mean, nullptr, eps, var, nullptr);
    scale_kernel<<<(units + 255) / 256, 256, 0, st>>>(var, units, 1.0f / (float)rows);
    hrb::count_launches(3);
    HRB_LAUNCH_CHECK();
  }
  dice_apply_kernel<<<ew_grid(rows * units), 256, 0, st>>>(x, rows * units, units, alpha, mean, var, eps, y);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_dice_bwd(const float* x, const float* dy, int64_t rows, int32_t units, const float* alpha,
                         const float* mean, const float* var, float eps, int32_t training, float* dx, float* dalpha,
                         float* scratch, void* stream) {
  HRB_REQUIRE(x && dy && alpha && mean && var && dx && rows >= 0 && units > 0, "hrb_dice_bwd: null/negative argument");
  HRB_REQUIRE(!training || scratch != nullptr, "hrb_dice_bwd: training mode needs a 2*units float scratch");
  cudaStream_t st = (cudaStream_t)stream;
  if (dalpha != nullptr) HRB_CUDA(cudaMemsetAsync(dalpha, 0, sizeof(float) * units, st));
  if (rows == 0) return HRB_OK;
  dim3 grid;
  int64_t rpb;
  slab_grid(rows, units, grid, rpb);
  if (training) {
    HRB_CUDA(cudaMemsetAsync(scratch, 0, sizeof(float) * 2 * units, st));
    dice_colstat_kernel<2><<<grid, 256, 0, st>>>(x, dy, rows, units, rpb, alpha, mean, var, eps, scratch, scratch + units);
    HRB_LAUNCH_CHECK();
  }
  dice_bwd_kernel<<<grid, 256, 0, st>>>(x, dy, rows, units, rpb, alpha, mean, var, eps, training, scratch, dx, dalpha);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_pack_dense(const void* src, int32_t src_is_int32, int64_t src_ld, int64_t batch, int32_t n, int32_t n_pad,
                           float* dst, int64_t dst_ld, void* stream) {
  HRB_REQUIRE(batch >= 0 && n >= 0 && n_pad >= n && src_ld >= n && dst_ld >= n_pad, "hrb_pack_dense: bad sizes");
  if (batch == 0 || n_pad == 0) return HRB_OK;
  HRB_REQUIRE(src && dst, "hrb_pack_dense: null pointer");
  if (src_is_int32)
    pack_dense_kernel<int32_t><<<ew_grid(batch * n_pad), 256, 0, (cudaStream_t)stream>>>((const int32_t*)src, src_ld, batch, n, n_pad, dst, dst_ld);
  else
    pack_dense_kernel<float><<<ew_grid(batch * n_pad), 256, 0, (cudaStream_t)stream>>>((const float*)src, src_ld, batch, n, n_pad, dst, dst_ld);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
