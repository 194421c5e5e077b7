// layers_misc.cu -- the remaining pieces of the Keras-layer face: BatchNormalization and Dropout of the DNN
// (layers/core.py:71-73), the DIN attention input [q, k, q-k, q*k] and the masked weighted key sum
// (layers/sequence.py:94-101, models/ranking/sequential/DIN.py:93), forward and backward.
// All HBM-bound element-wise / column-statistics kernels.
#include "common.cuh"

namespace hrb {

static inline unsigned ew_grid2(int64_t n) {
  int64_t b = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

// column sums over a row slab: MODE 0: sum x; 1: sum (x-mean)^2; 2: {sum dy, sum dy*xhat}
template <int MODE>
__global__ void __launch_bounds__(256) bn_colstat_kernel(const float* __restrict__ x, const float* __restrict__ dy, int64_t rows,
                                                        int32_t units, int64_t rows_per_block, const float* __restrict__ mean,
                                                        const float* __restrict__ var, float eps, float* __restrict__ out0,
                                                        float* __restrict__ out1) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  __shared__ float r0s[8][33], r1s[8][33];
  const int64_t rbeg = (int64_t)blockIdx.y * rows_per_block, rend = min(rows, rbeg + rows_per_block);
  float s0 = 0.f, s1 = 0.f;
  if (n < units) {
    const float mu = MODE >= 1 ? mean[n] : 0.f;
    const float rstd = MODE == 2 ? rsqrtf(var[n] + eps) : 0.f;
    for (int64_t r = rbeg + ry; r < rend; r += 8) {
      const float v = __ldg(x + r * units + n);
      if (MODE == 0) s0 += v;
      else if (MODE == 1) s0 = fmaf(v - mu, v - mu, s0);
      else {
        const float g = __ldg(dy + r * units + n);
        s0 += g;
        s1 = fmaf(g, (v - mu) * rstd, s1);
      }
    }
  }
  r0s[ry][threadIdx.x & 31] = s0;
  r1s[ry][threadIdx.x & 31] = s1;
  __syncthreads();
  if (ry == 0 && n < units) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) { a += r0s[k][threadIdx.x & 31]; b += r1s[k][threadIdx.x & 31]; }
    atomicAdd(out0 + n, a);
    if (MODE == 2) atomicAdd(out1 + n, b);
  }
}

__global__ void bn_scale_kernel(float* __restrict__ v, int32_t n, float s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= s;
}

__global__ void __launch_bounds__(256) bn_apply_kernel(const float* __restrict__ x, int64_t total, int32_t units,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      const float* __restrict__ mean, const float* __restrict__ var, float eps,
                                                      float* __restrict__ y) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i % units);
    float v = (x[i] - mean[n]) * rsqrtf(var[n] + eps);
    if (gamma != nullptr) v *= gamma[n];
    if (beta != nullptr) v += beta[n];
    y[i] = v;
  }
}

// dx = gamma*rstd*(dy - mean(dy) - xhat*mean(dy*xhat)) (training) | gamma*rstd*dy (inference)
__global__ void __launch_bounds__(256) bn_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, int64_t total,
                                                    int32_t units, int64_t rows, const float* __restrict__ gamma,
                                                    const float* __restrict__ mean, const float* __restrict__ var, float eps,
                                                    int32_t training, const float* __restrict__ stat, float* __restrict__ dx) {
  const float inv_rows = 1.0f / (float)rows;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i % units);
    const float rstd = rsqrtf(var[n] + eps);
    const float gm = gamma != nullptr ? gamma[n] : 1.f;
    float d = dy[i];
    if (training) d = d - stat[n] * inv_rows - (x[i] - mean[n]) * rstd * stat[units + n] * inv_rows;
    dx[i] = gm * rstd * d;
  }
}

// Dropout: keep mask from a counter-based hash (seed, element index); y = x * keep / (1 - rate)
__global__ void __launch_bounds__(256) dropout_kernel(const float* __restrict__ x, int64_t n, float rate, uint32_t seed,
                                                     float* __restrict__ y) {
  const float scale = 1.0f / (1.0f - rate);
  const uint32_t thresh = (uint32_t)(rate * 4294967296.0);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t h = hash_u32((uint32_t)i ^ hash_u32((uint32_t)(i >> 32) + seed * 0x9E3779B9u + 0x7F4A7C15u));
    y[i] = h >= thresh ? x[i] * scale : 0.0f;
  }
}

// att_in[b,t,:] = [q, k, q-k, q*k]   (sequence.py:96-97)
__global__ void __launch_bounds__(256) att_input_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k, int64_t batch,
                                                           int32_t T, int32_t D, float* __restrict__ out) {
  const int64_t total = batch * T * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const int64_t bt = i / D;
    const int64_t b = bt / T;
    const float qv = q[b * D + d], kv = k[i];
    float* o = out + bt * 4 * D + d;
    o[0] = qv;
    o[D] = kv;
    o[2 * D] = qv - kv;
    o[3 * D] = qv * kv;
  }
}
// dk[b,t] = g1 - g2 + g3*q ; dq[b] = sum_t (g0 + g2 + g3*k)
__global__ void __launch_bounds__(256) att_input_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                           const float* __restrict__ g, int64_t batch, int32_t T, int32_t D,
                                                           float* __restrict__ dq, float* __restrict__ dk) {
  const int64_t total = batch * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const int64_t b = i / D;
    const float qv = q[i];
    float acc = 0.f;
    for (int t = 0; t < T; ++t) {
      const int64_t bt = b * T + t;
      const float* gp = g + bt * 4 * D + d;
      const float kv = k[bt * D + d];
      acc += gp[0] + gp[2 * D] + gp[3 * D] * kv;
      dk[bt * D + d] = gp[D] - gp[2 * D] + gp[3 * D] * qv;
    }
    dq[i] = acc;
  }
}

// scores (B,T) masked by ids != 0 (sequence.py:100-101): out[b,t] = mask ? s : 0 ; bwd is the same multiply
__global__ void __launch_bounds__(256) mask_scores_kernel(const float* __restrict__ s, const uint8_t* __restrict__ mask, int64_t n,
                                                         float* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = mask[i] ? s[i] : 0.0f;
}

// pooled[b,:] = sum_t s[b,t] * k[b,t,:]   (DIN.py:93, tf.matmul(att (B,1,T), keys (B,T,D)))
__global__ void __launch_bounds__(256) att_pool_fwd_kernel(const float* __restrict__ s, const float* __restrict__ k, int64_t batch,
                                                          int32_t T, int32_t D, float* __restrict__ out) {
  const int64_t total = batch * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const int64_t b = i / D;
    float acc = 0.f;
    for (int t = 0; t < T; ++t) acc = fmaf(s[b * T + t], k[(b * T + t) * D + d], acc);
    out[i] = acc;
  }
}
// ds[b,t] = dout[b,:] . k[b,t,:] ; dk[b,t,:] = s[b,t] * dout[b,:]
__global__ void __launch_bounds__(256) att_pool_bwd_kernel(const float* __restrict__ s, const float* __restrict__ k,
                                                          const float* __restrict__ dout, int64_t batch, int32_t T, int32_t D,
                                                          float* __restrict__ ds, float* __restrict__ dk) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t bt = warp0; bt < batch * T; bt += nwarps) {
    const int64_t b = bt / T;
    const float sv = s[bt];
    float acc = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float g = dout[b * D + d];
      acc = fmaf(g, k[bt * D + d], acc);
      dk[bt * D + d] = sv * g;
    }
    acc = warp_sum(acc);
    if (lane == 0) ds[bt] = acc;
  }
}

static inline void slab(int64_t rows, int32_t units, dim3& grid, int64_t& rpb) {
  int yb = (int)min((int64_t)sm_count() * 2, (rows + 63) / 64);
  if (yb < 1) yb = 1;
  rpb = (rows + yb - 1) / yb;
  grid = dim3((units + 31) / 32, yb);
}

}  // namespace hrb

using namespace hrb;

// Keras BatchNormalization on the last axis (core.py:71-72; defaults eps=1e-3).  training != 0: batch statistics
// (biased variance over all rows) are written to mean/var; otherwise they are read (moving statistics).
HRB_API int hrb_batchnorm_fwd(const float* x, int64_t rows, int32_t units, const float* gamma, const float* beta, float* mean,
                              float* var, float eps, int32_t training, float* y, void* stream) {
  HRB_REQUIRE(rows >= 0 && units > 0, "hrb_batchnorm_fwd: bad sizes");
  if (rows == 0) return HRB_OK;
  HRB_REQUIRE(x && mean && var && y, "hrb_batchnorm_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (training) {
    dim3 grid;
    int64_t rpb;
    slab(rows, units, grid, rpb);
    HRB_CUDA(cudaMemsetAsync(mean, 0, sizeof(float) * units, st));
    HRB_CUDA(cudaMemsetAsync(var, 0, sizeof(float) * units, st));
    bn_colstat_kernel<0><<<grid, 256, 0, st>>>(x, nullptr, rows, units, rpb, nullptr, nullptr, eps, mean, nullptr);
    bn_scale_kernel<<<(units + 255) / 256, 256, 0, st>>>(mean, units, 1.0f / (float)rows);
    bn_colstat_kernel<1><<<grid, 256, 0, st>>>(x, nullptr, rows, units, rpb, mean, nullptr, eps, var, nullptr);
    bn_scale_kernel<<<(units + 255) / 256, 256, 0, st>>>(var, units, 1.0f / (float)rows);
    count_launches(3);
    HRB_LAUNCH_CHECK();
  }
  bn_apply_kernel<<<ew_grid2(rows * units), 256, 0, st>>>(x, rows * units, units, gamma, beta, mean, var, eps, y);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_batchnorm_bwd(const float* x, const float* dy, int64_t rows, int32_t units, const float* gamma, const float* mean,
                              const float* var, float eps, int32_t training, float* dx, float* dgamma, float* dbeta,
                              float* scratch /* 2*units floats */, void* stream) {
  HRB_REQUIRE(rows >= 0 && units > 0, "hrb_batchnorm_bwd: bad sizes");
  HRB_REQUIRE(scratch && (rows == 0 || (x && dy && mean && var && dx)), "hrb_batchnorm_bwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  HRB_CUDA(cudaMemsetAsync(scratch, 0, sizeof(float) * 2 * units, st));
  if (rows > 0) {
    dim3 grid;
    int64_t rpb;
    slab(rows, units, grid, rpb);
    bn_colstat_kernel<2><<<grid, 256, 0, st>>>(x, dy, rows, units, rpb, mean, var, eps, scratch, scratch + units);
    HRB_LAUNCH_CHECK();
    bn_bwd_kernel<<<ew_grid2(rows * units), 256, 0, st>>>(x, dy, rows * units, units, rows, gamma, mean, var, eps, training, scratch, dx);
    HRB_LAUNCH_CHECK();
  }
  // dbeta = sum dy ; dgamma = sum dy*xhat  (already in scratch; zero for an empty batch)
  if (dbeta != nullptr) HRB_CUDA(cudaMemcpyAsync(dbeta, scratch, sizeof(float) * units, cudaMemcpyDeviceToDevice, st));
  if (dgamma != nullptr) HRB_CUDA(cudaMemcpyAsync(dgamma, scratch + units, sizeof(float) * units, cudaMemcpyDeviceToDevice, st));
  return HRB_OK;
}

// Keras Dropout (core.py:73): y = x * keep / (1-rate); the keep mask is a pure function of (seed, index), so the
// backward is the same call on the upstream gradient.
HRB_API int hrb_dropout(const float* x, int64_t n, float rate, uint32_t seed, float* y, void* stream) {
  HRB_REQUIRE(n >= 0 && rate >= 0.f && rate < 1.f, "hrb_dropout: bad argument");
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(x && y, "hrb_dropout: null pointer");
  dropout_kernel<<<ew_grid2(n), 256, 0, (cudaStream_t)stream>>>(x, n, rate, seed, y);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_att_input_fwd(const float* q, const float* k, int64_t batch, int32_t T, int32_t D, float* out, void* stream) {
  HRB_REQUIRE(batch >= 0 && T > 0 && D > 0, "hrb_att_input_fwd: bad sizes");
  if (batch == 0) return HRB_OK;
  HRB_REQUIRE(q && k && out, "hrb_att_input_fwd: null pointer");
  att_input_fwd_kernel<<<ew_grid2(batch * T * D), 256, 0, (cudaStream_t)stream>>>(q, k, batch, T, D, out);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
HRB_API int hrb_att_input_bwd(const float* q, const float* k, const float* g, int64_t batch, int32_t T, int32_t D, float* dq,
                              float* dk, void* stream) {
  HRB_REQUIRE(batch >= 0 && T > 0 && D > 0, "hrb_att_input_bwd: bad sizes");
  if (batch == 0) return HRB_OK;
  HRB_REQUIRE(q && k && g && dq && dk, "hrb_att_input_bwd: null pointer");
  att_input_bwd_kernel<<<ew_grid2(batch * D), 256, 0, (cudaStream_t)stream>>>(q, k, g, batch, T, D, dq, dk);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
HRB_API int hrb_mask_scores(const float* s, const uint8_t* mask, int64_t n, float* out, void* stream) {
  HRB_REQUIRE(n >= 0, "hrb_mask_scores: bad size");
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(s && mask && out, "hrb_mask_scores: null pointer");
  mask_scores_kernel<<<ew_grid2(n), 256, 0, (cudaStream_t)stream>>>(s, mask, n, out);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
HRB_API int hrb_att_pool_fwd(const float* s, const float* k, int64_t batch, int32_t T, int32_t D, float* out, void* stream) {
  HRB_REQUIRE(batch >= 0 && T > 0 && D > 0, "hrb_att_pool_fwd: bad sizes");
  if (batch == 0) return HRB_OK;
  HRB_REQUIRE(s && k && out, "hrb_att_pool_fwd: null pointer");
  att_pool_fwd_kernel<<<ew_grid2(batch * D), 256, 0, (cudaStream_t)stream>>>(s, k, batch, T, D, out);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
HRB_API int hrb_att_pool_bwd(const float* s, const float* k, const float* dout, int64_t batch, int32_t T, int32_t D, float* ds,
                             float* dk, void* stream) {
  HRB_REQUIRE(batch >= 0 && T > 0 && D > 0, "hrb_att_pool_bwd: bad sizes");
  if (batch == 0) return HRB_OK;
  HRB_REQUIRE(s && k && dout && ds && dk, "hrb_att_pool_bwd: null pointer");
  att_pool_bwd_kernel<<<ew_grid2(batch * T * 32), 256, 0, (cudaStream_t)stream>>>(s, k, dout, batch, T, D, ds, dk);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
