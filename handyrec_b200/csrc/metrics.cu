// metrics.cu -- Keras confusion-matrix and accuracy metrics counted on the device (tf.keras.metrics AUC / Precision / Recall /
// BinaryAccuracy, Keras 2.6 metrics_utils.update_confusion_matrix_variables).
//
// One launch per update, whatever the number of metrics:
//   every CTA copies the sorted thresholds into shared memory, classifies each sample by label (0, 1, other) and by bucket
//   (the number of thresholds p is strictly above, found by binary search; NaN lands in bucket 0), and counts into a
//   privatised shared histogram [3][T+1] with warp-aggregated increments (__match_any_sync: CTR predictions cluster in a few
//   buckets).  The CTA adds its non-zero bins into a global uint32 scratch with integer atomics (order-free, deterministic).
//   The last CTA to finish (threadfence + done counter) takes suffix sums above_c[j] = sum_{b > j} hist[c][b], adds every
//   variable's integer increment into its float32 variable with one rounding (Keras assign_add), and re-zeroes the scratch.
//   A prediction outside [0, 1] (or NaN) anywhere in the batch sets the flag of every tp / fp / tn / fn variable of the call, so
//   only the metrics that counted it report it, and resetting one metric clears its own flags.
#include <atomic>

#include "common.cuh"

namespace hrb {

constexpr int MET_THREADS = 256;
constexpr int MET_ITEMS = 8;  // samples per thread per grid-stride round

__device__ __forceinline__ uint32_t bucket_of(const float* __restrict__ thr, int T, float p) {
  // number of thresholds strictly below p: lower bound of p in the sorted list (NaN compares false everywhere -> 0)
  int lo = 0, len = T;
  while (len > 0) {
    const int half = len >> 1;
    const bool right = thr[lo + half] < p;
    lo = right ? lo + half + 1 : lo;
    len = right ? len - half - 1 : half;
  }
  return (uint32_t)lo;
}

// dst[i] = src[i] for i < n with MET_ITEMS loads in flight per thread (the last CTA's passes are bound by L2 latency otherwise)
template <typename T>
__device__ __forceinline__ void block_load(T* dst, const T* src, int n) {
  for (int base = threadIdx.x; base < n; base += MET_ITEMS * MET_THREADS) {
    T v[MET_ITEMS];
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      const int i = base + k * MET_THREADS;
      v[k] = i < n ? __ldcg(src + i) : T(0);
    }
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      const int i = base + k * MET_THREADS;
      if (i < n) dst[i] = v[k];
    }
  }
}

// exclusive suffix sum over the block's threads: returns sum of x over threads > threadIdx.x (ws: MET_THREADS / 32 entries)
__device__ __forceinline__ uint32_t block_suffix_exclusive(uint32_t x, uint32_t* ws) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_down_sync(0xffffffffu, inc, o);
    if (lane + o < 32) inc += t;
  }
  if (lane == 0) ws[w] = inc;  // the warp's total
  __syncthreads();
  uint32_t later = 0;
  for (int u = w + 1; u < MET_THREADS / 32; ++u) later += ws[u];
  __syncthreads();
  return inc - x + later;
}

__global__ void __launch_bounds__(MET_THREADS) metric_update_kernel(const float* __restrict__ prob, const float* __restrict__ label,
                                                                    int64_t n, const float* __restrict__ thresholds, int T,
                                                                    const int32_t* __restrict__ var_kind,
                                                                    const int32_t* __restrict__ var_thr, int n_vars,
                                                                    float* __restrict__ vars, uint32_t* __restrict__ scratch,
                                                                    int32_t* __restrict__ flags) {
  extern __shared__ uint32_t smem[];
  float* thr = reinterpret_cast<float*>(smem);
  uint32_t* hist = smem + T;  // [3][T+1]; the last CTA reuses it for the suffix sums
  const int NB = T + 1;
  const int nh = 3 * NB;
  __shared__ bool last;
  __shared__ uint32_t wsum[MET_THREADS / 32];

  block_load(thr, thresholds, T);
  for (int i = threadIdx.x; i < nh; i += blockDim.x) hist[i] = 0u;
  __syncthreads();

  const int lane = threadIdx.x & 31;
  bool bad = false;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * MET_ITEMS;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x * MET_ITEMS; base < n; base += stride) {
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      const int64_t i = base + (int64_t)k * blockDim.x + threadIdx.x;
      uint32_t key = 0xFFFFFFFFu;
      if (i < n) {
        const float p = __ldg(prob + i);
        const float y = __ldg(label + i);
        bad |= !(p >= 0.f && p <= 1.f);
        const uint32_t c = y == 0.f ? 0u : (y == 1.f ? 1u : 2u);  // NaN: "other", a positive (bool(NaN) is true)
        key = c * (uint32_t)NB + bucket_of(thr, T, p);
      }
      const uint32_t peers = __match_any_sync(0xffffffffu, key);
      if (key != 0xFFFFFFFFu && lane == __ffs(peers) - 1) atomicAdd(&hist[key], (uint32_t)__popc(peers));
    }
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(&scratch[nh + 1], 1u);  // scratch[nh + 1]: the batch had a bad prediction
  __syncthreads();

  for (int i = threadIdx.x; i < nh; i += blockDim.x)
    if (hist[i]) atomicAdd(&scratch[i], hist[i]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&scratch[nh], 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();

  // ---- last CTA: global histogram -> suffix sums (in place: hist[c][b] = sum_{b' >= b}) ----
  block_load(hist, scratch, nh);
  __syncthreads();
  const int chunk = (NB + MET_THREADS - 1) / MET_THREADS;  // each thread owns `chunk` consecutive buckets of every class
  for (int c = 0; c < 3; ++c) {
    uint32_t* h = hist + c * NB;
    const int b0 = min(threadIdx.x * chunk, NB), b1 = min(b0 + chunk, NB);
    uint32_t s = 0;
    for (int b = b0; b < b1; ++b) s += h[b];
    s = block_suffix_exclusive(s, wsum);
    for (int b = b1 - 1; b >= b0; --b) {
      s += h[b];
      h[b] = s;
    }
  }
  __syncthreads();

  // ---- every variable takes its integer increment with one float32 rounding (Keras assign_add) ----
  const uint32_t tot0 = hist[0], tot1 = hist[NB], tot2 = hist[2 * NB];
  const bool any_bad = __ldcg(&scratch[nh + 1]) != 0u;
  for (int base = threadIdx.x; base < n_vars; base += MET_ITEMS * MET_THREADS) {
    int kind[MET_ITEMS], j[MET_ITEMS];
    float var[MET_ITEMS];
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {  // every load of the group first
      const int v = base + k * MET_THREADS;
      kind[k] = v < n_vars ? __ldg(var_kind + v) : -1;
      j[k] = v < n_vars ? __ldg(var_thr + v) : 0;
      var[k] = v < n_vars ? vars[v] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      const int v = base + k * MET_THREADS;
      const int jj = kind[k] == HRB_METRIC_COUNT ? 0 : j[k];
      if (v >= n_vars || jj < 0 || jj >= T) continue;
      const uint32_t a0 = hist[jj + 1], a1 = hist[NB + jj + 1], a2 = hist[2 * NB + jj + 1];  // class c above thresholds[jj]
      uint32_t inc;
      switch (kind[k]) {
        case HRB_METRIC_TP: inc = a1 + a2; break;
        case HRB_METRIC_FP: inc = a0; break;
        case HRB_METRIC_TN: inc = tot0 - a0; break;
        case HRB_METRIC_FN: inc = tot1 + tot2 - (a1 + a2); break;
        case HRB_METRIC_CORRECT: inc = a1 + (tot0 - a0); break;
        case HRB_METRIC_COUNT: inc = (uint32_t)n; break;
        default: continue;
      }
      vars[v] = __fadd_rn(var[k], __uint2float_rn(inc));
      if (flags != nullptr && any_bad && kind[k] <= HRB_METRIC_FN) flags[v] = 1;
    }
  }

  // ---- leave the scratch zeroed for the next call (stream order makes the next launch see it) ----
  for (int i = threadIdx.x; i <= nh + 1; i += blockDim.x) scratch[i] = 0u;
}

}  // namespace hrb

HRB_API int hrb_metric_scratch_bytes(int32_t n_thr, size_t* bytes) {
  HRB_REQUIRE(bytes != nullptr, "hrb_metric_scratch_bytes: bytes is NULL");
  HRB_REQUIRE(n_thr >= 1 && n_thr <= HRB_METRIC_MAX_THRESHOLDS, "hrb_metric_scratch_bytes: n_thr = %d outside 1..%d", (int)n_thr,
              HRB_METRIC_MAX_THRESHOLDS);
  *bytes = (size_t)(3 * (n_thr + 1) + 2) * sizeof(uint32_t);  // histogram, done counter, bad-prediction word
  return HRB_OK;
}

HRB_API int hrb_metric_update(const float* prob, const float* label, int64_t n, const float* thresholds, int32_t n_thr,
                              const int32_t* var_kind, const int32_t* var_thr, int32_t n_vars, float* vars, void* scratch,
                              int32_t* flags, void* stream) {
  HRB_REQUIRE(prob && label && thresholds && var_kind && var_thr && vars && scratch, "hrb_metric_update: null pointer");
  HRB_REQUIRE(n >= 0 && n <= INT32_MAX, "hrb_metric_update: n = %lld outside 0..2^31-1", (long long)n);
  HRB_REQUIRE(n_thr >= 1 && n_thr <= HRB_METRIC_MAX_THRESHOLDS, "hrb_metric_update: n_thr = %d outside 1..%d", (int)n_thr,
              HRB_METRIC_MAX_THRESHOLDS);
  HRB_REQUIRE(n_vars >= 1, "hrb_metric_update: n_vars = %d, need at least one variable", (int)n_vars);
  if (n == 0) return HRB_OK;
  const size_t smem = (size_t)(n_thr + 3 * (n_thr + 1)) * sizeof(uint32_t);
  if (smem > 48 * 1024) {
    // the opt-in is a property of the kernel on a device, for the whole process: set it once per device to the largest size any
    // call can ask for (HRB_METRIC_MAX_THRESHOLDS), so that no thread can lower it under another
    constexpr size_t smem_max = (size_t)(HRB_METRIC_MAX_THRESHOLDS + 3 * (HRB_METRIC_MAX_THRESHOLDS + 1)) * sizeof(uint32_t);
    static std::atomic<bool> opted_in[64];
    int dev = 0;
    HRB_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !opted_in[dev].load(std::memory_order_acquire)) {
      HRB_CUDA(cudaFuncSetAttribute(hrb::metric_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
      if (dev < 64) opted_in[dev].store(true, std::memory_order_release);
    }
  }
  const int64_t per_cta = (int64_t)hrb::MET_THREADS * hrb::MET_ITEMS;
  int64_t blocks = (n + per_cta - 1) / per_cta;
  const int64_t cap = (int64_t)hrb::sm_count() * (smem > 100 * 1024 ? 1 : 2);
  if (blocks > cap) blocks = cap;
  hrb::metric_update_kernel<<<(unsigned)blocks, hrb::MET_THREADS, smem, (cudaStream_t)stream>>>(
      prob, label, n, thresholds, n_thr, var_kind, var_thr, n_vars, vars, (uint32_t*)scratch, flags);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
