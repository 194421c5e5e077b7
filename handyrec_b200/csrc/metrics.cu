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
//
// Weighted update (hrb_metric_update_weighted), two launches; float atomics would make the sums depend on the arrival order:
//   1. every CTA takes rounds of MET_THREADS * MET_ITEMS samples, sorts their (class * (T+1) + bucket, weight) pairs with a block
//      radix sort and reduces the runs of equal keys with a segmented block scan.  The last item of a run adds the run's fp64
//      weight sum into the CTA's own bins (one writer per bin and round) and its length into the global uint32 counts (integer
//      atomics, as above).
//   2. one thread per bin adds the CTAs' bins in CTA order (and zeroes them); the last CTA to finish takes the suffix sums of
//      counts and sums and updates every variable: counts as hrb_metric_update, weight sums rounded once to fp32.
#include <atomic>

#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

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

// the same in fp64, in a fixed order (the same bits on every call); the exclusive sum is shifted in, not formed as inc - x, which
// would lose the small terms next to a large x
__device__ __forceinline__ double block_suffix_exclusive(double x, double* ws) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_down_sync(0xffffffffu, inc, o);
    if (lane + o < 32) inc += t;
  }
  double excl = __shfl_down_sync(0xffffffffu, inc, 1);
  if (lane == 31) excl = 0.0;
  if (lane == 0) ws[w] = inc;
  __syncthreads();
  double later = 0.0;
  for (int u = MET_THREADS / 32 - 1; u > w; --u) later += ws[u];
  __syncthreads();
  return excl + later;
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


// ---- weighted update --------------------------------------------------------------------------------------------------------------
// One run of equal keys (or the part of it a span of sorted items holds): `head` says a run starts inside the span.  Combining a
// span with the span after it restarts at the later span's head, so an inclusive scan gives every item its run's sums so far.
struct WRun {
  int head;
  uint32_t cnt;
  double w;
};
struct WRunOp {
  __device__ __forceinline__ WRun operator()(const WRun& a, const WRun& b) const {
    return b.head ? b : WRun{a.head, a.cnt + b.cnt, a.w + b.w};
  }
};
typedef cub::BlockRadixSort<uint32_t, MET_THREADS, MET_ITEMS, double> WSort;
typedef cub::BlockScan<WRun, MET_THREADS> WScan;

// scratch of the weighted update: uint32 counts [3][T+1], bad-prediction word, done counter, (pad), fp64 sums [3][T+1], then one
// fp64 [3][T+1] bin block per CTA of launch 1 (at most metric_weighted_ctas())
__host__ __device__ __forceinline__ size_t wscratch_sums_offset(int nh) { return ((size_t)(nh + 2) * sizeof(uint32_t) + 7) / 8 * 8; }

__global__ void __launch_bounds__(MET_THREADS) metric_weighted_bins_kernel(const float* __restrict__ prob, const float* __restrict__ label,
                                                                           const float* __restrict__ weight, int64_t n,
                                                                           const float* __restrict__ thresholds, int T, int key_bits,
                                                                           uint32_t* __restrict__ counts, double* __restrict__ bins) {
  extern __shared__ uint32_t smem[];
  float* thr = reinterpret_cast<float*>(smem);
  __shared__ union {
    typename WSort::TempStorage sort;
    typename WScan::TempStorage scan;
  } tmp;
  __shared__ uint32_t first_key[MET_THREADS], last_key[MET_THREADS];
  const uint32_t NB = (uint32_t)T + 1u;
  const int nh = 3 * (int)NB;
  const uint32_t none = (1u << key_bits) - 1u;  // above every real key: out-of-range items sort last
  double* mine = bins + (size_t)blockIdx.x * nh;

  block_load(thr, thresholds, T);
  __syncthreads();

  const int lane = threadIdx.x & 31;
  bool bad = false;
  const int64_t per_round = (int64_t)MET_THREADS * MET_ITEMS;
  for (int64_t base = (int64_t)blockIdx.x * per_round; base < n; base += (int64_t)gridDim.x * per_round) {
    uint32_t key[MET_ITEMS];
    double w[MET_ITEMS];
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      const int64_t i = base + (int64_t)k * MET_THREADS + threadIdx.x;
      key[k] = none;
      w[k] = 0.0;
      if (i < n) {
        const float p = __ldg(prob + i);
        const float y = __ldg(label + i);
        bad |= !(p >= 0.f && p <= 1.f);
        const uint32_t c = y == 0.f ? 0u : (y == 1.f ? 1u : 2u);
        key[k] = c * NB + bucket_of(thr, T, p);
        w[k] = (double)__ldg(weight + i);
      }
    }
    __syncthreads();  // the previous round is done with tmp and the key arrays
    WSort(tmp.sort).Sort(key, w, 0, key_bits);  // blocked: this thread holds sorted items [8 t, 8 t + 8)
    first_key[threadIdx.x] = key[0];
    last_key[threadIdx.x] = key[MET_ITEMS - 1];
    __syncthreads();
    const uint32_t prev = threadIdx.x > 0 ? last_key[threadIdx.x - 1] : 0xFFFFFFFFu;
    const uint32_t next = threadIdx.x + 1 < MET_THREADS ? first_key[threadIdx.x + 1] : 0xFFFFFFFFu;
    const WRunOp op;
    WRun agg{0, 0u, 0.0};
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) agg = op(agg, WRun{key[k] != (k > 0 ? key[k - 1] : prev), 1u, w[k]});
    WRun run;
    WScan(tmp.scan).ExclusiveScan(agg, run, WRun{0, 0u, 0.0}, op);
#pragma unroll
    for (int k = 0; k < MET_ITEMS; ++k) {
      run = op(run, WRun{key[k] != (k > 0 ? key[k - 1] : prev), 1u, w[k]});
      const bool tail = key[k] != (k + 1 < MET_ITEMS ? key[k + 1] : next);
      if (tail && key[k] != none) {  // one writer per key and round; __syncthreads orders the rounds
        atomicAdd(&counts[key[k]], run.cnt);
        mine[key[k]] += run.w;
      }
    }
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(&counts[nh], 1u);
}

__global__ void __launch_bounds__(MET_THREADS) metric_weighted_finish_kernel(int64_t n, int T, int ctas, const int32_t* __restrict__ var_kind,
                                                                             const int32_t* __restrict__ var_thr, int n_vars,
                                                                             float* __restrict__ vars, uint32_t* __restrict__ counts,
                                                                             double* __restrict__ sums, double* __restrict__ bins,
                                                                             int32_t* __restrict__ flags) {
  __shared__ bool last;
  __shared__ uint32_t wsum_u[MET_THREADS / 32];
  __shared__ double wsum_d[MET_THREADS / 32];
  const int NB = T + 1;
  const int nh = 3 * NB;

  // ---- every bin: the CTAs' fp64 sums in CTA order; the bins are left zeroed ----
  for (int b = blockIdx.x * MET_THREADS + threadIdx.x; b < nh; b += gridDim.x * MET_THREADS) {
    double s = 0.0;
#pragma unroll 8
    for (int g = 0; g < ctas; ++g) {
      double* q = bins + (size_t)g * nh + b;
      s += __ldcg(q);
      *q = 0.0;
    }
    sums[b] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&counts[nh + 1], 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();

  // ---- last CTA: suffix sums of counts and sums, in place (h[c][b] = sum over b' >= b) ----
  const int chunk = (NB + MET_THREADS - 1) / MET_THREADS;
  for (int c = 0; c < 3; ++c) {
    uint32_t* h = counts + c * NB;
    double* hw = sums + c * NB;
    const int b0 = min((int)threadIdx.x * chunk, NB), b1 = min(b0 + chunk, NB);
    uint32_t s = 0;
    double sw = 0.0;
    for (int b = b1 - 1; b >= b0; --b) {
      s += __ldcg(h + b);
      sw += __ldcg(hw + b);
    }
    s = block_suffix_exclusive(s, wsum_u);
    sw = block_suffix_exclusive(sw, wsum_d);
    for (int b = b1 - 1; b >= b0; --b) {
      s += __ldcg(h + b);
      sw += __ldcg(hw + b);
      h[b] = s;
      hw[b] = sw;
    }
  }
  __syncthreads();

  // ---- every variable: counts as hrb_metric_update, weight sums rounded once to fp32 ----
  const uint32_t tot0 = __ldcg(counts), tot1 = __ldcg(counts + NB), tot2 = __ldcg(counts + 2 * NB);
  const double wt0 = __ldcg(sums), wt1 = __ldcg(sums + NB), wt2 = __ldcg(sums + 2 * NB);
  const bool any_bad = __ldcg(&counts[nh]) != 0u;
  for (int v = threadIdx.x; v < n_vars; v += MET_THREADS) {
    const int kind = __ldg(var_kind + v);
    const int jj = (kind == HRB_METRIC_COUNT || kind == HRB_METRIC_WCOUNT) ? 0 : __ldg(var_thr + v);
    if (jj < 0 || jj >= T) continue;
    const float var = vars[v];
    if (kind <= HRB_METRIC_COUNT) {
      const uint32_t a0 = __ldcg(counts + jj + 1), a1 = __ldcg(counts + NB + jj + 1), a2 = __ldcg(counts + 2 * NB + jj + 1);
      uint32_t inc;
      switch (kind) {
        case HRB_METRIC_TP: inc = a1 + a2; break;
        case HRB_METRIC_FP: inc = a0; break;
        case HRB_METRIC_TN: inc = tot0 - a0; break;
        case HRB_METRIC_FN: inc = tot1 + tot2 - (a1 + a2); break;
        case HRB_METRIC_CORRECT: inc = a1 + (tot0 - a0); break;
        case HRB_METRIC_COUNT: inc = (uint32_t)n; break;
        default: continue;
      }
      vars[v] = __fadd_rn(var, __uint2float_rn(inc));
    } else {
      const double a0 = __ldcg(sums + jj + 1), a1 = __ldcg(sums + NB + jj + 1), a2 = __ldcg(sums + 2 * NB + jj + 1);
      double inc;
      switch (kind) {
        case HRB_METRIC_WTP: inc = a1 + a2; break;
        case HRB_METRIC_WFP: inc = a0; break;
        case HRB_METRIC_WTN: inc = wt0 - a0; break;
        case HRB_METRIC_WFN: inc = (wt1 + wt2) - (a1 + a2); break;
        case HRB_METRIC_WCORRECT: inc = a1 + (wt0 - a0); break;
        case HRB_METRIC_WCOUNT: inc = wt0 + wt1 + wt2; break;
        default: continue;
      }
      vars[v] = __fadd_rn(var, __double2float_rn(inc));
    }
    if (flags != nullptr && any_bad && (kind <= HRB_METRIC_FN || (kind >= HRB_METRIC_WTP && kind <= HRB_METRIC_WFN))) flags[v] = 1;
  }

  // ---- leave the counts, the bad word and the done counter zeroed for the next call ----
  __syncthreads();
  for (int i = threadIdx.x; i <= nh + 1; i += MET_THREADS) counts[i] = 0u;
}

int metric_weighted_ctas() { return sm_count() * 2; }

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

HRB_API int hrb_metric_weighted_scratch_bytes(int32_t n_thr, size_t* bytes) {
  HRB_REQUIRE(bytes != nullptr, "hrb_metric_weighted_scratch_bytes: bytes is NULL");
  HRB_REQUIRE(n_thr >= 1 && n_thr <= HRB_METRIC_MAX_THRESHOLDS, "hrb_metric_weighted_scratch_bytes: n_thr = %d outside 1..%d",
              (int)n_thr, HRB_METRIC_MAX_THRESHOLDS);
  const int nh = 3 * (n_thr + 1);
  *bytes = hrb::wscratch_sums_offset(nh) + (size_t)(1 + hrb::metric_weighted_ctas()) * nh * sizeof(double);
  return HRB_OK;
}

HRB_API int hrb_metric_update_weighted(const float* prob, const float* label, const float* weight, int64_t n, const float* thresholds,
                                       int32_t n_thr, const int32_t* var_kind, const int32_t* var_thr, int32_t n_vars, float* vars,
                                       void* scratch, int32_t* flags, void* stream) {
  HRB_REQUIRE(prob && label && weight && thresholds && var_kind && var_thr && vars && scratch, "hrb_metric_update_weighted: null pointer");
  HRB_REQUIRE(n >= 0 && n <= INT32_MAX, "hrb_metric_update_weighted: n = %lld outside 0..2^31-1", (long long)n);
  HRB_REQUIRE(n_thr >= 1 && n_thr <= HRB_METRIC_MAX_THRESHOLDS, "hrb_metric_update_weighted: n_thr = %d outside 1..%d", (int)n_thr,
              HRB_METRIC_MAX_THRESHOLDS);
  HRB_REQUIRE(n_vars >= 1, "hrb_metric_update_weighted: n_vars = %d, need at least one variable", (int)n_vars);
  if (n == 0) return HRB_OK;
  const int nh = 3 * (n_thr + 1);
  int key_bits = 1;
  while ((1 << key_bits) - 1 < nh) ++key_bits;  // every key < nh < the out-of-range key (1 << key_bits) - 1
  const size_t smem = (size_t)n_thr * sizeof(float);
  {
    // static (sort / scan) + dynamic (thresholds) shared memory passes 48 KB at the larger n_thr: opt in once per device, to the
    // largest size any call asks for (see hrb_metric_update)
    static std::atomic<bool> opted_in[64];
    int dev = 0;
    HRB_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !opted_in[dev].load(std::memory_order_acquire)) {
      HRB_CUDA(cudaFuncSetAttribute(hrb::metric_weighted_bins_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(HRB_METRIC_MAX_THRESHOLDS * sizeof(float))));
      if (dev < 64) opted_in[dev].store(true, std::memory_order_release);
    }
  }
  uint32_t* counts = (uint32_t*)scratch;
  double* sums = (double*)((char*)scratch + hrb::wscratch_sums_offset(nh));
  double* bins = sums + nh;
  const int64_t per_cta = (int64_t)hrb::MET_THREADS * hrb::MET_ITEMS;
  int64_t blocks = (n + per_cta - 1) / per_cta;
  if (blocks > hrb::metric_weighted_ctas()) blocks = hrb::metric_weighted_ctas();
  hrb::metric_weighted_bins_kernel<<<(unsigned)blocks, hrb::MET_THREADS, smem, (cudaStream_t)stream>>>(
      prob, label, weight, n, thresholds, n_thr, key_bits, counts, bins);
  HRB_LAUNCH_CHECK();
  const int fin_blocks = (nh + hrb::MET_THREADS - 1) / hrb::MET_THREADS;
  hrb::metric_weighted_finish_kernel<<<fin_blocks, hrb::MET_THREADS, 0, (cudaStream_t)stream>>>(
      n, n_thr, (int)blocks, var_kind, var_thr, n_vars, vars, counts, sums, bins, flags);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}
