// lookup.cu -- embedding gather + mask + masked sequence pooling (forward), fused FM epilogue,
// and the embedding backward as sort -> segment-reduce -> per-unique-row update (no atomics).
//
// Reference arithmetic replaced (paths under /root/reference/handyrec/):
//   layers/tools.py:87-101      CustomEmbedding (gather, tiled != 0 mask)
//   layers/sequence.py:26-46    SequencePoolingLayer (masked mean / sum / max)
//   features/group.py:299-336   FeatureGroup.embedding_lookup (per-feature orchestration)
//   layers/interaction.py:26-39 FM (fused epilogue of the lookup for DeepFM)
//   TF autodiff of the above    IndexedSlices scatter-add (+ 2*l2*W), SURVEY a13
//
// Data layout in HBM: tables are row-major (rows, D) fp32, rows 16-byte aligned (D % 4 == 0);
// ids of a batch are one packed int32 matrix ids[B, ids_ld]; the pooled output of a whole group is
// ONE row-major matrix out[B, out_ld] whose column blocks are the features in reference order, so
// the DNN input (B, sum D) and the FM input (B, F, D) are the same bytes (layers/utils.py:40-96).
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <new>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "common.cuh"

#include "plan.cuh"

namespace hrb {

constexpr uint32_t kNotMine = 0xFFFFFFFFu;

// ---------------------------------------------------------------------------------------------
// a5: plain gather + tiled mask (layer face)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embedding_fwd_kernel(const float* __restrict__ table, int64_t vocab,
                                                            int32_t chunks /* dim/4 */,
                                                            const int32_t* __restrict__ ids, int64_t n_ids,
                                                            float* __restrict__ out, uint8_t* __restrict__ mask,
                                                            int32_t* __restrict__ oob) {
  const int64_t total = n_ids * chunks;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  constexpr int U = 4;
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; base < total; base += stride * U) {
    int32_t id[U];
    int64_t item[U];
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      item[u] = base + u * stride;
      id[u] = item[u] < total ? __ldg(ids + item[u] / chunks) : 0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (item[u] < total) {
        const int q = (int)(item[u] % chunks);
        if (id[u] >= 0 && id[u] < vocab) {
          v[u] = ldg_nc_na(reinterpret_cast<const float4*>(table + (int64_t)id[u] * chunks * 4) + q);
        } else if (oob != nullptr) {
          oob[0] = 1;
          oob[1] = (int32_t)(item[u] / chunks);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (item[u] < total) {
        stg_na(reinterpret_cast<float4*>(out) + item[u], v[u]);
        if (mask != nullptr) {
          const uint32_t m = id[u] != 0 ? 0x01010101u : 0u;
          reinterpret_cast<uint32_t*>(mask)[item[u]] = m;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// a6: pooling on a materialised (B,L,D) tensor + (B,L,D) mask (layer face)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) seq_pool_fwd_kernel(const float* __restrict__ x,
                                                           const uint8_t* __restrict__ mask, int64_t batch,
                                                           int32_t L, int32_t D, int32_t method,
                                                           float* __restrict__ out) {
  const int64_t total = batch * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / D;
    const int d = (int)(i - b * D);
    const float* xp = x + b * (int64_t)L * D + d;
    const uint8_t* mp = mask + b * (int64_t)L * D + d;
    if (method == HRB_POOL_MAX) {
      float best = -INFINITY;
      for (int l = 0; l < L; ++l) {
        const float m = mp[(int64_t)l * D] ? 1.0f : 0.0f;
        best = fmaxf(best, __fsub_rn(xp[(int64_t)l * D], __fmul_rn(1.0f - m, 1e9f)));  // sequence.py:35
      }
      out[i] = best;
    } else {
      float cnt = 0.f;
      for (int l = 0; l < L; ++l) cnt += mp[(int64_t)l * D] ? 1.0f : 0.0f;
      // mean: mask / mask_sum with divide_no_nan (sequence.py:43-44); sum: weight 1
      const float w = method == HRB_POOL_MEAN ? (cnt > 0.f ? __fdiv_rn(1.0f, cnt) : 0.0f) : 1.0f;
      float acc = 0.f;
      for (int l = 0; l < L; ++l)
        if (mp[(int64_t)l * D]) acc = __fadd_rn(acc, __fmul_rn(xp[(int64_t)l * D], w));
      out[i] = acc;
    }
  }
}

__global__ void __launch_bounds__(256) seq_pool_bwd_kernel(const float* __restrict__ x,
                                                           const uint8_t* __restrict__ mask,
                                                           const float* __restrict__ dout, int64_t batch,
                                                           int32_t L, int32_t D, int32_t method,
                                                           float* __restrict__ dx) {
  const int64_t total = batch * D;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / D;
    const int d = (int)(i - b * D);
    const int64_t off = b * (int64_t)L * D + d;
    const float g = dout[i];
    if (method == HRB_POOL_MAX) {
      float best = -INFINITY;
      for (int l = 0; l < L; ++l) {
        const float m = mask[off + (int64_t)l * D] ? 1.0f : 0.0f;
        best = fmaxf(best, __fsub_rn(x[off + (int64_t)l * D], __fmul_rn(1.0f - m, 1e9f)));
      }
      int ties = 0;
      for (int l = 0; l < L; ++l) {
        const float m = mask[off + (int64_t)l * D] ? 1.0f : 0.0f;
        ties += (__fsub_rn(x[off + (int64_t)l * D], __fmul_rn(1.0f - m, 1e9f)) == best);
      }
      const float share = g / (float)ties;  // TF reduce_max gradient: equal split among ties
      for (int l = 0; l < L; ++l) {
        const float m = mask[off + (int64_t)l * D] ? 1.0f : 0.0f;
        const bool hit = __fsub_rn(x[off + (int64_t)l * D], __fmul_rn(1.0f - m, 1e9f)) == best;
        dx[off + (int64_t)l * D] = hit ? share : 0.0f;
      }
    } else {
      float cnt = 0.f;
      for (int l = 0; l < L; ++l) cnt += mask[off + (int64_t)l * D] ? 1.0f : 0.0f;
      const float w = method == HRB_POOL_MEAN ? (cnt > 0.f ? __fdiv_rn(1.0f, cnt) : 0.0f) : 1.0f;
      for (int l = 0; l < L; ++l) dx[off + (int64_t)l * D] = mask[off + (int64_t)l * D] ? g * w : 0.0f;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// pooled vector of one (sample, field, 4-column group): the shared inner loop of every fused kernel
//   PARTIAL: ids are LOCAL rows of a shard, kNotMine marks "owned elsewhere / padding"; returns
//   the raw sum (or partial max) and the valid count instead of finalising.
// ---------------------------------------------------------------------------------------------
template <bool PARTIAL>
__device__ __forceinline__ float4 pooled_chunk(const FieldDev& f, const int32_t* __restrict__ ids_row, int q,
                                               float& n_valid, int32_t* __restrict__ oob, int64_t b) {
  const float4* __restrict__ tab = reinterpret_cast<const float4*>(f.table);
  const int64_t row_f4 = f.dim >> 2;
  const int L = f.seq_len;
  const int32_t* idp = ids_row + f.ids_col;
  float4 acc;
  if (f.pool == HRB_POOL_MAX)
    acc = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  else
    acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float cnt = 0.f;
  constexpr int U = 8;
  for (int l0 = 0; l0 < L; l0 += U) {
    int32_t id[U];
    bool ok[U];
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) id[u] = (l0 + u < L) ? __ldg(idp + l0 + u) : (PARTIAL ? (int32_t)kNotMine : 0);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      bool valid;
      if (PARTIAL)
        valid = (uint32_t)id[u] != kNotMine;
      else
        valid = (l0 + u < L) && (f.pool == HRB_POOL_NONE || id[u] != 0);
      const bool in_range = id[u] >= 0 && (int64_t)id[u] < f.rows;
      ok[u] = valid;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {
        if (in_range) {
          v[u] = ldg_nc_na(tab + (int64_t)id[u] * row_f4 + q);
        } else if (oob != nullptr) {
          oob[0] = 1;
          oob[1] = (int32_t)b;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (ok[u]) {
        cnt += 1.0f;
        if (f.pool == HRB_POOL_MAX) {
          acc.x = fmaxf(acc.x, v[u].x);
          acc.y = fmaxf(acc.y, v[u].y);
          acc.z = fmaxf(acc.z, v[u].z);
          acc.w = fmaxf(acc.w, v[u].w);
        } else {
          acc.x += v[u].x;
          acc.y += v[u].y;
          acc.z += v[u].z;
          acc.w += v[u].w;
        }
      }
    }
  }
  n_valid = cnt;
  if (PARTIAL) return acc;
  if (f.pool == HRB_POOL_MEAN) {
    // reference: sum_l x * (mask / mask_sum), divide_no_nan -> 0 for an all-padding row (sequence.py:43-46)
    const float w = cnt > 0.f ? __fdiv_rn(1.0f, cnt) : 0.0f;
    acc.x *= w;
    acc.y *= w;
    acc.z *= w;
    acc.w *= w;
  } else if (f.pool == HRB_POOL_MAX) {
    if (cnt < (float)L) {
      // padded positions contribute x0 - 1e9 where x0 = row 0 of the table (sequence.py:35-36):
      // an all-padding row therefore yields fl(W[0,d] - 1e9) (~ -1e9), not 0.
      const float4 z = ldg_nc_na(tab + q);
      acc.x = fmaxf(acc.x, __fsub_rn(z.x, 1e9f));
      acc.y = fmaxf(acc.y, __fsub_rn(z.y, 1e9f));
      acc.z = fmaxf(acc.z, __fsub_rn(z.z, 1e9f));
      acc.w = fmaxf(acc.w, __fsub_rn(z.w, 1e9f));
    }
  }
  return acc;
}

// ---------------------------------------------------------------------------------------------
// a7 generic: one thread per (sample, output 4-column chunk); stores of a warp are contiguous.
// Four items per thread are in flight together (ids first, then rows, then stores).
// ---------------------------------------------------------------------------------------------
template <bool PARTIAL>
__global__ void __launch_bounds__(256) lookup_items_kernel(const FieldDev* __restrict__ fields,
                                                          const int32_t* __restrict__ chunk_field,
                                                          const int32_t* __restrict__ chunk_q, int32_t n_chunks,
                                                          int32_t n_fields, const int32_t* __restrict__ ids,
                                                          int64_t ids_ld, int64_t batch, float* __restrict__ out,
                                                          int64_t out_ld, float* __restrict__ aux,
                                                          int32_t* __restrict__ oob) {
  const int64_t total = batch * n_chunks;
  for (int64_t item = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; item < total;
       item += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = item / n_chunks;
    const int c = (int)(item - b * n_chunks);
    const int fi = __ldg(chunk_field + c);
    const int q = __ldg(chunk_q + c);
    const FieldDev f = fields[fi];
    float n_valid;
    const float4 r = pooled_chunk<PARTIAL>(f, ids + b * ids_ld, q, n_valid, oob, b);
    stg_na(reinterpret_cast<float4*>(out + b * out_ld + f.out_col) + q, r);
    if (aux != nullptr && q == 0) {
      if (PARTIAL)
        aux[b * n_fields + fi] = n_valid;
      else
        aux[b * n_fields + fi] = f.pool == HRB_POOL_MEAN ? (n_valid > 0.f ? __fdiv_rn(1.0f, n_valid) : 0.f) : 1.0f;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// a7 + a9 fused, uniform D: G = D/4 lanes own one sample and walk its F fields, so the FM sums
// (sum_f x, sum_f x^2) stay in registers and the pooled (B,F,D) block is written exactly once.
//   LEN1: every field is a plain lookup (Criteo shape) -> FU rows per lane in flight.
// ---------------------------------------------------------------------------------------------
template <int G, bool LEN1, bool FM>
__global__ void __launch_bounds__(256) lookup_rows_kernel(const FieldDev* __restrict__ fields_g, int32_t n_fields,
                                                         const int32_t* __restrict__ ids, int64_t ids_ld,
                                                         int64_t batch, float* __restrict__ out, int64_t out_ld,
                                                         float* __restrict__ inv_count,
                                                         const float* __restrict__ fm_w,
                                                         const float* __restrict__ fm_w0,
                                                         float* __restrict__ fm_out, float* __restrict__ fm_sum,
                                                         int32_t* __restrict__ oob) {
  constexpr int SPB = 256 / G;  // samples per block pass
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FieldDev* fields = reinterpret_cast<FieldDev*>(smem_raw);  // descriptors are read F times per sample
  for (int i = threadIdx.x; i < n_fields * (int)(sizeof(FieldDev) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(fields)[i] = reinterpret_cast<const uint32_t*>(fields_g)[i];
  __syncthreads();
  const int q = threadIdx.x % G;
  const int s_in_block = threadIdx.x / G;
  float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float w0 = 0.f;
  if (FM) {
    w4 = __ldg(reinterpret_cast<const float4*>(fm_w) + q);
    w0 = __ldg(fm_w0);
  }
  // the loop bound is block-uniform; lanes past the end stay in it (valid == false) because the FM
  // epilogue shuffles with a full mask
  for (int64_t b0 = blockIdx.x * (int64_t)SPB; b0 < batch; b0 += (int64_t)gridDim.x * SPB) {
    const int64_t b = b0 + s_in_block;
    const bool valid = b < batch;
    const int32_t* ids_row = ids + (valid ? b : 0) * ids_ld;
    float* out_row = out + (valid ? b : 0) * out_ld;
    float4 S = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 Q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (LEN1) {
      constexpr int FU = 13;
      for (int f0 = 0; f0 < n_fields; f0 += FU) {
        int32_t id[FU];
        float4 v[FU];
#pragma unroll
        for (int u = 0; u < FU; ++u) id[u] = (valid && f0 + u < n_fields) ? __ldg(ids_row + fields[f0 + u].ids_col) : 0;
#pragma unroll
        for (int u = 0; u < FU; ++u) {
          v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (valid && f0 + u < n_fields) {
            const FieldDev& f = fields[f0 + u];
            if (id[u] >= 0 && (int64_t)id[u] < f.rows) {
              v[u] = ldg_nc_na(reinterpret_cast<const float4*>(f.table) + (int64_t)id[u] * G + q);
            } else if (oob != nullptr) {
              oob[0] = 1;
              oob[1] = (int32_t)b;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < FU; ++u) {
          if (valid && f0 + u < n_fields) {
            stg_na(reinterpret_cast<float4*>(out_row + fields[f0 + u].out_col) + q, v[u]);
            if (FM) {
              S.x += v[u].x; S.y += v[u].y; S.z += v[u].z; S.w += v[u].w;
              Q.x = fmaf(v[u].x, v[u].x, Q.x); Q.y = fmaf(v[u].y, v[u].y, Q.y);
              Q.z = fmaf(v[u].z, v[u].z, Q.z); Q.w = fmaf(v[u].w, v[u].w, Q.w);
            }
          }
        }
      }
      if (inv_count != nullptr && valid)
        for (int f = q; f < n_fields; f += G) inv_count[b * n_fields + f] = 1.0f;
    } else {
      for (int fi = 0; valid && fi < n_fields; ++fi) {
        const FieldDev f = fields[fi];
        float n_valid;
        const float4 r = pooled_chunk<false>(f, ids_row, q, n_valid, oob, b);
        stg_na(reinterpret_cast<float4*>(out_row + f.out_col) + q, r);
        if (inv_count != nullptr && q == 0)
          inv_count[b * n_fields + fi] =
              f.pool == HRB_POOL_MEAN ? (n_valid > 0.f ? __fdiv_rn(1.0f, n_valid) : 0.f) : 1.0f;
        if (FM) {
          S.x += r.x; S.y += r.y; S.z += r.z; S.w += r.w;
          Q.x = fmaf(r.x, r.x, Q.x); Q.y = fmaf(r.y, r.y, Q.y);
          Q.z = fmaf(r.z, r.z, Q.z); Q.w = fmaf(r.w, r.w, Q.w);
        }
      }
    }
    if (FM) {
      // interaction.py:29-39: part2 = (sum_f x).w ; part3 = 0.5*sum_d[(sum_f x)^2 - sum_f x^2]
      float p2 = S.x * w4.x + S.y * w4.y + S.z * w4.z + S.w * w4.w;
      float p3 = (S.x * S.x - Q.x) + (S.y * S.y - Q.y) + (S.z * S.z - Q.z) + (S.w * S.w - Q.w);
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) {
        p2 += __shfl_xor_sync(0xffffffffu, p2, o, G);
        p3 += __shfl_xor_sync(0xffffffffu, p3, o, G);
      }
      if (valid && q == 0) fm_out[b] = p2 + 0.5f * p3 + w0;
      if (valid && fm_sum != nullptr) reinterpret_cast<float4*>(fm_sum + b * (int64_t)(G * 4))[q] = S;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// a7 + a9, plain-lookup groups (Criteo shape), v2: the gather never touches registers.
//   One CTA owns tiles of 32 samples.  Every row is copied global -> shared with 16-byte cp.async (LDGSTS),
//   all F*D/4 copies of a thread in flight at once; the FM sums are taken from shared memory; each sample's
//   F*D-float output row leaves as ONE bulk TMA store (cp.async.bulk shared -> global, full lines).
//   Shared tile pitch = F*D*4 + pad so that two neighbouring samples sit 64 B apart mod 128 (conflict-free LDS.128).
//   ~54 KB per CTA at F=26, D=16 -> 4 CTAs/SM, 200+ KB of gathers in flight per SM with ~40 registers/thread.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int G, bool FM, bool PEER>
__global__ void __launch_bounds__(32 * G) lookup_tile_kernel(const FieldDev* __restrict__ fields_g, int32_t n_fields,
                                                            const int32_t* __restrict__ ids, int64_t ids_ld, int64_t batch,
                                                            float* __restrict__ out, int64_t out_ld, int32_t pitch /* floats */,
                                                            const float* __restrict__ fm_w, const float* __restrict__ fm_w0,
                                                            float* __restrict__ fm_out, float* __restrict__ fm_sum,
                                                            int32_t* __restrict__ oob, const float* const* __restrict__ peer_tab,
                                                            const int64_t* __restrict__ full_rows, int32_t n_ranks, int32_t n_tables) {
  constexpr int TS = 32;            // samples per tile
  constexpr int NT = 32 * G;        // threads: G lanes per sample
  constexpr int D = 4 * G;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* tile = reinterpret_cast<float*>(smem_raw);                                   // [TS][pitch]
  FieldDev* fields = reinterpret_cast<FieldDev*>(smem_raw + (size_t)TS * pitch * 4);  // descriptors
  for (int i = threadIdx.x; i < n_fields * (int)(sizeof(FieldDev) / 4); i += NT)
    reinterpret_cast<uint32_t*>(fields)[i] = reinterpret_cast<const uint32_t*>(fields_g)[i];
  __syncthreads();
  const int q = threadIdx.x % G, s = threadIdx.x / G;
  float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float w0 = 0.f;
  if (FM) {
    w4 = __ldg(reinterpret_cast<const float4*>(fm_w) + q);
    w0 = __ldg(fm_w0);
  }
  const int out_col0 = fields[0].out_col;
  const uint32_t row_bytes = (uint32_t)(n_fields * D * 4);
  const int64_t n_tiles = (batch + TS - 1) / TS;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t b = t * TS + s;
    const bool valid = b < batch;
    const int32_t* ids_row = ids + (valid ? b : 0) * ids_ld;
    float* my_row = tile + (size_t)s * pitch;
    // gather: ids first (independent loads), then one 16-byte async copy per (field, chunk).  (A 64-byte 1-D bulk copy per row and a
    // plain ld.global.nc + st.shared variant were measured too: within 2 % locally and over NVLink, so the simplest form stays.)
    constexpr int FU = 13;
    for (int f0 = 0; f0 < n_fields; f0 += FU) {
      int32_t id[FU];
#pragma unroll
      for (int u = 0; u < FU; ++u) id[u] = (valid && f0 + u < n_fields) ? __ldg(ids_row + fields[f0 + u].ids_col) : 0;
#pragma unroll
      for (int u = 0; u < FU; ++u) {
        if (f0 + u < n_fields) {
          const FieldDev& f = fields[f0 + u];
          float* dst = my_row + (f0 + u) * D + q * 4;
          // a table without peer pointers is replicated: read the local copy
          const bool remote = PEER && peer_tab[f.table_idx] != nullptr;
          const int64_t vocab = remote ? __ldg(full_rows + f.table_idx) : f.rows;
          if (valid && id[u] >= 0 && (int64_t)id[u] < vocab) {
            const float* src;
            if (remote)  // row-sharded table: the row lives on rank id % N (NVLink peer mapping) at local row id / N
              src = peer_tab[(id[u] % n_ranks) * n_tables + f.table_idx] + (int64_t)(id[u] / n_ranks) * D + q * 4;
            else
              src = f.table + (int64_t)id[u] * D + q * 4;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr_u32(dst)), "l"(src) : "memory");
          } else {
            *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid && oob != nullptr) {
              oob[0] = 1;
              oob[1] = (int32_t)b;
            }
          }
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // rows must be visible to the bulk-store engine
    __syncthreads();
    // one bulk store per sample row (1664 B at F=26, D=16): shared -> global, full lines
    if (q == 0 && valid)
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out + b * out_ld + out_col0),
                   "r"(smem_addr_u32(my_row)), "r"(row_bytes)
                   : "memory");
    if (q == 0) asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    if (FM) {
      float4 S = make_float4(0.f, 0.f, 0.f, 0.f), Q = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4* r4 = reinterpret_cast<const float4*>(my_row) + q;
#pragma unroll 2
      for (int f = 0; f < n_fields; ++f) {
        const float4 v = r4[f * G];
        S.x += v.x; S.y += v.y; S.z += v.z; S.w += v.w;
        Q.x = fmaf(v.x, v.x, Q.x); Q.y = fmaf(v.y, v.y, Q.y); Q.z = fmaf(v.z, v.z, Q.z); Q.w = fmaf(v.w, v.w, Q.w);
      }
      float p2 = S.x * w4.x + S.y * w4.y + S.z * w4.z + S.w * w4.w;
      float p3 = (S.x * S.x - Q.x) + (S.y * S.y - Q.y) + (S.z * S.z - Q.z) + (S.w * S.w - Q.w);
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) {
        p2 += __shfl_xor_sync(0xffffffffu, p2, o, G);
        p3 += __shfl_xor_sync(0xffffffffu, p3, o, G);
      }
      if (valid && q == 0) fm_out[b] = p2 + 0.5f * p3 + w0;
      if (valid && fm_sum != nullptr) reinterpret_cast<float4*>(fm_sum + b * (int64_t)D)[q] = S;
    }
    // the tile is rewritten next iteration: the bulk stores must have finished READING it
    if (q == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// a13 backward.  Step 1: keys.  One thread per (sample, field): key = key_base(table) + id for
// every valid position, SENTINEL (= total rows, sorts last) for padding; scale = 1/n_valid (mean).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bwd_keys_kernel(const FieldDev* __restrict__ fields, int32_t n_fields,
                                                      int32_t pos_cols, const int32_t* __restrict__ ids,
                                                      int64_t ids_ld, int64_t batch, uint32_t sentinel,
                                                      uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                      float* __restrict__ scale) {
  const int64_t total = batch * n_fields;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_fields;
    const int fi = (int)(i - b * n_fields);
    const FieldDev& f = fields[fi];
    const int32_t* idp = ids + b * ids_ld + f.ids_col;
    const int64_t p0 = b * pos_cols + f.pos_col;
    int cnt = 0;
    for (int l = 0; l < f.seq_len; ++l) {
      const int32_t id = idp[l];
      const bool valid = (f.pool == HRB_POOL_NONE || id != 0) && id >= 0 && (int64_t)id < f.rows;
      cnt += valid;
      keys[p0 + l] = valid ? f.key_base + (uint32_t)id : sentinel;
      vals[p0 + l] = (uint32_t)(p0 + l);
    }
    scale[i] = f.pool == HRB_POOL_MEAN ? (cnt > 0 ? __fdiv_rn(1.0f, (float)cnt) : 0.f) : 1.0f;
  }
}

__global__ void __launch_bounds__(256) flat_keys_kernel(const int32_t* __restrict__ ids, int64_t n, int64_t vocab,
                                                       uint32_t sentinel, uint32_t* __restrict__ keys,
                                                       uint32_t* __restrict__ vals) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t id = ids[i];
    keys[i] = (id >= 0 && id < vocab) ? (uint32_t)id : sentinel;
    vals[i] = (uint32_t)i;
  }
}

// gradient sources -----------------------------------------------------------------------------
struct PlanGrad {  // gradient of position p comes from dout[b, out_col_f : +D] * scale[b,f]
  const FieldDev* fields;
  const int32_t* pos_field;
  const float* dout;
  const float* scale;
  int64_t dout_ld;
  int32_t pos_cols, n_fields;
  __device__ __forceinline__ float4 load(uint32_t p, int q, float& s) const {
    const int64_t b = p / (uint32_t)pos_cols;
    const int c = (int)(p - (uint32_t)b * (uint32_t)pos_cols);
    const int fi = __ldg(pos_field + c);
    s = __ldg(scale + b * n_fields + fi);
    if (q * 4 >= fields[fi].dim) return make_float4(0.f, 0.f, 0.f, 0.f);  // narrower table than the widest one
    return __ldg(reinterpret_cast<const float4*>(dout + b * dout_ld + fields[fi].out_col) + q);
  }
};
struct FlatGrad {  // gradient of position p is dout[p, :]
  const float* dout;
  int32_t dim;
  __device__ __forceinline__ float4 load(uint32_t p, int q, float& s) const {
    s = 1.0f;
    return __ldg(reinterpret_cast<const float4*>(dout + (int64_t)p * dim) + q);
  }
};

// row updates ----------------------------------------------------------------------------------
struct ApplyCtx {
  const TableDev* tables;
  int32_t n_tables;
  hrb_opt_params opt;
  float* dense_out;  // for the dense-gradient face
  float lr_t;        // adam: lr*sqrt(bc2)/bc1
};

__device__ __forceinline__ int find_table(const TableDev* __restrict__ t, int n, uint32_t key) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (t[mid].key_base <= key) lo = mid; else hi = mid - 1;
  }
  return lo;
}

template <int MODE>  // UpdMode: sgd, adam lazy, adagrad, ftrl, or dense gradient add
__device__ __forceinline__ void apply_row(const ApplyCtx& c, uint32_t key, int q, float4 g) {
  if (MODE == UPD_DENSE_ADD) {
    float4* p = reinterpret_cast<float4*>(c.dense_out + (int64_t)key * c.tables[0].dim) + q;
    float4 o = *p;
    o.x += g.x; o.y += g.y; o.z += g.z; o.w += g.w;
    *p = o;
    return;
  }
  const int ti = find_table(c.tables, c.n_tables, key);
  const TableDev& t = c.tables[ti];
  apply_table_row<MODE>(t, c.opt, c.lr_t, (int64_t)(key - t.key_base), q, g);
}

// Rows of tiny tables (vocab <= HOT_MAX_ROWS) collect thousands of duplicates per step (65536/V each at the Criteo
// shape).  They are taken out of the chunk/merge path: one CTA per such row finds the row's run in the sorted keys by
// binary search and reduces it with all its lanes (fixed assignment + fixed-order tree -> deterministic).
constexpr int HOT_MAX_ROWS = 128;   // 65536/128 = 512 duplicates per row at the bench batch: chains of >= 32 chunks
constexpr int HOT_SLICES = 8;      // CTAs per hot row (stage 1); stage 2 adds the slices in order
constexpr int HOT_MAX_RANGES = 32;
struct HotInfo {
  int32_t n_ranges;
  uint32_t lo[HOT_MAX_RANGES];
  uint32_t len[HOT_MAX_RANGES];
  const uint32_t* keys;  // key of hot row i (nullptr: key = i)
  int32_t n_keys;
};
__device__ __forceinline__ bool is_hot(const HotInfo& h, uint32_t key) {
  bool hot = false;
  for (int r = 0; r < h.n_ranges; ++r) hot |= (key - h.lo[r]) < h.len[r];
  return hot;
}

// lower_bound over sorted keys by a whole CTA: every round probes blockDim.x evenly spaced positions and keeps the one gap that
// brackets the answer.  All threads return the same value.
__device__ __forceinline__ int64_t block_lower_bound(const uint32_t* __restrict__ keys, int64_t n, uint32_t target) {
  int64_t lo = 0, hi = n;
  while (hi > lo) {
    const int nt = (int)blockDim.x;
    const int64_t step = (hi - lo + nt - 1) / nt;
    const int64_t p = lo + (int64_t)threadIdx.x * step;
    const bool less = p < hi && __ldg(keys + p) < target;
    const int c = __syncthreads_count(less);  // the predicate is monotone: probes 0..c-1 are below the target
    const int64_t nlo = c > 0 ? lo + (int64_t)(c - 1) * step + 1 : lo;
    const int64_t pc = lo + (int64_t)c * step;
    hi = (c < nt && pc < hi) ? pc : hi;
    lo = nlo;
  }
  return lo;
}

// stage 1: CTA (row, slice) reduces its slice of the row's run -> hot_partial[(row*HOT_SLICES + slice)][G*4]
template <typename GradSrc>
__global__ void __launch_bounds__(256) bwd_hot_slice_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                           int64_t n, int G, GradSrc src, HotInfo hot, float* __restrict__ hot_partial,
                                                           const uint32_t* __restrict__ dyn_count) {
  __shared__ float4 red[256];
  const int row = blockIdx.x / HOT_SLICES, slice = blockIdx.x % HOT_SLICES;
  if (dyn_count != nullptr && (uint32_t)row >= __ldg(dyn_count)) return;  // run-time list: rows past its end do not exist
  const uint32_t key = hot.keys != nullptr ? hot.keys[row] : (uint32_t)row;
  // the row's run [s_lo, s_hi) in the sorted keys: two 256-ary searches by the whole CTA (3 rounds of one load each at n = 1.7 M
  // instead of 2 x 21 dependent loads by one thread)
  const int64_t s_lo = block_lower_bound(keys, n, key);
  const int64_t s_hi = block_lower_bound(keys, n, key + 1u);
  const int64_t len = s_hi - s_lo;
  const int64_t lo = s_lo + len * slice / HOT_SLICES, hi = s_lo + len * (slice + 1) / HOT_SLICES;
  const int groups = blockDim.x / G;
  const int q = threadIdx.x % G, g = threadIdx.x / G;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (g < groups) {
    constexpr int U = 4;
    for (int64_t i0 = lo + g; i0 < hi; i0 += (int64_t)groups * U) {
      float4 v[U];
      float sc[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + (int64_t)u * groups;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        sc[u] = 0.f;
        if (i < hi) v[u] = src.load(__ldg(vals + i), q, sc[u]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        acc.x = fmaf(v[u].x, sc[u], acc.x); acc.y = fmaf(v[u].y, sc[u], acc.y);
        acc.z = fmaf(v[u].z, sc[u], acc.z); acc.w = fmaf(v[u].w, sc[u], acc.w);
      }
    }
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int stride = 128; stride >= G; stride >>= 1) {  // fixed-order tree over the groups (same q: G apart)
    if (threadIdx.x < stride && threadIdx.x + stride < groups * G) {
      const float4 o = red[threadIdx.x + stride];
      float4 m = red[threadIdx.x];
      m.x += o.x; m.y += o.y; m.z += o.z; m.w += o.w;
      red[threadIdx.x] = m;
    }
    __syncthreads();
  }
  if (threadIdx.x < G) reinterpret_cast<float4*>(hot_partial + (size_t)blockIdx.x * (G * 4))[threadIdx.x] = red[threadIdx.x];
  if (threadIdx.x == 0 && slice == 0) hot_partial[(size_t)gridDim.x * (G * 4) + row] = (float)(len > 0);  // touched flag
}
// stage 2: one group per hot row adds its slices in order and updates the row
template <int MODE>
__global__ void __launch_bounds__(256) bwd_hot_apply_kernel(int n_rows, int G, ApplyCtx ctx, HotInfo hot, const float* __restrict__ hot_partial,
                                                           const uint32_t* __restrict__ dyn_count) {
  const int gpb = blockDim.x / G;
  const int row = blockIdx.x * gpb + threadIdx.x / G, q = threadIdx.x % G;
  if (threadIdx.x / G >= gpb || row >= n_rows) return;
  if (dyn_count != nullptr && (uint32_t)row >= __ldg(dyn_count)) return;
  if (hot_partial[(size_t)n_rows * HOT_SLICES * (G * 4) + row] == 0.f) return;  // row not touched by this batch
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int sl = 0; sl < HOT_SLICES; ++sl) {
    const float4 v = reinterpret_cast<const float4*>(hot_partial + ((size_t)row * HOT_SLICES + sl) * (G * 4))[q];
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  apply_row<MODE>(ctx, hot.keys != nullptr ? hot.keys[row] : (uint32_t)row, q, acc);
}

// Long runs found at run time.  A row whose run in the sorted keys covers two consecutive sample points (every LONG_STEP-th
// position), i.e. any run of >= 2*LONG_STEP positions and some of LONG_STEP+1..2*LONG_STEP-1, is "long": skewed ids (Zipf
// histories, popular items) produce runs of 10^4..10^5 positions, whose chunk partials the merge kernel would add one after the
// other (measured: 2.8 of DIN's 4.9 ms of GPU time per step).  Long rows leave the chunk/merge path like the host-known hot rows
// above: bwd_long_detect_kernel lists them (one entry per row), HOT_SLICES CTAs per row reduce slices of the run, one group adds
// the slices in order.  The classification is a pure function of the sorted keys, so every kernel agrees on it.
constexpr int LONG_STEP = 256;
struct LongInfo {
  uint32_t* keys;  // [max] rows found by bwd_long_detect_kernel
  uint32_t* count; // [1]
  int32_t max;     // 0: disabled
};
// key k at sorted position i (k = keys[i]) -- does its run cover two consecutive sample points?  Only the four sample points
// around i can be involved: the run contains i, so if it holds two consecutive sample points it holds one next to i.
__device__ __forceinline__ bool run_is_long(const uint32_t* __restrict__ keys, int64_t n, uint32_t sentinel, int64_t i, uint32_t k) {
  const int64_t p0 = i / LONG_STEP * LONG_STEP;
  const uint32_t s0 = __ldg(keys + p0);
  const uint32_t s1 = p0 + LONG_STEP < n ? __ldg(keys + p0 + LONG_STEP) : sentinel;
  if (s0 == k && s1 == k) return true;
  if (s0 == k) return p0 >= LONG_STEP && __ldg(keys + p0 - LONG_STEP) == k;
  if (s1 == k) return p0 + 2 * LONG_STEP < n && __ldg(keys + p0 + 2 * LONG_STEP) == k;
  return false;
}

__global__ void __launch_bounds__(256) bwd_long_detect_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t sentinel, HotInfo hot,
                                                             LongInfo lg) {
  const int64_t n_pts = (n + LONG_STEP - 1) / LONG_STEP;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j + 1 < n_pts; j += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = __ldg(keys + j * LONG_STEP);
    if (k == sentinel || is_hot(hot, k)) continue;
    if (__ldg(keys + (j + 1) * LONG_STEP) != k) continue;
    if (j > 0 && __ldg(keys + (j - 1) * LONG_STEP) == k) continue;  // the first pair of the run reports it
    const uint32_t slot = atomicAdd(lg.count, 1u);
    if (slot < (uint32_t)lg.max) lg.keys[slot] = k;
  }
}

// Step 3: chunk kernel.  G lanes own CH consecutive sorted positions.  Runs (equal keys) that lie
// strictly inside the chunk are final and update their row at once; the (at most two) runs that
// touch a chunk edge and continue across it go to the partial buffer (slot 0 = head, 1 = tail).
constexpr int CH = 8;
constexpr uint32_t PF_VALID = 1u, PF_CONT = 2u, PF_ROPEN = 4u;

template <int MODE, typename GradSrc>
__global__ void __launch_bounds__(256) bwd_chunk_kernel(const uint32_t* __restrict__ keys,
                                                       const uint32_t* __restrict__ vals, int64_t n,
                                                       uint32_t sentinel, int G, GradSrc src, ApplyCtx ctx,
                                                       float* __restrict__ partial /* (2*chunks, G*4) */,
                                                       uint32_t* __restrict__ pkey, uint32_t* __restrict__ pflag, HotInfo hot,
                                                       bool long_rows) {
  const int groups_per_block = blockDim.x / G;
  const int q = threadIdx.x % G;
  const int g_in_block = threadIdx.x / G;
  if (g_in_block >= groups_per_block) return;
  const int64_t n_chunks = (n + CH - 1) / CH;
  for (int64_t chunk = blockIdx.x * (int64_t)groups_per_block + g_in_block; chunk < n_chunks;
       chunk += (int64_t)gridDim.x * groups_per_block) {
    const int64_t i0 = chunk * CH;
    uint32_t k[CH];
    float4 g[CH];
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      k[j] = (i0 + j < n) ? __ldg(keys + i0 + j) : sentinel;
      if (k[j] != sentinel && is_hot(hot, k[j])) k[j] = sentinel;  // rows of tiny tables belong to bwd_hot_kernel
    }
    if (long_rows) {  // positions of long runs belong to the slice kernels (a chunk never straddles a sample block: LONG_STEP % CH == 0)
      bool lr = false;
      uint32_t kl = sentinel;
#pragma unroll
      for (int j = 0; j < CH; ++j) {
        if (k[j] == sentinel) continue;
        if (k[j] != kl) {  // one test per distinct key of the chunk
          kl = k[j];
          lr = run_is_long(keys, n, sentinel, i0 + j, kl);
        }
        if (lr) k[j] = sentinel;
      }
    }
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k[j] != sentinel) {
        float s;
        const float4 v = src.load(__ldg(vals + i0 + j), q, s);
        g[j] = make_float4(v.x * s, v.y * s, v.z * s, v.w * s);
      }
    }
    uint32_t kprev = i0 > 0 ? __ldg(keys + i0 - 1) : sentinel;
    uint32_t knext = (i0 + CH < n) ? __ldg(keys + i0 + CH) : sentinel;
    if (kprev != sentinel && is_hot(hot, kprev)) kprev = sentinel;
    if (knext != sentinel && is_hot(hot, knext)) knext = sentinel;
    if (q == 0) {
      pflag[2 * chunk] = 0;
      pflag[2 * chunk + 1] = 0;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int run_start = 0;
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      acc.x += g[j].x; acc.y += g[j].y; acc.z += g[j].z; acc.w += g[j].w;
      const bool last = (j == CH - 1);
      const uint32_t kn = last ? knext : k[j + 1];
      if (last || kn != k[j]) {  // run [run_start, j] ends here (inside this chunk)
        if (k[j] != sentinel) {
          const bool lopen = (run_start == 0) && (i0 > 0) && (kprev == k[j]);
          const bool ropen = last && (kn == k[j]);
          if (!lopen && !ropen) {
            apply_row<MODE>(ctx, k[j], q, acc);
          } else {
            const int slot = (run_start == 0) ? 0 : 1;
            reinterpret_cast<float4*>(partial + (2 * chunk + slot) * (int64_t)(G * 4))[q] = acc;
            if (q == 0) {
              pkey[2 * chunk + slot] = k[j];
              pflag[2 * chunk + slot] = PF_VALID | (lopen ? PF_CONT : 0u) | (ropen ? PF_ROPEN : 0u);
            }
          }
        }
        acc = make_float4(0.f, 0.f, 0.f, 0.f);
        run_start = j + 1;
      }
    }
  }
}

// Step 4: merge kernel.  A partial that does not continue a previous chunk starts a chain; its group
// walks the head slots of the following chunks in order (fixed order -> deterministic) and updates the row.
template <int MODE>
__global__ void __launch_bounds__(256) bwd_merge_kernel(int64_t n_chunks, int G, ApplyCtx ctx,
                                                       const float* __restrict__ partial,
                                                       const uint32_t* __restrict__ pkey,
                                                       const uint32_t* __restrict__ pflag) {
  const int groups_per_block = blockDim.x / G;
  const int q = threadIdx.x % G;
  const int g_in_block = threadIdx.x / G;
  if (g_in_block >= groups_per_block) return;
  const int64_t n_slots = 2 * n_chunks;
  for (int64_t slot = blockIdx.x * (int64_t)groups_per_block + g_in_block; slot < n_slots;
       slot += (int64_t)gridDim.x * groups_per_block) {
    const uint32_t fl = __ldg(pflag + slot);
    if (!(fl & PF_VALID) || (fl & PF_CONT)) continue;
    float4 acc = reinterpret_cast<const float4*>(partial + slot * (int64_t)(G * 4))[q];
    if (fl & PF_ROPEN) {
      // hot rows span hundreds of chunks: fetch 8 head partials at a time (independent loads), add them in
      // chunk order and stop at the first one that does not continue to the right
      constexpr int W = 8;
      bool open = true;
      for (int64_t c0 = slot / 2 + 1; open && c0 < n_chunks; c0 += W) {
        uint32_t f2[W];
        float4 v[W];
#pragma unroll
        for (int u = 0; u < W; ++u) {
          const bool in = c0 + u < n_chunks;
          f2[u] = in ? __ldg(pflag + 2 * (c0 + u)) : 0u;
          v[u] = in ? __ldg(reinterpret_cast<const float4*>(partial + (2 * (c0 + u)) * (int64_t)(G * 4)) + q)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < W; ++u) {
          if (open && c0 + u < n_chunks) {
            acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
            if (!(f2[u] & PF_ROPEN)) open = false;
          }
        }
      }
    }
    apply_row<MODE>(ctx, __ldg(pkey + slot), q, acc);
  }
}

__global__ void __launch_bounds__(256) dense_grad_init_kernel(const float* __restrict__ table, float l2_scale,
                                                             int64_t n, float* __restrict__ dtable) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dtable[i] = table != nullptr ? l2_scale * table[i] : 0.0f;
}

static inline unsigned grid_for(int64_t work_items, int threads, int waves = 8) {
  int64_t blocks = (work_items + threads - 1) / threads;
  const int64_t cap = (int64_t)sm_count() * waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

struct BwdWorkspace {
  uint32_t *keys_in, *keys_out, *vals_in, *vals_out, *pkey, *pflag;
  float *scale, *partial, *hot_partial, *long_partial;
  uint32_t *long_keys, *long_count;
  int32_t long_max;
  void* cub_tmp;
  size_t cub_bytes;
  size_t total;
};

static int carve_bwd_ws(int64_t n, int64_t scale_elems, int max_dim, int key_bits, void* base, BwdWorkspace& w) {
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? (void*)((char*)base + off) : nullptr;
    off += align_up(bytes);
    return p;
  };
  const int64_t n_chunks = (n + CH - 1) / CH;
  w.keys_in = (uint32_t*)take((size_t)n * 4);
  w.keys_out = (uint32_t*)take((size_t)n * 4);
  w.vals_in = (uint32_t*)take((size_t)n * 4);
  w.vals_out = (uint32_t*)take((size_t)n * 4);
  w.scale = (float*)take((size_t)scale_elems * 4);
  w.partial = (float*)take((size_t)n_chunks * 2 * max_dim * 4);
  w.pkey = (uint32_t*)take((size_t)n_chunks * 2 * 4);
  w.pflag = (uint32_t*)take((size_t)n_chunks * 2 * 4);
  w.hot_partial = (float*)take((size_t)HOT_MAX_RANGES * HOT_MAX_ROWS * (HOT_SLICES * max_dim + 1) * 4);
  w.long_max = (int32_t)(n / (2 * LONG_STEP) + 2);  // a listed row covers two sample points of its own: at most n / LONG_STEP / 2 rows
  w.long_keys = (uint32_t*)take((size_t)w.long_max * 4);
  w.long_count = (uint32_t*)take(4);
  w.long_partial = (float*)take((size_t)w.long_max * (HOT_SLICES * max_dim + 1) * 4);
  size_t cub_bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, key_bits);
  if (e != cudaSuccess) return fail(HRB_CUDA_ERROR, "cub temp size query: %s", cudaGetErrorString(e));
  w.cub_bytes = cub_bytes;
  w.cub_tmp = take(cub_bytes);
  w.total = off;
  return HRB_OK;
}

static int bits_for(uint64_t max_value) {
  int b = 1;
  while (b < 32 && (max_value >> b) != 0) ++b;
  return b;
}

static HotInfo hot_from_plan(const hrb_plan* plan) {
  HotInfo h{};
  h.n_ranges = (int32_t)plan->hot_lo.size();
  for (int i = 0; i < h.n_ranges; ++i) {
    h.lo[i] = plan->hot_lo[i];
    h.len[i] = plan->hot_len[i];
  }
  h.keys = plan->d_hot_keys;
  h.n_keys = plan->n_hot_keys;
  return h;
}

template <typename GradSrc>
static int run_sorted_update(int mode, const BwdWorkspace& w, int64_t n, uint32_t sentinel, int key_bits, int G,
                             GradSrc src, ApplyCtx ctx, const HotInfo& hot_in, cudaStream_t st) {
  HotInfo hot = hot_in;
  if ((G & (G - 1)) != 0 || G > 128) {  // the hot-row tree reduction pairs lanes a power of two apart
    hot.n_keys = 0;
    hot.n_ranges = 0;
  }
  size_t cub_bytes = w.cub_bytes;
  HRB_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, cub_bytes, w.keys_in, w.keys_out, w.vals_in, w.vals_out,
                                           (int)n, 0, key_bits, st));
  count_launches(1 + (key_bits + 7) / 8);  // CUB onesweep: one histogram pass + one pass per 8 key bits
  const int64_t n_chunks = (n + CH - 1) / CH;
  const int threads = 256;
  const int gpb = threads / G;
  const unsigned grid1 = grid_for(n_chunks * G, gpb * G, 16);
  const unsigned grid2 = grid_for(2 * n_chunks * G, gpb * G, 16);
  const int launch_threads = gpb * G;
  // run-time long rows: worth a pass once a run can span two sample points at all
  const bool long_rows = (G & (G - 1)) == 0 && G <= 128 && n >= 4 * LONG_STEP;
  LongInfo lg{w.long_keys, w.long_count, long_rows ? w.long_max : 0};
  HotInfo dyn{};
  dyn.keys = w.long_keys;
  dyn.n_keys = w.long_max;
  if (long_rows) {
    HRB_CUDA(cudaMemsetAsync(w.long_count, 0, 4, st));
    bwd_long_detect_kernel<<<grid_for((n + LONG_STEP - 1) / LONG_STEP, 256), 256, 0, st>>>(w.keys_out, n, sentinel, hot, lg);
    HRB_LAUNCH_CHECK();
  }
#define HRB_RUN_MODE(M)                                                                                        \
  bwd_chunk_kernel<M, GradSrc><<<grid1, launch_threads, 0, st>>>(w.keys_out, w.vals_out, n, sentinel, G, src, \
                                                                 ctx, w.partial, w.pkey, w.pflag, hot, long_rows); \
  HRB_LAUNCH_CHECK();                                                                                          \
  if (hot.n_keys > 0) {                                                                                        \
    bwd_hot_slice_kernel<GradSrc><<<hot.n_keys * HOT_SLICES, launch_threads, 0, st>>>(w.keys_out, w.vals_out, n, G, src, hot, w.hot_partial, nullptr); \
    HRB_LAUNCH_CHECK();                                                                                        \
    bwd_hot_apply_kernel<M><<<(hot.n_keys + gpb - 1) / gpb, launch_threads, 0, st>>>(hot.n_keys, G, ctx, hot, w.hot_partial, nullptr); \
    HRB_LAUNCH_CHECK();                                                                                        \
  }                                                                                                            \
  if (long_rows) {                                                                                             \
    bwd_hot_slice_kernel<GradSrc><<<w.long_max * HOT_SLICES, launch_threads, 0, st>>>(w.keys_out, w.vals_out, n, G, src, dyn, w.long_partial, w.long_count); \
    HRB_LAUNCH_CHECK();                                                                                        \
    bwd_hot_apply_kernel<M><<<(w.long_max + gpb - 1) / gpb, launch_threads, 0, st>>>(w.long_max, G, ctx, dyn, w.long_partial, w.long_count); \
    HRB_LAUNCH_CHECK();                                                                                        \
  }                                                                                                            \
  bwd_merge_kernel<M><<<grid2, launch_threads, 0, st>>>(n_chunks, G, ctx, w.partial, w.pkey, w.pflag);         \
  HRB_LAUNCH_CHECK();
  if (mode == UPD_SGD) {
    HRB_RUN_MODE(UPD_SGD)
  } else if (mode == UPD_ADAM) {
    HRB_RUN_MODE(UPD_ADAM)
  } else if (mode == UPD_ADAGRAD) {
    HRB_RUN_MODE(UPD_ADAGRAD)
  } else if (mode == UPD_FTRL) {
    HRB_RUN_MODE(UPD_FTRL)
  } else {
    HRB_RUN_MODE(UPD_DENSE_ADD)
  }
#undef HRB_RUN_MODE
  return HRB_OK;
}

}  // namespace hrb

using namespace hrb;

// =============================================================================================
// C ABI
// =============================================================================================
HRB_API int hrb_embedding_fwd(const float* table, int64_t vocab, int32_t dim, const int32_t* ids, int64_t n_ids,
                              float* out, uint8_t* mask, int32_t* oob, void* stream) {
  HRB_REQUIRE(vocab > 0 && dim > 0 && n_ids >= 0, "hrb_embedding_fwd: null/negative argument");
  if (n_ids == 0) return HRB_OK;  // empty batch: nothing to read or write (pointers may be NULL)
  HRB_REQUIRE(table && ids && out, "hrb_embedding_fwd: null/negative argument");
  if (dim % 4 != 0) return fail(HRB_UNSUPPORTED, "hrb_embedding_fwd: dim %d is not a multiple of 4", dim);
  HRB_REQUIRE(aligned16(table) && aligned16(out), "hrb_embedding_fwd: table/out must be 16-byte aligned");
  HRB_REQUIRE(mask == nullptr || (reinterpret_cast<uintptr_t>(mask) & 3u) == 0, "hrb_embedding_fwd: mask must be 4-byte aligned");
  if (n_ids == 0) return HRB_OK;
  const int chunks = dim / 4;
  const unsigned grid = grid_for((n_ids * chunks + 3) / 4, 256, 8);
  embedding_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(table, vocab, chunks, ids, n_ids, out, mask, oob);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_seq_pool_fwd(const float* x, const uint8_t* mask, int64_t batch, int32_t seq_len, int32_t dim,
                             int32_t method, float* out, void* stream) {
  HRB_REQUIRE(x && out && batch >= 0 && seq_len > 0 && dim > 0, "hrb_seq_pool_fwd: null/negative argument");
  HRB_REQUIRE(mask != nullptr, "hrb_seq_pool_fwd: mask is NULL (Embedding layer should set `mask_zero` as True)");
  HRB_REQUIRE(method == HRB_POOL_MEAN || method == HRB_POOL_SUM || method == HRB_POOL_MAX,
              "hrb_seq_pool_fwd: Pooling method should be `mean`, `max`, or `sum`");
  if (batch == 0) return HRB_OK;
  seq_pool_fwd_kernel<<<grid_for(batch * dim, 256), 256, 0, (cudaStream_t)stream>>>(x, mask, batch, seq_len, dim,
                                                                                    method, out);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_seq_pool_bwd(const float* x, const uint8_t* mask, const float* dout, int64_t batch, int32_t seq_len,
                             int32_t dim, int32_t method, float* dx, void* stream) {
  HRB_REQUIRE(x && mask && dout && dx && batch >= 0 && seq_len > 0 && dim > 0, "hrb_seq_pool_bwd: null/negative argument");
  HRB_REQUIRE(method == HRB_POOL_MEAN || method == HRB_POOL_SUM || method == HRB_POOL_MAX,
              "hrb_seq_pool_bwd: Pooling method should be `mean`, `max`, or `sum`");
  if (batch == 0) return HRB_OK;
  seq_pool_bwd_kernel<<<grid_for(batch * dim, 256), 256, 0, (cudaStream_t)stream>>>(x, mask, dout, batch, seq_len,
                                                                                    dim, method, dx);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_plan_create(const hrb_table_desc* tables_host, int32_t n_tables, const hrb_field_desc* fields_host,
                            int32_t n_fields, hrb_plan** plan_out) {
  HRB_REQUIRE(tables_host && fields_host && plan_out && n_tables > 0 && n_fields > 0, "hrb_plan_create: null/empty argument");
  hrb_plan* p = new (std::nothrow) hrb_plan();
  HRB_REQUIRE(p != nullptr, "hrb_plan_create: out of host memory");
  p->n_tables = n_tables;
  p->n_fields = n_fields;
  p->tables.assign(tables_host, tables_host + n_tables);
  p->fields.assign(fields_host, fields_host + n_fields);
  uint64_t base = 0;
  p->tdev_host.resize(n_tables);
  for (int t = 0; t < n_tables; ++t) {
    const hrb_table_desc& td = p->tables[t];
    if (!td.weight || td.rows <= 0 || td.dim <= 0 || td.dim % 4 != 0 || !aligned16(td.weight) ||
        (td.adam_m && !aligned16(td.adam_m)) || (td.adam_v && !aligned16(td.adam_v))) {
      delete p;
      return fail(td.dim % 4 ? HRB_UNSUPPORTED : HRB_BAD_ARG,
                  "hrb_plan_create: table %d needs a 16-byte aligned weight, rows>0 and dim%%4==0 (dim=%d)", t, td.dim);
    }
    p->tdev_host[t] = TableDev{td.weight, td.adam_m, td.adam_v, td.rows, (uint32_t)base, td.dim, nullptr};
    base += (uint64_t)td.rows;
    if (td.dim > p->max_dim) p->max_dim = td.dim;
  }
  if (base >= 0xFFFFFFFFull) {
    delete p;
    return fail(HRB_UNSUPPORTED, "hrb_plan_create: %llu total rows do not fit 32-bit sort keys", (unsigned long long)base);
  }
  p->total_rows = base;
  p->key_bits = bits_for(base);
  p->fdev_host.resize(n_fields);
  std::vector<int32_t> chunk_field, chunk_q, pos_field;
  const int32_t dim0 = p->tables[p->fields[0].table < n_tables && p->fields[0].table >= 0 ? p->fields[0].table : 0].dim;
  for (int f = 0; f < n_fields; ++f) {
    const hrb_field_desc& fd = p->fields[f];
    if (fd.table < 0 || fd.table >= n_tables || fd.seq_len <= 0 || fd.ids_col < 0 || fd.out_col < 0 ||
        fd.out_col % 4 != 0 || fd.pool < HRB_POOL_NONE || fd.pool > HRB_POOL_MAX ||
        (fd.pool == HRB_POOL_NONE && fd.seq_len != 1)) {
      delete p;
      return fail(HRB_BAD_ARG, "hrb_plan_create: field %d is malformed (table/seq_len/cols/pool)", f);
    }
    const TableDev& td = p->tdev_host[fd.table];
    p->fdev_host[f] = FieldDev{td.w, td.rows, td.key_base, td.dim, fd.seq_len, fd.pool, fd.ids_col, fd.out_col,
                               p->pos_cols, fd.table};
    for (int l = 0; l < fd.seq_len; ++l) pos_field.push_back(f);
    p->pos_cols += fd.seq_len;
    for (int q = 0; q < td.dim / 4; ++q) {
      chunk_field.push_back(f);
      chunk_q.push_back(q);
    }
    if (td.dim != dim0) p->uniform_dim = false;
    if (fd.out_col != p->fields[0].out_col + f * dim0) p->contiguous_out = false;
    if (fd.seq_len != 1 || fd.pool != HRB_POOL_NONE) p->all_len1 = false;
    if (fd.pool == HRB_POOL_MAX) p->has_max = true;
  }
  if (!p->uniform_dim) p->contiguous_out = false;
  p->out_chunks = (int32_t)chunk_field.size();
  // tiny tables: their rows are reduced by bwd_hot_kernel (one CTA per row)
  std::vector<uint32_t> hot_keys;
  for (int t = 0; t < n_tables && (int)p->hot_lo.size() < 32; ++t) {
    const TableDev& td = p->tdev_host[t];
    if (td.rows <= 128) {
      p->hot_lo.push_back(td.key_base);
      p->hot_len.push_back((uint32_t)td.rows);
      for (int64_t r = 0; r < td.rows; ++r) hot_keys.push_back(td.key_base + (uint32_t)r);
    }
  }
  p->n_hot_keys = (int32_t)hot_keys.size();
  // one device blob: fields | tables | chunk_field | chunk_q | pos_field | hot_keys
  const size_t sz_f = align_up(sizeof(FieldDev) * n_fields), sz_t = align_up(sizeof(TableDev) * n_tables);
  const size_t sz_c = align_up(sizeof(int32_t) * chunk_field.size()), sz_p = align_up(sizeof(int32_t) * pos_field.size());
  const size_t sz_h = align_up(sizeof(uint32_t) * (hot_keys.size() + 1));
  // position columns grouped by table (embedding_bwd.cu: a unit scans every column of its table)
  std::vector<ColDev> cols;
  p->col_start_host.assign(n_tables + 1, 0);
  p->unit_path_ok = true;
  for (int t = 0; t < n_tables; ++t) {
    p->col_start_host[t] = (int32_t)cols.size();
    for (int f = 0; f < n_fields; ++f) {
      if (p->fields[f].table != t) continue;
      for (int l = 0; l < p->fields[f].seq_len; ++l)
        cols.push_back(ColDev{p->fdev_host[f].pos_col + l, p->fields[f].out_col, f, 0});
      if (p->fields[f].pool == HRB_POOL_MEAN) p->has_mean = true;
    }
    const int g = p->tdev_host[t].dim / 4;
    if ((int)cols.size() - p->col_start_host[t] > 256 || (g & (g - 1)) != 0 || g > 32) p->unit_path_ok = false;
  }
  p->col_start_host[n_tables] = (int32_t)cols.size();
  const size_t sz_cols = align_up(sizeof(ColDev) * (cols.size() + 1)), sz_cs = align_up(sizeof(int32_t) * (n_tables + 1));
  const size_t total = sz_f + sz_t + 2 * sz_c + sz_p + sz_h + sz_cols + sz_cs;
  std::vector<char> blob(total, 0);
  memcpy(blob.data(), p->fdev_host.data(), sizeof(FieldDev) * n_fields);
  memcpy(blob.data() + sz_f, p->tdev_host.data(), sizeof(TableDev) * n_tables);
  memcpy(blob.data() + sz_f + sz_t, chunk_field.data(), sizeof(int32_t) * chunk_field.size());
  memcpy(blob.data() + sz_f + sz_t + sz_c, chunk_q.data(), sizeof(int32_t) * chunk_q.size());
  memcpy(blob.data() + sz_f + sz_t + 2 * sz_c, pos_field.data(), sizeof(int32_t) * pos_field.size());
  if (!hot_keys.empty()) memcpy(blob.data() + sz_f + sz_t + 2 * sz_c + sz_p, hot_keys.data(), sizeof(uint32_t) * hot_keys.size());
  if (!cols.empty()) memcpy(blob.data() + sz_f + sz_t + 2 * sz_c + sz_p + sz_h, cols.data(), sizeof(ColDev) * cols.size());
  memcpy(blob.data() + sz_f + sz_t + 2 * sz_c + sz_p + sz_h + sz_cols, p->col_start_host.data(), sizeof(int32_t) * (n_tables + 1));
  cudaError_t e = cudaMalloc(&p->dev_blob, total);
  if (e == cudaSuccess) e = cudaMemcpy(p->dev_blob, blob.data(), total, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (p->dev_blob) cudaFree(p->dev_blob);
    delete p;
    return fail(HRB_CUDA_ERROR, "hrb_plan_create: %s", cudaGetErrorString(e));
  }
  char* d = (char*)p->dev_blob;
  p->d_fields = (FieldDev*)d;
  p->d_tables = (TableDev*)(d + sz_f);
  p->d_chunk_field = (int32_t*)(d + sz_f + sz_t);
  p->d_chunk_q = (int32_t*)(d + sz_f + sz_t + sz_c);
  p->d_pos_field = (int32_t*)(d + sz_f + sz_t + 2 * sz_c);
  p->d_hot_keys = (uint32_t*)(d + sz_f + sz_t + 2 * sz_c + sz_p);
  p->d_cols = (ColDev*)(d + sz_f + sz_t + 2 * sz_c + sz_p + sz_h);
  p->d_col_start = (int32_t*)(d + sz_f + sz_t + 2 * sz_c + sz_p + sz_h + sz_cols);
  *plan_out = p;
  return HRB_OK;
}

HRB_API int hrb_plan_destroy(hrb_plan* plan) {
  if (plan == nullptr) return HRB_OK;
  if (plan->dev_blob) cudaFree(plan->dev_blob);
  if (plan->d_peer_tab) cudaFree((void*)plan->d_peer_tab);
  if (plan->d_full_rows) cudaFree(plan->d_full_rows);
  if (plan->units.d_blob) cudaFree(plan->units.d_blob);
  delete plan;
  return HRB_OK;
}

static int check_lookup_args(const char* who, const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch,
                             const float* out, int64_t out_ld) {
  HRB_REQUIRE(plan && ids && out && batch >= 0, "%s: null/negative argument", who);
  HRB_REQUIRE(aligned16(out) && out_ld % 4 == 0, "%s: out must be 16-byte aligned with out_ld %% 4 == 0", who);
  for (const auto& f : plan->fdev_host) {
    HRB_REQUIRE(f.ids_col + f.seq_len <= ids_ld, "%s: ids_ld %lld too small for a field ending at column %d", who,
                (long long)ids_ld, f.ids_col + f.seq_len);
    HRB_REQUIRE(f.out_col + f.dim <= out_ld, "%s: out_ld %lld too small for a field ending at column %d", who,
                (long long)out_ld, f.out_col + f.dim);
  }
  return HRB_OK;
}

template <bool FM>
static int launch_rows(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* out,
                       int64_t out_ld, float* inv_count, const float* fm_w, const float* fm_w0, float* fm_out,
                       float* fm_sum, int32_t* oob, cudaStream_t st) {
  const int G = plan->max_dim / 4;
  // v2 tile kernel for plain-lookup groups laid out contiguously (the Criteo shape)
#ifdef HRB_DEVTOOLS
  static int use_tile = -1;
  if (use_tile < 0) {
    const char* e = getenv("HRB_LOOKUP_KERNEL");
    use_tile = (e != nullptr && strcmp(e, "rows") == 0) ? 0 : 1;
  }
#else
  const int use_tile = 1;
#endif
  if (use_tile && inv_count == nullptr && plan->all_len1 && plan->contiguous_out && (G == 2 || G == 4 || G == 8 || G == 16) && aligned16(out) &&
      (out_ld % 4 == 0) && (plan->fdev_host[0].out_col % 4 == 0)) {
    int pitch = plan->n_fields * plan->max_dim;       // floats
    while ((pitch / 4) % 8 != 4) pitch += 4;            // neighbouring samples 64 B apart mod 128
    const size_t smem = (size_t)32 * pitch * 4 + sizeof(FieldDev) * (size_t)plan->n_fields;
    if (smem <= 100 * 1024) {
      const int per_sm = (int)((220 * 1024) / (smem + 1024));
      int64_t tiles = (batch + 31) / 32;
      int64_t grid = (int64_t)sm_count() * (per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm));
      if (grid > tiles) grid = tiles;
#define HRB_TILE_P(GG, PP)                                                                                                    \
  {                                                                                                                           \
    static bool attr = false;                                                                                                 \
    if (!attr) {                                                                                                              \
      HRB_CUDA(cudaFuncSetAttribute(lookup_tile_kernel<GG, FM, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); \
      attr = true;                                                                                                            \
    }                                                                                                                         \
    lookup_tile_kernel<GG, FM, PP><<<(unsigned)grid, 32 * GG, smem, st>>>(plan->d_fields, plan->n_fields, ids, ids_ld, batch, \
                                                                          out, out_ld, pitch, fm_w, fm_w0, fm_out, fm_sum,    \
                                                                          oob, plan->d_peer_tab, plan->d_full_rows,           \
                                                                          plan->n_ranks, plan->n_tables);                     \
  }
#define HRB_TILE(GG)                                                                                                          \
  if (plan->d_peer_tab != nullptr) HRB_TILE_P(GG, true) else HRB_TILE_P(GG, false)
      switch (G) {
        case 2: HRB_TILE(2) break;
        case 4: HRB_TILE(4) break;
        case 8: HRB_TILE(8) break;
        default: HRB_TILE(16) break;
      }
#undef HRB_TILE_P
#undef HRB_TILE
      HRB_LAUNCH_CHECK();
      return HRB_OK;
    }
  }
  if (plan->d_peer_tab != nullptr)
    return fail(HRB_UNSUPPORTED, "peer-mapped (row-sharded) lookup is implemented for plain-lookup groups laid out contiguously only");
  const int spb = 256 / G;
  // enough CTAs for every SM to hold its full complement, persistent-style grid-stride over samples
  int64_t blocks = (batch + spb - 1) / spb;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  const size_t smem = sizeof(FieldDev) * (size_t)plan->n_fields;
  if (smem > 40 * 1024) return fail(HRB_UNSUPPORTED, "fused row kernel: too many fields (%d)", plan->n_fields);
#define HRB_ROWS(GG)                                                                                              \
  if (plan->all_len1)                                                                                             \
    lookup_rows_kernel<GG, true, FM><<<(unsigned)blocks, 256, smem, st>>>(plan->d_fields, plan->n_fields, ids, ids_ld, \
                                                                      batch, out, out_ld, inv_count, fm_w, fm_w0, \
                                                                      fm_out, fm_sum, oob);                       \
  else                                                                                                            \
    lookup_rows_kernel<GG, false, FM><<<(unsigned)blocks, 256, smem, st>>>(plan->d_fields, plan->n_fields, ids,      \
                                                                       ids_ld, batch, out, out_ld, inv_count,     \
                                                                       fm_w, fm_w0, fm_out, fm_sum, oob);
  switch (G) {
    case 1: HRB_ROWS(1) break;
    case 2: HRB_ROWS(2) break;
    case 4: HRB_ROWS(4) break;
    case 8: HRB_ROWS(8) break;
    case 16: HRB_ROWS(16) break;
    case 32: HRB_ROWS(32) break;
    default: return fail(HRB_UNSUPPORTED, "fused row kernel needs dim/4 in {1,2,4,8,16,32}, got dim=%d", plan->max_dim);
  }
#undef HRB_ROWS
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_lookup_fwd(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* out,
                           int64_t out_ld, float* inv_count, int32_t* oob, void* stream) {
  int rc = check_lookup_args("hrb_lookup_fwd", plan, ids, ids_ld, batch, out, out_ld);
  if (rc != HRB_OK) return rc;
  if (batch == 0) return HRB_OK;
  if (inv_count == nullptr && plan->all_len1 && plan->uniform_dim && plan->contiguous_out) {
    const int G = plan->max_dim / 4;
    if (G == 2 || G == 4 || G == 8 || G == 16)  // plain-lookup group: the cp.async / bulk-store tile kernel without the FM epilogue
      return launch_rows<false>(plan, ids, ids_ld, batch, out, out_ld, nullptr, nullptr, nullptr, nullptr, nullptr, oob, (cudaStream_t)stream);
  }
  const unsigned grid = grid_for(batch * plan->out_chunks, 256, 8);
  lookup_items_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(plan->d_fields, plan->d_chunk_field,
                                                                    plan->d_chunk_q, plan->out_chunks, plan->n_fields,
                                                                    ids, ids_ld, batch, out, out_ld, inv_count, oob);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_lookup_fm_fwd(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* out,
                              int64_t out_ld, float* inv_count, const float* fm_w, const float* fm_w0, float* fm_out,
                              float* fm_sum, int32_t* oob, void* stream) {
  int rc = check_lookup_args("hrb_lookup_fm_fwd", plan, ids, ids_ld, batch, out, out_ld);
  if (rc != HRB_OK) return rc;
  HRB_REQUIRE(fm_w && fm_w0 && fm_out, "hrb_lookup_fm_fwd: fm_w / fm_w0 / fm_out is NULL");
  HRB_REQUIRE(aligned16(fm_w) && (fm_sum == nullptr || aligned16(fm_sum)), "hrb_lookup_fm_fwd: fm_w/fm_sum must be 16-byte aligned");
  if (!plan->uniform_dim)
    return fail(HRB_UNSUPPORTED, "hrb_lookup_fm_fwd: FM needs every field to have the same embedding dim");
  if (batch == 0) return HRB_OK;
  return launch_rows<true>(plan, ids, ids_ld, batch, out, out_ld, inv_count, fm_w, fm_w0, fm_out, fm_sum, oob,
                           (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Touched rows for Ftrl, whose step with a zero gradient is not a no-op.  Keras gathers id 0 at the padding positions of a
// pooled field, so row 0 is in the IndexedSlices gradient (with a zero gradient) and steps; the backward above drops those
// positions.  mark_rows_kernel flags the touched rows of dense-updated tables; pad_flags_kernel notes per table whether the
// batch holds padding (flags[2t]) and whether a valid position names row 0 (flags[2t+1], then the backward steps row 0 with
// the gradient sum); ftrl_pad_kernel gives row 0 its zero-gradient step where only padding named it.  Every writer of a flag
// stores the same value, so plain stores suffice.
// ---------------------------------------------------------------------------------------------
constexpr int MARK_MAX_TABLES = 512;
struct TouchedPtrs {
  float* p[MARK_MAX_TABLES];
};

__global__ void __launch_bounds__(256) mark_rows_kernel(const FieldDev* __restrict__ fields, int32_t n_fields, const int32_t* __restrict__ ids,
                                                       int64_t ids_ld, int64_t batch, const TouchedPtrs tp) {
  const int64_t total = batch * n_fields;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_fields;
    const FieldDev& f = fields[i - b * n_fields];
    float* touched = tp.p[f.table_idx];
    if (touched == nullptr) continue;
    const int32_t* idp = ids + b * ids_ld + f.ids_col;
    for (int l = 0; l < f.seq_len; ++l) {
      const int32_t id = idp[l];
      if (id >= 0 && (int64_t)id < f.rows) touched[id] = 1.0f;
    }
  }
}

__global__ void __launch_bounds__(256) pad_flags_kernel(const FieldDev* __restrict__ fields, int32_t n_fields, const int32_t* __restrict__ ids,
                                                       int64_t ids_ld, int64_t batch, float* __restrict__ flags) {
  const int64_t total = batch * n_fields;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_fields;
    const FieldDev& f = fields[i - b * n_fields];
    const int32_t* idp = ids + b * ids_ld + f.ids_col;
    bool zero = false;
    for (int l = 0; l < f.seq_len; ++l) zero |= idp[l] == 0;
    float* fl = flags + 2 * f.table_idx + (f.pool == HRB_POOL_NONE ? 1 : 0);  // id 0 of a pooled field is padding
    if (zero && *fl == 0.f) *fl = 1.0f;
  }
}

// one CTA: row 0 of every row-updated table whose batch held padding and no valid id 0 takes a zero-gradient step
__global__ void __launch_bounds__(256) ftrl_pad_kernel(const TableDev* __restrict__ tables, int32_t n_tables, const float* __restrict__ flags,
                                                      const hrb_opt_params opt) {
  for (int32_t ti = 0; ti < n_tables; ++ti) {
    const TableDev& t = tables[ti];
    if (t.grad != nullptr || flags[2 * ti] == 0.f || flags[2 * ti + 1] != 0.f) continue;
    for (int e = threadIdx.x; e < t.dim; e += blockDim.x) {
      const float w = t.w[e];
      float a = t.m[e], l = t.v[e];
      t.w[e] = ftrl_elem(w, a, l, fmaf(opt.l2_scale, w, 0.f), opt.lr, opt.l1, opt.l2, opt.lr_power, opt.l2_shrinkage);
      t.m[e] = a;
      t.v[e] = l;
    }
  }
}

static bool has_pooled(const hrb_plan* plan) {
  for (const auto& f : plan->fdev_host)
    if (f.pool != HRB_POOL_NONE) return true;
  return false;
}
// the padding flags of hrb_lookup_bwd_update under Ftrl sit in the last bytes of its workspace
static size_t pad_flag_bytes(const hrb_plan* plan) { return has_pooled(plan) ? align_up((size_t)plan->n_tables * 8) : 0; }

static int ftrl_tables_ok(const hrb_plan* plan, const char* who) {
  for (const auto& t : plan->tdev_host)
    HRB_REQUIRE(t.grad || (t.m && t.v), "%s: Ftrl needs an accumulator (adam_m) and a linear slot (adam_v) for every row-updated table", who);
  return HRB_OK;
}

static int launch_pad_flags(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* flags, cudaStream_t st) {
  HRB_CUDA(cudaMemsetAsync(flags, 0, (size_t)plan->n_tables * 8, st));
  pad_flags_kernel<<<grid_for(batch * plan->n_fields, 256), 256, 0, st>>>(plan->d_fields, plan->n_fields, ids, ids_ld, batch, flags);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

static int launch_ftrl_pad(const hrb_plan* plan, const float* flags, const hrb_opt_params& opt, cudaStream_t st) {
  ftrl_pad_kernel<<<1, 256, 0, st>>>(plan->d_tables, plan->n_tables, flags, opt);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_plan_mark_rows(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* const* touched_host,
                               void* stream) {
  HRB_REQUIRE(plan && ids && touched_host && batch >= 0, "hrb_plan_mark_rows: null/negative argument");
  if (plan->n_tables > MARK_MAX_TABLES) return fail(HRB_UNSUPPORTED, "hrb_plan_mark_rows: more than %d tables", MARK_MAX_TABLES);
  TouchedPtrs tp{};
  bool any = false;
  for (int32_t t = 0; t < plan->n_tables; ++t) {
    tp.p[t] = touched_host[t];
    any |= touched_host[t] != nullptr;
  }
  if (batch == 0 || !any) return HRB_OK;
  mark_rows_kernel<<<grid_for(batch * plan->n_fields, 256), 256, 0, (cudaStream_t)stream>>>(plan->d_fields, plan->n_fields, ids, ids_ld,
                                                                                           batch, tp);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_plan_pad_flags(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* flags, void* stream) {
  HRB_REQUIRE(plan && ids && flags && batch >= 0, "hrb_plan_pad_flags: null/negative argument");
  if (batch == 0) return HRB_OK;
  pad_flags_kernel<<<grid_for(batch * plan->n_fields, 256), 256, 0, (cudaStream_t)stream>>>(plan->d_fields, plan->n_fields, ids, ids_ld,
                                                                                           batch, flags);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_plan_ftrl_pad_step(const hrb_plan* plan, const float* flags, const hrb_opt_params* opt_host, void* stream) {
  HRB_REQUIRE(plan && flags && opt_host, "hrb_plan_ftrl_pad_step: null argument");
  HRB_REQUIRE(opt_host->opt == HRB_OPT_FTRL, "hrb_plan_ftrl_pad_step: needs HRB_OPT_FTRL, got %d", opt_host->opt);
  int rc = ftrl_tables_ok(plan, "hrb_plan_ftrl_pad_step");
  if (rc != HRB_OK) return rc;
  return launch_ftrl_pad(plan, flags, load_opt(opt_host), (cudaStream_t)stream);
}

HRB_API int hrb_lookup_bwd_workspace(const hrb_plan* plan, int64_t ids_ld, int64_t batch, size_t* bytes) {
  HRB_REQUIRE(plan && bytes && batch >= 0, "hrb_lookup_bwd_workspace: null/negative argument");
  (void)ids_ld;
  const int64_t n = batch * plan->pos_cols;
  HRB_REQUIRE(n < 0x7FFFFFFFll, "hrb_lookup_bwd_workspace: batch*sum(seq_len) = %lld exceeds 2^31-1", (long long)n);
  BwdWorkspace w;
  int rc = carve_bwd_ws(n > 0 ? n : 1, batch * plan->n_fields + 1, plan->max_dim, plan->key_bits, nullptr, w);
  if (rc != HRB_OK) return rc;
  *bytes = w.total;
  if (unit_path_supported(plan, batch)) *bytes = std::max(w.total, unit_workspace_bytes(plan, batch));
  if (const size_t fb = pad_flag_bytes(plan)) *bytes = align_up(*bytes) + fb;  // hrb_lookup_bwd_update keeps the flags in the last fb bytes
  return HRB_OK;
}

static int run_plan_sorted_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const float* dout,
                                  int64_t dout_ld, const hrb_opt_params& opt, void* workspace, size_t workspace_bytes, cudaStream_t st);

HRB_API int hrb_lookup_bwd_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch,
                                  const float* dout, int64_t dout_ld, const float* inv_count,
                                  const hrb_opt_params* opt_host, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  (void)inv_count;  // recomputed from ids; accepted for symmetry with the forward
  HRB_REQUIRE(plan && ids && dout && opt_host && workspace && batch >= 0, "hrb_lookup_bwd_update: null/negative argument");
  HRB_REQUIRE(aligned16(dout) && dout_ld % 4 == 0, "hrb_lookup_bwd_update: dout must be 16-byte aligned, dout_ld %% 4 == 0");
  if (plan->has_max)
    return fail(HRB_UNSUPPORTED, "hrb_lookup_bwd_update: max-pooled fields go through hrb_seq_pool_bwd + hrb_embedding_bwd_dense");
  const hrb_opt_params opt = load_opt(opt_host);
  HRB_REQUIRE(opt.opt == HRB_OPT_SGD || opt.opt == HRB_OPT_ADAM_LAZY || opt.opt == HRB_OPT_ADAGRAD || opt.opt == HRB_OPT_FTRL,
              "hrb_lookup_bwd_update: unknown optimiser %d", opt.opt);
  if (opt.opt == HRB_OPT_ADAM_LAZY)
    for (const auto& t : plan->tdev_host)
      HRB_REQUIRE(t.grad || (t.m && t.v), "hrb_lookup_bwd_update: lazy Adam needs adam_m/adam_v for every table");
  if (opt.opt == HRB_OPT_ADAGRAD)
    for (const auto& t : plan->tdev_host)
      HRB_REQUIRE(t.grad || t.m, "hrb_lookup_bwd_update: Adagrad needs an accumulator (adam_m) for every row-updated table");
  if (opt.opt == HRB_OPT_FTRL) {
    int rc = ftrl_tables_ok(plan, "hrb_lookup_bwd_update");
    if (rc != HRB_OK) return rc;
  }
  const int G = plan->max_dim / 4;
  if (G > 256) return fail(HRB_UNSUPPORTED, "hrb_lookup_bwd_update: dim %d too large", plan->max_dim);
  if (batch == 0) return HRB_OK;
  const int64_t n = batch * plan->pos_cols;
  HRB_REQUIRE(n < 0x7FFFFFFFll, "hrb_lookup_bwd_update: batch*sum(seq_len) exceeds 2^31-1");
  cudaStream_t st = (cudaStream_t)stream;
  // Ftrl with pooled fields: the padding flags come from the ids before the backward, row 0 takes its padding step after it
  float* pad_flags = nullptr;
  if (opt.opt == HRB_OPT_FTRL && has_pooled(plan)) {
    const size_t fb = pad_flag_bytes(plan);
    if (workspace_bytes < fb) return fail(HRB_WORKSPACE, "hrb_lookup_bwd_update: workspace %zu < %zu bytes of padding flags", workspace_bytes, fb);
    workspace_bytes = (workspace_bytes - fb) / 256 * 256;
    pad_flags = (float*)((char*)workspace + workspace_bytes);
    int rc = launch_pad_flags(plan, ids, ids_ld, batch, pad_flags, st);
    if (rc != HRB_OK) return rc;
  }
  int rc = HRB_OK;
  if (plan->bwd_algo != HRB_BWD_SORT && unit_path_supported(plan, batch))  // two-level partition, one CTA per row range (embedding_bwd.cu)
    rc = run_unit_update(plan, ids, ids_ld, batch, dout, dout_ld, opt, workspace, workspace_bytes, st);
  else
    rc = run_plan_sorted_update(plan, ids, ids_ld, batch, dout, dout_ld, opt, workspace, workspace_bytes, st);
  if (rc != HRB_OK || pad_flags == nullptr) return rc;
  return launch_ftrl_pad(plan, pad_flags, opt, st);
}

// the SORT algorithm of hrb_lookup_bwd_update (global radix sort of the (table,row) keys)
static int run_plan_sorted_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const float* dout,
                                  int64_t dout_ld, const hrb_opt_params& opt, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int G = plan->max_dim / 4;
  const int64_t n = batch * plan->pos_cols;
  BwdWorkspace w;
  int rc = carve_bwd_ws(n, batch * plan->n_fields + 1, plan->max_dim, plan->key_bits, workspace, w);
  if (rc != HRB_OK) return rc;
  if (w.total > workspace_bytes)
    return fail(HRB_WORKSPACE, "hrb_lookup_bwd_update: workspace %zu < required %zu bytes", workspace_bytes, w.total);
  const uint32_t sentinel = (uint32_t)plan->total_rows;
  bwd_keys_kernel<<<grid_for(batch * plan->n_fields, 256), 256, 0, st>>>(plan->d_fields, plan->n_fields, plan->pos_cols,
                                                                        ids, ids_ld, batch, sentinel, w.keys_in,
                                                                        w.vals_in, w.scale);
  HRB_LAUNCH_CHECK();
  PlanGrad src{plan->d_fields, plan->d_pos_field, dout, w.scale, dout_ld, plan->pos_cols, plan->n_fields};
  ApplyCtx ctx{plan->d_tables, plan->n_tables, opt, nullptr, 0.f};
  if (opt.opt == HRB_OPT_ADAM_LAZY)
    ctx.lr_t = opt.lr * sqrtf(opt.bias_corr2) / opt.bias_corr1;
  return run_sorted_update(upd_mode(opt.opt), w, n, sentinel, plan->key_bits, G, src, ctx, hot_from_plan(plan), st);
}

HRB_API int hrb_embedding_bwd_dense_workspace(int64_t n_ids, int32_t dim, size_t* bytes) {
  HRB_REQUIRE(bytes && n_ids >= 0 && dim > 0, "hrb_embedding_bwd_dense_workspace: bad argument");
  HRB_REQUIRE(n_ids < 0x7FFFFFFFll, "hrb_embedding_bwd_dense_workspace: n_ids exceeds 2^31-1");
  BwdWorkspace w;
  int rc = carve_bwd_ws(n_ids > 0 ? n_ids : 1, 1, dim, 32, nullptr, w);
  if (rc != HRB_OK) return rc;
  *bytes = w.total + align_up(sizeof(TableDev));
  return HRB_OK;
}

HRB_API int hrb_embedding_bwd_dense(const int32_t* ids, int64_t n_ids, const float* dout, int64_t vocab, int32_t dim,
                                    const float* table, float l2_scale, float* dtable, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  HRB_REQUIRE(ids && dout && dtable && workspace && n_ids >= 0 && vocab > 0 && dim > 0, "hrb_embedding_bwd_dense: null/negative argument");
  if (dim % 4 != 0) return fail(HRB_UNSUPPORTED, "hrb_embedding_bwd_dense: dim %d is not a multiple of 4", dim);
  HRB_REQUIRE(aligned16(dout) && aligned16(dtable), "hrb_embedding_bwd_dense: dout/dtable must be 16-byte aligned");
  HRB_REQUIRE(vocab < 0xFFFFFFFFll && n_ids < 0x7FFFFFFFll, "hrb_embedding_bwd_dense: sizes exceed 32-bit keys");
  cudaStream_t st = (cudaStream_t)stream;
  dense_grad_init_kernel<<<grid_for(vocab * dim, 256), 256, 0, st>>>(l2_scale != 0.f ? table : nullptr, l2_scale,
                                                                    vocab * (int64_t)dim, dtable);
  HRB_LAUNCH_CHECK();
  if (n_ids == 0) return HRB_OK;
  const int key_bits = bits_for((uint64_t)vocab);
  BwdWorkspace w;
  int rc = carve_bwd_ws(n_ids, 1, dim, key_bits, workspace, w);
  if (rc != HRB_OK) return rc;
  const size_t need = w.total + align_up(sizeof(TableDev));
  if (need > workspace_bytes)
    return fail(HRB_WORKSPACE, "hrb_embedding_bwd_dense: workspace %zu < required %zu bytes", workspace_bytes, need);
  TableDev* d_t = (TableDev*)((char*)workspace + w.total);
  TableDev t{dtable, nullptr, nullptr, vocab, 0u, dim};
  HRB_CUDA(cudaMemcpyAsync(d_t, &t, sizeof(t), cudaMemcpyHostToDevice, st));
  const uint32_t sentinel = (uint32_t)vocab;
  flat_keys_kernel<<<grid_for(n_ids, 256), 256, 0, st>>>(ids, n_ids, vocab, sentinel, w.keys_in, w.vals_in);
  HRB_LAUNCH_CHECK();
  FlatGrad src{dout, dim};
  ApplyCtx ctx{d_t, 1, hrb_opt_params{}, dtable, 0.f};
  HotInfo hot{};
  if (vocab <= HOT_MAX_ROWS) {  // the whole (tiny) table goes through the one-CTA-per-row kernel
    hot.n_ranges = 1;
    hot.lo[0] = 0;
    hot.len[0] = (uint32_t)vocab;
    hot.keys = nullptr;
    hot.n_keys = (int32_t)vocab;
  }
  return run_sorted_update(UPD_DENSE_ADD, w, n_ids, sentinel, key_bits, dim / 4, src, ctx, hot, st);
}

// =============================================================================================
// (e) compact row exchange for row-sharded tables: owner(r) = r % N, local row r / N.
//   requester: route (owner, owner-side key per position) -> sort by owner -> keys in send order
//   owner:     rows by key (forward) / keyed sorted-segment update (backward)
//   requester: scatter the received rows (forward) / gather the per-position gradients (backward)
// All NCCL calls are made by the host between these kernels (handyrec_b200/sharded.py).
// =============================================================================================
namespace hrb {

__device__ __forceinline__ bool routed_id_valid(const FieldDev& f, int32_t id, const int64_t* __restrict__ full_rows) {
  return (f.pool == HRB_POOL_NONE || id != 0) && id >= 0 && (full_rows == nullptr || (int64_t)id < full_rows[f.table_idx]);
}

// one thread per (sample, position column): owner rank and the key in the OWNER's shard key space
__global__ void __launch_bounds__(256) route_kernel(const FieldDev* __restrict__ fields, const int32_t* __restrict__ pos_field,
                                                   int32_t pos_cols, const int32_t* __restrict__ ids, int64_t ids_ld, int64_t batch,
                                                   int32_t n_ranks, const uint32_t* __restrict__ key_base /* [n_ranks][n_tables] */,
                                                   int32_t n_tables, const int64_t* __restrict__ full_rows, uint32_t* __restrict__ owner,
                                                   uint32_t* __restrict__ key, uint32_t* __restrict__ pos) {
  const int64_t total = batch * pos_cols;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / pos_cols;
    const int c = (int)(i - b * pos_cols);
    const FieldDev& f = fields[pos_field[c]];
    const int32_t id = ids[b * ids_ld + f.ids_col + (c - f.pos_col)];
    // same validity rule as the single-GPU path (bwd_prep_kernel / the forward): padding, negative and out-of-vocabulary ids
    // are nobody's; without the full vocabulary sizes (hrb_plan_set_full_rows) only the lower bound can be checked
    const bool valid = routed_id_valid(f, id, full_rows);
    const uint32_t o = valid ? (uint32_t)(id % n_ranks) : (uint32_t)n_ranks;  // n_ranks = "nobody": sorts last
    owner[i] = o;
    key[i] = valid ? key_base[o * n_tables + f.table_idx] + (uint32_t)(id / n_ranks) : 0xFFFFFFFFu;
    pos[i] = (uint32_t)i;
  }
}

// counts[r] = number of sorted owners equal to r (r in [0, n_ranks]); one thread per rank, binary search
__global__ void owner_counts_kernel(const uint32_t* __restrict__ sorted_owner, int64_t n, int32_t n_ranks,
                                    int64_t* __restrict__ counts) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_ranks) return;
  auto lower = [&](uint32_t v) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (sorted_owner[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
  };
  counts[r] = lower((uint32_t)r + 1) - lower((uint32_t)r);
}

__global__ void __launch_bounds__(256) gather_u32_kernel(const uint32_t* __restrict__ src, const uint32_t* __restrict__ perm,
                                                        int64_t n, uint32_t* __restrict__ dst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[perm[i]];
}

// owner side: out[j, :] = shard row addressed by keys[j]
__global__ void __launch_bounds__(256) rows_by_key_kernel(const TableDev* __restrict__ tables, int32_t n_tables, int32_t chunks,
                                                         const uint32_t* __restrict__ keys, int64_t n, float* __restrict__ out) {
  const int64_t total = n * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / chunks;
    const int q = (int)(i - j * chunks);
    const uint32_t k = __ldg(keys + j);
    const int ti = find_table(tables, n_tables, k);
    const TableDev& t = tables[ti];
    const int64_t row = (int64_t)(k - t.key_base);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < t.rows && q * 4 < t.dim) v = ldg_nc_na(reinterpret_cast<const float4*>(t.w) + row * (t.dim >> 2) + q);
    stg_na(reinterpret_cast<float4*>(out) + i, v);
  }
}

// requester side, forward: received row j belongs to position perm[j]; plain features go straight to the output
// block, positions of pooled features go to the position-ordered buffer for pool_positions_kernel
__global__ void __launch_bounds__(256) scatter_rows_kernel(const FieldDev* __restrict__ fields, const int32_t* __restrict__ pos_field,
                                                          int32_t pos_cols, int32_t chunks, const uint32_t* __restrict__ perm,
                                                          int64_t n, const float* __restrict__ rows, float* __restrict__ out,
                                                          int64_t out_ld, float* __restrict__ pos_rows) {
  const int64_t total = n * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / chunks;
    const int q = (int)(i - j * chunks);
    const uint32_t p = __ldg(perm + j);
    const int64_t b = p / (uint32_t)pos_cols;
    const int c = (int)(p - (uint32_t)b * (uint32_t)pos_cols);
    const FieldDev& f = fields[__ldg(pos_field + c)];
    const float4 v = __ldg(reinterpret_cast<const float4*>(rows) + i);
    if (f.pool == HRB_POOL_NONE)
      *(reinterpret_cast<float4*>(out + b * out_ld + f.out_col) + q) = v;
    else
      *(reinterpret_cast<float4*>(pos_rows) + (int64_t)p * chunks + q) = v;
  }
}

// pooled features from the position-ordered rows (same arithmetic as pooled_chunk)
__global__ void __launch_bounds__(256) pool_positions_kernel(const FieldDev* __restrict__ fields, int32_t n_fields, int32_t pos_cols,
                                                            int32_t chunks, const int32_t* __restrict__ ids, int64_t ids_ld,
                                                            int64_t batch, const float* __restrict__ pos_rows,
                                                            float* __restrict__ out, int64_t out_ld, const int64_t* __restrict__ full_rows) {
  const int64_t total = batch * n_fields * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int q = (int)(i % chunks);
    const int64_t bf = i / chunks;
    const int fi = (int)(bf % n_fields);
    const int64_t b = bf / n_fields;
    const FieldDev& f = fields[fi];
    if (f.pool == HRB_POOL_NONE) continue;
    const int32_t* idp = ids + b * ids_ld + f.ids_col;
    const float4* pr = reinterpret_cast<const float4*>(pos_rows) + (b * pos_cols + f.pos_col) * (int64_t)chunks + q;
    float4 acc = f.pool == HRB_POOL_MAX ? make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY) : make_float4(0.f, 0.f, 0.f, 0.f);
    float cnt = 0.f;
    for (int l = 0; l < f.seq_len; ++l) {
      if (routed_id_valid(f, idp[l], full_rows)) {
        const float4 v = __ldg(pr + (int64_t)l * chunks);
        cnt += 1.f;
        if (f.pool == HRB_POOL_MAX) {
          acc.x = fmaxf(acc.x, v.x); acc.y = fmaxf(acc.y, v.y); acc.z = fmaxf(acc.z, v.z); acc.w = fmaxf(acc.w, v.w);
        } else {
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
      }
    }
    if (f.pool == HRB_POOL_MEAN) {
      const float w = cnt > 0.f ? __fdiv_rn(1.0f, cnt) : 0.0f;
      acc.x *= w; acc.y *= w; acc.z *= w; acc.w *= w;
    } else if (f.pool == HRB_POOL_MAX && cnt < (float)f.seq_len) {
      acc.x = fmaxf(acc.x, -1e9f); acc.y = fmaxf(acc.y, -1e9f); acc.z = fmaxf(acc.z, -1e9f); acc.w = fmaxf(acc.w, -1e9f);
    }
    *(reinterpret_cast<float4*>(out + b * out_ld + f.out_col) + q) = acc;
  }
}

// requester side, backward: gradient of position perm[j] = dout[b, field cols] * (1/n_valid for mean)
__global__ void __launch_bounds__(256) gather_grads_kernel(const FieldDev* __restrict__ fields, const int32_t* __restrict__ pos_field,
                                                          int32_t pos_cols, int32_t chunks, const int32_t* __restrict__ ids,
                                                          int64_t ids_ld, const uint32_t* __restrict__ perm, int64_t n,
                                                          const float* __restrict__ dout, int64_t dout_ld, float* __restrict__ send,
                                                          const int64_t* __restrict__ full_rows) {
  const int64_t total = n * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / chunks;
    const int q = (int)(i - j * chunks);
    const uint32_t p = __ldg(perm + j);
    const int64_t b = p / (uint32_t)pos_cols;
    const int c = (int)(p - (uint32_t)b * (uint32_t)pos_cols);
    const FieldDev& f = fields[__ldg(pos_field + c)];
    float s = 1.0f;
    if (f.pool == HRB_POOL_MEAN) {
      const int32_t* idp = ids + b * ids_ld + f.ids_col;
      int cnt = 0;
      for (int l = 0; l < f.seq_len; ++l) cnt += routed_id_valid(f, idp[l], full_rows);
      s = cnt > 0 ? __fdiv_rn(1.0f, (float)cnt) : 0.f;
    }
    float4 v = __ldg(reinterpret_cast<const float4*>(dout + b * dout_ld + f.out_col) + q);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    reinterpret_cast<float4*>(send)[i] = v;
  }
}

// requester side, backward, fused with the exchange: the gradient row of position perm[j] and its owner-side key are stored
// straight into the OWNER's receive buffers (peer mappings over NVLink; the local rank's own pointer for its own rows).  Rows for
// owner d are perm[send_off[d] .. send_off[d+1]) and land at rows dst_off[d].. of d's buffers, i.e. in the layout an all-to-all
// (ordered by sender) would produce.  Consecutive threads write consecutive 16-byte chunks: 512 contiguous bytes per warp.
struct PeerScatterArgs {
  float* grads[HRB_MAX_PEERS];
  uint32_t* keys[HRB_MAX_PEERS];
  int64_t send_off[HRB_MAX_PEERS + 1];
  int64_t dst_off[HRB_MAX_PEERS];
  int32_t n_ranks;
};

__global__ void __launch_bounds__(256) scatter_grads_to_owners_kernel(const FieldDev* __restrict__ fields, const int32_t* __restrict__ pos_field,
                                                                      int32_t pos_cols, int32_t chunks, const int32_t* __restrict__ ids,
                                                                      int64_t ids_ld, const uint32_t* __restrict__ perm,
                                                                      const uint32_t* __restrict__ send_keys, int64_t n,
                                                                      const float* __restrict__ dout, int64_t dout_ld,
                                                                      const int64_t* __restrict__ full_rows, const PeerScatterArgs a) {
  const int64_t total = n * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / chunks;
    const int q = (int)(i - j * chunks);
    int d = 0;
    while (d + 1 < a.n_ranks && j >= a.send_off[d + 1]) ++d;
    const int64_t r = a.dst_off[d] + (j - a.send_off[d]);
    const uint32_t p = __ldg(perm + j);
    const int64_t b = p / (uint32_t)pos_cols;
    const int c = (int)(p - (uint32_t)b * (uint32_t)pos_cols);
    const FieldDev& f = fields[__ldg(pos_field + c)];
    float s = 1.0f;
    if (f.pool == HRB_POOL_MEAN) {
      const int32_t* idp = ids + b * ids_ld + f.ids_col;
      int cnt = 0;
      for (int l = 0; l < f.seq_len; ++l) cnt += routed_id_valid(f, idp[l], full_rows);
      s = cnt > 0 ? __fdiv_rn(1.0f, (float)cnt) : 0.f;
    }
    float4 v = __ldg(reinterpret_cast<const float4*>(dout + b * dout_ld + f.out_col) + q);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    reinterpret_cast<float4*>(a.grads[d])[r * chunks + q] = v;
    if (q == 0) a.keys[d][r] = __ldg(send_keys + j);
  }
}

}  // namespace hrb

static int route_ws(int64_t n, size_t* cub_bytes, size_t* total) {
  size_t cb = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, cb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                                  (uint32_t*)nullptr, (int)(n > 0 ? n : 1), 0, 8);
  if (e != cudaSuccess) return fail(HRB_CUDA_ERROR, "cub temp size query: %s", cudaGetErrorString(e));
  *cub_bytes = cb;
  *total = align_up((size_t)(n > 0 ? n : 1) * 4) * 4 + align_up(cb);
  return HRB_OK;
}

HRB_API int hrb_route_workspace(const hrb_plan* plan, int64_t batch, size_t* bytes) {
  HRB_REQUIRE(plan && bytes && batch >= 0, "hrb_route_workspace: bad argument");
  size_t cb, tot;
  int rc = route_ws(batch * plan->pos_cols, &cb, &tot);
  if (rc != HRB_OK) return rc;
  *bytes = tot;
  return HRB_OK;
}

// perm[j] (positions in send order, grouped by owner), send_keys[j] (owner-side key of perm[j]),
// counts[r] for r in [0, n_ranks] (the last entry counts padding positions, which are not sent)
HRB_API int hrb_route_ids(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, int32_t n_ranks,
                          const uint32_t* key_base, uint32_t* perm, uint32_t* send_keys, int64_t* counts, void* workspace,
                          size_t workspace_bytes, void* stream) {
  HRB_REQUIRE(plan && ids && key_base && perm && send_keys && counts && workspace && batch >= 0 && n_ranks > 0 && n_ranks < 255,
              "hrb_route_ids: bad argument");
  const int64_t n = batch * plan->pos_cols;
  HRB_REQUIRE(n < 0x7FFFFFFFll, "hrb_route_ids: batch*sum(seq_len) exceeds 2^31-1");
  size_t cb, tot;
  int rc = route_ws(n, &cb, &tot);
  if (rc != HRB_OK) return rc;
  if (workspace_bytes < tot) return fail(HRB_WORKSPACE, "hrb_route_ids: workspace %zu < required %zu bytes", workspace_bytes, tot);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    HRB_CUDA(cudaMemsetAsync(counts, 0, sizeof(int64_t) * (n_ranks + 1), st));
    return HRB_OK;
  }
  const size_t seg = align_up((size_t)n * 4);
  uint32_t* owner = (uint32_t*)workspace;
  uint32_t* key = (uint32_t*)((char*)workspace + seg);
  uint32_t* pos = (uint32_t*)((char*)workspace + 2 * seg);
  uint32_t* owner_sorted = (uint32_t*)((char*)workspace + 3 * seg);
  void* cub_tmp = (char*)workspace + 4 * seg;
  route_kernel<<<grid_for(n, 256), 256, 0, st>>>(plan->d_fields, plan->d_pos_field, plan->pos_cols, ids, ids_ld, batch, n_ranks, key_base,
                                               plan->n_tables, plan->d_full_rows, owner, key, pos);
  HRB_LAUNCH_CHECK();
  int bits = 1;
  while ((1 << bits) <= n_ranks) ++bits;
  HRB_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, owner, owner_sorted, pos, perm, (int)n, 0, bits, st));
  count_launches(2);
  owner_counts_kernel<<<1, 256, 0, st>>>(owner_sorted, n, n_ranks, counts);
  HRB_LAUNCH_CHECK();
  gather_u32_kernel<<<grid_for(n, 256), 256, 0, st>>>(key, perm, n, send_keys);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_rows_by_key(const hrb_plan* plan, const uint32_t* keys, int64_t n, float* out, void* stream) {
  HRB_REQUIRE(plan && n >= 0, "hrb_rows_by_key: bad argument");
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(keys && out && aligned16(out), "hrb_rows_by_key: null/misaligned pointer");
  if (!plan->uniform_dim) return fail(HRB_UNSUPPORTED, "hrb_rows_by_key: the row exchange needs one embedding dim");
  const int chunks = plan->max_dim / 4;
  rows_by_key_kernel<<<grid_for(n * chunks, 256), 256, 0, (cudaStream_t)stream>>>(plan->d_tables, plan->n_tables, chunks, keys, n, out);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_scatter_rows(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const uint32_t* perm, int64_t n,
                             const float* rows, float* out, int64_t out_ld, float* pos_rows, void* stream) {
  HRB_REQUIRE(plan && ids && out && batch >= 0 && n >= 0, "hrb_scatter_rows: bad argument");
  HRB_REQUIRE(aligned16(out) && out_ld % 4 == 0, "hrb_scatter_rows: out must be 16-byte aligned, out_ld %% 4 == 0");
  if (!plan->uniform_dim) return fail(HRB_UNSUPPORTED, "hrb_scatter_rows: the row exchange needs one embedding dim");
  HRB_REQUIRE(plan->all_len1 || pos_rows != nullptr, "hrb_scatter_rows: pooled features need the position buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = plan->max_dim / 4;
  if (n > 0) {
    HRB_REQUIRE(perm && rows && aligned16(rows), "hrb_scatter_rows: null/misaligned pointer");
    scatter_rows_kernel<<<grid_for(n * chunks, 256), 256, 0, st>>>(plan->d_fields, plan->d_pos_field, plan->pos_cols, chunks, perm, n, rows,
                                                                  out, out_ld, pos_rows);
    HRB_LAUNCH_CHECK();
  }
  if (!plan->all_len1 && batch > 0) {
    pool_positions_kernel<<<grid_for(batch * plan->n_fields * chunks, 256), 256, 0, st>>>(plan->d_fields, plan->n_fields, plan->pos_cols,
                                                                                         chunks, ids, ids_ld, batch, pos_rows, out, out_ld, plan->d_full_rows);
    HRB_LAUNCH_CHECK();
  }
  return HRB_OK;
}

HRB_API int hrb_gather_grads(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, const uint32_t* perm, int64_t n,
                             const float* dout, int64_t dout_ld, float* send, void* stream) {
  HRB_REQUIRE(plan && n >= 0, "hrb_gather_grads: bad argument");
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(ids && perm && dout && send && aligned16(dout) && aligned16(send) && dout_ld % 4 == 0, "hrb_gather_grads: null/misaligned pointer");
  if (!plan->uniform_dim || plan->has_max) return fail(HRB_UNSUPPORTED, "hrb_gather_grads: needs one embedding dim and no max pooling");
  const int chunks = plan->max_dim / 4;
  gather_grads_kernel<<<grid_for(n * chunks, 256), 256, 0, (cudaStream_t)stream>>>(plan->d_fields, plan->d_pos_field, plan->pos_cols, chunks,
                                                                                  ids, ids_ld, perm, n, dout, dout_ld, send, plan->d_full_rows);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_scatter_grads_to_owners(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, const uint32_t* perm,
                                        const uint32_t* send_keys, const float* dout, int64_t dout_ld, int32_t n_ranks,
                                        const int64_t* send_counts_host, const int64_t* dst_off_host, void* const* peer_grads_host,
                                        void* const* peer_keys_host, void* stream) {
  HRB_REQUIRE(plan && n_ranks >= 1 && n_ranks <= HRB_MAX_PEERS && send_counts_host && dst_off_host && peer_grads_host && peer_keys_host,
              "hrb_scatter_grads_to_owners: bad argument");
  if (!plan->uniform_dim || plan->has_max) return fail(HRB_UNSUPPORTED, "hrb_scatter_grads_to_owners: needs one embedding dim and no max pooling");
  hrb::PeerScatterArgs a{};
  a.n_ranks = n_ranks;
  int64_t n = 0;
  for (int d = 0; d < n_ranks; ++d) {
    HRB_REQUIRE(send_counts_host[d] >= 0 && dst_off_host[d] >= 0, "hrb_scatter_grads_to_owners: negative count / offset for rank %d", d);
    HRB_REQUIRE(send_counts_host[d] == 0 || (peer_grads_host[d] && peer_keys_host[d] && aligned16(peer_grads_host[d])),
                "hrb_scatter_grads_to_owners: null/misaligned receive buffer of rank %d", d);
    a.grads[d] = (float*)peer_grads_host[d];
    a.keys[d] = (uint32_t*)peer_keys_host[d];
    a.send_off[d] = n;
    a.dst_off[d] = dst_off_host[d];
    n += send_counts_host[d];
  }
  a.send_off[n_ranks] = n;
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(ids && perm && send_keys && dout && aligned16(dout) && dout_ld % 4 == 0, "hrb_scatter_grads_to_owners: null/misaligned pointer");
  const int chunks = plan->max_dim / 4;
  hrb::scatter_grads_to_owners_kernel<<<grid_for(n * chunks, 256), 256, 0, (cudaStream_t)stream>>>(
      plan->d_fields, plan->d_pos_field, plan->pos_cols, chunks, ids, ids_ld, perm, send_keys, n, dout, dout_ld, plan->d_full_rows, a);
  HRB_LAUNCH_CHECK();
  return HRB_OK;
}

HRB_API int hrb_keyed_bwd_workspace(const hrb_plan* plan, int64_t n, size_t* bytes) {
  HRB_REQUIRE(plan && bytes && n >= 0 && n < 0x7FFFFFFFll, "hrb_keyed_bwd_workspace: bad argument");
  BwdWorkspace w;
  int rc = carve_bwd_ws(n > 0 ? n : 1, 1, plan->max_dim, plan->key_bits, nullptr, w);
  if (rc != HRB_OK) return rc;
  *bytes = w.total;
  return HRB_OK;
}

// owner side, backward: (key, gradient row) pairs -> sort -> segment-reduce -> row update of the shard tables
HRB_API int hrb_keyed_bwd_update(const hrb_plan* plan, const uint32_t* keys, const float* grads, int64_t n, const hrb_opt_params* opt_host,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  HRB_REQUIRE(plan && opt_host && workspace && n >= 0 && n < 0x7FFFFFFFll, "hrb_keyed_bwd_update: bad argument");
  if (n == 0) return HRB_OK;
  HRB_REQUIRE(keys && grads && aligned16(grads), "hrb_keyed_bwd_update: null/misaligned pointer");
  if (!plan->uniform_dim) return fail(HRB_UNSUPPORTED, "hrb_keyed_bwd_update: needs one embedding dim");
  const hrb_opt_params opt = load_opt(opt_host);
  HRB_REQUIRE(opt.opt == HRB_OPT_SGD || opt.opt == HRB_OPT_ADAM_LAZY || opt.opt == HRB_OPT_ADAGRAD || opt.opt == HRB_OPT_FTRL,
              "hrb_keyed_bwd_update: unknown optimiser %d", opt.opt);
  if (opt.opt == HRB_OPT_ADAM_LAZY)
    for (const auto& t : plan->tdev_host) HRB_REQUIRE(t.m && t.v, "hrb_keyed_bwd_update: lazy Adam needs adam_m/adam_v for every table");
  if (opt.opt == HRB_OPT_ADAGRAD)
    for (const auto& t : plan->tdev_host) HRB_REQUIRE(t.m, "hrb_keyed_bwd_update: Adagrad needs an accumulator (adam_m) for every table");
  if (opt.opt == HRB_OPT_FTRL)
    for (const auto& t : plan->tdev_host)
      HRB_REQUIRE(t.m && t.v, "hrb_keyed_bwd_update: Ftrl needs an accumulator (adam_m) and a linear slot (adam_v) for every table");
  BwdWorkspace w;
  int rc = carve_bwd_ws(n, 1, plan->max_dim, plan->key_bits, workspace, w);
  if (rc != HRB_OK) return rc;
  if (w.total > workspace_bytes) return fail(HRB_WORKSPACE, "hrb_keyed_bwd_update: workspace %zu < required %zu bytes", workspace_bytes, w.total);
  cudaStream_t st = (cudaStream_t)stream;
  // keys_in = keys (anything outside the shard's key space becomes the sentinel), vals_in = 0..n-1 (gradient row index)
  HRB_REQUIRE(plan->total_rows < 0x7FFFFFFFull, "hrb_keyed_bwd_update: shard key space exceeds 2^31");
  flat_keys_kernel<<<grid_for(n, 256), 256, 0, st>>>(reinterpret_cast<const int32_t*>(keys), n, (int64_t)plan->total_rows,
                                                    (uint32_t)plan->total_rows, w.keys_in, w.vals_in);
  HRB_LAUNCH_CHECK();
  FlatGrad src{grads, plan->max_dim};
  ApplyCtx ctx{plan->d_tables, plan->n_tables, opt, nullptr, 0.f};
  if (opt.opt == HRB_OPT_ADAM_LAZY) ctx.lr_t = opt.lr * sqrtf(opt.bias_corr2) / opt.bias_corr1;
  return run_sorted_update(upd_mode(opt.opt), w, n, (uint32_t)plan->total_rows, plan->key_bits, plan->max_dim / 4, src, ctx,
                           hot_from_plan(plan), st);
}

// Row-sharded tables read in place over NVLink: `peer_tables_host[r*n_tables + t]` is the device pointer of rank r's shard
// of table t as mapped into THIS process (own shards: the local pointers; other ranks: CUDA-IPC / symmetric-memory mappings);
// `full_rows_host[t]` is the full vocabulary size.  Afterwards hrb_lookup_fwd / hrb_lookup_fm_fwd take GLOBAL ids and gather
// row id from rank id % n_ranks at local row id / n_ranks -- no all-to-all in the forward pass.
HRB_API int hrb_plan_set_dense_grads(hrb_plan* plan, float* const* grads_host) {
  HRB_REQUIRE(plan && grads_host, "hrb_plan_set_dense_grads: bad argument");
  for (int32_t t = 0; t < plan->n_tables; ++t) {
    HRB_REQUIRE(aligned16(grads_host[t]), "hrb_plan_set_dense_grads: gradient buffer of table %d is not 16-byte aligned", t);
    plan->tdev_host[t].grad = grads_host[t];
  }
  HRB_CUDA(cudaMemcpy(plan->d_tables, plan->tdev_host.data(), sizeof(hrb::TableDev) * plan->n_tables, cudaMemcpyHostToDevice));
  return HRB_OK;
}

HRB_API int hrb_plan_set_peers(hrb_plan* plan, int32_t n_ranks, const void* const* peer_tables_host, const int64_t* full_rows_host) {
  HRB_REQUIRE(plan && n_ranks >= 1 && peer_tables_host && full_rows_host, "hrb_plan_set_peers: bad argument");
  if (!(plan->all_len1 && plan->uniform_dim && plan->contiguous_out))
    return fail(HRB_UNSUPPORTED, "hrb_plan_set_peers: implemented for plain-lookup groups laid out contiguously only");
  const size_t np = (size_t)n_ranks * plan->n_tables;
  for (int32_t t = 0; t < plan->n_tables; ++t)  // a table is sharded (pointers on every rank) or replicated (NULL on every rank)
    for (int32_t r = 1; r < n_ranks; ++r)
      HRB_REQUIRE((peer_tables_host[(size_t)r * plan->n_tables + t] == nullptr) == (peer_tables_host[t] == nullptr),
                  "hrb_plan_set_peers: table %d has peer pointers on some ranks only", t);
  if (plan->d_peer_tab) cudaFree((void*)plan->d_peer_tab);
  if (plan->d_full_rows) cudaFree(plan->d_full_rows);
  plan->d_peer_tab = nullptr;
  plan->d_full_rows = nullptr;
  HRB_CUDA(cudaMalloc((void**)&plan->d_peer_tab, np * sizeof(void*)));
  HRB_CUDA(cudaMalloc((void**)&plan->d_full_rows, plan->n_tables * sizeof(int64_t)));
  HRB_CUDA(cudaMemcpy((void*)plan->d_peer_tab, peer_tables_host, np * sizeof(void*), cudaMemcpyHostToDevice));
  HRB_CUDA(cudaMemcpy(plan->d_full_rows, full_rows_host, plan->n_tables * sizeof(int64_t), cudaMemcpyHostToDevice));
  plan->n_ranks = n_ranks;
  return HRB_OK;
}

// Full vocabulary sizes of the tables of a plan whose `rows` are shard sizes (the requester side of the row exchange):
// hrb_route_ids / hrb_scatter_rows / hrb_gather_grads then treat ids >= full_rows[table] as invalid, exactly like the
// single-GPU path does with `rows`.
HRB_API int hrb_plan_set_full_rows(hrb_plan* plan, const int64_t* full_rows_host) {
  HRB_REQUIRE(plan && full_rows_host, "hrb_plan_set_full_rows: bad argument");
  if (plan->d_full_rows == nullptr) HRB_CUDA(cudaMalloc((void**)&plan->d_full_rows, plan->n_tables * sizeof(int64_t)));
  HRB_CUDA(cudaMemcpy(plan->d_full_rows, full_rows_host, plan->n_tables * sizeof(int64_t), cudaMemcpyHostToDevice));
  return HRB_OK;
}

HRB_API int hrb_plan_set_bwd_algo(hrb_plan* plan, int32_t algo) {
  HRB_REQUIRE(plan && algo >= HRB_BWD_AUTO && algo <= HRB_BWD_SORT, "hrb_plan_set_bwd_algo: bad argument");
  plan->bwd_algo = algo;
  return HRB_OK;
}
