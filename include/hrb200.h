/*
 * hrb200.h -- C ABI of libhrb200.so: the B200 (sm_100a) implementation of HandyRec's
 * data-parallel hot path (embedding lookup + masked sequence pooling -> FM / DIN
 * attention / dense towers, and the embedding backward).
 *
 * HandyRec (TF 2.6 / Keras, pure Python) has no FFI today; the path sits behind the
 * Keras Layer protocol.  Each entry point below names the reference interface whose
 * arithmetic it replaces (paths relative to /root/reference/).  The reference-side
 * binding a maintainer would add (TF custom op / ctypes) is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - floats are fp32, ids are int32 (features/type.py:76,128), sizes are int64_t;
 *   - the caller owns every buffer, including tables and workspaces; the library
 *     allocates nothing except the small opaque hrb_plan (hrb_plan_create/destroy);
 *   - every compute entry takes a cudaStream_t as `void* stream`, is asynchronous and
 *     never synchronises the device; no internal streams;
 *   - return value: 0 = HRB_OK, otherwise an hrb_status code; never throws or aborts.
 *     hrb_last_error() returns a thread-local detail string.
 */
#ifndef HRB200_H_
#define HRB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HRB_ABI_VERSION 1

typedef enum hrb_status {
  HRB_OK = 0,
  HRB_BAD_ARG = 1,      /* null pointer, negative size, misaligned buffer ...            */
  HRB_UNSUPPORTED = 2,  /* valid request the kernels do not cover (stated in the message) */
  HRB_CUDA_ERROR = 3,   /* a CUDA runtime call failed (message holds cudaGetErrorString)  */
  HRB_WORKSPACE = 4     /* workspace too small                                            */
} hrb_status;

/* pooling methods: layers/sequence.py:19-23 ("mean" | "max" | "sum"); NONE = plain lookup (L must be 1) */
typedef enum hrb_pool { HRB_POOL_NONE = 0, HRB_POOL_MEAN = 1, HRB_POOL_SUM = 2, HRB_POOL_MAX = 3 } hrb_pool;

/* activations: layers/utils.py:117-133 -> keras Activation(name); "dice" is its own entry point */
typedef enum hrb_act {
  HRB_ACT_LINEAR = 0,
  HRB_ACT_RELU = 1,
  HRB_ACT_SIGMOID = 2,
  HRB_ACT_TANH = 3,
  HRB_ACT_DICE = 4 /* only inside hrb_lau_fwd (inference statistics); standalone Dice is hrb_dice_fwd/bwd */
} hrb_act;

int hrb_abi_version(void);
const char* hrb_status_str(int status);
const char* hrb_last_error(void);
/* number of CUDA kernels this library has launched in this process (every <<<>>> is counted) */
int hrb_launch_count(int64_t* count);

/* ------------------------------------------------------------------------------------------
 * Synthetic tables.  table[r,c] = lo + u*(hi-lo), u = (hash(seed, (row_start+r*row_step)*dim+c)>>8)*2^-24.
 * Bit-identical to oracle/layers_ref.py:hash_uniform_table.  Replaces Keras Embedding's
 * `uniform` initialiser (features/group.py:285-293) for benchmarks and parity runs.
 * ------------------------------------------------------------------------------------------ */
int hrb_init_uniform(float* table, int64_t rows, int32_t dim, uint32_t seed, float lo, float hi,
                     int64_t row_start, int64_t row_step, void* stream);

/* ------------------------------------------------------------------------------------------
 * a5  CustomEmbedding.__call__ + compute_mask   (layers/tools.py:87-101)
 *   out[i,:] = table[ids[i],:]  (row 0 is gathered like any row);
 *   mask[i,d] = ids[i] != 0 tiled over dim (uint8 0/1), only when mask != NULL.
 *   oob (nullable, int32[2], caller-zeroed): set to {1, first offending flat index seen} when an id
 *   is outside [0,vocab); such rows are written as zeros (TF-GPU behaviour), TF-CPU raises.
 * ------------------------------------------------------------------------------------------ */
int hrb_embedding_fwd(const float* table, int64_t vocab, int32_t dim, const int32_t* ids, int64_t n_ids,
                      float* out, uint8_t* mask, int32_t* oob, void* stream);

/* Embedding backward as a DENSE table gradient (layer face; TF autodiff of a5, SURVEY a13):
 *   dtable[r,:] = sum_{i: ids[i]==r} dout[i,:]   (+ l2_scale * table[r,:] when table != NULL)
 * Sorted-segment reduction, no atomics, deterministic.  dtable (vocab x dim) is fully overwritten. */
int hrb_embedding_bwd_dense_workspace(int64_t n_ids, int32_t dim, size_t* bytes);
int hrb_embedding_bwd_dense(const int32_t* ids, int64_t n_ids, const float* dout, int64_t vocab, int32_t dim,
                            const float* table, float l2_scale, float* dtable, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a6  SequencePoolingLayer.call   (layers/sequence.py:26-46)
 *   x (B,L,D), mask (B,L,D) uint8 as produced by a5 -> out (B,1,D).  method: hrb_pool (not NONE).
 *   mean: sum_l x*(mask/sum_l mask), divide_no_nan; sum: sum_l x*mask; max: max_l (x-(1-mask)*1e9).
 *   bwd: dx (B,L,D) given dout (B,D); max distributes equally among ties (TF reduce_max gradient).
 * ------------------------------------------------------------------------------------------ */
int hrb_seq_pool_fwd(const float* x, const uint8_t* mask, int64_t batch, int32_t seq_len, int32_t dim,
                     int32_t method, float* out, void* stream);
int hrb_seq_pool_bwd(const float* x, const uint8_t* mask, const float* dout, int64_t batch, int32_t seq_len,
                     int32_t dim, int32_t method, float* dx, void* stream);

/* ------------------------------------------------------------------------------------------
 * a7  FeatureGroup.embedding_lookup   (features/group.py:299-336), fused: ids -> pooled (B, sum D)
 *   A plan describes every sparse / sparse-sequence feature of a group: which table, where its ids
 *   sit in the packed id matrix ids[B, ids_ld] (column ids_col .. ids_col+seq_len), the pooling
 *   method, and the output column.  One launch does gather + mask + pool for all features; the
 *   (B,L,D) tensor and its mask are never materialised.
 * ------------------------------------------------------------------------------------------ */
typedef struct hrb_table_desc {
  float* weight;  /* (rows, dim) fp32, 16-byte aligned                        */
  float* adam_m;  /* optimiser state: Adam m / Adagrad or Ftrl accumulator (same shape) or NULL */
  float* adam_v;  /* Adam second moment / Ftrl linear (same shape) or NULL; NULL under Adagrad */
  int64_t rows;   /* vocab_size                                               */
  int32_t dim;    /* embedding dim                                            */
  int32_t pad_;
} hrb_table_desc;

typedef struct hrb_field_desc {
  int32_t table;    /* index into the plan's table array                                          */
  int32_t seq_len;  /* 1 for SparseFeature; L for SparseSeqFeature                                */
  int32_t pool;     /* hrb_pool; NONE => every id valid (mask_zero has no effect on the values)    */
  int32_t ids_col;  /* first column of this feature in ids[B, ids_ld]                             */
  int32_t out_col;  /* first output column (floats) in out[B, out_ld]                             */
  int32_t pad_;
} hrb_field_desc;

typedef struct hrb_plan hrb_plan;

int hrb_plan_create(const hrb_table_desc* tables_host, int32_t n_tables, const hrb_field_desc* fields_host,
                    int32_t n_fields, hrb_plan** plan);
int hrb_plan_destroy(hrb_plan* plan);

/* fwd: out[b, out_col_f : +D_f] for every field.  inv_count (nullable): (B, n_fields) fp32, 1/n_valid
 * (0 when none) for mean fields, 1 otherwise -- saved for the backward.  oob as in a5. */
int hrb_lookup_fwd(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* out,
                   int64_t out_ld, float* inv_count, int32_t* oob, void* stream);

/* fwd fused with a9 FM (layers/interaction.py:26-39) for the DeepFM case where the FM group and
 * the DNN group hold the same features (models/ranking/context_aware/DeepFM.py:62-63): requires
 * equal dims D and fields laid out contiguously (out_col_f = out_col_0 + f*D).
 *   fm_out[b] = w0 + sum_f x_f . w + 0.5*sum_d[(sum_f x)^2 - sum_f x^2];  fm_sum[b,:] = sum_f x_f (for bwd) */
int hrb_lookup_fm_fwd(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* out,
                      int64_t out_ld, float* inv_count, const float* fm_w, const float* fm_w0, float* fm_out,
                      float* fm_sum, int32_t* oob, void* stream);

/* a13 embedding backward + row update, fused plan face.
 *   dout (B, dout_ld): gradient w.r.t. the pooled outputs (same column layout as out).
 *   Sort (table,row) keys -> segment-reduce -> per-unique-row update, no atomics.
 *   opt = HRB_OPT_SGD:       w[r] -= lr * (g[r] + l2_scale*w[r])        (touched rows only)
 *   opt = HRB_OPT_ADAM_LAZY: Adam moments/weights updated for touched rows only (needs adam_m/adam_v)
 *   opt = HRB_OPT_ADAGRAD:   g' = g[r] + l2_scale*w[r]; acc[r] += g'^2; w[r] -= lr * g' / (sqrt(acc[r]) + eps)
 *                            (touched rows only, acc in adam_m; Keras ResourceSparseApplyAdagradV2 on the summed rows)
 *   opt = HRB_OPT_FTRL:      Keras Ftrl (ResourceSparseApplyFtrl / V2) on the summed rows, accum in adam_m, linear in adam_v:
 *                            g' = g[r] + l2_scale*w[r]; gs = g' + 2*l2_shrinkage*w[r]; acc' = acc + g'^2;
 *                            linear += gs - (p(acc') - p(acc)) / lr * w[r], p(a) = a^(-lr_power);
 *                            w[r] = |linear| > l1 ? (sign(linear)*l1 - linear) / (p(acc') / lr + 2*l2) : 0; acc = acc'.
 *                            Touched rows: every in-range id of a plain field and every position of a pooled field -- the
 *                            padding id 0 included, with a zero gradient (Keras gathers row 0 there): when a batch holds
 *                            padding for a row-updated table, row 0 of that table takes exactly one step.
 *   max-pooled fields are not supported here (use a6 bwd + hrb_embedding_bwd_dense). */
typedef enum hrb_opt { HRB_OPT_SGD = 0, HRB_OPT_ADAM_LAZY = 1, HRB_OPT_ADAGRAD = 2, HRB_OPT_FTRL = 3 } hrb_opt;
typedef struct hrb_opt_params {
  int32_t opt;
  float lr, beta1, beta2, eps, l2_scale; /* l2_scale = 2*l2_embd (features/group.py:289) */
  float bias_corr1, bias_corr2;          /* 1-beta1^t, 1-beta2^t */
  /* read only when opt == HRB_OPT_FTRL: Keras' l1 / l2 / learning_rate_power / l2_shrinkage strengths, l2 with beta / (2*lr)
   * already added */
  float l1, l2, lr_power, l2_shrinkage;
} hrb_opt_params;
int hrb_lookup_bwd_workspace(const hrb_plan* plan, int64_t ids_ld, int64_t batch, size_t* bytes);
int hrb_lookup_bwd_update(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch,
                          const float* dout, int64_t dout_ld, const float* inv_count,
                          const hrb_opt_params* opt_host, void* workspace, size_t workspace_bytes,
                          void* stream);

/* Two implementations of hrb_lookup_bwd_update with identical semantics (both deterministic, no atomics on gradients):
 *   UNITS  two-level radix partition; the second level (one CTA per row range) sorts in shared memory and is fused with the
 *          segmented reduction and the row update (csrc/embedding_bwd.cu) -- fastest when ids spread over the tables;
 *   SORT   global radix sort of (table,row) keys, then chunked segmented reduction + merge (csrc/lookup.cu) -- robust when a
 *          few rows collect most of the batch (Zipf ids).
 * AUTO = UNITS whenever the plan / batch is covered by it.  The host may time both on its own data and pin one. */
typedef enum hrb_bwd_algo { HRB_BWD_AUTO = 0, HRB_BWD_UNITS = 1, HRB_BWD_SORT = 2 } hrb_bwd_algo;
int hrb_plan_set_bwd_algo(hrb_plan* plan, int32_t algo);

/* Dense-updated tables: grads_host[t] != NULL (rows*dim fp32, 16-byte aligned) makes hrb_lookup_bwd_update ADD the
 * per-row gradient sums of table t into that buffer and leave weight/moments alone -- the caller zeroes the buffer,
 * (all-reduces it when the table is replicated over ranks) and runs its dense optimiser step over the table, which is
 * exactly what Keras does for an IndexedSlices gradient under Adam (dense moment decay).  NULL keeps the in-place
 * touched-rows update.  The array has n_tables entries. */
int hrb_plan_set_dense_grads(hrb_plan* plan, float* const* grads_host);

/* Touched rows of a batch, for optimisers whose step with a zero gradient is not a no-op (Ftrl): for every table t with
 * touched_host[t] != NULL (one float per row, caller-zeroed), store 1.0f at every row a position of the batch names --
 * every in-range id of a plain field, every position of a pooled field, the padding id 0 included.  Plain stores: every
 * writer stores the same value.  The array has n_tables entries. */
int hrb_plan_mark_rows(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* const* touched_host,
                       void* stream);
/* Row 0 and the padding of pooled fields, for callers that apply the row update themselves (the owner of row 0 of a
 * row-sharded table): hrb_plan_pad_flags stores 1.0f in flags[2t] when a pooled field of table t holds padding in the batch
 * and in flags[2t+1] when a valid position names row 0 of table t (2*n_tables floats, caller-zeroed, plain stores; flags of
 * several batches may be summed).  hrb_plan_ftrl_pad_step then gives row 0 of every row-updated table t with
 * flags[2t] != 0 and flags[2t+1] == 0 its zero-gradient Ftrl step (opt_host->opt must be HRB_OPT_FTRL).
 * hrb_lookup_bwd_update does both itself. */
int hrb_plan_pad_flags(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* flags, void* stream);
int hrb_plan_ftrl_pad_step(const hrb_plan* plan, const float* flags, const hrb_opt_params* opt_host, void* stream);

/* ------------------------------------------------------------------------------------------
 * a9  FM.call   (layers/interaction.py:15-39) on a materialised (B,F,D) tensor.
 *   x rows are x_ld floats apart (x_ld >= F*D).  out (B).  fm_sum (nullable) (B,D).
 *   bwd: dx[b,f,:] (+)= dout[b]*(w + S[b] - x[b,f,:]); dw[d] = sum_b dout[b]*S[b,d]; dw0 = sum_b dout[b].
 *   dw_dw0: D+1 floats, overwritten.  accumulate!=0 adds into dx instead of overwriting.
 * ------------------------------------------------------------------------------------------ */
int hrb_fm_fwd(const float* x, int64_t x_ld, int64_t batch, int32_t fields, int32_t dim, const float* w,
               const float* w0, float* out, float* fm_sum, void* stream);
int hrb_fm_bwd(const float* x, int64_t x_ld, int64_t batch, int32_t fields, int32_t dim, const float* w,
               const float* dout, float* dx, int64_t dx_ld, int32_t accumulate, float* dw_dw0, void* stream);

/* ------------------------------------------------------------------------------------------
 * a11  Dense layers of DNN   (layers/core.py:53-78; Keras Dense = x@W+b)
 *   fwd:   y[M,N] = act(x[M,K] @ w[K,N] + bias[N])
 *   bwd_x: dx[M,K] = dz[M,N] @ w[K,N]^T, optionally * act'(a_prev) where a_prev[M,K] is the
 *          previous layer's post-activation output (relu/sigmoid/tanh derivative from the output)
 *   bwd_w: dw[K,N] = x[M,K]^T @ dz[M,N]; dbias[N] = sum_m dz[m,n]   (split over M, fixed-order reduce)
 *   precision: fp32 FFMA (HRB_GEMM_FP32) or tcgen05 3xTF32 error-compensated (HRB_GEMM_3XTF32).
 * ------------------------------------------------------------------------------------------ */
typedef enum hrb_gemm_mode { HRB_GEMM_AUTO = 0, HRB_GEMM_FP32 = 1, HRB_GEMM_3XTF32 = 2 } hrb_gemm_mode;
int hrb_dense_fwd(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* bias, int64_t M,
                  int32_t K, int32_t N, int32_t act, float* y, int64_t ldy, int32_t mode, void* stream);
int hrb_dense_bwd_x(const float* dz, int64_t lddz, const float* w, int64_t ldw, int64_t M, int32_t K,
                    int32_t N, const float* a_prev, int64_t lda_prev, int32_t act_prev, float* dx,
                    int64_t lddx, int32_t mode, void* stream);
int hrb_dense_bwd_w_workspace(int64_t M, int32_t K, int32_t N, size_t* bytes);
int hrb_dense_bwd_w(const float* x, int64_t ldx, const float* dz, int64_t lddz, int64_t M, int32_t K,
                    int32_t N, float* dw, int64_t lddw, float* dbias, void* workspace, size_t workspace_bytes,
                    int32_t mode, void* stream);
/* tcgen05 "TN" variants (3xTF32 error-compensated, fp32 accumulate in TMEM): every operand has its reduction
 * dimension contiguous, so the caller keeps transposed copies -- wt[N,K] = w^T for the forward, xt[K,M] and
 * dzt[N,M] for the weight gradient.  yt / dxt (nullable) receive the transposed copy of the output for the
 * next weight gradient.  Shapes the tensor-core kernel does not cover return HRB_UNSUPPORTED (use hrb_dense_*). */
int hrb_transpose(const float* src, int64_t rows, int32_t cols, int64_t lds, float* dst, int64_t ldd, void* stream);
/* relu_mask (nullable): uint32 words [M][ceil(units/32)], bit j of word [m][c] = (activation[m][32c+j] > 0).  The relu
 * forward writes it; the backward of the layer above reads it instead of re-reading the activations (a_prev is then unused). */
int hrb_dense_fwd_t(const float* x, int64_t ldx, const float* wt, int64_t ldwt, const float* bias, int64_t M, int32_t K,
                    int32_t N, int32_t act, float* y, int64_t ldy, float* yt, int64_t ldyt, uint32_t* relu_mask, void* stream);
int hrb_dense_bwd_x_t(const float* dz, int64_t lddz, const float* w, int64_t ldw, int64_t M, int32_t K, int32_t N,
                      const float* a_prev, int64_t lda_prev, int32_t act_prev, const uint32_t* relu_mask, float* dx, int64_t lddx,
                      float* dxt, int64_t lddxt, void* stream);
int hrb_dense_bwd_w_t_workspace(int64_t M, int32_t K, int32_t N, size_t* bytes);
int hrb_dense_bwd_w_t(const float* xt, int64_t ldxt, const float* dzt, int64_t lddzt, const float* dz, int64_t lddz, int64_t M,
                      int32_t K, int32_t N, float* dw, int64_t lddw, float* dbias, void* workspace, size_t workspace_bytes,
                      void* stream);
/* The same weight gradient from x as the forward stored it (x[M,K] row-major): no x^T copy has to exist, the kernel
 * transposes the tile on its way into tensor memory.  Workspace as hrb_dense_bwd_w_t_workspace. */
int hrb_dense_bwd_w_xn(const float* x, int64_t ldx, const float* dzt, int64_t lddzt, int64_t M, int32_t K, int32_t N, float* dw,
                       int64_t lddw, float* dbias, void* workspace, size_t workspace_bytes, void* stream);

/* The 1-unit logit layer (models/ranking/context_aware/DeepFM.py:59-60): GEMV forward y[m] = x[m,:].w + b and a fused
 * backward dz_prev = dy (x) w * act'(x) (+ transposed copy), dw = x^T dy, dbias = sum dy (fixed-order reductions). */
int hrb_dense1_fwd(const float* x, int64_t ldx, const float* w, const float* bias, int64_t M, int32_t K, float* y, void* stream);
int hrb_dense1_bwd_workspace(int64_t M, int32_t K, size_t* bytes);
int hrb_dense1_bwd(const float* x, int64_t ldx, const float* w, const float* dy, int64_t M, int32_t K, int32_t act_prev,
                   float* dz_prev, int64_t lddz, float* dz_prev_t, int64_t lddzt, float* dw, float* dbias, void* workspace,
                   size_t workspace_bytes, void* stream);

/* dz = dy * act'(y) in place-capable elementwise (used at the head of a backward chain) */
int hrb_act_bwd(const float* y, const float* dy, int64_t n, int32_t act, float* dz, void* stream);

/* Dice   (layers/activation.py:27-42): p = sigmoid((x-mean)*rsqrt(var+eps)); y = p*x + (1-p)*alpha*x.
 * training != 0: mean/var are computed over all rows (biased) and written to batch_mean/batch_var;
 * otherwise mean/var are read from them (moving statistics). */
int hrb_dice_fwd(const float* x, int64_t rows, int32_t units, const float* alpha, float* mean, float* var,
                 float eps, int32_t training, float* y, void* stream);
int hrb_dice_bwd(const float* x, const float* dy, int64_t rows, int32_t units, const float* alpha,
                 const float* mean, const float* var, float eps, int32_t training, float* dx, float* dalpha,
                 float* scratch /* 2*units floats, training only */, void* stream);

/* Keras BatchNormalization (layers/core.py:71-72; last axis, biased batch variance in training) and Dropout
 * (core.py:73; the keep mask is a pure function of (seed, element index): the backward is the same call on dy). */
int hrb_batchnorm_fwd(const float* x, int64_t rows, int32_t units, const float* gamma, const float* beta, float* mean,
                      float* var, float eps, int32_t training, float* y, void* stream);
int hrb_batchnorm_bwd(const float* x, const float* dy, int64_t rows, int32_t units, const float* gamma, const float* mean,
                      const float* var, float eps, int32_t training, float* dx, float* dgamma, float* dbeta,
                      float* scratch /* 2*units floats */, void* stream);
int hrb_dropout(const float* x, int64_t n, float rate, uint32_t seed, float* y, void* stream);

/* ------------------------------------------------------------------------------------------
 * a10  LocalActivationUnit.call + SqueezeMask + tf.matmul(att, keys)
 *      (layers/sequence.py:92-102, layers/tools.py:104-113, models/ranking/sequential/DIN.py:87-93)
 *   Fused per sample: att_in=[q,k,q-k,q*k] built on the fly (never materialised), MLP
 *   [4D -> 4D -> h1 -> ... -> 1] with an elementwise activation (relu/sigmoid/tanh/linear, or dice in
 *   inference mode via dice_* arrays), mask by ids != 0, no softmax; pooled[b,:] = sum_t score[b,t]*k[b,t,:].
 *   The MLP is described by n_layers weight matrices packed back to back in `params`:
 *   for layer i: W_i (in_i x out_i, row-major), b_i (out_i), then -- only when act == HRB_ACT_DICE and
 *   i is not the last layer -- alpha_i, moving_mean_i, moving_var_i (out_i each); the running offset is
 *   rounded up to a multiple of 4 floats after every layer.  in_0 = 4D; layer_out_host[0] is normally 4D
 *   (core.py:57 prepends Dense(in)); the last layer must have 1 unit.
 * ------------------------------------------------------------------------------------------ */
int hrb_lau_fwd(const float* table, int64_t vocab, int32_t dim, const int32_t* query_ids,
                const int32_t* key_ids, int64_t batch, int32_t seq_len, const float* params,
                const int32_t* layer_out_host, int32_t n_layers, int32_t act, float* score, float* pooled,
                void* stream);

/* a10, layer face (training path; the MLP between them is hrb_dense_* / hrb_dice_*):
 *   att_input  out[b,t,:] = [q, k, q-k, q*k]  (sequence.py:96-97) and its backward (dq, dk)
 *   mask_scores  out = mask ? s : 0           (sequence.py:100-101; its own backward)
 *   att_pool   out[b,:] = sum_t s[b,t]*k[b,t,:]  (DIN.py:93) and its backward (ds, dk) */
int hrb_att_input_fwd(const float* q, const float* k, int64_t batch, int32_t T, int32_t D, float* out, void* stream);
int hrb_att_input_bwd(const float* q, const float* k, const float* g, int64_t batch, int32_t T, int32_t D, float* dq,
                      float* dk, void* stream);
int hrb_mask_scores(const float* s, const uint8_t* mask, int64_t n, float* out, void* stream);
int hrb_att_pool_fwd(const float* s, const float* k, int64_t batch, int32_t T, int32_t D, float* out, void* stream);
int hrb_att_pool_bwd(const float* s, const float* k, const float* dout, int64_t batch, int32_t T, int32_t D, float* ds,
                     float* dk, void* stream);

/* a10, training path without the (B,T,4D) tensor.  With W = [Wa; Wb; Wc; Wd] (first Dense of the LAU MLP, core.py:57):
 *   [q, k, q-k, q*k] . W + b  =  (q.(Wa+Wc) + b)  +  [k | q*k] . [Wb-Wc; Wd]
 * = a per-sample term (B x U) + a B*T-row GEMM over 2D columns (half the flops), summed in the GEMM epilogue:
 *   hrb_lau_split_weights   wq (D,U) = Wa+Wc, wp (2D,U) = [Wb-Wc; Wd], wpt = wp^T (U,2D) for the TN GEMM
 *   hrb_lau_pack_fwd        A'[b*T+t] = [k[b,t] | q[b]*k[b,t]]                         (B*T, 2D)
 *   hrb_dense_fwd_t_grouped y = act(A' . wpt^T + qterm[m / T])                         tcgen05 3xTF32, bias per group of T rows
 *   hrb_group_sum           dqterm[b] = sum_t dz[b*T+t]                                 fixed order
 *   hrb_lau_pack_bwd        dk = dA'[:, :D] + dA'[:, D:]*q;  dq (+)= sum_t dA'[:, D:]*k  fixed order
 *   hrb_lau_merge_wgrads    dWa = dwq, dWb = dwp[:D], dWc = dwq - dwp[:D], dWd = dwp[D:] */
int hrb_lau_split_weights(const float* w, int64_t ldw, int32_t dim, int32_t units, float* wq, float* wp, float* wpt, void* stream);
int hrb_lau_merge_wgrads(const float* dwq, const float* dwp, int32_t dim, int32_t units, float* dw, int64_t ldw, void* stream);
int hrb_lau_pack_fwd(const float* q, const float* k, int64_t batch, int32_t T, int32_t dim, float* out, void* stream);
int hrb_lau_pack_bwd(const float* q, const float* k, const float* da, int64_t batch, int32_t T, int32_t dim, int32_t accumulate_dq,
                     float* dq, float* dk, void* stream);
int hrb_group_sum(const float* x, int64_t ldx, int64_t groups, int32_t group_rows, int32_t n, float* out, void* stream);
int hrb_dense_fwd_t_grouped(const float* x, int64_t ldx, const float* wt, int64_t ldwt, const float* group_bias, int64_t ldgb,
                            int32_t group_rows, int64_t M, int32_t K, int32_t N, int32_t act, float* y, int64_t ldy, void* stream);

/* ------------------------------------------------------------------------------------------
 * DeepFM head + loss   (models/ranking/context_aware/DeepFM.py:86-88 + Keras binary_crossentropy)
 *   logit = dnn[b] + fm[b]; p = sigmoid(logit); loss_sum += bce(logit,y); dlogit[b] = (p-y)*grad_scale
 *   loss_sum: one float, caller-zeroed, accumulated with a fixed-order block reduction + one atomic per block.
 * ------------------------------------------------------------------------------------------ */
int hrb_sigmoid_bce(const float* dnn_logit, const float* fm_logit, const float* label, int64_t batch,
                    float grad_scale, float* prob, float* dlogit, float* loss_sum, void* stream);

/* Keras binary_crossentropy on probabilities (the fallback Keras takes when the prediction is not the direct output of a sigmoid,
 * e.g. DNN(..., use_bn=True, output_activation="sigmoid"): layers/core.py:66-73 puts BN / Dropout behind the activation):
 *   p = clip(prob, eps, 1-eps); loss_sum += -(y log p + (1-y) log(1-p)); dprob = d loss / d prob * grad_scale (0 where clipped). */
int hrb_clipped_bce(const float* prob, const float* label, int64_t n, float eps, float grad_scale, float* dprob,
                    float* loss_sum, void* stream);

/* Keras sample weights (losses_utils.compute_weighted_loss): the entries above with one fp32 weight per sample,
 *   loss_sum += w*l;  dlogit (dprob) = d l / d logit (prob) * w * grad_scale.
 * The caller divides loss_sum by the batch size, not by sum(w), and passes grad_scale = 1 / (batch * ranks) as above.
 * w = 1 gives prob and dlogit (dprob) bit-equal to the unweighted entries. */
int hrb_sigmoid_bce_weighted(const float* dnn_logit, const float* fm_logit, const float* label, const float* weight, int64_t batch,
                             float grad_scale, float* prob, float* dlogit, float* loss_sum, void* stream);
int hrb_clipped_bce_weighted(const float* prob, const float* label, const float* weight, int64_t n, float eps, float grad_scale,
                             float* dprob, float* loss_sum, void* stream);

/* Keras regression losses (keras/losses.py mean_squared_error, mean_absolute_error, huber; the head of DeepFM(task="regression"),
 * DeepFM.py:86-88 without the sigmoid):
 *   pred = pred_a (+ pred_b when not null); e = pred - label, elementwise over (batch, cols);
 *   loss 0 (MSE): e^2, de = 2e;  1 (MAE): |e|, de = sign(e) (0 at e = 0);
 *   2 (Huber):  0.5 q^2 + delta (|e| - q), q = min(|e|, delta), de = e for |e| <= delta (the tie takes the quadratic branch),
 *               delta sign(e) otherwise;
 *   per-sample loss l = mean over cols (Keras' mean over the last axis); loss_sum = sum_b w_b l_b (w = 1 unweighted), written (not
 *   accumulated) and reduced in float64 in a fixed order, so it is the same bits from run to run;
 *   dpred = de * w * grad_scale / cols (grad_scale = 1 / (batch * ranks): Keras' sum(w * l) / B, B the batch size, not sum(w)).
 * pred, dpred, loss_sum may be null; label may be null when dpred and loss_sum are (a forward alone).  The workspace (size from
 * hrb_regression_loss_workspace) is needed with loss_sum; it must be zeroed once before its first use and is left zeroed.
 * The weighted entry takes one fp32 weight per sample (batch of them); w = 1 gives the unweighted bits. */
int hrb_regression_loss_workspace(int64_t n, size_t* bytes);
int hrb_regression_loss(int32_t loss, float delta, const float* pred_a, const float* pred_b, const float* label, int64_t batch, int32_t cols,
                        float grad_scale, float* pred, float* dpred, float* loss_sum, void* workspace, size_t workspace_bytes, void* stream);
int hrb_regression_loss_weighted(int32_t loss, float delta, const float* pred_a, const float* pred_b, const float* label, const float* weight,
                                 int64_t batch, int32_t cols, float grad_scale, float* pred, float* dpred, float* loss_sum, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * (f1) retrieval loss: SampledSoftmaxLayer.call = tf.nn.sampled_softmax_loss (layers/tools.py:56-75), TF defaults:
 *   num_true = 1, remove_accidental_hits, subtract log Q, log-uniform candidates drawn unique.
 *   true_logit[b] = <user_b, item_label(b)> (hrb_rowdot), sampled_logit[b,j] = <user_b, item_sampled(j)> (hrb_dense_bwd_x as A.B^T);
 *   this entry applies - log Q, masks sampled(j) == label(b) with -FLT_MAX and takes the softmax cross-entropy against class 0:
 *   loss[b] = logsumexp(z) - z_0; with gradient buffers also d_true_logit / d_sampled_logit (times gout[b], NULL = 1).
 *   Q(k) = -expm1(num_tries*log1p(-p_k)), p_k = log((k+2)/(k+1))/log(range_max+1) -- or the caller's own expected counts
 *   (true_expected (B), sampled_expected (S); both or none), which is how `sampled_values` are injected for parity tests.
 * tf.nn.l2_normalize(x) WITHOUT an axis, as DSSM calls it (models/retrieval/DSSM.py:105-106): y = x * rsqrt(max(sum x^2, eps))
 *   over the whole tensor; stat (1 float) keeps the factor for the backward; scratch: 256 floats; fixed-order reductions.
 * ------------------------------------------------------------------------------------------ */
int hrb_sampled_softmax(const float* true_logit, const float* sampled_logit, int64_t ld, const int32_t* labels,
                        const int32_t* sampled, int64_t batch, int32_t num_sampled, const float* true_expected,
                        const float* sampled_expected, float num_tries, int64_t range_max, int32_t remove_accidental_hits,
                        const float* gout, float* loss, float* d_true_logit, float* d_sampled_logit, void* stream);
int hrb_rowdot(const float* a, int64_t lda, const float* b, int64_t ldb, int64_t M, int32_t K, float* out, void* stream);
int hrb_rowscale(const float* x, int64_t ldx, const float* s, int64_t M, int32_t K, float* out, int64_t ldo, void* stream);
int hrb_l2_normalize_fwd(const float* x, int64_t n, float eps, float* y, float* stat, float* scratch, void* stream);
int hrb_l2_normalize_bwd(const float* y, const float* dy, int64_t n, const float* stat, float* dx, float* scratch, void* stream);

/* ------------------------------------------------------------------------------------------
 * (f4) top-n inner-product search: faiss.IndexFlatIP.search(user_embd, n) of handyrec/models/utils.py:7-51.
 *   The caller computes the scores of a chunk of items (queries . items^T, e.g. hrb_dense_bwd_x_t) and folds every chunk into the
 *   running lists: best_val / best_idx (queries, k), ordered by (score descending, item index ascending); hrb_topk_init first.
 * ------------------------------------------------------------------------------------------ */
int hrb_topk_init(float* best_val, int32_t* best_idx, int64_t queries, int32_t k, void* stream);
int hrb_topk_merge(const float* scores, int64_t ld, int64_t queries, int32_t n_cols, int64_t col_base, int32_t k, float* best_val,
                   int32_t* best_idx, void* stream);

/* ------------------------------------------------------------------------------------------
 * Keras metrics tf.keras.metrics.{AUC, Precision, Recall, BinaryAccuracy} (Keras 2.6
 * metrics_utils.update_confusion_matrix_variables and the MeanMetricWrapper of binary_accuracy), one launch per update.
 *   thresholds (n_thr fp32, ascending, distinct -- not checked, the pointer is a device pointer; 1 <= n_thr <= 8192): the
 *   union of every metric's thresholds.  Variable v is vars[v] (fp32), of kind var_kind[v] at threshold thresholds[var_thr[v]]
 *   (ignored for COUNT).  With above_c(j) = #{i : label class c, prob[i] > thresholds[j]} (strict, fp32), classes
 *   0: label == 0, 1: label == 1, 2: any other label (NaN included; bool(label) is true for classes 1 and 2):
 *     TP = above_1 + above_2      FP = above_0      TN = tot_0 - above_0      FN = tot_1 + tot_2 - TP
 *     CORRECT = above_1 + tot_0 - above_0 (binary_accuracy's sum)           COUNT = n
 *   and vars[v] = fl(vars[v] + (float)increment): the batch's integer count, added with one fp32 rounding (Keras assign_add).
 *   flags (nullable, n_vars int32, caller-zeroed): when a prob of the batch is outside [0, 1] or NaN, flags[v] = 1 for every
 *   TP / FP / TN / FN variable v (Keras asserts 0 <= y_pred <= 1 for the confusion metrics; accuracy variables are never
 *   flagged).  scratch: hrb_metric_scratch_bytes(n_thr), zeroed by the caller once; every call leaves it zeroed (calls sharing a
 *   scratch must be stream-ordered).  n = 0 launches nothing. */
#define HRB_METRIC_MAX_THRESHOLDS 8192
typedef enum hrb_metric_kind {
  HRB_METRIC_TP = 0,
  HRB_METRIC_FP = 1,
  HRB_METRIC_TN = 2,
  HRB_METRIC_FN = 3,
  HRB_METRIC_CORRECT = 4,
  HRB_METRIC_COUNT = 5,
  HRB_METRIC_WTP = 6, /* the weighted kinds: hrb_metric_update_weighted only */
  HRB_METRIC_WFP = 7,
  HRB_METRIC_WTN = 8,
  HRB_METRIC_WFN = 9,
  HRB_METRIC_WCORRECT = 10,
  HRB_METRIC_WCOUNT = 11
} hrb_metric_kind;
int hrb_metric_scratch_bytes(int32_t n_thr, size_t* bytes);
int hrb_metric_update(const float* prob, const float* label, int64_t n, const float* thresholds, int32_t n_thr,
                      const int32_t* var_kind, const int32_t* var_thr, int32_t n_vars, float* vars, void* scratch, int32_t* flags,
                      void* stream);

/* Keras metrics with sample weights (update_confusion_matrix_variables with sample_weight, the Mean of binary_accuracy): as
 * hrb_metric_update with one fp32 weight per sample.  Kinds 0..5 add the same integer counts, bit-equal to hrb_metric_update on
 * the same batch.  Kinds WTP..WCOUNT add the same sums with every sample counted as its weight instead of 1 (WCOUNT = sum w):
 * each per-(class, bucket) sum is accumulated in fp64, the suffix sums are taken in fp64, and each variable adds its increment
 * rounded once to fp32 (Keras assign_add).  Negative, zero and NaN weights are taken as given.  Flags: as hrb_metric_update, for
 * WTP..WFN too.  The variables are bit-reproducible: every CTA sorts its samples by (class, bucket) with a block radix sort and
 * sums the runs in sorted order into its own fp64 bins; a second launch adds the bins over the CTAs in CTA order, takes the
 * suffix sums and updates the variables.  scratch: hrb_metric_weighted_scratch_bytes(n_thr) for the CURRENT device, zeroed by
 * the caller once; every call leaves it zeroed (calls sharing a scratch must be stream-ordered).  Two launches; n = 0 launches
 * nothing. */
int hrb_metric_weighted_scratch_bytes(int32_t n_thr, size_t* bytes);
int hrb_metric_update_weighted(const float* prob, const float* label, const float* weight, int64_t n, const float* thresholds,
                               int32_t n_thr, const int32_t* var_kind, const int32_t* var_thr, int32_t n_vars, float* vars,
                               void* scratch, int32_t* flags, void* stream);

/* a8 concat glue (layers/utils.py:28-36,70-84): dense features (fp32, or int32 cast to fp32) go to the
 * head columns of the DNN input row; columns [n, n_pad) are zero-filled (alignment padding). */
int hrb_pack_dense(const void* src, int32_t src_is_int32, int64_t src_ld, int64_t batch, int32_t n, int32_t n_pad,
                   float* dst, int64_t dst_ld, void* stream);

/* a3 input glue, HOST side (the only entry points that take host pointers and run on the CPU; no device work).
 * FeatureGroup.construct_inputs (features/group.py:218-248) hands Keras one array per feature; the fused lookup takes one
 * packed int32 id matrix and one fp32 dense matrix per batch (a7/a8).  Rows [row_start, row_start+rows) of every column array
 * cols_host[c] (row-major, ld_host[c] elements per row, width_host[c] used; dtype_host[c]: 0 int32, 1 int64, 2 float32, 3
 * float64) are converted and written side by side into dst_host[rows, dst_ld] by a persistent thread pool (n_threads <= 0: all). */
int hrb_host_pack_i32(const void* const* cols_host, const int32_t* dtype_host, const int64_t* width_host, const int64_t* ld_host,
                      int32_t n_cols, int64_t row_start, int64_t rows, int32_t* dst_host, int64_t dst_ld, int32_t n_threads);
int hrb_host_pack_f32(const void* const* cols_host, const int32_t* dtype_host, const int64_t* width_host, const int64_t* ld_host,
                      int32_t n_cols, int64_t row_start, int64_t rows, float* dst_host, int64_t dst_ld, int32_t n_threads);

/* The packers write every finished block of dst_host back from the CPU caches to memory (x86 clwb / clflushopt), because the
 * next reader is the GPU's copy engine and dirty lines in the packing cores' private caches slow that DMA.  on = 0 turns the
 * write-back off (measurements); returns what the CPU offers: 2 clwb, 1 clflushopt, 0 neither (then the call has no effect). */
int hrb_host_pack_set_writeback(int32_t on);

/* Dense-parameter optimisers on a flat fp32 buffer (Keras Adam / SGD / Adagrad formulas).  Adagrad (ResourceApplyAdagradV2):
 * g' = grad + l2_scale*param; acc += g'^2; param -= lr * g' / (sqrt(acc) + eps), acc starting at initial_accumulator_value. */
int hrb_adam_step(float* param, const float* grad, float* m, float* v, int64_t n, float lr, float beta1,
                  float beta2, float eps, float bias_corr1, float bias_corr2, float l2_scale, void* stream);
int hrb_sgd_step(float* param, const float* grad, int64_t n, float lr, float l2_scale, void* stream);
int hrb_adagrad_step(float* param, const float* grad, float* acc, int64_t n, float lr, float eps, float l2_scale, void* stream);
/* Keras Ftrl (ResourceApplyFtrl, or V2 when l2_shrinkage > 0) with the arithmetic of HRB_OPT_FTRL above; l2 with beta / (2*lr)
 * added.  row_touched NULL: every element steps.  Otherwise it holds one float per row of `dim` elements (n % dim == 0) and
 * the elements of rows whose value is 0 are left bit-identical (param, acc and lin): a dense-updated embedding table steps the
 * rows its IndexedSlices gradient lists (hrb_plan_mark_rows) and no others. */
int hrb_ftrl_step(float* param, const float* grad, float* acc, float* lin, int64_t n, float lr, float l1, float l2, float lr_power,
                  float l2_shrinkage, float l2_scale, const float* row_touched, int32_t dim, void* stream);
/* The same steps for `count` parameter tensors in one launch per HRB_MULTI_MAX tensors (host arrays of device pointers / sizes /
 * per-tensor l2 scales; l2_scale_host may be NULL).  The layer-by-layer models (DIN, the retrieval towers) hold 12-27 small
 * tensors; Keras applies one optimiser op per variable (keras optimizer_v2 _resource_apply_dense), here they share a launch. */
#define HRB_MULTI_MAX 32
int hrb_adam_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* m_host,
                        float* const* v_host, const int64_t* n_host, const float* l2_scale_host, float lr, float beta1,
                        float beta2, float eps, float bias_corr1, float bias_corr2, void* stream);
int hrb_sgd_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, const int64_t* n_host,
                       const float* l2_scale_host, float lr, void* stream);
int hrb_adagrad_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* acc_host,
                           const int64_t* n_host, const float* l2_scale_host, float lr, float eps, void* stream);
int hrb_ftrl_step_multi(int32_t count, float* const* param_host, const float* const* grad_host, float* const* acc_host,
                        float* const* lin_host, const int64_t* n_host, const float* l2_scale_host, float lr, float l1, float l2,
                        float lr_power, float l2_shrinkage, void* stream);

/* ------------------------------------------------------------------------------------------
 * Gradient clipping: Keras 2.6 OptimizerV2 `clipvalue`, `clipnorm`, `global_clipnorm` (optimizer_v2.py
 * `_transform_gradients`: clipvalue first, then clipnorm, then global_clipnorm).  In-place passes that run after every
 * gradient of a step is known and before the optimiser steps above (which are unchanged); the caller then steps with l2 = 0
 * wherever the prepare pass folded a regulariser in.  Squared norms are summed in float64 in a fixed order (the same bits on
 * every run) and added to sumsq[var] (fp32, caller-zeroed per step) with one rounding per call.
 *   workspace: hrb_clip_workspace_bytes(n_tables of the plan, or 0), zeroed by the caller once.  It holds one completion
 *   counter per entry point (each call leaves its counter zeroed) and the partial sums, so hrb_clip_prepare_multi and
 *   hrb_plan_clip_grads may share one workspace sized for the plan (calls sharing it must be stream-ordered).
 *   clipvalue = +INFINITY: no clamp.
 *
 * hrb_clip_prepare_multi   tf.clip_by_value on dense gradients with the regulariser folded in, and their squared norms:
 *     per segment i (host arrays as in hrb_*_step_multi, any count; w_host / l2_scale_host nullable, w_host[i] NULL needs l2 0):
 *     g[j] = clamp(fmaf(l2_scale[i], w[j], g[j]), -clipvalue, clipvalue);  sumsq[var[i]] += sum_j g[j]^2 (sumsq nullable).
 *     NaN passes the clamp unchanged.
 * hrb_plan_clip_grads      the same for the IndexedSlices gradient of the plan's tables (tf.clip_by_value and the norm of
 *     clip_by_norm over the un-deduplicated values), where the DNN part of a field's gradient is in dx and the FM part in fm
 *     (DeepFM looks every table up twice; Keras concatenates the two lookups' values, backprop_util.AggregateIndexedSlicesGradients).
 *     Per sample b, field f, element: p = part * inv with inv = 1/n_valid (mean pooling) or 1, clamped per part; dx receives the
 *     sum of the two parts in the form the backward reads (a part whose clamp does not bind is kept unchanged, a bound one
 *     becomes +-clipvalue * n_valid for mean pooling, +-clipvalue otherwise), and sumsq[table] += n_valid * (p_dnn'^2 + p_fm'^2).
 *     n_valid counts the positions the backward reads: in-range ids, and ids != 0 for pooled fields.  fm (nullable; needs
 *     contiguous field columns) holds field f at column out_col_f - out_col_0; sumsq (n_tables floats) nullable.  No max pooling.
 * hrb_clip_scales          tf.clip_by_norm / tf.clip_by_global_norm as a scale: scale[k] = c / max(sqrt(sumsq[k]), c) per
 *     variable, or (global != 0) every scale[k] = c / max(sqrt(sum_k sumsq[k]), c), NaN when that norm is not finite (TF's
 *     `scale + (norm - norm)`).  A norm <= c gives exactly 1; norm 0 with c = 0 gives NaN, as in TF.  One launch, no host sync.
 * hrb_clip_apply_multi     g[j] *= scale[var[i]] over segments.
 * hrb_plan_clip_apply      dx[b, columns of field f] *= scale[table of f] (the plan's layout as in hrb_lookup_bwd_update).
 * ------------------------------------------------------------------------------------------ */
int hrb_clip_workspace_bytes(int32_t n_tables, size_t* bytes);
int hrb_clip_prepare_multi(int32_t count, float* const* g_host, const float* const* w_host, const int64_t* n_host,
                           const float* l2_scale_host, const int32_t* var_host, float clipvalue, float* sumsq, void* workspace,
                           size_t workspace_bytes, void* stream);
int hrb_plan_clip_grads(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, float* dx, int64_t dx_ld,
                        const float* fm, int64_t fm_ld, float clipvalue, float* sumsq, void* workspace, size_t workspace_bytes,
                        void* stream);
int hrb_clip_scales(const float* sumsq, int32_t n_vars, float clipnorm, int32_t global, float* scale, void* stream);
int hrb_clip_apply_multi(int32_t count, float* const* g_host, const int64_t* n_host, const int32_t* var_host, const float* scale,
                         void* stream);
int hrb_plan_clip_apply(const hrb_plan* plan, float* dx, int64_t dx_ld, int64_t batch, const float* scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * (e) row-sharded tables: owner(r) = r % n_ranks, local row r / n_ranks  (SURVEY §8e).
 * ------------------------------------------------------------------------------------------ */

/* Compact row exchange (what handyrec_b200/sharded.py runs between NCCL all-to-alls):
 *   requester  hrb_route_ids     owner rank + owner-side key of every position, grouped by owner (stable):
 *                                perm[j] = position (b*sum_L + column), send_keys[j], counts[0..n_ranks] (last = padding).
 *                                key_base[r*n_tables + t] = first key of table t in rank r's shard key space.
 *   owner      hrb_rows_by_key   out[j,:] = shard row addressed by keys[j]
 *   requester  hrb_scatter_rows  rows -> output block (plain features) / position buffer + pooling (sequence features)
 *   requester  hrb_gather_grads  send[j,:] = dout[b, field(perm[j]) columns] * (1/n_valid for mean pooling)
 *   owner      hrb_keyed_bwd_update  (key, gradient row) pairs -> sort -> segment-reduce -> SGD / lazy-Adam / Adagrad / Ftrl row update */
/* Peer-mapped lookup: peer_tables_host[r*n_tables + t] = device pointer of rank r's shard of table t as mapped into this
 * process (CUDA IPC / symmetric memory over NVLink), full_rows_host[t] = full vocabulary size.  After this call
 * hrb_lookup_fwd / hrb_lookup_fm_fwd take GLOBAL ids and read row id from rank id % n_ranks at local row id / n_ranks:
 * the forward needs no all-to-all (plain-lookup groups laid out contiguously only).  A table whose pointers are NULL on
 * EVERY rank is replicated: its rows are read from the plan's own copy (hrb_table_desc.weight, full row count). */
int hrb_enable_peer_access(int32_t peer_device); /* cudaDeviceEnablePeerAccess from the current device, idempotent */
int hrb_plan_set_peers(hrb_plan* plan, int32_t n_ranks, const void* const* peer_tables_host, const int64_t* full_rows_host);
/* Requester-side plans hold SHARD row counts; with the full vocabulary sizes set, the routing helpers below skip ids outside
 * [0, full_rows[table]) exactly like the single-GPU path skips ids outside [0, rows) (TF-GPU gather semantics, a5). */
int hrb_plan_set_full_rows(hrb_plan* plan, const int64_t* full_rows_host);
int hrb_route_workspace(const hrb_plan* plan, int64_t batch, size_t* bytes);
int hrb_route_ids(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, int32_t n_ranks,
                  const uint32_t* key_base, uint32_t* perm, uint32_t* send_keys, int64_t* counts, void* workspace,
                  size_t workspace_bytes, void* stream);
int hrb_rows_by_key(const hrb_plan* plan, const uint32_t* keys, int64_t n, float* out, void* stream);
int hrb_scatter_rows(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, int64_t batch, const uint32_t* perm, int64_t n,
                     const float* rows, float* out, int64_t out_ld, float* pos_rows, void* stream);
int hrb_gather_grads(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, const uint32_t* perm, int64_t n,
                     const float* dout, int64_t dout_ld, float* send, void* stream);
/* hrb_gather_grads fused with the exchange (one node, NVLink): the gradient row and the owner-side key of position perm[j] are
 * stored directly into the OWNER's receive buffers through peer mappings (symmetric memory) instead of into a local send buffer
 * that an all-to-all then moves.  perm / send_keys come from hrb_route_ids (grouped by owner); send_counts_host[d] = entries
 * for owner d, dst_off_host[d] = first row this rank writes in d's buffers (= entries of lower-ranked senders for d, so that
 * every owner ends up with the layout of an all-to-all ordered by sender); peer_grads_host[d] / peer_keys_host[d] = owner d's
 * buffers as mapped into this process ([rows, D] fp32 / [rows] uint32; d = own rank: the local pointers).  The caller orders
 * the stores before the owners' reads with a cross-GPU barrier (sharded.py: symmetric-memory signal barrier). */
#define HRB_MAX_PEERS 16
int hrb_scatter_grads_to_owners(const hrb_plan* plan, const int32_t* ids, int64_t ids_ld, const uint32_t* perm,
                                const uint32_t* send_keys, const float* dout, int64_t dout_ld, int32_t n_ranks,
                                const int64_t* send_counts_host, const int64_t* dst_off_host, void* const* peer_grads_host,
                                void* const* peer_keys_host, void* stream);
int hrb_keyed_bwd_workspace(const hrb_plan* plan, int64_t n, size_t* bytes);
int hrb_keyed_bwd_update(const hrb_plan* plan, const uint32_t* keys, const float* grads, int64_t n, const hrb_opt_params* opt_host,
                         void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HRB200_H_ */
