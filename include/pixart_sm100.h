/* pixart_sm100.h -- C ABI of libpixart_sm100.so: hand-written sm_100a (B200) kernels for the
 * PixArt-Sigma DiT denoiser hot path  PixArtMS.forward -> 28 x PixArtMSBlock.forward.
 *
 * The reference (PixArt-alpha/PixArt-sigma) is pure Python and has NO FFI / plugin interface; its GPU math is
 * reached through library calls (torch nn.Linear / LayerNorm / GELU, xformers memory_efficient_attention).
 * Each entry point below replaces one such call site (file:line relative to the reference root) and is what a
 * ctypes binding inside diffusion/model/nets/PixArt_blocks.py would bind (see INTEGRATION.md).
 *
 * Contract (all entry points):
 *   - plain pointers and sizes only; every buffer (inputs, outputs, workspace) is owned by the caller and is
 *     DEVICE memory; the library never allocates, frees or synchronises and launches only on `stream`
 *     (a cudaStream_t passed as void*), so calls are CUDA-graph capturable;
 *   - returns 0 on success, a negative PXA_ERR_* otherwise; pxa_last_error() gives the message (thread local);
 *   - bf16 operands, fp32 accumulation / statistics / softmax; pointers must be 16-byte aligned;
 *   - requires an sm_100 device (PXA_ERR_ARCH otherwise). There is no CPU or non-Blackwell path.
 */
#ifndef PIXART_SM100_H_
#define PIXART_SM100_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PXA_OK 0
#define PXA_ERR_ARG (-1)     /* bad shape / null pointer / unsupported option */
#define PXA_ERR_ALIGN (-2)   /* pointer or stride not 16-byte aligned */
#define PXA_ERR_ARCH (-3)    /* device is not sm_100 */
#define PXA_ERR_CUDA (-4)    /* CUDA runtime / driver error (launch, tensor-map encode) */

#define PXA_DTYPE_BF16 0
#define PXA_DTYPE_F32 1

int pxa_version(void);
const char* pxa_last_error(void);
/* Number of kernel launches issued by this library since load (all streams) -- bench.py's `gpu_launches`. */
uint64_t pxa_launch_count(void);

/* ------------------------------------------------------------------------------------------------- GEMM
 * out = epilogue( A[M,K] . W[N,K]^T + bias[N] ),  A/W bf16 K-contiguous (W is the nn.Linear weight as stored).
 * tcgen05 (UMMA 128xBNx16, fp32 accumulators in TMEM), TMA-fed smem ring, persistent, warp-specialised.
 *
 * Replaces: attn.qkv PixArt_blocks.py:130 | attn.proj + gate + residual PixArt_blocks.py:155, PixArtMS.py:75 |
 *   cross_attn.q_linear / kv_linear / proj (+residual) PixArt_blocks.py:47,48,55, PixArtMS.py:76 |
 *   mlp.fc1 + GELU(tanh) / fc2 + gate + residual (timm Mlp; PixArtMS.py:67,77) | y_embedder.y_proj PixArt_blocks.py:406.
 */
#define PXA_EPI_BIAS 0          /* out = acc + bias                                   */
#define PXA_EPI_BIAS_GELU 1     /* out = gelu_tanh(acc + bias)                        */
#define PXA_EPI_BIAS_RESIDUAL 2 /* out = residual + gate[row/rows_per_batch, n] * (acc + bias); gate NULL -> 1 */
/* Training fusions of the MLP (timm Mlp, PixArtMS.py:67,77).  EXPERIMENTAL: compiled, but not yet validated on a B200 --
 * no default path calls them (pixart_sigma_b200.autograd uses them only with PXA_EXPERIMENTAL_FUSED_MLP=1) and their
 * GPU tests are skipped unless PXA_EXPERIMENTAL=1. */
#define PXA_EPI_BIAS_GELU_AUX 3 /* out = gelu_tanh(acc + bias), out_aux_bf16 = acc + bias (pre-activation kept for the backward) */
#define PXA_EPI_MUL_DGELU 4     /* out = acc * gelu_tanh'(pre), pre = `residual` as bf16 [M, N] row stride ldo; bias must be NULL  */
/* adaLN-single modulate FUSED into the projection that follows it (norm1 + t2i_modulate + attn.qkv, PixArtMS.py:75 with
 * PixArt_blocks.py:24-25,130; norm2 + t2i_modulate + mlp.fc1, PixArtMS.py:77): the LayerNorm'ed, modulated activations
 * are never materialised.  With mu_r / rstd_r the LayerNorm statistics of row r of the fp32 residual stream x and
 * (shift_b, scale_b) the modulation of its sample b,
 *     sum_k [ (x[r,k] - mu_r) rstd_r (1 + scale_b[k]) + shift_b[k] ] W[n,k] + bias[n]
 *   = rstd_r * ( acc[r,n] - mu_r * u_b[n] ) + v_b[n],     acc = A W^T,  A[r,k] = bf16( x[r,k] (1 + scale_b[k]) ),
 *     u_b[n] = sum_k (1 + scale_b[k]) W[n,k],   v_b[n] = sum_k shift_b[k] W[n,k] + bias[n].
 * A and the per-row statistics are by-products of the residual epilogue that produced x (`aux_scale`, `row_stats_out`
 * below) or of pxa_ln_prepare; u_b / v_b are two tiny per-sample GEMVs per forward. */
#define PXA_EPI_LN_BIAS 5       /* out = rstd*(acc - mu*u) + v            (`ln_*` fields; bias must be NULL: it is inside v) */
#define PXA_EPI_LN_BIAS_GELU 6  /* out = gelu_tanh(rstd*(acc - mu*u) + v)                                                   */
#define PXA_LN_STAT_PARTS 8     /* row statistics are kept as 8 partial (sum x, sum x^2) pairs per row: fp32 [M][8][2]      */

typedef struct PxaGemmArgs {
  const void* a;        /* bf16 [M, K], row stride lda (elements)                                   */
  const void* w;        /* bf16 [N, K], row stride ldw (elements)                                   */
  const void* bias;     /* bf16 [N] or NULL                                                         */
  void* out;            /* [M, N], row stride ldo (elements), dtype out_dtype                       */
  void* out_aux_bf16;   /* optional second bf16 copy of out (row stride ldo) or NULL                */
  const void* residual; /* EPI_BIAS_RESIDUAL: [M, N] row stride ldo, dtype out_dtype (may alias out)*/
  const float* gate;    /* EPI_BIAS_RESIDUAL: fp32, element (b, n) at gate[b*gate_batch_stride + n], or NULL */
  int64_t gate_batch_stride;
  int32_t rows_per_batch; /* rows of A per sample (tokens N); row r belongs to sample r / rows_per_batch */
  int32_t M, N, K;
  int32_t lda, ldw, ldo;
  int32_t epilogue;     /* PXA_EPI_*            */
  int32_t out_dtype;    /* PXA_DTYPE_*          */
  int32_t block_n;      /* 0 = auto (192 when it divides N, else 128); or 128 / 192 / 256           */
  int32_t max_ctas;     /* 0 = one CTA per SM; >0 caps the persistent grid (tests)                  */
  int32_t cta_pair;     /* 0 = auto, 1 = single-CTA UMMA (128 x BN tiles), 2 = CTA-pair UMMA (256 x BN tiles) */
  int64_t* debug_trace; /* NULL in production. Else device int64[4096]: cycle stamps of CTA 0's epilogue issuer thread */
  int32_t operands_mn_major; /* 1: weight-gradient form out[M, N] += A^T . W with a = [K, M] (row stride lda) and
                                w = [K, N] (row stride ldw), i.e. the contraction runs over the ROWS of both operands
                                (dW = dY^T X straight from the activations' natural layouts; no transposes).  Requires
                                EPI_BIAS_RESIDUAL, fp32 out, residual == out (in-place accumulate), no bias / gate / aux. */
  int32_t k_splits;     /* operands_mn_major only: 0 = auto (fill the 148 SMs), else the number of K splits        */
  int32_t aux_is_branch; /* EPI_BIAS_RESIDUAL with out_aux_bf16: 1 = the aux output receives acc + bias (the un-gated
                            branch output, which the backward of the gate needs) instead of a bf16 copy of out          */
  /* --- producer side of the fused LayerNorm-modulate (EPI_BIAS_RESIDUAL, fp32 out, out_aux_bf16 set) */
  const float* aux_scale;   /* fp32 or NULL: the bf16 aux copy becomes out[r,n] * aux_scale[b*aux_scale_batch_stride + n]
                               (pass 1 + scale of the NEXT modulate: the aux output is then the A operand above)          */
  int64_t aux_scale_batch_stride;
  float* row_stats_out;     /* fp32 [M][PXA_LN_STAT_PARTS][2] or NULL: partial (sum, sum of squares) of each row of `out`
                               over the columns of one output tile, part = the tile's column index; unused parts zeroed     */
  /* --- consumer side (EPI_LN_BIAS / EPI_LN_BIAS_GELU) */
  const float* ln_stats;    /* fp32 [M][PXA_LN_STAT_PARTS][2] partial sums of the rows of x (row_stats_out / pxa_ln_prepare) */
  const float* ln_u;        /* fp32, u_b[n] at ln_u[b*ln_uv_batch_stride + n]                                                */
  const float* ln_v;        /* fp32, v_b[n] at ln_v[b*ln_uv_batch_stride + n]                                                */
  int64_t ln_uv_batch_stride;
  int32_t ln_dim;           /* row length C of x the statistics were taken over                                              */
  float ln_eps;
  int32_t res_epilogue;     /* EPI_BIAS_RESIDUAL, fp32 out, CTA pair: 0 = auto, 1 = register-staged residual (coalesced
                               loads, smem transpose), 2 = residual tile streamed through smem by TMA (row per thread)       */
  int32_t epi_warps;        /* CTA pair, bf16 epilogues: 0 = auto (8: two epilogue warps per TMEM lane quarter), 4 or 8     */
  int32_t reverse_tiles;    /* 1: visit the output tiles from the LAST row block to the first.  A GEMM whose A operand was
                               written front to back by the previous kernel (mlp.fc2 after mlp.fc1) then starts on the rows
                               that are still in the 126 MB L2 instead of the ones already evicted to HBM                   */
} PxaGemmArgs;
int pxa_gemm_bf16(const PxaGemmArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------- fused Mlp
 * x32[r, :] += gate[b, :] * ( gelu_tanh(x[r, :] W1^T + b1) W2^T + b2 )        b = r / rows_per_batch
 * The timm Mlp of PixArtMSBlock with its gate and residual (PixArtMS.py:67,77) as ONE persistent kernel: both GEMMs in one
 * tile list, the second one group of 256-row panels behind the first, the [M, N1] hidden activations kept in a small ring
 * (hidden_ws) that lives in L2 instead of streaming through HBM (mlp_sm100.cu).  x = the normalised, modulated bf16
 * activations (pxa_ln_modulate output); x32 = the fp32 residual stream, updated in place (TMA reduce-add).
 */
typedef struct PxaMlpArgs {
  const void* x;         /* bf16 [M, K1], row stride ldx                                   */
  const void* w1;        /* bf16 [N1, K1] (mlp.fc1.weight), row stride ldw1                 */
  const void* b1;        /* bf16 [N1] or NULL                                              */
  const void* w2;        /* bf16 [N2, N1] (mlp.fc2.weight), row stride ldw2                 */
  const void* b2;        /* bf16 [N2] or NULL                                              */
  float* x32;            /* fp32 [M, N2], row stride ldo: residual stream, updated in place */
  const float* gate;     /* fp32 (b, n) at gate[b*gate_batch_stride + n], or NULL           */
  int64_t gate_batch_stride;
  void* hidden_ws;       /* bf16 scratch, >= ring * group * 256 * N1 elements               */
  int64_t hidden_ws_bytes;
  void* flags_ws;        /* int32 scratch, >= 2 * ceil(M/256) + ceil(ceil(M/256)/group) ints (zeroed by the call) */
  int64_t flags_ws_bytes;
  int32_t rows_per_batch;
  int32_t M, K1, N1, N2; /* N1 % 256 == 0, N2 % 192 == 0                                   */
  int32_t ldx, ldw1, ldw2, ldo;
  int32_t group;         /* 256-row panels per group (0 = 4)                               */
  int32_t ring;          /* groups held by hidden_ws (0 = lag + 2)                         */
  int32_t max_ctas;      /* 0 = one CTA per SM; > 0 caps the persistent grid (tests)       */
  int32_t lag;           /* fc2 runs `lag` groups behind fc1 in the tile list (0 = 1); ring > lag, ring >= lag + 2 keeps
                            fc1 from waiting on the slot it is about to overwrite (ring 0 = lag + 2)                      */
  int32_t k_splits;      /* fc2 tiles reduce over N1 / k_splits each and are summed by the reduce-add epilogue (0 = auto:
                            the split that makes a fc2 tile cost what a fc1 tile costs, 3 for 1152 -> 4608 -> 1152)        */
} PxaMlpArgs;
int pxa_mlp_fused_bf16(const PxaMlpArgs* args, void* stream);

/* ------------------------------------------------------------------------------------ LayerNorm + modulate
 * out[r,:] = LN(x[r,:]; eps, no affine) * (1 + scale[b,:]) + shift[b,:]  with b = r / rows_per_batch, bf16 out.
 * Replaces norm1/norm2 + t2i_modulate (PixArtMS.py:58,64,75,77; PixArt_blocks.py:24-25) and the final-layer
 * modulate (PixArt_blocks.py:218-219).  HBM-bound: reads x once, writes out once.
 */
typedef struct PxaLnModArgs {
  const void* x;        /* [M, C] row stride ldx, dtype x_dtype */
  void* out;            /* bf16 [M, C] contiguous                */
  const float* shift;   /* fp32, (b, c) at shift[b*mod_batch_stride + c] */
  const float* scale;   /* fp32, same addressing                  */
  int64_t mod_batch_stride;
  int32_t rows_per_batch;
  int32_t M, C, ldx;
  int32_t x_dtype;      /* PXA_DTYPE_* */
  float eps;
  int32_t reverse_rows; /* 1: CTAs take the rows from the last to the first (start on the rows of x that the front-to-back
                           residual GEMM before it wrote last, i.e. the ones still in L2)                        */
  int32_t max_ctas;     /* 0 = auto: a grid-stride launch of two 8-warp CTAs per SM, every warp prefetching its next row;
                           > 0 caps / widens the grid (M / 8 or more = one row per warp)                               */
} PxaLnModArgs;
int pxa_ln_modulate(const PxaLnModArgs* args, void* stream);

/* First link of the fused LayerNorm-modulate chain (see PXA_EPI_LN_BIAS): for the residual stream x as the patch embedding
 * leaves it (PixArtMS.py:184), writes the A operand  a[r,:] = bf16( x[r,:] * mult[b,:] ), mult = 1 + scale (the same
 * multiplier PxaGemmArgs.aux_scale takes), and the row statistics
 * stats[r][0] = (sum_k x[r,k], sum_k x[r,k]^2), stats[r][1..7] = 0  that the QKV GEMM of block 0 consumes.  Later links
 * get both from the residual epilogues (PxaGemmArgs.aux_scale / row_stats_out).  HBM-bound: one read of x, one bf16 write.
 */
typedef struct PxaLnPrepareArgs {
  const float* x;       /* fp32 [M, C] row stride ldx                 */
  void* a_out;          /* bf16 [M, C] contiguous                     */
  float* stats_out;     /* fp32 [M][PXA_LN_STAT_PARTS][2]             */
  const float* scale;   /* fp32 multiplier 1 + scale_b, (b, c) at scale[b*mod_batch_stride + c] */
  int64_t mod_batch_stride;
  int32_t rows_per_batch;
  int32_t M, C, ldx;
} PxaLnPrepareArgs;
int pxa_ln_prepare(const PxaLnPrepareArgs* args, void* stream);

/* In-place LayerNorm(C = 1152, affine weight / bias bf16, fp32 statistics) on M bf16 rows of stride ld (elements):
 * q_norm / k_norm of AttentionKVCompress (`qk_norm=True`, PixArt_blocks.py:91-95,133-134) on the q and k column slices
 * of the qkv GEMM output.  HBM-bound: one read and one write of the slice. */
int pxa_layernorm_affine_bf16(void* x, const void* weight, const void* bias, int32_t M, int32_t C, int64_t ld, float eps,
                              void* stream);

/* RMS norm of the T5-v1.1-XXL caption encoder (transformers `T5LayerNorm`, eps 1e-6; reference call site diffusion/model/t5.py:107-110):
 * out[r, c] = bf16(x[r, c] * rsqrt(mean_c(x[r, :]^2) + eps) * weight[c]) on M rows of the fp32 residual stream (row strides ldx /
 * ldo in elements, C a multiple of 4).  HBM-bound: 4 C + 2 C bytes per row. */
int pxa_rmsnorm_bf16(const float* x, const void* weight, void* out, int32_t M, int32_t C, int64_t ldx, int64_t ldo, float eps,
                     void* stream);

/* Self-attention of the T5-v1.1-XXL caption encoder (transformers `T5Attention.forward`; reference call site
 * diffusion/model/t5.py:107-110): out[b, i, h, :] = softmax_j(q_i . k_j * scale + bias[h, i, j] + key_bias[b, j]) v_j for head_dim 64
 * and L <= 384 tokens per sample (T5 uses scale = 1 and a learned relative-position bias; key_bias carries the additive padding mask:
 * 0 for real tokens, a large negative number for padding).  q / k / v: bf16, element (b, i, h, d) at x[(b*L + i)*x_sn + h*x_sh + d]
 * (strided views of a fused qkv GEMM output are fine); out: bf16 [(b*L + i)*ldo + h*64 + d].  Logits, bias add, softmax and the
 * accumulation are fp32; P enters P V as bf16. */
typedef struct PxaT5AttnArgs {
  const void* q; const void* k; const void* v;
  void* out;
  const float* bias;      /* fp32 [H, L, L]; may be NULL when rel_bias is given                                              */
  const float* key_bias;  /* fp32 [B, L] or NULL                                                                             */
  int64_t q_sn, q_sh, k_sn, k_sh, v_sn, v_sh, ldo;
  int32_t B, H, L;
  float scale;
  const float* rel_bias;  /* fp32 [H, 2L-1] or NULL: the Toeplitz form bias[h, i, j] = rel_bias[h, j - i + L - 1] that T5's relative
                             position bias has; staged in shared memory (used instead of `bias` when non-NULL)              */
} PxaT5AttnArgs;
int pxa_t5_attn_d64_bf16(const PxaT5AttnArgs* args, void* stream);

/* GroupNorm (+ SiLU) on an NHWC bf16 image: the prologue of each 3x3 convolution of the SDXL-VAE decoder ResnetBlock2D
 * (diffusers GroupNorm(32, eps 1e-6) -> SiLU; reference call site scripts/inference.py:136).  out[b,p,c] =
 * silu((x[b,p,c] - mean[b,g]) * rstd[b,g] * gamma[c] + beta[c]), g = c / (C / groups), statistics over the HW pixels and the
 * C / groups channels of the group (fp32).  stats_ws: caller-owned fp32 [B][groups][2] scratch (zeroed by the call, on the
 * stream).  Two launches: statistics, apply.  HBM-bound: 2 reads + 1 write of the image. */
int pxa_groupnorm_silu_nhwc_bf16(const void* x, void* out, const void* gamma, const void* beta, float* stats_ws, int32_t B,
                                 int32_t HW, int32_t C, int32_t groups, float eps, int32_t silu, void* stream);

/* AdamW on a flat fp32 bucket (torch.optim.AdamW semantics: decoupled weight decay, bias-corrected moments) -- the optimizer
 * the reference trains with (configs/PixArt_xl2_internal.py:48 `AdamW(lr=2e-5, weight_decay=3e-2, eps=1e-10)`, built by
 * diffusion/utils/optimizer.py:236-245), applied to the gradient buckets of pixart_sigma_b200.parallel.GradBucketReducer in one
 * launch per bucket; optionally writes the bf16 copy of the updated parameters that the GEMMs read.  All pointers device. */
typedef struct PxaAdamWArgs {
  float* param;          /* fp32 [n], updated in place          */
  const float* grad;     /* fp32 [n]                            */
  float* exp_avg;        /* fp32 [n], updated in place          */
  float* exp_avg_sq;     /* fp32 [n], updated in place          */
  void* shadow_bf16;     /* bf16 [n] or NULL                    */
  int64_t n;             /* multiple of 4                       */
  int32_t step;          /* 1-based step count (bias correction) */
  float lr, beta1, beta2, eps, weight_decay;
  float grad_scale;      /* gradients are multiplied by this first (1 / loss scale, or 1) */
} PxaAdamWArgs;
int pxa_adamw_flat(const PxaAdamWArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------- attention
 * out[b, i, h, :] = softmax_j( q[b,i,h,:] . k[b,j,h,:] * scale ) v[b,j,h,:],  j < kv_len[b],  head_dim 72.
 * Flash-style: TMA-staged K/V ring, S = QK^T and O += PV on tcgen05 with S/P/O in TMEM, fp32 online softmax.
 * One kernel serves self-attention (PixArt_blocks.py:153, optionally KV-compressed: Nk < Nq) and the packed
 * var-len T5 cross-attention (PixArt_blocks.py:50-53, BlockDiagonalMask semantics via kv_off/kv_len).
 * Rows with kv_len == 0 produce zeros (xformers behaviour).
 */
typedef struct PxaAttnArgs {
  const void* q;  /* bf16, element (b, i, h, d) at q[(b*Nq + i)*q_sn + h*q_sh + d] */
  const void* k;  /* bf16, element (row, h, d) at k[row*k_sn + h*k_sh + d], row = kv_off[b] + j (see below) */
  const void* v;  /* bf16, same addressing as k with v_sn / v_sh */
  void* out;      /* bf16, element (b, i, h, d) at out[(b*Nq + i)*ldo + h*72 + d] */
  const int32_t* kv_len; /* device [B] or NULL (-> Nk for every sample)                                */
  const int32_t* kv_off; /* device [B] first key row of sample b, or NULL (-> b*Nk: padded/unpacked)   */
  int64_t q_sn, q_sh;
  int64_t k_sn, k_sh, v_sn, v_sh;
  int64_t kv_rows;  /* total rows addressable through k / v (B*Nk unpacked, sum(kv_len) packed)          */
  int32_t B, H, Nq, Nk; /* Nk = max keys per sample (loop bound) */
  int32_t ldo;
  float scale;      /* softmax scale, 72^-0.5 */
  int64_t* debug_trace; /* NULL in production. Else device int64[16 warps + 2][kTraceMax] cycle stamps of CTA (0,0,0) */
  float* lse;       /* optional fp32 [B, H, Nq]: log2-domain log-sum-exp of the scaled scores, the softmax statistic the
                       backward pass recomputes P from (training); NULL for inference                              */
  int32_t reverse_batch; /* 1: CTAs take the samples from the last to the first (same L2 argument as PxaGemmArgs.reverse_tiles:
                            the qkv rows of the last samples are the ones the QKV GEMM has just written)                   */
  int32_t variant;  /* 0 = auto (= 4).  Work item = 256 query rows of one (sample, head), two 128-row tiles with a double-buffered S:
                       4 = persistent grid, one CTA per SM walks the items; the next item's loads and first Q K^T overlap the
                           current item's epilogue; for Nk <= 1024 the output leaves as one TMA tensor store per 128-row tile;
                       2 = one CTA per item (same arithmetic, bit-identical results);
                       3 = three tiles per CTA, single S buffer each, three softmax warps per sub-partition (attn3_sm100.cu);
                       5 / 6 / 7 = experiment forms of 4 (no tile-B stagger / direct output stores always / tile stores always) */
  int32_t p_precision; /* 0 = P rounded to bf16 before P V (up to 2^-8 relative; the default).
                          1 = `fp32_attention` semantics (PixArt_blocks.py:145-147: q / k / v and hence P kept in fp32): P enters
                              the tensor pipe as bf16 hi + lo terms (2^-17 relative), two P V products per 16 keys; logits,
                              softmax and accumulation are fp32 in both modes.  Not available for variant 3.                  */
  int32_t reserved0;   /* must be 0 */
} PxaAttnArgs;
int pxa_flash_attn_d72_bf16(const PxaAttnArgs* args, void* stream);

/* ------------------------------------------------------------------------------------- KV token compression
 * out[b, p, c] = LN_c( bias[c] + sum_{dy,dx<2} w[c,dy,dx] * in[b, (2py+dy)*W + 2px+dx, c] ) * gamma[c] + beta[c]
 * Depthwise conv k=s=2 + LayerNorm(affine, eps 1e-5) on K and V (PixArt_blocks.py:84-89, 115-117), both tensors in
 * one launch.  in: bf16 rows of `ld_in` elements (k and v are column slices of the qkv GEMM output).
 */
typedef struct PxaKvCompressArgs {
  const void* k_in; const void* v_in; /* bf16, token row stride ld_in, batch stride H*W*ld_in */
  void* k_out; void* v_out;           /* bf16 [B, (H/2)*(W/2), C] contiguous                   */
  const void* conv_w;   /* bf16 [C, 1, 2, 2] */
  const void* conv_b;   /* bf16 [C]          */
  const void* ln_w;     /* bf16 [C]          */
  const void* ln_b;     /* bf16 [C]          */
  int32_t B, H, W, C, ld_in;
  float eps;
} PxaKvCompressArgs;
int pxa_kv_compress_conv2_ln(const PxaKvCompressArgs* args, void* stream);

/* ------------------------------------------------------------------------------------ 3x3 convolution (SDXL-VAE decoder)
 * out[b,y,x,:] = (residual[b,y,x,:] +) bias + sum_{dy,dx,c} w[:, dy, dx, c] * x[b, y+dy-1, x+dx-1, c]   (zero padding 1)
 * Implicit GEMM on the tcgen05 GEMM kernel: M = B*H*W pixels, N = Cout, K = 9*Cin; the A tiles are 128-pixel blocks of
 * the NHWC image fetched by a 4-D TMA tensor map whose out-of-bounds fill implements the padding (no im2col buffer).
 * Replaces the conv1 / conv2 of the decoder ResBlocks of diffusers' AutoencoderKL (reference call site
 * scripts/inference.py:136 `vae.decode`; GroupNorm + SiLU stay PyTorch).
 * Requirements: Cin % 64 == 0, Cout % 8 == 0.  Any H x W: widths that are a power of two <= 128 (with H a multiple of 128 / W) or a
 * multiple of 128 tile exactly; the others run over a virtual width rounded up to 128 (W / Wp of the MMA work is useful).
 */
typedef struct PxaConv3x3Args {
  const void* x;        /* bf16 NHWC [B, H, W, Cin] contiguous (torch channels_last)                         */
  const void* w;        /* bf16 [Cout, 3, 3, Cin] contiguous = checkpoint weight [Cout, Cin, 3, 3] permuted    */
  const void* bias;     /* bf16 [Cout] or NULL                                                               */
  void* out;            /* bf16 NHWC [B, H, W, Cout]                                                         */
  const void* residual; /* bf16 NHWC [B, H, W, Cout] or NULL                                                 */
  int32_t B, H, W, Cin, Cout;
} PxaConv3x3Args;
int pxa_conv3x3_nhwc_bf16(const PxaConv3x3Args* args, void* stream);

/* ------------------------------------------------------------------------------------ DPM-Solver++ sampler step
 * One fused elementwise pass per sampling step of the multistep DPM-Solver++ (2M) loop the reference runs in PyTorch
 * (diffusion/model/dpm_solver.py: CFG combine :326-332, data prediction :435-444, first-order update :565-577,
 * second-order multistep update :822-840; loop :1196-1241; call site scripts/inference.py:102-118):
 *     eps   = eps_uncond + cfg_scale * (eps_cond - eps_uncond)
 *     x0    = (x - sigma_s * eps) * inv_alpha_s                      (data prediction at the current time s)
 *     x    <- a * x - b * x0 - c * (x0 - x0_prev)                    (c = 0: first-order update)
 *     x0_prev <- x0
 * with host-computed scalars a = sigma_t / sigma_s, b = alpha_t * expm1(-h), c = 0.5 * b / r0.
 * `model_out` is the denoiser output of the CFG batch [uncond (n) ; cond (n)]: element (i, ch, p) at
 * model_out[i * out_batch_stride + ch * hw + p], ch < 4 (so the 8-channel learn-sigma output can be passed as is).
 * fp32 arithmetic; x, x0_prev: fp32 [n, 4, hw] contiguous, updated in place.  HBM-bound: 24 (fp32 out) / 16 (bf16 out)
 * algorithmic bytes per latent element.
 */
typedef struct PxaDpmStepArgs {
  const void* model_out;    /* [2n, >=4, hw], dtype out_dtype                         */
  float* x;                 /* fp32 [n, 4, hw] in/out                                 */
  float* x0_prev;           /* fp32 [n, 4, hw] in/out (ignored on input when c == 0)  */
  int64_t out_batch_stride; /* elements                                               */
  int32_t n, hw;
  int32_t out_dtype;        /* PXA_DTYPE_*                                            */
  float cfg_scale, sigma_s, inv_alpha_s, a, b, c;
} PxaDpmStepArgs;
int pxa_dpm_solver_pp_step(const PxaDpmStepArgs* args, void* stream);

/* ------------------------------------------------------------------------------------ SA-Solver sampler step
 * One fused elementwise pass per denoiser evaluation i of the SA-Solver "few steps" loop (predictor order 2, corrector
 * order 2, PEC) the reference runs in PyTorch (diffusion/model/sa_solver.py: CFG combine :310-318, data prediction
 * :377-386, predictor :644-698, corrector :700-753, loop :755-909; wrapper diffusion/sa_sampler.py:75-92):
 *     eps   = eps_uncond + cfg_scale * (eps_cond - eps_uncond)      (eps_cond alone when cond_row_offset == 0)
 *     x0    = (x_pred - sigma * eps) * inv_alpha                    (data prediction at t_i, x_pred = the denoiser input)
 *     x_c   = has_corr ? cA * x + (c0 * x0 + c1 * x0_prev) + cN * noise : x_pred        (corrector of step i)
 *     x_pred <- pA * x_c + (p0 * x0 + p1 * x0_prev) + pN * noise_next                   (predictor of step i + 1)
 *     x <- x_c,  x0_prev <- x0
 * with host-computed scalars (pixart_sigma_b200/sampler.py, SASolverSampler.plan); p1 = 0 for a first-order predictor.
 * After the last evaluation x_pred holds the sample.  Every product and sum is rounded separately, in the order above
 * (the reference's float32 tensor ops), so only the reciprocal inv_alpha differs from it.
 * `model_out`: the unconditional output of image j at row j, the conditional one at row j + cond_row_offset (n for the
 * CFG batch [uncond (n) ; cond (n)], 0 for a single conditional evaluation); element (row, ch, p) at
 * model_out[row * out_batch_stride + ch * hw + p], ch < 4 (the 8-channel learn-sigma output can be passed as is).
 * fp32 arithmetic; x, x_pred, x0_prev, noise, noise_next: fp32 [n, 4, hw] contiguous; x, x_pred, x0_prev updated in place.
 * x and noise are not read when has_corr == 0, x0_prev not read when has_corr == 0 and p1 == 0.
 * HBM-bound: 40 (fp32 CFG output) / 36 (bf16) algorithmic bytes per latent element.
 */
typedef struct PxaSaStepArgs {
  const void* model_out;    /* [cond_row_offset + n, >=4, hw], dtype out_dtype        */
  float* x;                 /* fp32 [n, 4, hw] in/out: corrected state                */
  float* x_pred;            /* fp32 [n, 4, hw] in/out: predicted state                */
  float* x0_prev;           /* fp32 [n, 4, hw] in/out: previous data prediction       */
  const float* noise;       /* fp32 [n, 4, hw]: noise of step i (corrector)           */
  const float* noise_next;  /* fp32 [n, 4, hw]: noise of step i + 1 (predictor)       */
  int64_t out_batch_stride; /* elements                                               */
  int32_t n, hw;
  int32_t cond_row_offset;  /* 0 or n                                                 */
  int32_t out_dtype;        /* PXA_DTYPE_*                                            */
  int32_t has_corr;         /* 0 at the first evaluation                              */
  float cfg_scale, sigma, inv_alpha;
  float cA, c0, c1, cN;     /* corrector of step i                                    */
  float pA, p0, p1, pN;     /* predictor of step i + 1                                */
} PxaSaStepArgs;
int pxa_sa_solver_step(const PxaSaStepArgs* args, void* stream);

/* =============================================================================================== training backward
 * The reference trains through torch autograd (train_scripts/train.py:197 `accelerator.backward(loss)`, per-block
 * activation checkpointing diffusion/model/utils.py:28-45).  The entry points below are the backward twins of the forward
 * ops above; `pixart_sigma_b200/autograd.py` binds them as torch.autograd.Function s.  The dgrad / wgrad matrix products
 * run on pxa_gemm_bf16 itself (dX = dY . W  ==  gemm(A = dY, W' = W^T);  dW += dY^T . X  ==  gemm(A = dY^T, W' = X^T) with the
 * fp32 residual epilogue adding into the gradient buffer), fed by pxa_transpose_bf16.
 */

/* out[C, R] = in[R, C]^T (bf16; 32-bit accesses when R, C, ldi, ldo are even, element-wise otherwise). */
int pxa_transpose_bf16(const void* in, void* out, int32_t R, int32_t C, int64_t ldi, int64_t ldo, void* stream);

/* GELU(approximate='tanh') on n bf16 elements (n % 8 == 0): dh == NULL: out = gelu(pre);  else out = dh * gelu'(pre).
 * Replaces timm Mlp.act (PixArtMS.py:67) forward (training path, which keeps `pre` for the backward) and backward. */
int pxa_gelu_tanh_bf16(const void* pre, const void* dh, void* out, int64_t n, void* stream);

/* Gated residual add of the block (PixArtMS.py:75-77) on the fp32 residual stream, and its backward.
 *   fwd: out[r,:] = x[r,:] + gate[b,:] * y[r,:]                      (x, out fp32; y bf16; gate NULL -> 1)
 *   bwd: x = dout (fp32), out = dy (bf16) = dout * gate[b,:];  dgate[b,:] += sum_{r in b} dout[r,:] * y[r,:]  (if dgate)  */
typedef struct PxaGateResidualArgs {
  const void* x;        /* fp32 [M, C] contiguous (fwd: residual stream; bwd: incoming gradient)               */
  const void* y;        /* bf16 [M, C] contiguous branch output (bwd: only needed with dgate)                   */
  const float* gate;    /* fp32 (b, c) at gate[b*gate_batch_stride + c], or NULL                                */
  void* out;            /* fwd: fp32 [M, C];  bwd: bf16 [M, C]                                                  */
  float* dgate;         /* bwd only: fp32 [B, C] contiguous, accumulated into (atomics); or NULL                */
  int64_t gate_batch_stride;
  int32_t rows_per_batch;
  int32_t M, C;
} PxaGateResidualArgs;
int pxa_gate_residual_fwd(const PxaGateResidualArgs* args, void* stream);
int pxa_gate_residual_bwd(const PxaGateResidualArgs* args, void* stream);

/* Backward of pxa_ln_modulate w.r.t. x, shift and scale (C = 1152):
 *   dx = LN-backward((1 + scale[b]) * dxn);  dshift[b,:] += sum_r dxn[r,:];  dscale[b,:] += sum_r dxn[r,:] * xhat[r,:]  */
typedef struct PxaLnModBwdArgs {
  const void* x;        /* fp32 [M, C] contiguous: the forward input                                            */
  const void* dxn;      /* bf16 [M, C] contiguous: gradient of the forward output                               */
  const float* scale;   /* fp32 (b, c) at scale[b*mod_batch_stride + c]                                         */
  void* dx;             /* fp32 [M, C] contiguous (written)                                                     */
  float* dshift;        /* fp32 [B, C] contiguous (accumulated, atomics)                                        */
  float* dscale;        /* fp32 [B, C] contiguous (accumulated, atomics)                                        */
  int64_t mod_batch_stride;
  int32_t rows_per_batch;
  int32_t M, C;
  float eps;
  const float* add_in;  /* optional fp32 [M, C]: dx = add_in + (gradient through the LayerNorm): the gradient of the residual
                           stream that by-passes the norm (x feeds both the norm and the residual add), folded in       */
} PxaLnModBwdArgs;
int pxa_ln_modulate_bwd(const PxaLnModBwdArgs* args, void* stream);

/* Backward of pxa_kv_compress_conv2_ln (depthwise conv k=s=2 + LayerNorm(affine) on K and V, PixArt_blocks.py:84-89,
 * 115-117): input gradients written to the 4 input rows of every output token, parameter gradients (shared by K and V)
 * ACCUMULATED into fp32 buffers (atomics).  The LN bias does not influence any gradient and is not needed. */
typedef struct PxaKvCompressBwdArgs {
  const void* k_in; const void* v_in;     /* bf16 forward inputs, token row stride ld_in                           */
  const void* dk_out; const void* dv_out; /* bf16 [B, (H/2)*(W/2), C] gradients of the compressed K / V             */
  void* dk_in; void* dv_in;               /* bf16 gradients of the inputs, token row stride ld_din (written)        */
  const void* conv_w; const void* conv_b; const void* ln_w;   /* bf16 parameters as in the forward                  */
  float* d_conv_w;      /* fp32 [C, 1, 2, 2] accumulated */
  float* d_conv_b;      /* fp32 [C] accumulated           */
  float* d_ln_w;        /* fp32 [C] accumulated           */
  float* d_ln_b;        /* fp32 [C] accumulated           */
  int32_t B, H, W, C, ld_in, ld_din;
  float eps;
} PxaKvCompressBwdArgs;
int pxa_kv_compress_conv2_ln_bwd(const PxaKvCompressBwdArgs* args, void* stream);

/* out[c] += sum_r a[r, c]  (bias gradients; a bf16 [M, N] row stride lda, N % 8 == 0; out fp32 [N], atomics). */
int pxa_colsum_bf16(const void* a, float* out, int32_t M, int32_t N, int64_t lda, void* stream);

/* delta[(b*H + h)*Nq + i] = sum_d dO[b,i,h,d] * O[b,i,h,d]  (o / dO bf16 [B*Nq, H*72] with row strides ldo / lddo). */
int pxa_attn_delta_d72(const void* o, const void* d_o, float* delta, int32_t B, int32_t H, int32_t Nq, int64_t ldo,
                       int64_t lddo, void* stream);

/* Backward of pxa_flash_attn_d72_bf16: dq, dk, dv from (q, k, v, o, dO, lse).  Flash-attention-2 recomputation on
 * tcgen05 (two passes: dK/dV per key tile, dQ per query tile); nothing N x N reaches HBM.  Same addressing as the
 * forward (strided bf16 views, packed var-len keys through kv_off / kv_len), any Nq / Nk.
 * dk / dv rows of keys >= kv_len[b] are not written.  `delta` is caller-owned workspace.                         */
typedef struct PxaAttnBwdArgs {
  const void* q; const void* k; const void* v;   /* as PxaAttnArgs                                              */
  const void* o;        /* bf16 forward output, (b, i, h, d) at o[(b*Nq + i)*ldo + h*72 + d]                      */
  const void* d_o;      /* bf16 gradient of o, row stride lddo                                                   */
  const float* lse;     /* fp32 [B, H, Nq] written by the forward (PxaAttnArgs.lse)                              */
  float* delta;         /* fp32 [B, H, Nq] workspace                                                             */
  void* dq; void* dk; void* dv;                  /* bf16, addressed like q / k / v with the strides below        */
  const int32_t* kv_len; const int32_t* kv_off;
  int64_t q_sn, q_sh, k_sn, k_sh, v_sn, v_sh;
  int64_t dq_sn, dq_sh, dk_sn, dk_sh, dv_sn, dv_sh;
  int64_t ldo, lddo;
  int64_t kv_rows;
  int32_t B, H, Nq, Nk;
  float scale;
} PxaAttnBwdArgs;
int pxa_flash_attn_d72_bwd_bf16(const PxaAttnBwdArgs* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PIXART_SM100_H_ */
