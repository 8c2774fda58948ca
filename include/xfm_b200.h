/*
 * xfm_b200 — C-ABI of the B200-native XFM hot path (libxfm_b200.so).
 *
 * Every entry point takes plain device pointers, sizes and a cudaStream_t (passed as void*);
 * no torch types cross this boundary.  All functions return 0 on success or a non-zero
 * cudaError_t / negative xfm error code; the Python host side (xfm_b200/lib.py) raises on != 0.
 *
 * The reference (zhangxinsong-nlp/XFM) is pure PyTorch: the "FFI" this library replaces is the
 * set of ATen calls made from the modules below (file:line relative to the reference root).
 * Each declaration cites the reference code whose arithmetic it reproduces.
 *
 * Conventions: activations are row-major [rows, features]; "bf16" = __nv_bfloat16; "f32" = float.
 */
#ifndef XFM_B200_H
#define XFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XFM_ERR_BAD_ARG (-2)
#define XFM_ERR_NO_DRIVER (-3)

/* ------------------------------------------------------------------------------------------------
 * Library
 * ---------------------------------------------------------------------------------------------- */
/* Returns the ABI version (monotonic integer). */
int xfm_version(void);
/* Resolves driver entry points and sets kernel attributes on the current device.  Must be called
 * once per process after the CUDA context exists. */
int xfm_init(void);
/* Number of kernels launched by this library since process start (all entry points). */
int64_t xfm_launch_count(void);
/* Human-readable description of the last error recorded by this library on this thread. */
const char* xfm_last_error(void);
/* Seed salt: a device-resident 64-bit word (per device, initially 0) that every kernel drawing random numbers (dropout in
 * the GEMM / attention / LayerNorm-backward kernels, hard-negative sampling) ADDS to the seed it is given.  CUDA-graph
 * replays repeat kernel arguments verbatim; xfm_seed_salt_bump (a one-thread kernel, capturable) advances the word so each
 * replayed step draws fresh masks, while the forward and backward kernels of one step still see the same value. */
int xfm_seed_salt_bump(uint64_t inc, void* stream);
int xfm_seed_salt_set(uint64_t value, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1 — tcgen05 GEMM with fused epilogue.
 *   C[M,N] = epilogue( A[M,K] · B[N,K]^T )
 * Replaces torch addmm / F.linear at: beit2.py:132,160 (qkv, proj), beit2.py:62-69 (Mlp),
 * xroberta.py:211,224-225,233-234 (query/key/value), :301 (SelfOutput.dense), :368 (Intermediate),
 * :382 (Output.dense), :1325-1333 (LM head), xfm.py:115-121,500-501 (heads), model_vqkd.py:86-90,
 * and their autograd backward (dgrad / wgrad) GEMMs.
 *
 * Operand layouts (bf16):
 *   a_mn_major == 0 : A stored [M, K] row-major, leading dimension lda (elements).
 *   a_mn_major == 1 : A stored [K, M] row-major (i.e. the transpose is in memory), lda = row stride.
 *   b_mn_major == 0 : B stored [N, K] row-major (a torch Linear weight), ldb.
 *   b_mn_major == 1 : B stored [K, N] row-major, ldb.
 * Leading dimensions must be multiples of 8 elements and base pointers 16-byte aligned (TMA).
 *
 * Epilogue, applied per element in this order (each step optional):
 *   v  = acc (+ bias[n])
 *   aux_out[m,n] = bf16(v)                         (pre-activation / pre-scale copy for backward)
 *   v  = act(v)            act: 0 none | 1 GELU(erf) | 2 v * GELU'(aux_in[m,n]) | 3 tanh
 *   v *= col_scale[n]                              (BEiT LayerScale gamma, beit2.py:204-205)
 *   v *= row_group_scale[m / rows_per_group]       (DropPath keep/keep_prob per sample)
 *   v  = dropout(v; p, seed, element index)        (xroberta.py:302,383)
 *   v += residual[m,n]                             (bf16 or f32)
 *   C[m,n] (+)= v                                  (bf16 or f32; accumulate / split-K use f32 atomics)
 * ---------------------------------------------------------------------------------------------- */
typedef struct xfm_gemm_params {
  const void* A;
  const void* B;
  void* C;
  int64_t lda, ldb, ldc;
  int32_t M, N, K;
  int32_t a_mn_major, b_mn_major;
  int32_t c_dtype;    /* 0 = bf16, 1 = f32 */
  int32_t split_k;    /* >= 1; > 1 requires c_dtype == 1 and accumulate == 1 (atomic f32 adds), and no bias, residual,
                         aux_out or act: every K slice applies the epilogue to its partial sum, so only col_scale,
                         row_group_scale and dropout (linear, same factor in every slice) may be combined with it */
  int32_t accumulate; /* 0: C = v, 1: C += v (f32 only) */
  int32_t act;        /* 0 none, 1 gelu, 2 dgelu(aux_in), 3 tanh */
  int32_t res_dtype;  /* 0 = bf16, 1 = f32 */
  int32_t rows_per_group;
  int32_t block_n;    /* 0 = auto, else 64 / 128 / 256 */
  const float* bias;
  const void* aux_in;
  void* aux_out;
  int64_t ld_aux_in, ld_aux_out, ld_res;
  const float* col_scale;
  const float* row_group_scale;
  const void* residual;
  float dropout_p;
  uint64_t dropout_seed;
} xfm_gemm_params;

int xfm_gemm_bf16(const xfm_gemm_params* p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2/K3/K4 — flash-style attention, head_dim 64 (scores never written to HBM).
 * Replaces beit2.py:133-159 (q*scale, q@k^T, + relative_position_bias, softmax, @v),
 * xroberta.py:237-284 (q/sqrt(d), + (1-m)*-1e4 mask, softmax, dropout, @v) and the cross-attention
 * call at xroberta.py:448-455, plus their autograd backward.
 *   q rows of sample b: q + (b*Lq + i)*q_stride + h*64;  k/v rows: k + (kv_row*Lk + j)*k_stride + h*64,
 *   kv_row = kv_index ? kv_index[b] : b  (several samples may attend to one image's K/V).
 *   logits = scale * q.k + bias[h,i,j] + kmask[b,j]
 * Backward needs lse (saved by the forward), a [B,H,Lq] f32 scratch `delta`, and writes bf16 dq/dk/dv.
 * ds_dump (optional, bf16 [B,H,Lq,ds_ld]) receives dS for the relative-position-bias gradient.
 * kv_offsets/kv_samples: CSR inverse of kv_index over the Bkv K/V rows (null = identity); the backward requires them
 * whenever kv_index is given.  K/V rows that no sample references get zero dk/dv.
 * ---------------------------------------------------------------------------------------------- */
typedef struct xfm_attn_params {
  const void *q, *k, *v;
  void* out;
  float* lse;
  const float* bias;
  const float* kmask;
  const int32_t* kv_index;
  int64_t q_stride, k_stride, v_stride, o_stride, bias_ld;
  int32_t B, H, Lq, Lk, head_dim, Bkv;
  float scale, dropout_p;
  uint64_t dropout_seed;
  /* backward */
  const void* dout;
  float* delta;
  void *dq, *dk, *dv, *ds_dump;
  int64_t do_stride, dq_stride, dk_stride, dv_stride, ds_ld;
  const int32_t* kv_offsets;
  const int32_t* kv_samples;
  /* BEiT relative position bias in closed form (beit2.py:94-116): table [ (2W-1)^2 + 3, H ] f32 and the window side W
   * (Lq = Lk = W*W + 1).  When given (and no mask / dropout / kv_index is), the forward runs on the tcgen05 kernel and
   * gathers the bias from the table instead of reading `bias`; `bias` must then hold the same values (backward). */
  const float* rel_table;
  int32_t rel_window;
  int32_t allow_tc; /* 1: use a tcgen05 / TMEM kernel when the problem fits one; 0: always the mma.sync kernels */
  /* Forward scratch for rows processed in key blocks (577 keys at 384 px: 3 blocks; 901 at 480 px: 5): bf16 [nb, B*Lq, H*64]
   * block-normalised partial outputs and f32 [nb, B, H, Lq] block lse, merged into out / lse by a last kernel, with nb from
   * xfm_attention_fwd_parts.  Without them these forwards run on the mma.sync kernel. */
  void* part_out;
  float* part_lse;
} xfm_attn_params;

int xfm_attention_fwd(const xfm_attn_params* p, void* stream);
int xfm_attention_bwd(const xfm_attn_params* p, void* stream);
/* Number of key blocks nb whose partial results the forward of *p would write to part_out / part_lse if they were given
 * (0: the path xfm_attention_fwd chooses needs no scratch).  Host-only, needs no device; part_out / part_lse are ignored. */
int xfm_attention_fwd_parts(const xfm_attn_params* p);

/* ------------------------------------------------------------------------------------------------
 * K4v — packed variable-length self-attention, head_dim 64 (RoBERTa sequence classification over GLUE batches, whose
 * sentences are padded to max_seq_length but mostly much shorter).  n sequences of 1..128 tokens are packed back to back,
 * with no padding rows: sequence s occupies rows [cu_seqlens[s], cu_seqlens[s+1]) of the q / k / v / out column slices
 * (T = cu_seqlens[n] rows); a query sees exactly the keys of its own sequence.
 *   logits = scale * q.k;  lse / delta f32 [H, T]
 * Tiles: a tile is a maximal run of consecutive sequences of at most 128 rows in total; tiles int32 [n_tiles + 1] holds
 * the first sequence of every tile, then n.  xfm_attention_varlen_plan computes cu_seqlens and tiles from the lengths
 * (host-only, no device; HOST pointers, cu_seqlens [n + 1], tiles room for n + 1 entries) and rejects lengths outside
 * 1..128.  The fwd / bwd entry points read DEVICE copies of both.
 * Dropout: element (s, h, query i, key j) is numbered ((s H + h) Lpad + i) ((Lpad + 1) & ~1) + j, the index the
 * xfm_attention_* kernels give it in the padded [n, Lpad] layout, so both draw the same mask for the same seed.
 * The backward writes delta itself (bf16 dq / dk / dv; every row is written exactly once: no accumulation).
 * ---------------------------------------------------------------------------------------------- */
typedef struct xfm_varlen_params {
  const void *q, *k, *v;
  void* out;
  float* lse;
  int64_t q_stride, k_stride, v_stride, o_stride;
  const int32_t* cu_seqlens;
  const int32_t* tiles;
  int32_t n, n_tiles, H, Lpad, T;
  float scale, dropout_p;
  uint64_t dropout_seed;
  /* backward */
  const void* dout;
  float* delta;
  void *dq, *dk, *dv;
  int64_t do_stride, dq_stride, dk_stride, dv_stride;
} xfm_varlen_params;

int xfm_attention_varlen_plan(const int32_t* lengths, int n, int32_t* cu_seqlens, int32_t* tiles, int32_t* n_tiles);
int xfm_attention_varlen_fwd(const xfm_varlen_params* p, void* stream);
int xfm_attention_varlen_bwd(const xfm_varlen_params* p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K6 — LayerNorm (torch layer_norm at beit2.py:201-205,458; xroberta.py:135,303,384,1328; xfm.py:118).
 * dtype codes: 0 = bf16, 1 = f32.  stats = [M,2] f32 (mean, rstd).  y2_f32: optional second f32 copy.
 * bwd: dx = LN'(dy) (+ add_in); dw/db accumulate (+=) with f32 atomics.
 * ---------------------------------------------------------------------------------------------- */
int xfm_layernorm_fwd(const void* x, int x_dtype, const float* w, const float* b, void* y, int y_dtype, float* y2_f32,
                      float* stats, int M, int D, float eps, void* stream);
int xfm_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                      const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, int M, int D,
                      void* stream);
/* LayerNorm backward of a RobertaSelfOutput / RobertaOutput site (xroberta.py:300-304,381-385: LayerNorm(dropout(dense(.)) +
 * residual)) that also emits what the dense layer's own backward needs: dx16 = bf16(mask * dx / (1 - drop_p)) with the
 * forward's dropout mask re-derived from (drop_seed, row * D + col) as in the GEMM epilogue, and dbias += column sums of
 * dx16 (the dense bias gradient).  dx (f32 / bf16) is still written: it is the gradient of the residual branch. */
int xfm_layernorm_bwd_dense(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                            const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, void* dx16_bf16,
                            float* dbias, float drop_p, uint64_t drop_seed, int M, int D, void* stream);
/* LayerScale / DropPath backward (beit2.py:204-205): dz = dx_out*gamma*rs; dgamma += sum dx_out*rs*z; dbias += sum dz. */
int xfm_layerscale_bwd(const float* dx_out, const void* z_bf16, const float* gamma, const float* row_group_scale,
                       int rows_per_group, void* dz_bf16, float* dgamma, float* dbias, int M, int D, void* stream);
/* out[c] += sum_rows in[row,c]  (bias gradients of every Linear). */
int xfm_colsum_bf16(const void* in, int64_t ld, float* out, int M, int N, void* stream);
int xfm_cast_f32_to_bf16(const float* in, void* out, size_t n, void* stream);
int xfm_cast_bf16_to_f32(const void* in, float* out, size_t n, void* stream);
int xfm_scale_by_scalar(const void* in, void* out, int dtype, const float* scalar, size_t n, void* stream); /* out may alias in */
/* fp32-grade GEMM operands for the bf16 tensor cores: every f32 row [K] becomes a bf16 row [6K] holding the three-term
 * split x = h + m + l in the block order l,m,h,m,h,h (role 0, left operand) or h,m,l,h,m,h (role 1, right operand), so that
 * xfm_gemm_bf16 over K' = 6K sums the six products of order <= 2, smallest first (the tensor-core accumulator truncates:
 * error ~ (K/16) 2^-24 of max|C|, the level of an fp32 library GEMM).  act: 0 none, 1 tanh first.
 * Replaces the autocast(enabled=False) fp32 Linear-Tanh-Linear of model_vqkd.py:86-90,154-155 (encode_task_layer) and the
 * fp32 similarity of xfm.py:696-697. */
int xfm_split_bf16x3(const float* in_f32, void* out_bf16, int M, int K, int role, int act, void* stream);

/* Stand-alone GELU(erf) forward / backward (xfm.py:115-121 ITM head; xroberta.py:1325-1328 LM head) and the
 * dropout mask re-application used by the backward of the GEMM dropout epilogue (same (seed, row*N+col) stream). */
int xfm_gelu_fwd(const void* x, int x_dtype, void* y_bf16, size_t n, void* stream);
int xfm_gelu_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, void* dx_bf16, size_t n, void* stream);
int xfm_dropout_apply(const void* x, int x_dtype, void* y_bf16, size_t n, float p, uint64_t seed, void* stream);

/* K7 — text embeddings (word + token-type row 0 + position) + LayerNorm and the scatter-add backward.
 * absolute_pos = 0: RoBERTa position ids cumsum(ids != pad) * (ids != pad) + pad (xroberta.py:104-137, :1747-1757);
 * absolute_pos = 1: BERT position ids 0..L-1 (xbert.py:167-221).  word_pad / pos_pad: padding_idx rows of the word / position
 * tables that receive no gradient (-1 = none): RoBERTa pad_id for both, BERT pad_token_id for the words only. */
int xfm_roberta_embed_fwd(const int64_t* ids, const float* word, const float* pos, const float* type0, const float* ln_w,
                          const float* ln_b, void* y_bf16, float* pre_ln, float* stats, int32_t* pos_ids, int B, int L,
                          int D, int pad_id, int absolute_pos, float eps, void* stream);
int xfm_roberta_embed_bwd(const float* dpre, const int64_t* ids, const int32_t* pos_ids, float* dword, float* dpos,
                          float* dtype0, int rows, int D, int word_pad, int pos_pad, void* stream);

/* K8/K9 — patch-embed im2col (beit2.py:229), token assembly with mask-token blend + CLS (+ abs pos) (beit2.py:438-449),
 * mean-pool pseudo-CLS (beit2.py:456-466) and their backward. */
/* pre_mul: null, or a DEVICE scalar m: pixels become x * m / 127.5 - 1 before the cast (model_vqkd.py:125-131; m is the
 * result of the reference's data-dependent `if data.max() <= 1` rule, evaluated on the device). */
int xfm_im2col(const float* image, void* out_bf16, int B, int C, int H, int W, int P, const float* pre_mul, void* stream);
int xfm_assemble_tokens(const float* patch, const float* cls, const float* mask_token, const uint8_t* mask, const float* pos,
                        float* x, int B, int np, int D, void* stream);
int xfm_assemble_tokens_bwd(const float* dx, const uint8_t* mask, void* dpatch_bf16, float* dcls, float* dmask_token, int B,
                            int np, int D, void* stream);
int xfm_meanpool_fwd(void* y_bf16, float* y_f32, int B, int np, int D, void* stream);
int xfm_meanpool_bwd(const float* dout, float* dy, int B, int np, int D, void* stream);

/* K12 — row gather / scatter-add (xfm.py:758-786 negatives, xroberta.py:1215-1216 masked positions, xfm.py:629 masked patches). */
int xfm_gather_rows(const void* in, int in_dtype, const int64_t* index, void* out, int out_dtype, int n, int D, void* stream);
int xfm_scatter_add_rows(const void* in, int in_dtype, const int64_t* index, float* out, int n, int D, void* stream);

/* Relative position bias gather (beit2.py:139-144) and its backward; batch reduction of the attention dS dump. */
int xfm_relpos_bias_fwd(const float* table, const int64_t* index, float* bias, int N, int ld, int H, void* stream);
int xfm_relpos_bias_bwd(const float* dbias, const int64_t* index, float* dtable, int N, int ld, int H, void* stream);
int xfm_batch_sum_bf16(const void* in, float* out, int B, size_t per, void* stream);

/* K13/K14 — softmax cross-entropy with ignore_index=-100 (xroberta.py:1298-1299; xfm.py:629,800-802).
 * fwd: row_loss[R], lse[R], *loss = mean over valid rows, *count = #valid.  bwd: dlogits (bf16, ld = ldd) =
 * (softmax - onehot) * (*upstream) / count. */
int xfm_ce_fwd(const float* logits, int64_t ld, const int64_t* labels, int R, int V, float* row_loss, float* lse, float* loss,
               float* count, void* stream);
int xfm_ce_bwd(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* count,
               const float* upstream, void* dlogits_bf16, int64_t ldd, int R, int V, void* stream);
/* CrossEntropyLoss(reduction='none') followed by a weighted sum over rows — the VQA answer loss (xroberta.py:1104-1110,
 * model_generation.py:130-131): dlogits = (softmax - onehot) * row_scale[row] * (*upstream); rows with label < 0 get 0. */
int xfm_ce_bwd_rows(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* row_scale,
                    const float* upstream, void* dlogits_bf16, int64_t ldd, int R, int V, void* stream);

/* K10 — ITC (xfm.py:683-715) on gathered features [n,E] f32: loss and, in the same call, the gradients wrt the LOCAL
 * slice [local_off, local_off+local_n) of image/text features (AllGather.backward, xfm.py:93-98) and wrt temp, for an
 * upstream gradient of 1.  work: f32 scratch of xfm_itc_workspace(n) elements. */
size_t xfm_itc_workspace(int n);
int xfm_itc_loss_fused(const float* image_all, const float* text_all, int n, int E, const int64_t* idx_all, const float* temp,
                       int local_off, int local_n, float* work, float* loss, float* d_image_local, float* d_text_local,
                       float* dtemp, void* stream);

/* K11 — ITM hard negatives (xfm.py:717-746): weights (optional outputs, [B,B] f32) and one on-device draw per row. */
int xfm_hard_negatives(const float* image_feat, const float* text_feat, int B, int E, const float* temp, const int64_t* idx,
                       uint64_t seed, float* w_i2t, float* w_t2i, int64_t* text_neg_idx, int64_t* image_neg_idx, void* stream);

/* K15 — VQ-KD codebook argmin (norm_ema_quantizer.py:149-162): z [R,32] f32 (un-normalised), codebook [K,32] f32,
 * ids [R] int64.  Bit-exact contract: exact fp32 arithmetic, first index on ties. */
int xfm_vq_argmin(const float* z, const float* codebook, int64_t* ids, int R, int K, int C, void* stream);

/* Exact-fp32 small GEMM with element strides: C[m,n] (+)= sum_k A[m*sam + k*sak] * B[n*sbn + k*sbk] (+ bias[n]).
 * Used for the latency-bound [B,768]x[768,256] ITC projections (xfm.py:614-621, self.vision_proj / self.text_proj) and
 * their backward, where bf16 operand rounding would be amplified by 1/temp in the contrastive logits. */
int xfm_sgemm_f32(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbn, int64_t sbk, float* C, int64_t ldc,
                  int M, int N, int K, const float* bias, int accumulate, void* stream);

/* ITC feature normalisation (F.normalize, xfm.py:614-621): y = x / max(||x||_2, 1e-12), inv_norm[R] saved for the
 * backward dx = (dy - y <y,dy>) * inv_norm. */
int xfm_l2norm_fwd(const float* x, float* y, float* inv_norm, int R, int E, void* stream);
int xfm_l2norm_bwd(const float* dy, const float* y, const float* inv_norm, float* dx, int R, int E, void* stream);

/* K14 — MIM loss, MSE variant (xfm.py:631-635): x, t f32 [B, np+1, D]; mask u8 [B, np].  Writes *loss, *count (number
 * of masked patches) and dx = dloss/dx for an upstream gradient of 1 (zero outside the selected rows). */
int xfm_mim_mse(const float* x, const float* t, const uint8_t* mask, int B, int np, int D, int with_cls, float* count,
                float* loss, float* dx, void* stream);

/* Region / bounding-box branch (SURVEY.md §8 f4).
 * xfm_region_pool_fwd: models/beit2.py:468-475 — y f32 [n_img, N, D] vision tokens (token 0 = full-image mean), idx int64
 *   [bsz] sample -> image, atts int64 [bsz, N] region masks: out[b, 1+j] = y[idx[b], 1+j]; out[b, 0] = the atts-weighted mean
 *   of those patch tokens.  out_bf16 (optional) receives the same values in bf16.  _bwd accumulates (+=, atomics) into dy.
 * xfm_sigmoid_fwd/bwd: bbox_head(...).sigmoid() (models/xfm.py:852-853).
 * xfm_bbox_loss: models/xfm.py:815-840 with models/box_ops.py (cxcywh -> xyxy, generalized IoU, diagonal only): L1 and
 *   1 - GIoU summed over the kept samples / num_boxes; is_image f32 [n] or null; a degenerate box anywhere zeroes the GIoU
 *   loss (decided on the device).  d_bbox / d_giou [n, 4]: gradients wrt coord for upstream gradients of 1.
 * xfm_axpby_scalars: out = a * sa[0] + b * sb[0] (sa / sb device scalars, null = 0). */
int xfm_region_pool_fwd(const float* y, const int64_t* idx, const int64_t* atts, float* out, void* out_bf16, int bsz, int N,
                        int D, void* stream);
int xfm_region_pool_bwd(const float* dout, const int64_t* idx, const int64_t* atts, float* dy, int bsz, int N, int D,
                        void* stream);
int xfm_sigmoid_fwd(const float* x, float* y, int n, void* stream);
int xfm_sigmoid_bwd(const float* dy, const float* y, float* dx, int n, void* stream);
int xfm_bbox_loss(const float* coord, const float* target, const float* is_image, int n, float* loss_bbox, float* loss_giou,
                  float* d_bbox, float* d_giou, void* stream);
int xfm_axpby_scalars(const float* a, const float* sa, const float* b, const float* sb, float* out, int n, void* stream);

/* Batch feeder, device half (SURVEY.md §8 f4, loader side): the tail of the reference's image transform —
 * transforms.ToTensor() + transforms.Normalize(mean, std) (dataset/__init__.py:26-35; the same two lines close every Compose
 * there) and optionally the RandomHorizontalFlip of that Compose — on the uint8 crops the decode workers produce.
 *   in   u8  [B, H, W, 3]  device, 4-byte aligned (HWC as PIL / numpy hand it over); W % 4 == 0
 *   out  f32 [B, 3, H, W]  device, 16-byte aligned: out[b, c, y, x] = (in[b, y, x', c] / 255 - mean[c]) / std[c], IEEE
 *                          round-to-nearest divisions as in the CPU transform (bit-identical results)
 *   flip u8  [B] or null   1 = x' = W - 1 - x (torchvision hflip), 0 = x' = x
 *   mean, stdv             HOST pointers to 3 floats each (baked into the launch; graph-capturable) */
int xfm_image_u8_to_f32(const uint8_t* in, float* out, const uint8_t* flip, int B, int H, int W, const float* mean,
                        const float* stdv, void* stream);
/* Crop + bicubic resize of B ragged uint8 RGB images to [OH, OW]: RandomResizedCrop / Resize with InterpolationMode.BICUBIC
 * (dataset/__init__.py:28-30,63-67) and crop + resize of dataset/pretrain_dataset.py:470-483, i.e. Pillow's ImagingResample
 * (third party, reached through torchvision): horizontal then vertical pass in 8.22 fixed point with a uint8 intermediate.
 *   src   u8 packed images, each [h, w, 3]           desc  int64 [B, 8]: {byte offset in src, image width, crop x0, crop y0,
 *   hb/vb int32 [B, OW|OH, 2]: first tap, tap count        crop width, crop height, byte offset of the image's rows in tmp, 0}
 *   hk/vk int32 [B, OW|OH, KH|KV]: taps * 2^22 (Pillow's precompute_coeffs + normalize_coeffs_8bpc, computed on the host)
 *   tmp   u8 scratch, sum_b crop_height_b * OW * 3 bytes   out   u8 [B, OH, OW, 3]      max_rows = max_b crop height
 * All pointers are device pointers.  Bit-identical to PIL.Image.crop(box).resize((OW, OH), BICUBIC). */
/* Host-only helper of the batch feeder: copy n byte ranges back to back into dst (normally pinned staging memory) with up to
 * `threads` threads (equal byte spans across segment boundaries).  No CUDA call; all pointers are HOST pointers. */
int xfm_host_pack(const void* const* srcs, const int64_t* nbytes, int n, void* dst, int threads);
/* xfm_resize_taps fills hb / hk / vb / vk on the device from desc (crop width / height per image): Pillow's precompute_coeffs +
 * normalize_coeffs_8bpc for BICUBIC in float64 with explicitly rounded operations — the integers Pillow computes on the host.
 * KH / KV >= ceil(2 * max(crop / out, 1)) * 2 + 1 for every image (the caller sizes the tables). */
int xfm_resize_taps(const int64_t* desc, int32_t* hb, int32_t* hk, int KH, int32_t* vb, int32_t* vk, int KV, int B, int OH, int OW,
                    void* stream);
int xfm_resize_bicubic_u8(const uint8_t* src, const int64_t* desc, const int32_t* hb, const int32_t* hk, int KH, const int32_t* vb,
                          const int32_t* vk, int KV, uint8_t* tmp, uint8_t* out, int B, int max_rows, int OH, int OW, void* stream);

/* Baseline JPEG decode of the batch feeder (csrc/jpeg.cu): file bytes -> RGB, bit-identical to Pillow's
 * Image.open(f).convert("RGB") over libjpeg-turbo (jdhuff.c decode_mcu, jidctint.c ISLOW as its SIMD code computes it,
 * jdsample.c h2v1 / h2v2 fancy upsampling, jdcolor.c ycc_rgb_convert) for the device subset: SOF0 / SOF1 8-bit, one
 * sequential Huffman scan, grayscale or YCbCr (libjpeg's default_decompress_parms rule), sampling 4:4:4 / 4:2:2 / 4:2:0,
 * with or without DRI.  Every other stream gets a non-zero status and is decoded by the caller (feed.py: Pillow).
 * Two host-only calls (no CUDA call; all pointers HOST pointers, images spread over up to `threads` threads):
 *   xfm_jpeg_plan    info int64 [n, XFM_JPEG_INFO] = {status (0 = device path), width, height, restart intervals,
 *                    coefficient blocks, component plane bytes, 0, 0}; width / height are 0 when the header was not read.
 *   xfm_jpeg_tables  offs int64 [n, 4] = {byte offset of the blob in the device byte buffer, first coefficient block, first
 *                    plane byte (multiple of 8), byte offset of the image in out}; fills desc (n * xfm_jpeg_desc_bytes(),
 *                    16-byte aligned: Huffman look-up tables, natural-order quantisation tables, geometry) and intervals
 *                    int64 [sum of info[:, 3], 2] (byte range of every restart interval in the device byte buffer).
 * xfm_jpeg_decode (device pointers; three launches on `stream`, graph-capturable):
 *   bytes    u8 packed blobs           coef   int16 [sum blocks, 64] scratch (16-byte aligned)
 *   planes   u8 scratch, sum plane bytes                out  u8: image b is [height, width, 3] at byte offs[b][3]
 *   status   int32 [n]: 0 on entry for device-path images; the entropy stage ORs in a code (invalid Huffman code 16, run
 *            past coefficient 63 32, data ending before the interval's last MCU 64, unexpected marker 128) — such an image
 *            must be decoded again by the caller.  Images with info status != 0 are not touched (out included).
 *   max_blocks / max_w / max_h: the largest coefficient block count, width and height of a device-path image. */
#define XFM_JPEG_INFO 8
int xfm_jpeg_plan(const void* const* blobs, const int64_t* nbytes, int n, int64_t* info, int threads);
size_t xfm_jpeg_desc_bytes(void);
int xfm_jpeg_tables(const void* const* blobs, const int64_t* nbytes, int n, const int64_t* info, const int64_t* offs, void* desc,
                    int64_t* intervals, int threads);
int xfm_jpeg_decode(const uint8_t* bytes, const void* desc, const int64_t* intervals, int n, int16_t* coef, uint8_t* planes,
                    uint8_t* out, int32_t* status, int64_t max_blocks, int max_w, int max_h, void* stream);

/* Flat-buffer optimizer step (accelerators/ddp_accelerator.py:89-98 clip_grad_norm_ + optimizer.step with the
 * transformers AdamW of optim.py:4-50).  P/G/M/V: f32 buffers of nchunks*64 elements, S: bf16 shadow (may be null).
 *   chunk_seg[nchunks] int32  static: parameter segment of every 64-element chunk, -1 = frozen / padding (never touched)
 *   seg_group[nseg]    uint8  per step: hyper-parameter group 0..3 of the segment ({decay, no-decay} x {lr, lr*mult},
 *                             optim.py:10-46), 255 = no gradient since the last zero_grad (skipped like a None grad)
 *   seg_step[nseg]     int32  device-resident per-parameter step counters (AdamW's state['step']), advanced by
 *                             xfm_grad_sumsq for every live segment
 *   seg_bc[nseg]       float2 bias corrections (1 - beta1^t, 1 - beta2^t) written by xfm_grad_sumsq, read by the update
 *   hp                 16 f32 in DEVICE memory: lr[4] | weight_decay[4] | beta1 beta2 eps max_grad_norm | grad_mul
 *                             correct_bias 0 0   (max_grad_norm <= 0: no clipping; grad_mul = 1/world for DDP averaging)
 * xfm_grad_sumsq: *out (+)= sum of g^2 over live chunks (deterministic order).  xfm_adamw_flat: if sumsq != null the
 * gradient is scaled by grad_mul and clipped to max_grad_norm (total norm written to *norm_out when non-null). */
int xfm_grad_sumsq(const float* g, const int32_t* chunk_seg, const uint8_t* seg_group, size_t nchunks, int32_t* seg_step,
                   float* seg_bc, int nseg, const float* hp, float* out, int accumulate, void* stream);
int xfm_adamw_flat(float* P, const float* G, float* M, float* V, void* S_bf16, const int32_t* chunk_seg,
                   const uint8_t* seg_group, const float* seg_bc, size_t nchunks, const float* sumsq, float* norm_out,
                   const float* hp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XFM_B200_H */
