// xfm_b200 — host-side internals shared by the .cu translation units (not part of the C-ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "../../include/xfm_b200.h"

namespace xfm {

typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn get_tensor_map_encoder();
void set_error(const char* fmt, ...);
int num_sms();
void count_launch(int n = 1);
// Device word (one per device, zero until xfm_seed_salt_* is used) that every kernel drawing a dropout mask / a hard
// negative adds to its host-supplied seed.  A CUDA graph bakes kernel arguments, seeds included; advancing this word
// on the device between replays (xfm_seed_salt_bump, itself a graph node) gives every replayed step fresh masks while
// forward and backward of one step still agree.
const uint64_t* seed_salt_ptr();

int gemm_bf16(const xfm_gemm_params* p, cudaStream_t stream);
int attention_fwd(const xfm_attn_params* p, cudaStream_t s);
int attention_bwd(const xfm_attn_params* p, cudaStream_t s);
bool vit_attention_tc_supported(const xfm_attn_params* p, bool bwd = false);
int vit_attention_fwd_tc(const xfm_attn_params* p, cudaStream_t s);
int vit_attention_bwd_tc(const xfm_attn_params* p, cudaStream_t s);
// TMA maps of the tcgen05 attention kernels (attention_tc.cu): a bf16 activation of `cols` columns with a row stride of ld_elems
// elements, SWIZZLE_128B boxes of 64 columns.  2D: [rows] rows, boxes of box_rows rows.  3D: [samples][rows_per_sample] rows
// (samples sample_stride_rows rows apart, default rows_per_sample), boxes of 128 rows that clip at a sample's last row.
int encode_rows(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_rows);
int encode_rows_3d(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows_per_sample, uint64_t samples,
                   uint64_t ld_elems, uint64_t sample_stride_rows = 0);
// out / lse from nb key-block partials (bf16 [nb, B*L, H*64], f32 [nb, B, H, L]); attention_tc.cu
int launch_merge_parts(int nb, const void* part_out, const float* part_lse, void* out, int64_t o_stride, float* lse, int B, int H,
                       int L, cudaStream_t s);
// Key blocks of the tcgen05 attention kernels (attention_tc.cu, attention_xtc.cu).  Up to 208 keys are one block.  Longer rows
// are split into blocks of 192 keys (one launch each); a remainder of at most 16 keys joins the last block, a longer one is a
// block of its own.  577 keys (384 px) -> 192 / 192 / 193, 901 keys (480 px) -> 4 x 192 + 133.
struct KeyBlocks {
  static constexpr int KBS_MAX = 192;
  static constexpr int nb(int L) { return L <= 208 ? 1 : (L % KBS_MAX <= 16 ? L / KBS_MAX : L / KBS_MAX + 1); }
  static constexpr int kbs(int L) { return L <= 208 ? L : KBS_MAX; }                  // keys of every block but the last
  static constexpr int last(int L) { return L - (nb(L) - 1) * kbs(L); }             // keys of the last block
  static constexpr int lpad(int L) {                                                 // score columns: round16(widest block)
    return ((kbs(L) > last(L) ? kbs(L) : last(L)) + 15) / 16 * 16;
  }
};
static_assert(KeyBlocks::nb(577) == 3 && KeyBlocks::last(577) == 193 && KeyBlocks::lpad(577) == 208, "384 px key blocks");
static_assert(KeyBlocks::nb(901) == 5 && KeyBlocks::last(901) == 133 && KeyBlocks::lpad(901) == 192, "480 px key blocks");
static_assert(KeyBlocks::nb(197) == 1 && KeyBlocks::lpad(197) == 208, "224 px: one block");
// Partial-result blocks the forward of *p needs in part_out / part_lse when they are given (0: none; the chosen path writes
// out / lse directly).  Host-only: evaluates the same dispatch as attention_fwd.
int attention_fwd_parts(const xfm_attn_params* p);
bool cross_attention_tc_supported(const xfm_attn_params* p, bool bwd = false);
int cross_attention_fwd_tc(const xfm_attn_params* p, cudaStream_t s);
int cross_attention_bwd_tc(const xfm_attn_params* p, cudaStream_t s);
bool self_attention_tc_supported(const xfm_attn_params* p);
int self_attention_fwd_tc(const xfm_attn_params* p, cudaStream_t s);
int self_attention_bwd_tc(const xfm_attn_params* p, cudaStream_t s);
// Packed variable-length self-attention (attention_vtc.cu): host tile planner, forward, backward (delta kernel included).
int varlen_plan(const int32_t* lengths, int n, int32_t* cu_seqlens, int32_t* tiles, int32_t* n_tiles);
int varlen_attention_fwd(const xfm_varlen_params* p, cudaStream_t s);
int varlen_attention_bwd(const xfm_varlen_params* p, cudaStream_t s);

typedef __nv_bfloat16 bf16_t;
// delta[b, h, i] = rowsum(dO o O) of the attention backward (attention.cu)
int launch_attn_delta(const bf16_t* dout, int64_t do_stride, const bf16_t* out, int64_t o_stride, float* delta, int B, int H,
                      int Lq, cudaStream_t s);
int layernorm_fwd(const void* x, int x_dtype, const float* w, const float* b, void* y, int y_dtype, float* y2, float* stats,
                  int M, int D, float eps, cudaStream_t s);
int layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                  const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, int M, int D,
                  cudaStream_t s);
int layernorm_bwd_dense(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                        const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, bf16_t* dx16,
                        float* dbias, float drop_p, uint64_t drop_seed, int M, int D, cudaStream_t s);
int layerscale_bwd(const float* dxo, const bf16_t* z, const float* gamma, const float* rs, int rpg, bf16_t* dz, float* dgamma,
                   float* dbias, int M, int D, cudaStream_t s);
int colsum_bf16(const bf16_t* in, int64_t ld, float* out, int M, int N, cudaStream_t s);
int cast_f32_to_bf16(const float* in, bf16_t* out, size_t n, cudaStream_t s);
int cast_bf16_to_f32(const bf16_t* in, float* out, size_t n, cudaStream_t s);
int scale_by_scalar(const void* in, void* out, int dtype, const float* scalar, size_t n, cudaStream_t s);
int split_bf16x3(const float* in, bf16_t* out, int M, int K, int role, int act, cudaStream_t s);
int gelu_fwd(const void* x, int x_dtype, bf16_t* y, size_t n, cudaStream_t s);
int gelu_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, bf16_t* dx, size_t n, cudaStream_t s);
int dropout_apply(const void* x, int x_dtype, bf16_t* y, size_t n, float p, uint64_t seed, cudaStream_t s);
int roberta_embed_fwd(const int64_t* ids, const float* word, const float* pos, const float* type0, const float* w,
                      const float* b, bf16_t* y, float* pre_ln, float* stats, int32_t* pos_ids, int B, int L, int D,
                      int pad_id, int absolute_pos, float eps, cudaStream_t s);
int roberta_embed_bwd(const float* dpre, const int64_t* ids, const int32_t* pos_ids, float* dword, float* dpos,
                      float* dtype0, int rows, int D, int word_pad, int pos_pad, cudaStream_t s);
int im2col(const float* img, bf16_t* out, int B, int C, int H, int W, int P, const float* pre_mul, cudaStream_t s);
int assemble_tokens(const float* patch, const float* cls, const float* mask_token, const uint8_t* mask, const float* pos,
                    float* x, int B, int np, int D, cudaStream_t s);
int assemble_tokens_bwd(const float* dx, const uint8_t* mask, bf16_t* dpatch, float* dcls, float* dmask_token, int B, int np,
                        int D, cudaStream_t s);
int meanpool_fwd(bf16_t* y, float* y32, int B, int np, int D, cudaStream_t s);
int meanpool_bwd(const float* dout, float* dy, int B, int np, int D, cudaStream_t s);
int gather_rows(const void* in, int in_dtype, const int64_t* index, void* out, int out_dtype, int n, int D, cudaStream_t s);
int scatter_add_rows(const void* in, int in_dtype, const int64_t* index, float* out, int n, int D, cudaStream_t s);
int relpos_bias_fwd(const float* table, const int64_t* index, float* bias, int N, int ld, int H, cudaStream_t s);
int relpos_bias_bwd(const float* dbias, const int64_t* index, float* dtable, int N, int ld, int H, cudaStream_t s);
int batch_sum_bf16(const bf16_t* in, float* out, int B, size_t per, cudaStream_t s);
int ce_fwd(const float* logits, int64_t ld, const int64_t* labels, int R, int V, float* row_loss, float* lse, float* loss,
           float* count, cudaStream_t s);
int ce_bwd(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* count, const float* upstream,
           bf16_t* dlogits, int64_t ldd, int R, int V, cudaStream_t s);
int ce_bwd_rows(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* row_scale,
                const float* upstream, bf16_t* dlogits, int64_t ldd, int R, int V, cudaStream_t s);
int itc_loss_fused(const float* image_all, const float* text_all, int n, int E, const int64_t* idx_all, const float* temp,
                   int local_off, int local_n, float* work, float* loss, float* d_image_local, float* d_text_local,
                   float* dtemp, cudaStream_t s);
int hard_negatives(const float* image_feat, const float* text_feat, int B, int E, const float* temp, const int64_t* idx,
                   uint64_t seed, float* w_i2t, float* w_t2i, int64_t* text_neg, int64_t* image_neg, cudaStream_t s);
int vq_argmin(const float* z, const float* codebook, int64_t* ids, int R, int K, int C, cudaStream_t s);
int sgemm_f32(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbn, int64_t sbk, float* C, int64_t ldc,
              int M, int N, int K, const float* bias, int accumulate, cudaStream_t s);
int l2norm_fwd(const float* x, float* y, float* inv_norm, int R, int E, cudaStream_t s);
int l2norm_bwd(const float* dy, const float* y, const float* inv_norm, float* dx, int R, int E, cudaStream_t s);
int mim_mse(const float* x, const float* t, const uint8_t* mask, int B, int np, int D, int with_cls, float* count,
            float* loss, float* dx, cudaStream_t s);
int region_pool_fwd(const float* y, const int64_t* idx, const int64_t* atts, float* out, bf16_t* out16, int bsz, int N, int D,
                    cudaStream_t s);
int region_pool_bwd(const float* dout, const int64_t* idx, const int64_t* atts, float* dy, int bsz, int N, int D,
                    cudaStream_t s);
int sigmoid_fwd(const float* x, float* y, int n, cudaStream_t s);
int sigmoid_bwd(const float* dy, const float* y, float* dx, int n, cudaStream_t s);
int bbox_loss(const float* coord, const float* target, const float* is_image, int n, float* loss_bbox, float* loss_giou,
              float* d_bbox, float* d_giou, cudaStream_t s);
int axpby_scalars(const float* a, const float* sa, const float* b, const float* sb, float* out, int n, cudaStream_t s);
int resize_bicubic_u8(const uint8_t* src, const int64_t* desc, const int32_t* hb, const int32_t* hk, int KH, const int32_t* vb,
                      const int32_t* vk, int KV, uint8_t* tmp, uint8_t* out, int B, int max_rows, int OH, int OW, cudaStream_t s);
int resize_taps(const int64_t* desc, int32_t* hb, int32_t* hk, int KH, int32_t* vb, int32_t* vk, int KV, int B, int OH, int OW,
                cudaStream_t s);
int jpeg_plan(const void* const* blobs, const int64_t* nbytes, int n, int64_t* info, int threads);
size_t jpeg_desc_bytes();
int jpeg_tables(const void* const* blobs, const int64_t* nbytes, int n, const int64_t* info, const int64_t* offs, void* desc,
                int64_t* intervals, int threads);
int jpeg_decode(const uint8_t* bytes, const void* desc, const int64_t* intervals, int n, int16_t* coef, uint8_t* planes, uint8_t* out,
                int32_t* status, int64_t max_blocks, int max_w, int max_h, cudaStream_t s);
int image_u8_to_f32(const uint8_t* in, float* out, const uint8_t* flip, int B, int H, int W, const float* mean, const float* stdv,
                    cudaStream_t s);
int grad_sumsq(const float* g, const int32_t* chunk_seg, const uint8_t* seg_group, size_t nchunks, int32_t* seg_step,
               float* seg_bc, int nseg, const float* hp, float* out, int accumulate, cudaStream_t s);
int adamw_flat(float* P, const float* G, float* M, float* V, bf16_t* S, const int32_t* chunk_seg, const uint8_t* seg_group,
               const float* seg_bc, size_t nchunks, const float* sumsq, float* norm_out, const float* hp, cudaStream_t s);

}  // namespace xfm
