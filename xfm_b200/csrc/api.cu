// xfm_b200 — extern "C" entry points (the C-ABI declared in include/xfm_b200.h).
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <thread>
#include <vector>
#include "internal.h"

namespace xfm {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};
static TensorMapEncodeFn g_encode = nullptr;
static int g_num_sms = 0;
static uint64_t* g_salt[64] = {nullptr};

__global__ void seed_salt_bump_kernel(uint64_t* salt, uint64_t inc) { *salt += inc; }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
TensorMapEncodeFn get_tensor_map_encoder() { return g_encode; }
int num_sms() { return g_num_sms > 0 ? g_num_sms : 148; }
const uint64_t* seed_salt_ptr() {
  int dev = 0;
  cudaGetDevice(&dev);
  return g_salt[dev & 63];
}

}  // namespace xfm

using namespace xfm;

extern "C" {

int xfm_version(void) { return 1; }

int xfm_init(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return (int)e; }
  e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) { set_error("cudaDeviceGetAttribute: %s", cudaGetErrorString(e)); return (int)e; }
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled entry point not available");
      return XFM_ERR_NO_DRIVER;
    }
    g_encode = (TensorMapEncodeFn)fn;
  }
  if (!g_salt[dev & 63]) {
    e = cudaMalloc((void**)&g_salt[dev & 63], sizeof(uint64_t));
    if (e != cudaSuccess) { set_error("cudaMalloc(seed salt): %s", cudaGetErrorString(e)); return (int)e; }
    e = cudaMemset(g_salt[dev & 63], 0, sizeof(uint64_t));
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

int xfm_seed_salt_bump(uint64_t inc, void* stream) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!g_salt[dev & 63]) { set_error("xfm_init was not called on this device"); return XFM_ERR_BAD_ARG; }
  seed_salt_bump_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(g_salt[dev & 63], inc);
  count_launch();
  return (int)cudaGetLastError();
}
int xfm_seed_salt_set(uint64_t value, void* stream) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!g_salt[dev & 63]) { set_error("xfm_init was not called on this device"); return XFM_ERR_BAD_ARG; }
  return (int)cudaMemcpyAsync(g_salt[dev & 63], &value, sizeof(value), cudaMemcpyHostToDevice, (cudaStream_t)stream);
}

int64_t xfm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* xfm_last_error(void) { return g_err; }

#define ST ((cudaStream_t)stream)
#define BF(p) ((bf16_t*)(p))
#define CBF(p) ((const bf16_t*)(p))

int xfm_gemm_bf16(const xfm_gemm_params* p, void* stream) { return gemm_bf16(p, ST); }
int xfm_attention_fwd(const xfm_attn_params* p, void* stream) { return attention_fwd(p, ST); }
int xfm_attention_bwd(const xfm_attn_params* p, void* stream) { return attention_bwd(p, ST); }
int xfm_attention_fwd_parts(const xfm_attn_params* p) { return attention_fwd_parts(p); }
int xfm_attention_varlen_plan(const int32_t* lengths, int n, int32_t* cu_seqlens, int32_t* tiles, int32_t* n_tiles) {
  return varlen_plan(lengths, n, cu_seqlens, tiles, n_tiles);
}
int xfm_attention_varlen_fwd(const xfm_varlen_params* p, void* stream) { return varlen_attention_fwd(p, ST); }
int xfm_attention_varlen_bwd(const xfm_varlen_params* p, void* stream) { return varlen_attention_bwd(p, ST); }

int xfm_layernorm_fwd(const void* x, int x_dtype, const float* w, const float* b, void* y, int y_dtype, float* y2_f32,
                      float* stats, int M, int D, float eps, void* stream) {
  return layernorm_fwd(x, x_dtype, w, b, y, y_dtype, y2_f32, stats, M, D, eps, ST);
}
int xfm_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                      const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, int M, int D,
                      void* stream) {
  return layernorm_bwd(dy, dy_dtype, x, x_dtype, stats, w, add_in, add_dtype, dx, dx_dtype, dw, db, M, D, ST);
}
int xfm_layernorm_bwd_dense(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* stats, const float* w,
                            const void* add_in, int add_dtype, void* dx, int dx_dtype, float* dw, float* db, void* dx16,
                            float* dbias, float drop_p, uint64_t drop_seed, int M, int D, void* stream) {
  return layernorm_bwd_dense(dy, dy_dtype, x, x_dtype, stats, w, add_in, add_dtype, dx, dx_dtype, dw, db, BF(dx16), dbias, drop_p,
                             drop_seed, M, D, ST);
}
int xfm_layerscale_bwd(const float* dx_out, const void* z, const float* gamma, const float* rs, int rpg, void* dz, float* dgamma,
                       float* dbias, int M, int D, void* stream) {
  return layerscale_bwd(dx_out, CBF(z), gamma, rs, rpg, BF(dz), dgamma, dbias, M, D, ST);
}
int xfm_colsum_bf16(const void* in, int64_t ld, float* out, int M, int N, void* stream) {
  return colsum_bf16(CBF(in), ld, out, M, N, ST);
}
int xfm_cast_f32_to_bf16(const float* in, void* out, size_t n, void* stream) { return cast_f32_to_bf16(in, BF(out), n, ST); }
int xfm_cast_bf16_to_f32(const void* in, float* out, size_t n, void* stream) { return cast_bf16_to_f32(CBF(in), out, n, ST); }
int xfm_scale_by_scalar(const void* in, void* out, int dtype, const float* scalar, size_t n, void* stream) {
  return scale_by_scalar(in, out, dtype, scalar, n, ST);
}
int xfm_split_bf16x3(const float* in, void* out, int M, int K, int role, int act, void* stream) {
  return split_bf16x3(in, BF(out), M, K, role, act, ST);
}
int xfm_gelu_fwd(const void* x, int x_dtype, void* y, size_t n, void* stream) { return gelu_fwd(x, x_dtype, BF(y), n, ST); }
int xfm_gelu_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, void* dx, size_t n, void* stream) {
  return gelu_bwd(dy, dy_dtype, x, x_dtype, BF(dx), n, ST);
}
int xfm_dropout_apply(const void* x, int x_dtype, void* y, size_t n, float p, uint64_t seed, void* stream) {
  return dropout_apply(x, x_dtype, BF(y), n, p, seed, ST);
}
int xfm_roberta_embed_fwd(const int64_t* ids, const float* word, const float* pos, const float* type0, const float* ln_w,
                          const float* ln_b, void* y, float* pre_ln, float* stats, int32_t* pos_ids, int B, int L, int D,
                          int pad_id, int absolute_pos, float eps, void* stream) {
  return roberta_embed_fwd(ids, word, pos, type0, ln_w, ln_b, BF(y), pre_ln, stats, pos_ids, B, L, D, pad_id, absolute_pos, eps, ST);
}
int xfm_roberta_embed_bwd(const float* dpre, const int64_t* ids, const int32_t* pos_ids, float* dword, float* dpos,
                          float* dtype0, int rows, int D, int word_pad, int pos_pad, void* stream) {
  return roberta_embed_bwd(dpre, ids, pos_ids, dword, dpos, dtype0, rows, D, word_pad, pos_pad, ST);
}
int xfm_im2col(const float* image, void* out, int B, int C, int H, int W, int P, const float* pre_mul, void* stream) {
  return im2col(image, BF(out), B, C, H, W, P, pre_mul, ST);
}
int xfm_assemble_tokens(const float* patch, const float* cls, const float* mask_token, const uint8_t* mask, const float* pos,
                        float* x, int B, int np, int D, void* stream) {
  return assemble_tokens(patch, cls, mask_token, mask, pos, x, B, np, D, ST);
}
int xfm_assemble_tokens_bwd(const float* dx, const uint8_t* mask, void* dpatch, float* dcls, float* dmask_token, int B, int np,
                            int D, void* stream) {
  return assemble_tokens_bwd(dx, mask, BF(dpatch), dcls, dmask_token, B, np, D, ST);
}
int xfm_meanpool_fwd(void* y, float* y_f32, int B, int np, int D, void* stream) { return meanpool_fwd(BF(y), y_f32, B, np, D, ST); }
int xfm_meanpool_bwd(const float* dout, float* dy, int B, int np, int D, void* stream) { return meanpool_bwd(dout, dy, B, np, D, ST); }
int xfm_gather_rows(const void* in, int in_dtype, const int64_t* index, void* out, int out_dtype, int n, int D, void* stream) {
  return gather_rows(in, in_dtype, index, out, out_dtype, n, D, ST);
}
int xfm_scatter_add_rows(const void* in, int in_dtype, const int64_t* index, float* out, int n, int D, void* stream) {
  return scatter_add_rows(in, in_dtype, index, out, n, D, ST);
}
int xfm_relpos_bias_fwd(const float* table, const int64_t* index, float* bias, int N, int ld, int H, void* stream) {
  return relpos_bias_fwd(table, index, bias, N, ld, H, ST);
}
int xfm_relpos_bias_bwd(const float* dbias, const int64_t* index, float* dtable, int N, int ld, int H, void* stream) {
  return relpos_bias_bwd(dbias, index, dtable, N, ld, H, ST);
}
int xfm_batch_sum_bf16(const void* in, float* out, int B, size_t per, void* stream) { return batch_sum_bf16(CBF(in), out, B, per, ST); }
int xfm_ce_fwd(const float* logits, int64_t ld, const int64_t* labels, int R, int V, float* row_loss, float* lse, float* loss,
               float* count, void* stream) {
  return ce_fwd(logits, ld, labels, R, V, row_loss, lse, loss, count, ST);
}
int xfm_ce_bwd(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* count,
               const float* upstream, void* dlogits, int64_t ldd, int R, int V, void* stream) {
  return ce_bwd(logits, ld, labels, lse, count, upstream, BF(dlogits), ldd, R, V, ST);
}
int xfm_ce_bwd_rows(const float* logits, int64_t ld, const int64_t* labels, const float* lse, const float* row_scale,
                    const float* upstream, void* dlogits, int64_t ldd, int R, int V, void* stream) {
  return ce_bwd_rows(logits, ld, labels, lse, row_scale, upstream, BF(dlogits), ldd, R, V, ST);
}
size_t xfm_itc_workspace(int n) { return (size_t)2 * n * n + (size_t)3 * n; }
int xfm_itc_loss_fused(const float* image_all, const float* text_all, int n, int E, const int64_t* idx_all, const float* temp,
                       int local_off, int local_n, float* work, float* loss, float* d_image_local, float* d_text_local,
                       float* dtemp, void* stream) {
  return itc_loss_fused(image_all, text_all, n, E, idx_all, temp, local_off, local_n, work, loss, d_image_local, d_text_local,
                        dtemp, ST);
}
int xfm_hard_negatives(const float* image_feat, const float* text_feat, int B, int E, const float* temp, const int64_t* idx,
                       uint64_t seed, float* w_i2t, float* w_t2i, int64_t* text_neg_idx, int64_t* image_neg_idx, void* stream) {
  return hard_negatives(image_feat, text_feat, B, E, temp, idx, seed, w_i2t, w_t2i, text_neg_idx, image_neg_idx, ST);
}
int xfm_vq_argmin(const float* z, const float* codebook, int64_t* ids, int R, int K, int C, void* stream) {
  return vq_argmin(z, codebook, ids, R, K, C, ST);
}
int xfm_sgemm_f32(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbn, int64_t sbk, float* C, int64_t ldc,
                  int M, int N, int K, const float* bias, int accumulate, void* stream) {
  return sgemm_f32(A, sam, sak, B, sbn, sbk, C, ldc, M, N, K, bias, accumulate, ST);
}
int xfm_l2norm_fwd(const float* x, float* y, float* inv_norm, int R, int E, void* stream) {
  return l2norm_fwd(x, y, inv_norm, R, E, ST);
}
int xfm_l2norm_bwd(const float* dy, const float* y, const float* inv_norm, float* dx, int R, int E, void* stream) {
  return l2norm_bwd(dy, y, inv_norm, dx, R, E, ST);
}
int xfm_mim_mse(const float* x, const float* t, const uint8_t* mask, int B, int np, int D, int with_cls, float* count,
                float* loss, float* dx, void* stream) {
  return mim_mse(x, t, mask, B, np, D, with_cls, count, loss, dx, ST);
}
int xfm_region_pool_fwd(const float* y, const int64_t* idx, const int64_t* atts, float* out, void* out_bf16, int bsz, int N,
                        int D, void* stream) {
  return region_pool_fwd(y, idx, atts, out, BF(out_bf16), bsz, N, D, ST);
}
int xfm_region_pool_bwd(const float* dout, const int64_t* idx, const int64_t* atts, float* dy, int bsz, int N, int D,
                        void* stream) {
  return region_pool_bwd(dout, idx, atts, dy, bsz, N, D, ST);
}
int xfm_sigmoid_fwd(const float* x, float* y, int n, void* stream) { return sigmoid_fwd(x, y, n, ST); }
int xfm_sigmoid_bwd(const float* dy, const float* y, float* dx, int n, void* stream) { return sigmoid_bwd(dy, y, dx, n, ST); }
int xfm_bbox_loss(const float* coord, const float* target, const float* is_image, int n, float* loss_bbox, float* loss_giou,
                  float* d_bbox, float* d_giou, void* stream) {
  return bbox_loss(coord, target, is_image, n, loss_bbox, loss_giou, d_bbox, d_giou, ST);
}
int xfm_axpby_scalars(const float* a, const float* sa, const float* b, const float* sb, float* out, int n, void* stream) {
  return axpby_scalars(a, sa, b, sb, out, n, ST);
}
int xfm_resize_bicubic_u8(const uint8_t* src, const int64_t* desc, const int32_t* hb, const int32_t* hk, int KH, const int32_t* vb,
                          const int32_t* vk, int KV, uint8_t* tmp, uint8_t* out, int B, int max_rows, int OH, int OW, void* stream) {
  return resize_bicubic_u8(src, desc, hb, hk, KH, vb, vk, KV, tmp, out, B, max_rows, OH, OW, ST);
}
// Host-side: gather n byte ranges into one (pinned) staging buffer with several threads — the packing step of the batch feeder
// (a single-threaded copy of a 96-image batch, 82 MB, costs 7.5 ms; the H2D copy that follows 1.6 ms).  The total is cut into
// equal byte spans, one per thread, across segment boundaries.  No CUDA calls: usable (and tested) without a device.
int xfm_host_pack(const void* const* srcs, const int64_t* nbytes, int n, void* dst, int threads) {
  if (n < 0 || (n > 0 && (!srcs || !nbytes || !dst))) { set_error("host_pack: null pointer"); return XFM_ERR_BAD_ARG; }
  std::vector<int64_t> start(n + 1, 0);
  for (int i = 0; i < n; ++i) {
    if (nbytes[i] < 0 || (nbytes[i] > 0 && !srcs[i])) { set_error("host_pack: bad segment %d", i); return XFM_ERR_BAD_ARG; }
    start[i + 1] = start[i] + nbytes[i];
  }
  const int64_t total = start[n];
  int T = threads < 1 ? 1 : threads;
  const int64_t by_size = total / (4 << 20) + 1;            // at least 4 MB per thread
  if (T > by_size) T = (int)by_size;
  auto span = [&](int64_t lo, int64_t hi) {
    int i = (int)(std::upper_bound(start.begin(), start.end(), lo) - start.begin()) - 1;
    while (lo < hi) {
      const int64_t end = start[i + 1] < hi ? start[i + 1] : hi;
      if (end > lo) std::memcpy((char*)dst + lo, (const char*)srcs[i] + (lo - start[i]), (size_t)(end - lo));
      lo = end;
      ++i;
    }
  };
  if (T == 1) { span(0, total); return 0; }
  std::vector<std::thread> pool;
  for (int t = 1; t < T; ++t) pool.emplace_back(span, total * t / T, total * (t + 1) / T);
  span(0, total / T);
  for (auto& th : pool) th.join();
  return 0;
}
// Host-side JPEG plan (two calls: sizes, then tables into caller buffers) and the device decode; csrc/jpeg.cu.
int xfm_jpeg_plan(const void* const* blobs, const int64_t* nbytes, int n, int64_t* info, int threads) {
  return jpeg_plan(blobs, nbytes, n, info, threads);
}
size_t xfm_jpeg_desc_bytes(void) { return jpeg_desc_bytes(); }
int xfm_jpeg_tables(const void* const* blobs, const int64_t* nbytes, int n, const int64_t* info, const int64_t* offs, void* desc,
                    int64_t* intervals, int threads) {
  return jpeg_tables(blobs, nbytes, n, info, offs, desc, intervals, threads);
}
int xfm_jpeg_decode(const uint8_t* bytes, const void* desc, const int64_t* intervals, int n, int16_t* coef, uint8_t* planes,
                    uint8_t* out, int32_t* status, int64_t max_blocks, int max_w, int max_h, void* stream) {
  return jpeg_decode(bytes, desc, intervals, n, coef, planes, out, status, max_blocks, max_w, max_h, ST);
}
int xfm_resize_taps(const int64_t* desc, int32_t* hb, int32_t* hk, int KH, int32_t* vb, int32_t* vk, int KV, int B, int OH, int OW,
                    void* stream) {
  return resize_taps(desc, hb, hk, KH, vb, vk, KV, B, OH, OW, ST);
}
int xfm_image_u8_to_f32(const uint8_t* in, float* out, const uint8_t* flip, int B, int H, int W, const float* mean,
                        const float* stdv, void* stream) {
  return image_u8_to_f32(in, out, flip, B, H, W, mean, stdv, ST);
}
int xfm_grad_sumsq(const float* g, const int32_t* chunk_seg, const uint8_t* seg_group, size_t nchunks, int32_t* seg_step,
                   float* seg_bc, int nseg, const float* hp, float* out, int accumulate, void* stream) {
  return grad_sumsq(g, chunk_seg, seg_group, nchunks, seg_step, seg_bc, nseg, hp, out, accumulate, ST);
}
int xfm_adamw_flat(float* P, const float* G, float* M, float* V, void* S, const int32_t* chunk_seg, const uint8_t* seg_group,
                   const float* seg_bc, size_t nchunks, const float* sumsq, float* norm_out, const float* hp, void* stream) {
  return adamw_flat(P, G, M, V, BF(S), chunk_seg, seg_group, seg_bc, nchunks, sumsq, norm_out, hp, ST);
}

}  // extern "C"
