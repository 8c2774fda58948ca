// K2/K3/K4 — flash-style multi-head attention (head_dim 64) forward + backward for sm_100a.
//
// One kernel family serves the three attention sites of the hot path:
//   * BEiT self-attention   (beit2.py:126-166): S = (q*d^-1/2) k^T + rel_pos_bias[h], no mask.
//   * RoBERTa self-attention (xroberta.py:237-284): S = (q/sqrt d) k^T + (1-m)*-1e4 key mask, prob dropout.
//   * Cross-attention        (xroberta.py:223-226,448-455): queries from text, K/V from image tokens;
//     several text samples may share one image's K/V (kv_index), which is how the ITM negatives and the MLM
//     pass reuse the K/V projection of the same B images instead of recomputing it.
//
// Scores never touch HBM: each warp owns 16 query rows, iterates over 64-key blocks held in shared memory
// (XOR-swizzled 128-byte rows, ldmatrix fragments), online softmax in registers, bf16 mma.sync with fp32
// accumulation.  The backward recomputes P from the saved log-sum-exp; kernel A produces dQ (and the bf16 dS
// dump used for the relative-position-bias gradient), kernel B produces dK/dV per key tile, looping over every
// sample that references that K/V.  (tcgen05/TMEM port of these kernels: next round — attention is 3.1 % of
// the step FLOPs, SURVEY.md §0.6.)
#include "common.cuh"
#include "internal.h"

namespace xfm {

constexpr int HD = 64;        // head dim
// CTAs of 4 or 8 warps x 16 rows (template parameter WARPS of the kernels below); keys / queries are walked in 64-row blocks
constexpr int AT_TILE = 64;
constexpr int ROW_BYTES = HD * 2;  // 128

struct AttnArgs {
  const bf16 *q, *k, *v;
  int64_t q_stride, k_stride, v_stride;
  bf16* out;
  int64_t o_stride;
  float* lse;          // [B, H, Lq]
  const float* bias;   // [H, Lq, bias_ld] or null
  int64_t bias_ld;
  const float* kmask;  // additive, [B, Lk] (per SAMPLE) or null
  const int32_t* kv_index;  // [B] sample -> K/V batch row, or null (identity)
  int B, H, Lq, Lk;
  float scale, dropout_p;
  uint64_t seed;
  const uint64_t* salt;  // device word added to the seed (see internal.h seed_salt_ptr)
  // backward only
  const bf16* dout;
  int64_t do_stride;
  const float* delta;  // [B, H, Lq] rowsum(dO * O)
  bf16 *dq, *dk, *dv;
  int64_t dq_stride, dk_stride, dv_stride;
  bf16* ds_dump;       // [B, H, Lq, ds_ld] or null
  int64_t ds_ld;
  const int32_t* kv_offsets;  // CSR over K/V batch rows: samples referencing row r are kv_samples[kv_offsets[r] .. kv_offsets[r+1])
  const int32_t* kv_samples;  // null => identity (sample r <-> row r)
  int Bkv;
};

XFM_DEVINL uint32_t swz(int row, int col) {  // byte offset of element (row, col) in a [rows][64] bf16 tile
  return (uint32_t)(row * ROW_BYTES + ((((col >> 3) ^ (row & 7)) << 4) | ((col & 7) << 1)));
}
XFM_DEVINL void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
XFM_DEVINL void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
XFM_DEVINL void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
XFM_DEVINL uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *(uint32_t*)&t;
}

// Copy `total` rows x 64 bf16 (row stride `stride` elements) into a swizzled tile; rows >= valid are zero-filled.
// Asynchronous (LDGSTS, 16 B per thread per op): every load of the tile is in flight at once instead of one
// global round trip per loop iteration; the caller waits with cp_async_wait_all() + __syncthreads().
XFM_DEVINL void load_tile(uint8_t* tile, const bf16* g, int64_t stride, int valid, int total) {
  const uint32_t base = smem_u32(tile);
  for (int i = threadIdx.x; i < total * 8; i += blockDim.x) {
    const int r = i >> 3, ch = i & 7;
    const bool ok = r < valid;
    const bf16* src = g + (int64_t)(ok ? r : 0) * stride + ch * 8;
    const uint32_t dst = base + r * ROW_BYTES + ((ch ^ (r & 7)) << 4);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0) : "memory");
  }
}
XFM_DEVINL void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// A-operand fragments (16 rows x 64 cols) of a swizzled tile: f[kk][0..3], rows row0..row0+15.
XFM_DEVINL void load_a_frags(uint32_t tile_addr, int row0, int lane, uint32_t (&f)[4][4]) {
  const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) ldsm_x4(tile_addr + swz(r, kk * 16 + (lane >> 4) * 8), f[kk][0], f[kk][1], f[kk][2], f[kk][3]);
}

// acc[nt] (16 x 64 block, 8 n-tiles) += A(16 x 64 over d) * Bt, where tile rows n0..n0+63 are the "n" index and the
// contraction runs over the 64 columns (d):  acc[row][n] = sum_d A[row][d] * tile[n0 + n][d].
// `lim`: rows n0 .. n0+lim-1 of the tile are real; 16-row groups beyond are skipped (their accumulators stay 0), which is
// most of the work for the 40-token text sequences inside 64-row tiles.
XFM_DEVINL void mma_rows_nt(float (&acc)[8][4], const uint32_t (&a)[4][4], uint32_t tile_addr, int n0, int lane, int lim = 64) {
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
    for (int ntp = 0; ntp < 4; ++ntp) {
      if (ntp * 16 >= lim) continue;
      uint32_t b00, b01, b10, b11;
      const int n = n0 + ntp * 16 + (lane & 7) + (lane >> 4) * 8;
      ldsm_x4(tile_addr + swz(n, kk * 16 + ((lane >> 3) & 1) * 8), b00, b01, b10, b11);
      mma16816(acc[2 * ntp], a[kk], b00, b01);
      mma16816(acc[2 * ntp + 1], a[kk], b10, b11);
    }
  }
}

// acc (16 x 64 over d) += P(16 x 64 over k) * tile[k0 + k][d]; P given as 4 k-step A fragments.
XFM_DEVINL void mma_rows_kd(float (&acc)[8][4], const uint32_t (&p)[4][4], uint32_t tile_addr, int k0, int lane, int lim = 64) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j * 16 >= lim) continue;   // the P / dS fragment of these k rows is all zero
#pragma unroll
    for (int dtp = 0; dtp < 4; ++dtp) {
      uint32_t r0, r1, r2, r3;
      const int kr = k0 + j * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
      ldsm_x4_t(tile_addr + swz(kr, dtp * 16 + (lane >> 4) * 8), r0, r1, r2, r3);
      mma16816(acc[2 * dtp], p[j], r0, r1);
      mma16816(acc[2 * dtp + 1], p[j], r2, r3);
    }
  }
}

XFM_DEVINL void c_to_a_frags(const float (&c)[8][4], uint32_t (&a)[4][4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    a[j][0] = pack_bf16(c[2 * j][0], c[2 * j][1]);
    a[j][1] = pack_bf16(c[2 * j][2], c[2 * j][3]);
    a[j][2] = pack_bf16(c[2 * j + 1][0], c[2 * j + 1][1]);
    a[j][3] = pack_bf16(c[2 * j + 1][2], c[2 * j + 1][3]);
  }
}

XFM_DEVINL float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
XFM_DEVINL float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

XFM_DEVINL bool drop_keep(const AttnArgs& a, int b, int h, int q, int key) {
  // element index with an EVEN row stride: keys (2k, 2k+1) of a row share one hash pair (the tcgen05 kernels evaluate the
  // mask pair-wise; both kernel families must index identically so forward and backward regenerate the same mask)
  const uint64_t idx = (((uint64_t)b * a.H + h) * a.Lq + q) * (uint64_t)((a.Lk + 1) & ~1) + key;
  return drop_keep_idx(a.seed + *a.salt, idx, a.dropout_p);
}

// Pair-wise evaluation of the same mask: pair base of a (b, h, q) row, then both keys (key, key+1), key even, at once.
XFM_DEVINL uint64_t drop_row_pair_base(const AttnArgs& a, int b, int h, int q) {
  return ((((uint64_t)b * a.H + h) * a.Lq + q) * (uint64_t)((a.Lk + 1) & ~1)) >> 1;
}
XFM_DEVINL uint32_t drop_pair_row(uint64_t pair_base, int key_even, uint32_t seed_mix, uint32_t thr) {
  const uint64_t pair = pair_base + (uint64_t)(key_even >> 1);
  return drop_keep_pair(seed_mix, (uint32_t)pair, (uint32_t)(pair >> 32), thr);
}

// Logit of (query row, key) after scale / bias / mask; -inf outside [0,Lk).
XFM_DEVINL float logit(const AttnArgs& a, float raw, int b, int h, int row, int key) {
  if (key >= a.Lk) return -INFINITY;
  float v = raw * a.scale;
  if (a.bias && row < a.Lq) v += __ldg(a.bias + ((int64_t)h * a.Lq + row) * a.bias_ld + key);
  if (a.kmask) v += __ldg(a.kmask + (int64_t)b * a.Lk + key);
  return v;
}

// Additive term (relative-position bias + key mask) of the 16 x 64 score fragment this thread owns, fetched BEFORE the
// score MMAs are issued so the global-load latency hides under them.  rows = query rows r0 / r1, keys kb + nt*8 + 2t (+1).
// Requires an even bias_ld (the host checks), so the float2 never straddles a row.
XFM_DEVINL void load_addend_rows(const AttnArgs& a, int b, int h, int r0, int r1, int kb, int t, float (&bb)[8][4]) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int key = kb + nt * 8 + 2 * t;
    float2 v0 = make_float2(0.f, 0.f), v1 = make_float2(0.f, 0.f);
    if (a.bias && key < a.bias_ld) {
      if (r0 < a.Lq) v0 = __ldg((const float2*)(a.bias + ((int64_t)h * a.Lq + r0) * a.bias_ld + key));
      if (r1 < a.Lq) v1 = __ldg((const float2*)(a.bias + ((int64_t)h * a.Lq + r1) * a.bias_ld + key));
    }
    if (a.kmask) {
      const float m0 = key < a.Lk ? __ldg(a.kmask + (int64_t)b * a.Lk + key) : 0.f;
      const float m1 = key + 1 < a.Lk ? __ldg(a.kmask + (int64_t)b * a.Lk + key + 1) : 0.f;
      v0.x += m0; v0.y += m1; v1.x += m0; v1.y += m1;
    }
    bb[nt][0] = v0.x; bb[nt][1] = v0.y; bb[nt][2] = v1.x; bb[nt][3] = v1.y;
  }
}
// Transposed ownership (dK/dV kernel): rows = keys key0 / key1, columns = queries qb + nt*8 + 2t (+1).
XFM_DEVINL void load_addend_cols(const AttnArgs& a, int b, int h, int key0, int key1, int qb, int t, float (&bb)[8][4]) {
  const float m0 = (a.kmask && key0 < a.Lk) ? __ldg(a.kmask + (int64_t)b * a.Lk + key0) : 0.f;
  const float m1 = (a.kmask && key1 < a.Lk) ? __ldg(a.kmask + (int64_t)b * a.Lk + key1) : 0.f;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int key = (e < 2) ? key0 : key1;
      const int qi = qb + nt * 8 + 2 * t + (e & 1);
      float v = (e < 2) ? m0 : m1;
      if (a.bias && qi < a.Lq && key < a.Lk) v += __ldg(a.bias + ((int64_t)h * a.Lq + qi) * a.bias_ld + key);
      bb[nt][e] = v;
    }
  }
}
XFM_DEVINL float logit2(const AttnArgs& a, float raw, float addend, int key) {
  return key < a.Lk ? raw * a.scale + addend : -INFINITY;
}

// ================================================================================================ forward
// WARPS x 16 query rows per CTA (4 or 8 warps): K / V of the whole sample are shared-memory resident, so at N = 577 (164 KB)
// only one CTA fits an SM and the warp count per CTA is the SM's occupancy.
// STREAM (rows whose K / V do not fit shared memory, e.g. 901 keys at 480 px): K / V pass through shared memory in chunks of
// KV_CHUNK keys.  The 64-key blocks, and therefore every operation and its order, are the resident kernel's.
constexpr int KV_CHUNK = 128;
template <int WARPS, bool STREAM>
__global__ void __launch_bounds__(WARPS * 32)
attn_fwd_kernel(const AttnArgs a) {
  constexpr int RT = WARPS * 16;
  extern __shared__ __align__(128) uint8_t smem[];
  const int LkP = (a.Lk + AT_TILE - 1) / AT_TILE * AT_TILE;
  const int KR = STREAM ? KV_CHUNK : LkP;   // key rows held in shared memory
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + RT * ROW_BYTES;
  uint8_t* sV = sK + KR * ROW_BYTES;
  const int q0 = blockIdx.x * RT, h = blockIdx.y, b = blockIdx.z;
  const int kvb = a.kv_index ? a.kv_index[b] : b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bf16* kg = a.k + (int64_t)kvb * a.Lk * a.k_stride + h * HD;
  const bf16* vg = a.v + (int64_t)kvb * a.Lk * a.v_stride + h * HD;
  load_tile(sQ, a.q + ((int64_t)b * a.Lq + q0) * a.q_stride + h * HD, a.q_stride, min(RT, a.Lq - q0), RT);
  if (!STREAM) {
    load_tile(sK, kg, a.k_stride, a.Lk, LkP);
    load_tile(sV, vg, a.v_stride, a.Lk, LkP);
  }
  cp_async_wait_all();
  __syncthreads();
  const bool live = q0 + warp * 16 < a.Lq;   // warp-uniform
  if (!STREAM && !live) return;              // no later block-wide barrier
  const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV);
  uint32_t qf[4][4];
  load_a_frags(aQ, warp * 16, lane, qf);
  const int g = lane >> 2, t = lane & 3;
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  const float inv_keep = a.dropout_p > 0.f ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
  const uint64_t dp0 = drop_row_pair_base(a, b, h, r0), dp1 = drop_row_pair_base(a, b, h, r1);
  for (int chunk0 = 0; chunk0 < LkP; chunk0 += KR) {
  if (STREAM) {   // the whole CTA: the previous chunk is consumed, then the next one lands
    __syncthreads();
    load_tile(sK, kg + (int64_t)chunk0 * a.k_stride, a.k_stride, min(KR, a.Lk - chunk0), KR);
    load_tile(sV, vg + (int64_t)chunk0 * a.v_stride, a.v_stride, min(KR, a.Lk - chunk0), KR);
    cp_async_wait_all();
    __syncthreads();
    if (!live) continue;
  }
  for (int kb = chunk0; kb < min(chunk0 + KR, LkP); kb += AT_TILE) {
    float s[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
    float bb[8][4];
    load_addend_rows(a, b, h, r0, r1, kb, t, bb);
    const int lim = a.Lk - kb;   // valid keys in this block
    mma_rows_nt(s, qf, aK, kb - chunk0, lane, lim);
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt * 8 >= lim) continue;   // all-padding key group: s stays 0 = probability 0
      const int key = kb + nt * 8 + 2 * t;
      s[nt][0] = logit2(a, s[nt][0], bb[nt][0], key);
      s[nt][1] = logit2(a, s[nt][1], bb[nt][1], key + 1);
      s[nt][2] = logit2(a, s[nt][2], bb[nt][2], key);
      s[nt][3] = logit2(a, s[nt][3], bb[nt][3], key + 1);
      mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
    }
    const float mn0 = fmaxf(m0, quad_max(mx0)), mn1 = fmaxf(m1, quad_max(mx1));
    const float c0 = __expf(m0 - mn0), c1 = __expf(m1 - mn1);  // m = -inf on the first block -> 0
    m0 = mn0;
    m1 = mn1;
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      o[nt][0] *= c0; o[nt][1] *= c0; o[nt][2] *= c1; o[nt][3] *= c1;
      if (nt * 8 >= lim) continue;
      s[nt][0] = __expf(s[nt][0] - mn0);
      s[nt][1] = __expf(s[nt][1] - mn0);
      s[nt][2] = __expf(s[nt][2] - mn1);
      s[nt][3] = __expf(s[nt][3] - mn1);
      sum0 += s[nt][0] + s[nt][1];
      sum1 += s[nt][2] + s[nt][3];
    }
    l0 = l0 * c0 + sum0;
    l1 = l1 * c1 + sum1;
    if (a.dropout_p > 0.f) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt * 8 >= lim) continue;
        const int key = kb + nt * 8 + 2 * t;   // even: (key, key+1) is one hash pair of each row
        const uint32_t k0 = drop_pair_row(dp0, key, seed_mix, thr), k1 = drop_pair_row(dp1, key, seed_mix, thr);
        s[nt][0] = (k0 & 1u) ? s[nt][0] * inv_keep : 0.f;
        s[nt][1] = (k0 & 2u) ? s[nt][1] * inv_keep : 0.f;
        s[nt][2] = (k1 & 1u) ? s[nt][2] * inv_keep : 0.f;
        s[nt][3] = (k1 & 2u) ? s[nt][3] * inv_keep : 0.f;
      }
    }
    uint32_t pf[4][4];
    c_to_a_frags(s, pf);
    mma_rows_kd(o, pf, aV, kb - chunk0, lane, lim);
  }
  }
  if (!live) return;
  l0 = quad_sum(l0);
  l1 = quad_sum(l1);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = h * HD + nt * 8 + 2 * t;
    if (r0 < a.Lq) *(uint32_t*)(a.out + ((int64_t)b * a.Lq + r0) * a.o_stride + col) = pack_bf16(o[nt][0] * i0, o[nt][1] * i0);
    if (r1 < a.Lq) *(uint32_t*)(a.out + ((int64_t)b * a.Lq + r1) * a.o_stride + col) = pack_bf16(o[nt][2] * i1, o[nt][3] * i1);
  }
  if (t == 0 && a.lse) {
    if (r0 < a.Lq) a.lse[((int64_t)b * a.H + h) * a.Lq + r0] = m0 + __logf(l0);
    if (r1 < a.Lq) a.lse[((int64_t)b * a.H + h) * a.Lq + r1] = m1 + __logf(l1);
  }
}

// ================================================================================================ backward
// delta[b,h,i] = sum_d dO[b,i,h*64+d] * O[b,i,h*64+d]; blockDim = (8*H, 4): 8 threads x 16 bytes per (row, head).
__global__ void attn_delta_kernel(const bf16* __restrict__ dout, int64_t do_stride, const bf16* __restrict__ out,
                                  int64_t o_stride, float* __restrict__ delta, int B, int H, int Lq) {
  const int row_raw = blockIdx.x * blockDim.y + threadIdx.y;  // b * Lq + i
  const bool valid = row_raw < B * Lq;
  const int row = valid ? row_raw : B * Lq - 1;  // keep every lane alive for the shuffles
  const int h = threadIdx.x >> 3, part = threadIdx.x & 7;
  const uint4 u = *(const uint4*)(dout + (int64_t)row * do_stride + h * HD + part * 8);
  const uint4 w = *(const uint4*)(out + (int64_t)row * o_stride + h * HD + part * 8);
  const __nv_bfloat162* x = (const __nv_bfloat162*)&u;
  const __nv_bfloat162* y = (const __nv_bfloat162*)&w;
  float s = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float2 f = __bfloat1622float2(x[q]), gq = __bfloat1622float2(y[q]);
    s += f.x * gq.x + f.y * gq.y;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (part == 0 && valid) {
    const int b = row / Lq, i = row % Lq;
    delta[((int64_t)b * H + h) * Lq + i] = s;
  }
}

int launch_attn_delta(const bf16* dout, int64_t do_stride, const bf16* out, int64_t o_stride, float* delta, int B, int H, int Lq,
                      cudaStream_t s) {
  if (8 * H * 4 > 1024) { set_error("attention_bwd: too many heads"); return XFM_ERR_BAD_ARG; }
  attn_delta_kernel<<<(B * Lq + 3) / 4, dim3(8 * H, 4), 0, s>>>(dout, do_stride, out, o_stride, delta, B, H, Lq);
  count_launch();
  return 0;
}

// Kernel A: dQ (+ optional bf16 dS dump).  Same tiling as the forward; STREAM: K / V in chunks, as there.
template <int WARPS, bool STREAM>
__global__ void __launch_bounds__(WARPS * 32)
attn_bwd_dq_kernel(const AttnArgs a) {
  constexpr int RT = WARPS * 16;
  extern __shared__ __align__(128) uint8_t smem[];
  const int LkP = (a.Lk + AT_TILE - 1) / AT_TILE * AT_TILE;
  const int KR = STREAM ? KV_CHUNK : LkP;
  uint8_t* sQ = smem;
  uint8_t* sdO = sQ + RT * ROW_BYTES;
  uint8_t* sK = sdO + RT * ROW_BYTES;
  uint8_t* sV = sK + KR * ROW_BYTES;
  const int q0 = blockIdx.x * RT, h = blockIdx.y, b = blockIdx.z;
  const int kvb = a.kv_index ? a.kv_index[b] : b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = min(RT, a.Lq - q0);
  const bf16* kg = a.k + (int64_t)kvb * a.Lk * a.k_stride + h * HD;
  const bf16* vg = a.v + (int64_t)kvb * a.Lk * a.v_stride + h * HD;
  load_tile(sQ, a.q + ((int64_t)b * a.Lq + q0) * a.q_stride + h * HD, a.q_stride, nq, RT);
  load_tile(sdO, a.dout + ((int64_t)b * a.Lq + q0) * a.do_stride + h * HD, a.do_stride, nq, RT);
  if (!STREAM) {
    load_tile(sK, kg, a.k_stride, a.Lk, LkP);
    load_tile(sV, vg, a.v_stride, a.Lk, LkP);
  }
  cp_async_wait_all();
  __syncthreads();
  const bool live = q0 + warp * 16 < a.Lq;
  if (!STREAM && !live) return;
  const uint32_t aQ = smem_u32(sQ), adO = smem_u32(sdO), aK = smem_u32(sK), aV = smem_u32(sV);
  uint32_t qf[4][4], dof[4][4];
  load_a_frags(aQ, warp * 16, lane, qf);
  load_a_frags(adO, warp * 16, lane, dof);
  const int g = lane >> 2, t = lane & 3;
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
  const int64_t st = ((int64_t)b * a.H + h) * a.Lq;
  const float lse0 = r0 < a.Lq ? a.lse[st + r0] : 0.f, lse1 = r1 < a.Lq ? a.lse[st + r1] : 0.f;
  const float dl0 = r0 < a.Lq ? a.delta[st + r0] : 0.f, dl1 = r1 < a.Lq ? a.delta[st + r1] : 0.f;
  const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
  const uint64_t dpb0 = drop_row_pair_base(a, b, h, r0), dpb1 = drop_row_pair_base(a, b, h, r1);
  const float inv_keep = a.dropout_p > 0.f ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  float dq[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
  for (int chunk0 = 0; chunk0 < LkP; chunk0 += KR) {
  if (STREAM) {
    __syncthreads();
    load_tile(sK, kg + (int64_t)chunk0 * a.k_stride, a.k_stride, min(KR, a.Lk - chunk0), KR);
    load_tile(sV, vg + (int64_t)chunk0 * a.v_stride, a.v_stride, min(KR, a.Lk - chunk0), KR);
    cp_async_wait_all();
    __syncthreads();
    if (!live) continue;
  }
  for (int kb = chunk0; kb < min(chunk0 + KR, LkP); kb += AT_TILE) {
    float s[8][4], dp[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
      dp[i][0] = dp[i][1] = dp[i][2] = dp[i][3] = 0.f;
    }
    float bb[8][4];
    load_addend_rows(a, b, h, r0, r1, kb, t, bb);
    const int lim = a.Lk - kb;
    mma_rows_nt(s, qf, aK, kb - chunk0, lane, lim);    // S  = Q K^T
    mma_rows_nt(dp, dof, aV, kb - chunk0, lane, lim);  // dP = dO V^T
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt * 8 >= lim) continue;   // all-padding key group: dS stays 0 (ds_dump beyond Lk is pre-zeroed by the caller)
      uint32_t keep[2] = {3u, 3u};
      if (a.dropout_p > 0.f) {
        const int key_even = kb + nt * 8 + 2 * t;
        keep[0] = drop_pair_row(dpb0, key_even, seed_mix, thr);
        keep[1] = drop_pair_row(dpb1, key_even, seed_mix, thr);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int row = (e < 2) ? r0 : r1;
        const int key = kb + nt * 8 + 2 * t + (e & 1);
        const float p = __expf(logit2(a, s[nt][e], bb[nt][e], key) - ((e < 2) ? lse0 : lse1));  // 0 for key >= Lk
        float dpe = dp[nt][e];
        if (a.dropout_p > 0.f) dpe = (key < a.Lk && ((keep[e >> 1] >> (e & 1)) & 1u)) ? dpe * inv_keep : 0.f;
        const float ds = (row < a.Lq) ? p * (dpe - ((e < 2) ? dl0 : dl1)) : 0.f;
        s[nt][e] = ds;
      }
      if (a.ds_dump) {
        const int key = kb + nt * 8 + 2 * t;
        if (key < a.ds_ld) {  // ds_ld is a multiple of 8 >= Lk: pairs never straddle the end
          if (r0 < a.Lq) *(uint32_t*)(a.ds_dump + (st + r0) * a.ds_ld + key) = pack_bf16(s[nt][0], s[nt][1]);
          if (r1 < a.Lq) *(uint32_t*)(a.ds_dump + (st + r1) * a.ds_ld + key) = pack_bf16(s[nt][2], s[nt][3]);
        }
      }
    }
    uint32_t dsf[4][4];
    c_to_a_frags(s, dsf);
    mma_rows_kd(dq, dsf, aK, kb - chunk0, lane, lim);  // dQ += dS K
  }
  }
  if (!live) return;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = h * HD + nt * 8 + 2 * t;
    if (r0 < a.Lq)
      *(uint32_t*)(a.dq + ((int64_t)b * a.Lq + r0) * a.dq_stride + col) = pack_bf16(dq[nt][0] * a.scale, dq[nt][1] * a.scale);
    if (r1 < a.Lq)
      *(uint32_t*)(a.dq + ((int64_t)b * a.Lq + r1) * a.dq_stride + col) = pack_bf16(dq[nt][2] * a.scale, dq[nt][3] * a.scale);
  }
}

// Kernel B: dK, dV for one 64-key tile of one (K/V batch row, head); loops over every referencing sample and over
// that sample's queries in blocks of 64.  Works on the transposed problem: rows = keys, columns = queries.
// STREAM: a sample's Q / dO (and lse / delta) pass through shared memory in chunks of KV_CHUNK queries.
template <int WARPS, bool STREAM>
__global__ void __launch_bounds__(WARPS * 32)
attn_bwd_dkv_kernel(const AttnArgs a) {
  constexpr int RT = WARPS * 16;
  extern __shared__ __align__(128) uint8_t smem[];
  const int LqP = (a.Lq + AT_TILE - 1) / AT_TILE * AT_TILE;
  const int QR = STREAM ? KV_CHUNK : LqP;   // query rows held in shared memory
  uint8_t* sK = smem;
  uint8_t* sV = sK + RT * ROW_BYTES;
  uint8_t* sQ = sV + RT * ROW_BYTES;
  uint8_t* sdO = sQ + QR * ROW_BYTES;
  float* sLse = (float*)(sdO + QR * ROW_BYTES);
  float* sDelta = sLse + QR;
  const int k0 = blockIdx.x * RT, h = blockIdx.y, kvb = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nk = min(RT, a.Lk - k0);
  load_tile(sK, a.k + ((int64_t)kvb * a.Lk + k0) * a.k_stride + h * HD, a.k_stride, nk, RT);
  load_tile(sV, a.v + ((int64_t)kvb * a.Lk + k0) * a.v_stride + h * HD, a.v_stride, nk, RT);
  const uint32_t aK = smem_u32(sK), aV = smem_u32(sV), aQ = smem_u32(sQ), adO = smem_u32(sdO);
  const int g = lane >> 2, t = lane & 3;
  const int key0 = k0 + warp * 16 + g, key1 = key0 + 8;
  const bool warp_active = k0 + warp * 16 < a.Lk;
  const float inv_keep = a.dropout_p > 0.f ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  float dk[8][4], dv[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
    dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
  }
  uint32_t kf[4][4], vf[4][4];
  bool frags = false;
  const int s_begin = a.kv_samples ? a.kv_offsets[kvb] : kvb;
  const int s_end = a.kv_samples ? a.kv_offsets[kvb + 1] : kvb + 1;
  for (int si = s_begin; si < s_end; ++si) {
    const int b = a.kv_samples ? a.kv_samples[si] : si;
    const int64_t st = ((int64_t)b * a.H + h) * a.Lq;
    for (int chunk0 = 0; chunk0 < LqP; chunk0 += QR) {
    const int nq = min(QR, a.Lq - chunk0);
    __syncthreads();  // previous sample's (chunk's) tiles fully consumed (also orders the K/V tile loads on the first pass)
    load_tile(sQ, a.q + ((int64_t)b * a.Lq + chunk0) * a.q_stride + h * HD, a.q_stride, nq, QR);
    load_tile(sdO, a.dout + ((int64_t)b * a.Lq + chunk0) * a.do_stride + h * HD, a.do_stride, nq, QR);
    for (int i = threadIdx.x; i < QR; i += blockDim.x) {
      sLse[i] = i < nq ? a.lse[st + chunk0 + i] : 0.f;
      sDelta[i] = i < nq ? a.delta[st + chunk0 + i] : 0.f;
    }
    cp_async_wait_all();
    __syncthreads();
    if (!warp_active) continue;
    if (!frags) {
      load_a_frags(aK, warp * 16, lane, kf);
      load_a_frags(aV, warp * 16, lane, vf);
      frags = true;
    }
    for (int qb = chunk0; qb < min(chunk0 + QR, LqP); qb += AT_TILE) {
      float s[8][4], dp[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
        dp[i][0] = dp[i][1] = dp[i][2] = dp[i][3] = 0.f;
      }
      float bb[8][4];
      load_addend_cols(a, b, h, key0, key1, qb, t, bb);
      const int lim = a.Lq - qb;   // valid queries in this block
      mma_rows_nt(s, kf, aQ, qb - chunk0, lane, lim);    // S^T  = K Q^T
      mma_rows_nt(dp, vf, adO, qb - chunk0, lane, lim);  // dP^T = V dO^T
      float pd[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt * 8 >= lim) {   // all-padding query group
#pragma unroll
          for (int e = 0; e < 4; ++e) pd[nt][e] = s[nt][e] = 0.f;
          continue;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = (e < 2) ? key0 : key1;
          const int qi = qb + nt * 8 + 2 * t + (e & 1);
          float p = 0.f;
          if (qi < a.Lq && key < a.Lk) p = __expf(s[nt][e] * a.scale + bb[nt][e] - sLse[qi - chunk0]);
          float keep = 1.f;
          if (a.dropout_p > 0.f) keep = (qi < a.Lq && key < a.Lk && drop_keep(a, b, h, qi, key)) ? inv_keep : 0.f;
          pd[nt][e] = p * keep;
          s[nt][e] = p * (dp[nt][e] * keep - sDelta[min(qi - chunk0, QR - 1)]);
        }
      }
      uint32_t pf[4][4], dsf[4][4];
      c_to_a_frags(pd, pf);
      c_to_a_frags(s, dsf);
      mma_rows_kd(dv, pf, adO, qb - chunk0, lane, lim);  // dV += P^T dO
      mma_rows_kd(dk, dsf, aQ, qb - chunk0, lane, lim);  // dK += dS^T Q
    }
    }
  }
  if (!warp_active) return;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = h * HD + nt * 8 + 2 * t;
    if (key0 < a.Lk) {
      *(uint32_t*)(a.dk + ((int64_t)kvb * a.Lk + key0) * a.dk_stride + col) = pack_bf16(dk[nt][0] * a.scale, dk[nt][1] * a.scale);
      *(uint32_t*)(a.dv + ((int64_t)kvb * a.Lk + key0) * a.dv_stride + col) = pack_bf16(dv[nt][0], dv[nt][1]);
    }
    if (key1 < a.Lk) {
      *(uint32_t*)(a.dk + ((int64_t)kvb * a.Lk + key1) * a.dk_stride + col) = pack_bf16(dk[nt][2] * a.scale, dk[nt][3] * a.scale);
      *(uint32_t*)(a.dv + ((int64_t)kvb * a.Lk + key1) * a.dv_stride + col) = pack_bf16(dv[nt][2], dv[nt][3]);
    }
  }
}

// ------------------------------------------------------------------------------------------ host
static int attn_check(const xfm_attn_params* p) {
  if (!p || !p->q || !p->k || !p->v || p->B <= 0 || p->H <= 0 || p->Lq <= 0 || p->Lk <= 0) {
    set_error("attention: null pointer or non-positive shape");
    return XFM_ERR_BAD_ARG;
  }
  if (p->head_dim != HD) {
    set_error("attention: head_dim must be 64 (got %d)", p->head_dim);
    return XFM_ERR_BAD_ARG;
  }
  if (p->bias && (p->bias_ld & 1)) {
    set_error("attention: bias_ld must be even");
    return XFM_ERR_BAD_ARG;
  }
  if ((p->q_stride | p->k_stride | p->v_stride) & 7) {
    set_error("attention: row strides must be multiples of 8 elements");
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

static void fill_args(const xfm_attn_params* p, AttnArgs& a) {
  a.q = (const bf16*)p->q; a.k = (const bf16*)p->k; a.v = (const bf16*)p->v;
  a.q_stride = p->q_stride; a.k_stride = p->k_stride; a.v_stride = p->v_stride;
  a.out = (bf16*)p->out; a.o_stride = p->o_stride; a.lse = p->lse;
  a.bias = p->bias; a.bias_ld = p->bias_ld; a.kmask = p->kmask; a.kv_index = p->kv_index;
  a.B = p->B; a.H = p->H; a.Lq = p->Lq; a.Lk = p->Lk;
  a.scale = p->scale; a.dropout_p = p->dropout_p; a.seed = p->dropout_seed; a.salt = seed_salt_ptr();
  a.dout = (const bf16*)p->dout; a.do_stride = p->do_stride; a.delta = p->delta;
  a.dq = (bf16*)p->dq; a.dk = (bf16*)p->dk; a.dv = (bf16*)p->dv;
  a.dq_stride = p->dq_stride; a.dk_stride = p->dk_stride; a.dv_stride = p->dv_stride;
  a.ds_dump = (bf16*)p->ds_dump; a.ds_ld = p->ds_ld;
  a.kv_offsets = p->kv_offsets; a.kv_samples = p->kv_samples;
  a.Bkv = p->Bkv > 0 ? p->Bkv : p->B;
}

// The resident kernels hold a whole row of K / V (or Q / dO) in shared memory; past this, the streaming variants run.
constexpr size_t RESIDENT_SMEM_MAX = 220 * 1024;

template <int WARPS, bool STREAM>
static int launch_attn_fwd(const AttnArgs& a, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(attn_fwd_kernel<WARPS, STREAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const dim3 grid((a.Lq + WARPS * 16 - 1) / (WARPS * 16), a.H, a.B);
  attn_fwd_kernel<WARPS, STREAM><<<grid, WARPS * 32, smem, s>>>(a);
  count_launch();
  return (int)cudaGetLastError();
}

int attention_fwd_parts(const xfm_attn_params* p) {
  if (!p || !p->allow_tc || attn_check(p)) return 0;
  xfm_attn_params q = *p;   // as if the scratch were given: does the chosen tcgen05 path run in key blocks?
  static float dummy;
  q.part_out = &dummy;
  q.part_lse = &dummy;
  if (!vit_attention_tc_supported(&q) && !cross_attention_tc_supported(&q)) return 0;
  const int nb = KeyBlocks::nb(q.Lk);
  return nb > 1 ? nb : 0;
}

int attention_fwd(const xfm_attn_params* p, cudaStream_t s) {
  if (attn_check(p)) return XFM_ERR_BAD_ARG;
  if (p->allow_tc && vit_attention_tc_supported(p)) return vit_attention_fwd_tc(p, s);
  if (p->allow_tc && cross_attention_tc_supported(p)) return cross_attention_fwd_tc(p, s);
  if (p->allow_tc && self_attention_tc_supported(p)) return self_attention_fwd_tc(p, s);
  AttnArgs a;
  fill_args(p, a);
  const int LkP = (a.Lk + AT_TILE - 1) / AT_TILE * AT_TILE;
  const bool big = a.Lq > 256;   // 8 warps (128 query rows) per CTA when the resident K / V leave room for one CTA per SM only
  const int rt = big ? 128 : 64;
  const size_t smem = (size_t)(rt + 2 * LkP) * ROW_BYTES;
  if (smem > RESIDENT_SMEM_MAX) {
    const size_t smem_s = (size_t)(rt + 2 * KV_CHUNK) * ROW_BYTES;
    return big ? launch_attn_fwd<8, true>(a, smem_s, s) : launch_attn_fwd<4, true>(a, smem_s, s);
  }
  return big ? launch_attn_fwd<8, false>(a, smem, s) : launch_attn_fwd<4, false>(a, smem, s);
}

template <int WARPS, bool STREAM>
static int launch_attn_bwd_dq(const AttnArgs& a, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(attn_bwd_dq_kernel<WARPS, STREAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const dim3 grid((a.Lq + WARPS * 16 - 1) / (WARPS * 16), a.H, a.B);
  attn_bwd_dq_kernel<WARPS, STREAM><<<grid, WARPS * 32, smem, s>>>(a);
  count_launch();
  return (int)cudaGetLastError();
}

template <int WARPS, bool STREAM>
static int launch_attn_bwd_dkv(const AttnArgs& a, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(attn_bwd_dkv_kernel<WARPS, STREAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const dim3 grid((a.Lk + WARPS * 16 - 1) / (WARPS * 16), a.H, a.Bkv);
  attn_bwd_dkv_kernel<WARPS, STREAM><<<grid, WARPS * 32, smem, s>>>(a);
  count_launch();
  return (int)cudaGetLastError();
}

int attention_bwd(const xfm_attn_params* p, cudaStream_t s) {
  if (attn_check(p)) return XFM_ERR_BAD_ARG;
  if (!p->dout || !p->out || !p->lse || !p->delta || !p->dq || !p->dk || !p->dv) {
    set_error("attention_bwd: missing pointer");
    return XFM_ERR_BAD_ARG;
  }
  if (p->kv_index && (!p->kv_offsets || !p->kv_samples)) {   // dK / dV sum over the samples of each K/V row: the CSR lists them
    set_error("attention_bwd: kv_index needs kv_offsets and kv_samples");
    return XFM_ERR_BAD_ARG;
  }
  if (p->ds_dump && ((p->ds_ld & 7) || p->ds_ld < p->Lk)) {
    set_error("attention_bwd: ds_ld must be a multiple of 8 and >= Lk");
    return XFM_ERR_BAD_ARG;
  }
  AttnArgs a;
  fill_args(p, a);
  const int LkP = (a.Lk + AT_TILE - 1) / AT_TILE * AT_TILE;
  const int LqP = (a.Lq + AT_TILE - 1) / AT_TILE * AT_TILE;
  {
    const int rc = launch_attn_delta(a.dout, a.do_stride, a.out, a.o_stride, (float*)p->delta, a.B, a.H, a.Lq, s);
    if (rc) return rc;
  }
  if (p->allow_tc && vit_attention_tc_supported(p, true)) return vit_attention_bwd_tc(p, s);
  if (p->allow_tc && cross_attention_tc_supported(p, true)) return cross_attention_bwd_tc(p, s);
  if (p->allow_tc && self_attention_tc_supported(p) && !p->ds_dump) return self_attention_bwd_tc(p, s);
  const bool big_q = a.Lq > 256, big_k = a.Lk > 256;
  const int rq = big_q ? 128 : 64, rk = big_k ? 128 : 64;
  const size_t smem_a = (size_t)(2 * rq + 2 * LkP) * ROW_BYTES;
  const size_t smem_b = (size_t)(2 * rk + 2 * LqP) * ROW_BYTES + 2 * LqP * sizeof(float);
  int rc;
  if (smem_a > RESIDENT_SMEM_MAX) {
    const size_t sm = (size_t)(2 * rq + 2 * KV_CHUNK) * ROW_BYTES;
    rc = big_q ? launch_attn_bwd_dq<8, true>(a, sm, s) : launch_attn_bwd_dq<4, true>(a, sm, s);
  } else {
    rc = big_q ? launch_attn_bwd_dq<8, false>(a, smem_a, s) : launch_attn_bwd_dq<4, false>(a, smem_a, s);
  }
  if (rc) return rc;
  if (smem_b > RESIDENT_SMEM_MAX) {
    const size_t sm = (size_t)(2 * rk + 2 * KV_CHUNK) * ROW_BYTES + 2 * KV_CHUNK * sizeof(float);
    return big_k ? launch_attn_bwd_dkv<8, true>(a, sm, s) : launch_attn_bwd_dkv<4, true>(a, sm, s);
  }
  return big_k ? launch_attn_bwd_dkv<8, false>(a, smem_b, s) : launch_attn_bwd_dkv<4, false>(a, smem_b, s);
}

}  // namespace xfm
