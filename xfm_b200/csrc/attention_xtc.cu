// K4 — cross-attention (xroberta.py:223-226,243-284 called from :448-455) on tcgen05 + TMEM + TMA.
//
// Text queries attend to the image tokens of ONE image; several text samples share the same image (the ITM positives, the
// hard negatives that re-use that image, the MLM pass: kv_index / its CSR inverse kv_offsets, kv_samples).  The samples of
// one image are therefore STACKED along the query axis: up to GMAX samples x LQS (= 40) rows form the rows of two 128-row
// query tiles (slot g -> tile g % 2, rows (g / 2) * LQS ..), and the image's K / V tile is loaded once for all of them.
// Same pipeline as attention_tc.cu: warp 0 TMA, warp 1 single-thread tcgen05.mma (S = Q K^T into two TMEM score buffers,
// O = P V into a third region), two softmax warpgroups (one per query tile, thread = query row).  No bias; dropout on the
// probabilities uses the stateless (seed, (b, h, q, key)) hash shared with the mma.sync kernels, so forward and backward
// kernels of either family regenerate the same mask.  Images referenced by more than GMAX samples are processed in
// several chunks of GMAX.
#include "common.cuh"
#include "internal.h"

namespace xfm {

constexpr int XT_HD = 64;
constexpr int XT_THREADS = 64 + 256;
constexpr int XTF_THREADS = 64 + 512;   // fused backward: four element-wise / drain warpgroups

struct XAttnArgs {
  bf16* out;
  int64_t o_stride;
  float* lse;                 // [B, H, LQS]
  const int32_t* kv_offsets;  // [Bkv + 1]
  const int32_t* kv_samples;  // [B] sample ids grouped by K/V row
  int B, Bkv, H;
  float scale, dropout_p;
  uint64_t seed;
  const uint64_t* salt;
  int items_per_cta;
  // backward
  const float* delta;         // [B, H, LQS]
  bf16 *dq, *dk, *dv;
  int64_t dq_stride, dk_stride, dv_stride;
};

template <int LQS_, int LK_, int GMAX_>
struct XCfg {
  static constexpr int LQS = LQS_, LK = LK_, GMAX = GMAX_;
  static constexpr int PER_TILE = (GMAX + 1) / 2;            // sample slots per 128-row query tile
  static_assert(PER_TILE * LQS <= 128, "slots of one tile must fit 128 rows");
  static_assert((LQS * 128) % 1024 == 0, "a sample's rows must start on a swizzle-atom boundary (LQS multiple of 8)");
  // more than 208 keys (384 px: 577, 480 px: 901): one launch per key block (KeyBlocks), partial results merged afterwards
  // (forward) — see attention_tc.cu::VitFwdCfg
  static constexpr int NB = KeyBlocks::nb(LK);
  static constexpr bool BLOCKED = NB > 1;
  static constexpr int KBS = KeyBlocks::kbs(LK);
  static constexpr int LAST = KeyBlocks::last(LK);
  static constexpr int LPAD = KeyBlocks::lpad(LK);
  static_assert(LAST <= LPAD && (NB == 1 || KBS % 2 == 0), "key blocks");
  static constexpr int NKB = (LPAD + 63) / 64;
  static constexpr int Q_BYTES = 2 * 128 * 128;
  static constexpr int KV_BYTES = LPAD * 128;
  static constexpr int P_BYTES = NKB * 16384;
  static constexpr int SMEM_FWD = Q_BYTES + 2 * KV_BYTES + 2 * P_BYTES + 128;
  static constexpr int TMEM_O = 2 * LPAD;
  static_assert(2 * LPAD + 64 <= 512, "TMEM");
};

XFM_DEVINL void xt_ld32(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld_32x32(taddr, r); }

// One "unit" = (K/V row, head, chunk of <= GMAX samples).  Every role walks the same unit sequence.  With EMPTY, an image
// that no sample references is one unit with ns = 0 (the backward stores zero dK / dV for it); without, it is skipped.
struct XUnit {
  int r, h, first, ns;   // K/V row, head, index of the chunk's first entry in kv_samples, samples in the chunk
};
template <int GMAX, bool EMPTY = false>
struct XWalker {
  const XAttnArgs& a;
  int it, it_end, chunk, nchunks, off0, cnt;
  XFM_DEVINL XWalker(const XAttnArgs& a_, int it0, int it1) : a(a_), it(it0 - 1), it_end(it1), chunk(0), nchunks(0), off0(0), cnt(0) {}
  XFM_DEVINL bool next(XUnit& u) {
    ++chunk;
    while (chunk >= nchunks) {
      if (++it >= it_end) return false;
      const int r = it % a.Bkv;
      off0 = a.kv_offsets[r];
      cnt = a.kv_offsets[r + 1] - off0;
      nchunks = (cnt + GMAX - 1) / GMAX;
      if (EMPTY && nchunks == 0) nchunks = 1;
      chunk = 0;
    }
    u.r = it % a.Bkv;
    u.h = it / a.Bkv;
    u.first = off0 + chunk * GMAX;
    u.ns = min(GMAX, cnt - chunk * GMAX);
    return true;
  }
};

template <int LQS, int LK, int GMAX, int KB>
__global__ void __launch_bounds__(XT_THREADS, 1)
xattn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const XAttnArgs a) {
  using Cfg = XCfg<LQS, LK, GMAX>;
  constexpr int LPAD = Cfg::LPAD, PER_TILE = Cfg::PER_TILE;
  constexpr int K0 = KB * Cfg::KBS;                                   // first key of this launch's block
  constexpr int KLEN = KB == Cfg::NB - 1 ? Cfg::LAST : Cfg::KBS;      // its keys
  static_assert(KB < Cfg::NB, "key block");
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::Q_BYTES;
  uint8_t* sV = sK + Cfg::KV_BYTES;
  uint8_t* sP = sV + Cfg::KV_BYTES;   // [2][P_BYTES]
  uint64_t* bars = (uint64_t*)(sP + 2 * Cfg::P_BYTES);
  uint64_t *qk_full = bars, *qk_empty = bars + 1, *v_full = bars + 2, *v_empty = bars + 3;
  uint64_t *s_full = bars + 4, *p_full = bars + 6, *o_full = bars + 8, *o_empty = bars + 10;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 11);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < Cfg::Q_BYTES / 16; i += blockDim.x) ((uint4*)sQ)[i] = make_uint4(0u, 0u, 0u, 0u);  // unused slots stay finite
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    mbar_init(qk_full, 1);
    mbar_init(qk_empty, 1);
    mbar_init(v_full, 1);
    mbar_init(v_empty, 1);
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&p_full[t], 4);
      mbar_init(&o_full[t], 1);
    }
    mbar_init(o_empty, 4);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int n_items = a.Bkv * a.H;
  const int item0 = blockIdx.x * a.items_per_cta;
  const int item1 = min(n_items, item0 + a.items_per_cta);

  if (warp == 0) {
    if (lane == 0) {
      XWalker<GMAX> w(a, item0, item1);
      XUnit u;
      uint32_t ph = 0;
      while (w.next(u)) {
        mbar_wait_relaxed(qk_empty, ph ^ 1);
        mbar_arrive_expect_tx(qk_full, u.ns * LQS * 128 + Cfg::KV_BYTES);
        for (int g = 0; g < u.ns; ++g) {
          const int b = a.kv_samples[u.first + g];
          tma_load_2d(sQ + (g & 1) * 16384 + (g >> 1) * (LQS * 128), &map_q, qk_full, u.h * XT_HD, b * LQS);
        }
        tma_load_2d(sK, &map_k, qk_full, u.h * XT_HD, u.r * LK + K0);
        mbar_wait_relaxed(v_empty, ph ^ 1);
        mbar_arrive_expect_tx(v_full, Cfg::KV_BYTES);
        tma_load_2d(sV, &map_v, v_full, u.h * XT_HD, u.r * LK + K0);
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, LPAD, 0, 0);
      constexpr uint32_t idesc_o = make_idesc_bf16(128, XT_HD, 0, 1);
      const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV), aP = smem_u32(sP);
      XWalker<GMAX> w(a, item0, item1);
      XUnit u;
      uint32_t ph = 0;        // unit parity (qk_full / v_full / s_full / p_full / o_full[t] complete once per unit)
      uint32_t oe = 1;        // o_empty wait parity (completes once per tile)
      while (w.next(u)) {
        mbar_wait(qk_full, ph);
        tc_fence_after();
        for (int t = 0; t < 2; ++t) {   // S buffers are free: the previous unit's p_full[t] was consumed below
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + t * LPAD, make_smem_desc(aQ + t * 16384 + k * 32, 16, 1024),
                      make_smem_desc(aK + k * 32, 16, 1024), idesc_s, k > 0 ? 1u : 0u);
          umma_commit(&s_full[t]);
        }
        umma_commit(qk_empty);
        mbar_wait(v_full, ph);
        for (int t = 0; t < 2; ++t) {
          mbar_wait(&p_full[t], ph);
          mbar_wait(o_empty, oe);
          oe ^= 1;
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < LPAD / 16; ++k)
            umma_bf16(tmem_base + Cfg::TMEM_O, make_smem_desc(aP + t * Cfg::P_BYTES + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                      make_smem_desc(aV + k * 2048, 8192, 1024), idesc_o, k > 0 ? 1u : 0u);
          umma_commit(&o_full[t]);
        }
        umma_commit(v_empty);
        ph ^= 1;
      }
    }
    __syncwarp();
  } else {
    const int t = (warp - 2) >> 2;             // query tile of this warpgroup
    const int quad = warp & 3;
    const int r = quad * 32 + lane;            // row inside the tile
    const int slot_in_tile = r / LQS, q = r % LQS;
    const int g = 2 * slot_in_tile + t;        // sample slot of this row
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint32_t t_s = lane_base + (uint32_t)(t * LPAD), t_o = lane_base + (uint32_t)Cfg::TMEM_O;
    const float scale2 = a.scale * 1.4426950408889634f;
    const bool drop_on = a.dropout_p > 0.f;
    const float inv_keep = drop_on ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
    const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
    uint8_t* myP = sP + t * Cfg::P_BYTES + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    XWalker<GMAX> w(a, item0, item1);
    XUnit u;
    uint32_t ph = 0;
    while (w.next(u)) {
      const bool valid = slot_in_tile < PER_TILE && g < u.ns;
      const bool wv = __any_sync(0xffffffffu, valid);   // tcgen05.ld is warp-collective: decide per warp, mask per thread
      const int b = valid ? a.kv_samples[u.first + g] : 0;
      // dropout mask: element index ((b, h, q) row) * LKE + key with the even row stride LKE (attention.cu::drop_keep)
      constexpr int LKE = (LK + 1) & ~1;
      const uint64_t pair_base = ((((uint64_t)b * a.H + u.h) * LQS + q) * (uint64_t)LKE) >> 1;
      const uint32_t pb_lo = (uint32_t)pair_base, pb_hi = (uint32_t)(pair_base >> 32);
      mbar_wait(&s_full[t], ph);
      tc_fence_after();
      float m = -INFINITY, sum = 0.f;
      if (wv) {
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int c0 = 0; c0 < LPAD; c0 += 32) {
          uint32_t v[32];
          if (c0 + 32 <= LPAD) xt_ld32(t_s + c0, v);
          else tmem_ld_32x32_16(t_s + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (c0 + e < KLEN) m4[e & 3] = fmaxf(m4[e & 3], __uint_as_float(v[e]));
        }
        m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale2;   // scale2 > 0: max commutes with the scaling
      }
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c0 = 0; c0 < LPAD; c0 += 32) {
        uint32_t v[32];
        if (wv) {
          if (c0 + 32 <= LPAD) xt_ld32(t_s + c0, v);
          else tmem_ld_32x32_16(t_s + c0, v);
          tmem_ld_wait();
        }
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          if (c0 + g8 * 8 < LPAD) {
            float p[8];
#pragma unroll
            for (int e = 0; e < 8; e += 2) {
              const int j = c0 + g8 * 8 + e;   // even
              float p0 = 0.f, p1 = 0.f;
              if (valid && j < KLEN) {
                p0 = ex2_approx(fmaf(__uint_as_float(v[g8 * 8 + e]), scale2, -m));
                if (j + 1 < KLEN) p1 = ex2_approx(fmaf(__uint_as_float(v[g8 * 8 + e + 1]), scale2, -m));
                s4[e & 3] += p0;
                s4[(e + 1) & 3] += p1;
                if (drop_on) {
                  const uint32_t lo = pb_lo + (uint32_t)((K0 + j) >> 1);   // key index inside the whole row
                  const uint32_t keep = drop_keep_pair(seed_mix, lo, pb_hi + (lo < pb_lo ? 1u : 0u), thr);
                  p0 = (keep & 1u) ? p0 * inv_keep : 0.f;
                  p1 = (keep & 2u) ? p1 * inv_keep : 0.f;
                }
              }
              p[e] = p0;
              p[e + 1] = p1;
            }
            const int col8 = c0 + g8 * 8;
            st_bf16x8(myP + (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4), p);
          }
        }
      }
      sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[t]);
      mbar_wait(&o_full[t], ph);
      tc_fence_after();
      uint32_t o[2][32];
      if (wv) {
        tmem_ld_32x32(t_o, o[0]);
        tmem_ld_32x32(t_o + 32, o[1]);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
      if (valid) {
        const float inv = 1.0f / sum;
        bf16* orow = a.out + ((int64_t)b * LQS + q) * a.o_stride + u.h * XT_HD;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            float vv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) vv[k] = __uint_as_float(o[hh][e + k]) * inv;
            st_bf16x8((uint8_t*)(orow + hh * 32 + e), vv);
          }
        if (a.lse) a.lse[((int64_t)b * a.H + u.h) * LQS + q] = (m + log2f(sum)) * 0.6931471805599453f;
      }
      ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


// ================================================================================================ fused backward
// One kernel for dQ, dK and dV.  A unit is (image, head, chunk of <= 3 samples): ONE 128-row query tile (three 40-row slots).
// S = Q K^T and dP = dO V^T are computed once, P~ (dropout mask and 1/(1-p) applied) and dS are written to shared memory
// once, and dQ = dS K (dS read K-major), dK = dS^T Q, dV = P~^T dO (the same buffers read MN-major, keys as the M dimension
// in two 128-key tiles) are issued from them into the TMEM columns S / dP occupied, so the elementwise stage runs once per
// (query, key) pair.  Later chunks of the same image add their dK / dV to the rows the first chunk stored (same CTA, same
// thread per row: ordered without synchronisation).
template <int LQS, int LK>
struct XFusedCfg {
  static constexpr int GMAX = 3;
  static_assert(GMAX * LQS <= 128, "three samples per query tile");
  // Images with more than 208 tokens (384 px: 577, 480 px: 901) are processed one key block per launch, like the ViT backward
  // (attention_tc.cu::VitFusedCfg): P = 2^(S - lse) needs no online softmax; dQ accumulates across the launches.
  static constexpr int NB = KeyBlocks::nb(LK);
  static constexpr bool BLOCKED = NB > 1;
  static constexpr int KBS = KeyBlocks::kbs(LK);
  static constexpr int LAST = KeyBlocks::last(LK);
  static constexpr int LPAD = KeyBlocks::lpad(LK);
  static constexpr int NM = (LPAD + 127) / 128;
  static constexpr int KV_BYTES = LPAD * 128;
  static constexpr int PD_BYTES = 2 * NM * 16384;
  static constexpr int SMEM = 2 * 16384 + 2 * KV_BYTES + 2 * PD_BYTES + 128;
  static constexpr int TM_DQ = 0, TM_DK = 64, TM_DV = 64 + 64 * NM, TM_END = 64 + 128 * NM;
  static constexpr int UNITS = TM_END / 32;
  static_assert(LAST <= LPAD && (NB == 1 || KBS % 2 == 0) && 2 * LPAD <= 512 && TM_END <= 512, "TMEM / dropout pairs");
  static_assert(SMEM <= 232448, "shared memory");
};
static_assert(XFusedCfg<40, 577>::NB == 3 && XFusedCfg<40, 577>::LAST == 193 && XFusedCfg<40, 577>::LPAD == 208, "384 px");
static_assert(XFusedCfg<40, 901>::NB == 5 && XFusedCfg<40, 901>::LAST == 133 && XFusedCfg<40, 901>::LPAD == 192, "480 px");

template <int LQS, int LK, int KB>
__global__ void __launch_bounds__(XTF_THREADS, 1)
xattn_bwd_fused_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                          const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                          const __grid_constant__ CUtensorMap map_dq, const __grid_constant__ CUtensorMap map_dk,
                          const __grid_constant__ CUtensorMap map_dv, const XAttnArgs a) {
  using Cfg = XFusedCfg<LQS, LK>;
  static_assert((LQS * 128) % 1024 == 0, "a sample's slot must start on a swizzle-pattern boundary (TMA source of the dQ stores)");
  constexpr int LPAD = Cfg::LPAD, GMAX = Cfg::GMAX, NM = Cfg::NM;
  constexpr int K0 = KB * Cfg::KBS;                                   // first key of this launch's block
  constexpr int KLEN = KB == Cfg::NB - 1 ? Cfg::LAST : Cfg::KBS;      // its keys
  static_assert(KB < Cfg::NB, "key block");
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* sQ = smem;
  uint8_t* sdO = sQ + 16384;
  uint8_t* sK = sdO + 16384;
  uint8_t* sV = sK + Cfg::KV_BYTES;
  uint8_t* sdS = sV + Cfg::KV_BYTES;
  uint8_t* sP = sdS + Cfg::PD_BYTES;
  uint64_t* bars = (uint64_t*)(sP + Cfg::PD_BYTES);
  uint64_t *kv_full = bars, *kv_empty = bars + 1, *qdo_full = bars + 2, *qdo_empty = bars + 3, *sd_full = bars + 4,
           *ds_full = bars + 5, *out_full = bars + 6, *out_empty = bars + 7;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 2 * 16384 / 16; i += blockDim.x) ((uint4*)sQ)[i] = make_uint4(0u, 0u, 0u, 0u);  // unused slots stay finite
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_do);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    tma_prefetch_desc(&map_dq);
    tma_prefetch_desc(&map_dk);
    tma_prefetch_desc(&map_dv);
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    mbar_init(qdo_full, 1);
    mbar_init(qdo_empty, 1);
    mbar_init(sd_full, 1);
    mbar_init(ds_full, 16);
    mbar_init(out_full, 1);
    mbar_init(out_empty, 16);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  constexpr uint32_t TM_S = 0, TM_DP = LPAD;

  const int n_items = a.Bkv * a.H;
  const int item0 = blockIdx.x * a.items_per_cta;
  const int item1 = min(n_items, item0 + a.items_per_cta);

  // Every role walks the same unit sequence; K / V are loaded once per item (image, head), Q / dO once per unit.
  if (warp == 0) {
    if (lane == 0) {
      XWalker<GMAX, true> w(a, item0, item1);
      XUnit u;
      uint32_t up = 0, ip = 0;   // unit parity, item parity
      int cur = -1;
      while (w.next(u)) {
        const int id = u.h * a.Bkv + u.r;
        if (id != cur) {
          mbar_wait_relaxed(kv_empty, ip ^ 1);
          mbar_arrive_expect_tx(kv_full, 2 * Cfg::KV_BYTES);
          tma_load_2d(sK, &map_k, kv_full, u.h * XT_HD, u.r * LK + K0);
          tma_load_2d(sV, &map_v, kv_full, u.h * XT_HD, u.r * LK + K0);
          ip ^= 1;
          cur = id;
        }
        mbar_wait_relaxed(qdo_empty, up ^ 1);
        mbar_arrive_expect_tx(qdo_full, 2 * u.ns * LQS * 128);
        for (int g = 0; g < u.ns; ++g) {
          const int b = a.kv_samples[u.first + g];
          tma_load_2d(sQ + g * (LQS * 128), &map_q, qdo_full, u.h * XT_HD, b * LQS);
          tma_load_2d(sdO + g * (LQS * 128), &map_do, qdo_full, u.h * XT_HD, b * LQS);
        }
        up ^= 1;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, LPAD, 0, 0);
      constexpr uint32_t idesc_dq = make_idesc_bf16(128, XT_HD, 0, 1);
      constexpr uint32_t idesc_dkv = make_idesc_bf16(128, XT_HD, 1, 1);
      const uint32_t aQ = smem_u32(sQ), adO = smem_u32(sdO), aK = smem_u32(sK), aV = smem_u32(sV), adS = smem_u32(sdS),
                     aP = smem_u32(sP);
      XWalker<GMAX, true> w(a, item0, item1);
      XUnit u;
      uint32_t up = 0, ip = 1;
      int cur = -1;
      bool have = w.next(u);
      while (have) {
        const int id = u.h * a.Bkv + u.r;
        if (id != cur) {
          ip ^= 1;
          mbar_wait(kv_full, ip);
          cur = id;
        }
        const int ns = u.ns;
        XUnit nu;
        have = w.next(nu);
        const bool last_of_item = !have || (nu.h * a.Bkv + nu.r) != id;
        mbar_wait(qdo_full, up);
        mbar_wait(out_empty, up ^ 1);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base + TM_S, make_smem_desc(aQ + k * 32, 16, 1024), make_smem_desc(aK + k * 32, 16, 1024), idesc_s,
                    k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base + TM_DP, make_smem_desc(adO + k * 32, 16, 1024), make_smem_desc(aV + k * 32, 16, 1024), idesc_s,
                    k > 0 ? 1u : 0u);
        umma_commit(sd_full);
        mbar_wait(ds_full, up);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < LPAD / 16; ++k)
          umma_bf16(tmem_base + Cfg::TM_DQ, make_smem_desc(adS + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                    make_smem_desc(aK + k * 2048, 8192, 1024), idesc_dq, k > 0 ? 1u : 0u);
        const int nk = (ns * LQS + 15) / 16;
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          for (int k = 0; k < nk; ++k)
            umma_bf16(tmem_base + Cfg::TM_DK + m * 64, make_smem_desc(adS + m * 32768 + k * 2048, 16384, 1024),
                      make_smem_desc(aQ + k * 2048, 8192, 1024), idesc_dkv, k > 0 ? 1u : 0u);
          for (int k = 0; k < nk; ++k)
            umma_bf16(tmem_base + Cfg::TM_DV + m * 64, make_smem_desc(aP + m * 32768 + k * 2048, 16384, 1024),
                      make_smem_desc(adO + k * 2048, 8192, 1024), idesc_dkv, k > 0 ? 1u : 0u);
        }
        umma_commit(out_full);
        umma_commit(qdo_empty);
        if (last_of_item) umma_commit(kv_empty);
        up ^= 1;
        u = nu;
      }
    }
    __syncwarp();
  } else {
    const int wg = (warp - 2) >> 2;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const int slot = r / LQS, q = r % LQS;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const float scale2 = a.scale * 1.4426950408889634f;
    const bool drop_on = a.dropout_p > 0.f;
    const float inv_keep = drop_on ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
    const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
    uint8_t* myS = sdS + (r >> 3) * 1024 + (r & 7) * 128;
    uint8_t* myP = sP + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    constexpr int N16 = LPAD / 16;             // 16-column chunks of a score row, split in four runs
    const int ch_lo = (wg * N16) / 4, ch_hi = ((wg + 1) * N16) / 4;
    constexpr int LKE = (LK + 1) & ~1;
    const bool elected = threadIdx.x == 64;   // issues every TMA store of this CTA (bulk groups are per thread)
    XWalker<GMAX, true> w(a, item0, item1);
    XUnit u;
    uint32_t up = 0;
    int cur = -1, chunk_of_item = 0;
    while (w.next(u)) {
      const int id = u.h * a.Bkv + u.r;
      chunk_of_item = id == cur ? chunk_of_item + 1 : 0;
      cur = id;
      const bool valid = slot < GMAX && slot < u.ns;
      const bool wv = __any_sync(0xffffffffu, valid);
      const int b = valid ? a.kv_samples[u.first + slot] : 0;
      const int64_t st_row = ((int64_t)b * a.H + u.h) * LQS + q;
      const float lse2 = valid ? __ldg(a.lse + st_row) * 1.4426950408889634f : 0.f;
      const float dl = valid ? __ldg(a.delta + st_row) : 0.f;
      const uint64_t pair_base = ((uint64_t)st_row * (uint64_t)LKE) >> 1;
      const uint32_t pb_lo = (uint32_t)pair_base, pb_hi = (uint32_t)(pair_base >> 32);
      mbar_wait(sd_full, up);
      tc_fence_after();
      // the previous unit's output stores still read the P / dS buffers this unit is about to overwrite
      if (elected) tma_store_wait_read<0>();
      named_bar_sync(1, 512);
#pragma unroll 1
      for (int ch = ch_lo; ch < ch_hi; ++ch) {
        const int c0 = ch * 16;
        uint32_t vs[32], vp[32];                 // [0..15] used
        if (wv) {   // tcgen05.ld is warp-collective: decide per warp, mask per thread
          tmem_ld_32x32_16(lane_base + TM_S + c0, vs);
          tmem_ld_32x32_16(lane_base + TM_DP + c0, vp);
          tmem_ld_wait();
        }
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          float ds[8], pp[8];
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            const int j = c0 + g8 * 8 + e;   // even
            float d0 = 0.f, d1 = 0.f, p0 = 0.f, p1 = 0.f;
            if (valid && j < KLEN) {
              p0 = ex2_approx(fmaf(__uint_as_float(vs[g8 * 8 + e]), scale2, -lse2));
              p1 = j + 1 < KLEN ? ex2_approx(fmaf(__uint_as_float(vs[g8 * 8 + e + 1]), scale2, -lse2)) : 0.f;
              float k0 = 1.f, k1 = 1.f;
              if (drop_on) {
                const uint32_t lo = pb_lo + (uint32_t)((K0 + j) >> 1);   // key index inside the whole row (K0 is even)
                const uint32_t keep = drop_keep_pair(seed_mix, lo, pb_hi + (lo < pb_lo ? 1u : 0u), thr);
                k0 = (keep & 1u) ? inv_keep : 0.f;
                k1 = (keep & 2u) ? inv_keep : 0.f;
              }
              d0 = p0 * (__uint_as_float(vp[g8 * 8 + e]) * k0 - dl);
              d1 = p1 * (__uint_as_float(vp[g8 * 8 + e + 1]) * k1 - dl);
              p0 *= k0;
              p1 *= k1;
            }
            ds[e] = d0;
            ds[e + 1] = d1;
            pp[e] = p0;
            pp[e + 1] = p1;
          }
          const int col8 = c0 + g8 * 8;
          const int off8 = (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4);
          st_bf16x8(myS + off8, ds);
          st_bf16x8(myP + off8, pp);
        }
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
      mbar_wait(out_full, up);
      tc_fence_after();
      // Outputs (see attention_tc.cu's fused backward): every 64-column block is staged as bf16 in a SWIZZLE_128B [128 x 64]
      // tile — dK / dV in the consumed P buffer, dQ in block 0 of the consumed dS buffer — and stored by TMA: dQ one box of
      // LQS rows per stacked sample, dK / dV through [image, key, column] maps that clip at the image's last key; later
      // chunks of the same image go out as TMA reduce-adds onto the first chunk's rows.
      // Units per warpgroup: 0: {0, 1, 2} (dQ and the first dK unit), 1: {3, 4, 5}, 2: {6, 7}, 3: {8, 9} (UNITS = 10; 6: only 0 and 1).
      static_assert(Cfg::UNITS == 10 || Cfg::UNITS == 6, "unit lists below");
      const int n_mine = wg < 2 ? 3 : (Cfg::UNITS == 10 ? 2 : 0);
      const int u_first = wg < 2 ? 3 * wg : 2 + 2 * wg;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (i >= n_mine) continue;               // warp-uniform
        const int un = u_first + i;
        uint32_t o[32];
        xt_ld32(lane_base + (uint32_t)(un * 32), o);
        tmem_ld_wait();
        uint8_t* blk;
        float mul = a.scale;
        int half = un & 1;
        if (un < 2) {
          blk = sdS;
        } else {
          const bool is_dv = un >= 2 + 2 * NM;
          const int uu = is_dv ? un - 2 - 2 * NM : un - 2;
          blk = sP + ((is_dv ? NM : 0) + (uu >> 1)) * 16384;
          half = uu & 1;
          if (is_dv) mul = 1.0f;
        }
        uint8_t* row = blk + (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
        for (int e = 0; e < 32; e += 8) {
          float vv[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) vv[k] = u.ns > 0 ? __uint_as_float(o[e + k]) * mul : 0.f;   // no samples: accumulators never written
          st_bf16x8(row + (((half * 4 + (e >> 3)) ^ sw) << 4), vv);
        }
      }
      tc_fence_before();                         // every TMEM read of this warp is complete (tcgen05.wait::ld above)
      __syncwarp();
      if (lane == 0) mbar_arrive(out_empty);
      fence_proxy_async();
      named_bar_sync(1, 512);
      if (elected) {
        for (int g = 0; g < u.ns; ++g) {
          if (KB == 0) tma_store_2d(&map_dq, sdS + g * (LQS * 128), u.h * XT_HD, a.kv_samples[u.first + g] * LQS);
          else tma_reduce_add_2d(&map_dq, sdS + g * (LQS * 128), u.h * XT_HD, a.kv_samples[u.first + g] * LQS);   // earlier key blocks' launches
        }
        if (chunk_of_item == 0) {
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            tma_store_3d(&map_dk, sP + m * 16384, u.h * XT_HD, m * 128, u.r);
            tma_store_3d(&map_dv, sP + (NM + m) * 16384, u.h * XT_HD, m * 128, u.r);
          }
        } else {
          tma_store_wait_all<0>();               // the earlier chunks' dK / dV have landed
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            tma_reduce_add_3d(&map_dk, sP + m * 16384, u.h * XT_HD, m * 128, u.r);
            tma_reduce_add_3d(&map_dv, sP + (NM + m) * 16384, u.h * XT_HD, m * 128, u.r);
          }
        }
        tma_store_commit();
      }
      up ^= 1;
    }
    if (elected) tma_store_wait_all<0>();        // shared memory must outlive the reads; results complete before exit
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------ host
// Instantiated shapes: 40 text tokens attending to 197 image tokens (BASELINE configs[1]), up to 6 samples per chunk; and
// to 577 / 901 image tokens (384 / 480 px) in key blocks, where the forward needs the part scratch.  The backward writes no
// dS dump.
bool cross_attention_tc_supported(const xfm_attn_params* p, bool bwd) {
  const bool blocked = p->Lk == 577 || p->Lk == 901;
  return p->head_dim == XT_HD && p->Lq == 40 && (p->Lk == 197 || blocked) &&
         (bwd ? !p->ds_dump : (!blocked || (p->part_out && p->part_lse))) && !p->kmask && !p->bias && p->kv_offsets && p->kv_samples &&
         p->Bkv > 0 && ((uintptr_t)p->q & 15) == 0 && ((uintptr_t)p->k & 15) == 0 && ((uintptr_t)p->v & 15) == 0 &&
         ((p->q_stride | p->k_stride | p->v_stride | p->o_stride) & 7) == 0;
}

static void xt_fill(const xfm_attn_params* p, XAttnArgs& a) {
  a.out = (bf16*)p->out; a.o_stride = p->o_stride; a.lse = p->lse;
  a.kv_offsets = p->kv_offsets; a.kv_samples = p->kv_samples;
  a.B = p->B; a.Bkv = p->Bkv; a.H = p->H; a.scale = p->scale; a.dropout_p = p->dropout_p; a.seed = p->dropout_seed; a.salt = seed_salt_ptr();
  a.delta = p->delta;
  a.dq = (bf16*)p->dq; a.dk = (bf16*)p->dk; a.dv = (bf16*)p->dv;
  a.dq_stride = p->dq_stride; a.dk_stride = p->dk_stride; a.dv_stride = p->dv_stride;
  const int n_items = a.Bkv * a.H;
  const int ctas = n_items < num_sms() ? n_items : num_sms();
  a.items_per_cta = (n_items + ctas - 1) / ctas;
}

template <int LQS, int LK, int GMAX, int KB>
static int xt_launch_fwd_block(const xfm_attn_params* p, const XAttnArgs& a0, const CUtensorMap& mq, const CUtensorMap& mk,
                               const CUtensorMap& mv, cudaStream_t s) {
  using Cfg = XCfg<LQS, LK, GMAX>;
  XAttnArgs a = a0;
  if (Cfg::BLOCKED) {   // this block's partial output / lse
    a.out = (bf16*)p->part_out + KB * (int64_t)a.B * LQS * (a.H * XT_HD);
    a.o_stride = (int64_t)a.H * XT_HD;
    a.lse = p->part_lse + KB * (int64_t)a.B * a.H * LQS;
  }
  auto kern = xattn_fwd_tc_kernel<LQS, LK, GMAX, KB>;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_FWD);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  const int n_items = a.Bkv * a.H;
  const int grid = (n_items + a.items_per_cta - 1) / a.items_per_cta;
  kern<<<grid, XT_THREADS, Cfg::SMEM_FWD, s>>>(mq, mk, mv, a);
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if constexpr (KB + 1 < Cfg::NB) return xt_launch_fwd_block<LQS, LK, GMAX, KB + 1>(p, a0, mq, mk, mv, s);
  return 0;
}

template <int LQS, int LK, int GMAX>
static int xt_launch_fwd(const xfm_attn_params* p, cudaStream_t s) {
  using Cfg = XCfg<LQS, LK, GMAX>;
  XAttnArgs a;
  xt_fill(p, a);
  const uint64_t cols = (uint64_t)a.H * XT_HD;
  CUtensorMap mq, mk, mv;
  int rc = encode_rows(&mq, p->q, cols, (uint64_t)a.B * LQS, p->q_stride, LQS);
  if (!rc) rc = encode_rows(&mk, p->k, cols, (uint64_t)a.Bkv * LK, p->k_stride, Cfg::LPAD);
  if (!rc) rc = encode_rows(&mv, p->v, cols, (uint64_t)a.Bkv * LK, p->v_stride, Cfg::LPAD);
  if (rc) return rc;
  rc = xt_launch_fwd_block<LQS, LK, GMAX, 0>(p, a, mq, mk, mv, s);
  if (rc || !Cfg::BLOCKED) return rc;
  return launch_merge_parts(Cfg::NB, p->part_out, p->part_lse, p->out, p->o_stride, p->lse, a.B, a.H, LQS, s);
}

int cross_attention_fwd_tc(const xfm_attn_params* p, cudaStream_t s) {
  switch (p->Lk) {
    case 577: return xt_launch_fwd<40, 577, 6>(p, s);
    case 901: return xt_launch_fwd<40, 901, 6>(p, s);
  }
  return xt_launch_fwd<40, 197, 6>(p, s);
}

// Fused backward, one launch per key block.
template <int LQS, int LK, int KB>
static int xt_launch_fused_block(const xfm_attn_params* p, const XAttnArgs& a, const CUtensorMap& mq, const CUtensorMap& mdo,
                                 const CUtensorMap& mk_l, const CUtensorMap& mv_l, const CUtensorMap& m_dq, cudaStream_t s) {
  using FCfg = XFusedCfg<LQS, LK>;
  constexpr int K0 = KB * FCfg::KBS, KLEN = KB == FCfg::NB - 1 ? FCfg::LAST : FCfg::KBS;
  auto kf = xattn_bwd_fused_tc_kernel<LQS, LK, KB>;
  static bool fattr = false;
  if (!fattr) {
    cudaError_t e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, FCfg::SMEM);
    if (e != cudaSuccess) return (int)e;
    fattr = true;
  }
  const uint64_t cols = (uint64_t)a.H * XT_HD;
  CUtensorMap m_dk, m_dv;   // this block's key rows of every image
  int rc = encode_rows_3d(&m_dk, (const bf16*)p->dk + (int64_t)K0 * p->dk_stride, cols, KLEN, a.Bkv, p->dk_stride, LK);
  if (!rc) rc = encode_rows_3d(&m_dv, (const bf16*)p->dv + (int64_t)K0 * p->dv_stride, cols, KLEN, a.Bkv, p->dv_stride, LK);
  if (rc) return rc;
  const int n_items_f = a.Bkv * a.H;
  const int grid_f = (n_items_f + a.items_per_cta - 1) / a.items_per_cta;
  kf<<<grid_f, XTF_THREADS, FCfg::SMEM, s>>>(mq, mdo, mk_l, mv_l, m_dq, m_dk, m_dv, a);
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if constexpr (KB + 1 < FCfg::NB) return xt_launch_fused_block<LQS, LK, KB + 1>(p, a, mq, mdo, mk_l, mv_l, m_dq, s);
  return 0;
}

template <int LQS, int LK>
static int xt_launch_fused(const xfm_attn_params* p, cudaStream_t s) {
  using FCfg = XFusedCfg<LQS, LK>;
  XAttnArgs a;
  xt_fill(p, a);
  const uint64_t cols = (uint64_t)a.H * XT_HD;
  CUtensorMap mq, mdo, mk_l, mv_l, m_dq;
  int rc = encode_rows(&mq, p->q, cols, (uint64_t)a.B * LQS, p->q_stride, LQS);
  if (!rc) rc = encode_rows(&mdo, p->dout, cols, (uint64_t)a.B * LQS, p->do_stride, LQS);
  if (!rc) rc = encode_rows(&mk_l, p->k, cols, (uint64_t)a.Bkv * LK, p->k_stride, FCfg::LPAD);
  if (!rc) rc = encode_rows(&mv_l, p->v, cols, (uint64_t)a.Bkv * LK, p->v_stride, FCfg::LPAD);
  if (!rc) rc = encode_rows(&m_dq, p->dq, cols, (uint64_t)a.B * LQS, p->dq_stride, LQS);
  if (rc) return rc;
  return xt_launch_fused_block<LQS, LK, 0>(p, a, mq, mdo, mk_l, mv_l, m_dq, s);
}

int cross_attention_bwd_tc(const xfm_attn_params* p, cudaStream_t s) {
  if ((((uintptr_t)p->dout | (uintptr_t)p->dq | (uintptr_t)p->dk | (uintptr_t)p->dv) & 15) ||
      ((p->do_stride | p->dq_stride | p->dk_stride | p->dv_stride) & 7)) {
    set_error("cross attention bwd: operands must be 16-byte aligned with row strides that are multiples of 8");
    return XFM_ERR_BAD_ARG;
  }
  switch (p->Lk) {
    case 577: return xt_launch_fused<40, 577>(p, s);
    case 901: return xt_launch_fused<40, 901>(p, s);
  }
  return xt_launch_fused<40, 197>(p, s);
}

}  // namespace xfm
