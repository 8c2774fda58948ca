// K2 — BEiT / ViT self-attention forward on tcgen05 + TMEM + TMA (head_dim 64, Lq = Lk <= 208 tokens: one pass, no
// online softmax).  Reference arithmetic: beit2.py:126-166  (q*d^-1/2) k^T + relative_position_bias -> softmax -> @ v.
//
// One persistent CTA per SM walks a contiguous range of (head, sample) items; an item is NT query tiles of 128 rows.
//   warp 0      TMA: Q (NT*128 rows), K (LPAD rows), V (LPAD rows) boxes straight out of the fused qkv activation
//               (row stride 3*D) into SWIZZLE_128B shared-memory tiles.
//   warp 1      one thread issues tcgen05.mma.  Tiles ping-pong between two TMEM score buffers:
//               S[tau&1] = Q_t K^T (M=128, N=LPAD, K=64); O = P[tau&1] V (M=128, N=64, K=LPAD) into a third TMEM
//               region, so the score MMA of tile tau+2 is issued as soon as tile tau's probabilities are written and
//               overlaps the softmax of tile tau+1.
//   warps 2..9  two softmax warpgroups (tiles of even / odd parity), thread = query row.  Pass 1 pulls S out of TMEM,
//               applies scale + relative-position bias, writes the logits back to TMEM and tracks the row maximum;
//               pass 2 re-reads them, exponentiates (ex2), accumulates the row sum and stores bf16 P as the K-major A
//               operand of the second MMA; finally O / rowsum -> global, lse.
// The bias is gathered from the head's (2W-1)^2+3 entry table held in shared memory through the closed form of
// beit2.py:104-114's index: with the window side W a template constant the column part of the index is an immediate,
// so the gather is one LDS per score and the [H, N, N] bias tensor is never read.
// Scores, probabilities and the bias tensor never touch HBM.
#include <cstdio>
#include <cstdlib>
#include "common.cuh"
#include "internal.h"

namespace xfm {

constexpr int TC_HD = 64;
constexpr int TC_THREADS = 64 + 256;
constexpr int TCF_THREADS = 64 + 512;   // fused backward: four element-wise / drain warpgroups (four warps per scheduler)

struct VitAttnArgs {
  bf16* out;
  int64_t o_stride;
  float* lse;            // [B, H, L] natural-log sum-exp of the scaled + biased logits
  const float* table;    // [T, H] relative_position_bias_table or null
  int B, H;
  float scale;
  int items_per_cta;
  int ctas_per_head;     // key-blocked shapes: a CTA walks items of ONE head
  long long* prof;       // XFM_ATTN_PROF=1: per-phase clock64 totals of CTA 0's first softmax warp (null otherwise)
};

// Forward configuration.  Up to 208 keys: an item is one (sample, head) with all its query tiles.  More (384 px,
// W = 24, L = 577; 480 px, W = 30, L = 901): one launch per key block (KeyBlocks) writes a block-normalised partial output
// and the block's lse; the
// partials are merged afterwards (merge_parts_kernel).  An item is then a PAIR of query tiles of a (sample, head), a CTA
// stays on one head (one copy of the bias table, loaded once), and the K / V block is re-loaded per item (L2 hits).
template <int W>
struct VitFwdCfg {
  static constexpr int L = W * W + 1;
  static constexpr int NB = KeyBlocks::nb(L);
  static constexpr bool BLOCKED = NB > 1;
  static constexpr int KBS = KeyBlocks::kbs(L);
  static constexpr int LAST = KeyBlocks::last(L);
  static constexpr int LPAD = KeyBlocks::lpad(L);
  static constexpr int NT = BLOCKED ? 2 : (L + 127) / 128;          // query tiles per item
  static constexpr int NTP = BLOCKED ? ((L + 127) / 128 + 1) / 2 : 1;  // items per (sample, head)
  static constexpr int NKB = (LPAD + 63) / 64;
  static constexpr int T = (2 * W - 1) * (2 * W - 1) + 3;
  static constexpr int OFFMAX = (W - 1) * (2 * W - 1) + (W - 1);
  static constexpr int TAB_FLOATS = (OFFMAX + 1 + T + 7) & ~7;  // [OFFMAX+1 copies of table[T-3]] ++ [table]
  static constexpr int NTAB = BLOCKED ? 1 : 2;
  static constexpr int Q_BYTES = NT * 128 * 128;
  static constexpr int KV_BYTES = LPAD * 128;
  static constexpr int P_BYTES = NKB * 16384;
  static constexpr int SMEM_BYTES = Q_BYTES + 2 * KV_BYTES + 2 * P_BYTES + NTAB * TAB_FLOATS * 4 + 128;
  static constexpr int TMEM_O = 2 * LPAD;  // O accumulator columns; S buffers at 0 and LPAD
  static_assert(LAST <= LPAD && 2 * LPAD + 64 <= 512, "scores of two tiles + one output tile must fit TMEM");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
};
static_assert(VitFwdCfg<24>::NB == 3 && VitFwdCfg<24>::LAST == 193 && VitFwdCfg<24>::LPAD == 208, "384 px: 192 / 192 / 193");
static_assert(VitFwdCfg<30>::NB == 5 && VitFwdCfg<30>::LAST == 133 && VitFwdCfg<30>::LPAD == 192, "480 px: 4 x 192 + 133");
// column part of the relative-position index (beit2.py:104-108) of key j >= 1
template <int W>
XFM_DEVINL constexpr int rel_off(int j) {
  const int jj = (j < W * W + 1 ? j : W * W) - 1;
  return (jj / W) * (2 * W - 1) + jj % W;
}

XFM_DEVINL void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
XFM_DEVINL void tmem_st_32x32_16(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
XFM_DEVINL void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }


// HAS_TAB = false (no relative-position bias: the VQ-KD tokenizer's ViT): no bias gather, and the first pass only takes the
// maximum of the raw scores — nothing is written back to TMEM — because scale * s - m is one FMA in the second pass.
template <int W, int KB, bool HAS_TAB>
__global__ void __launch_bounds__(TC_THREADS, 1)
vit_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                       const __grid_constant__ CUtensorMap map_v, const VitAttnArgs a) {
  using Cfg = VitFwdCfg<W>;
  constexpr int L = Cfg::L, LPAD = Cfg::LPAD, NT = Cfg::NT;
  constexpr bool BLOCKED = Cfg::BLOCKED;
  constexpr int K0 = KB * Cfg::KBS;                                   // first key of this launch's block
  constexpr int KLEN = KB == Cfg::NB - 1 ? Cfg::LAST : Cfg::KBS;      // its keys
  static_assert(KB < Cfg::NB, "key block");
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();  // SWIZZLE_128B tiles need the 1024-byte alignment the declaration asks for
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::Q_BYTES;
  uint8_t* sV = sK + Cfg::KV_BYTES;
  uint8_t* sP = sV + Cfg::KV_BYTES;                          // [2][P_BYTES]
  float* tabs = (float*)(sP + 2 * Cfg::P_BYTES);             // [2 warpgroups][TAB_FLOATS] (key-blocked: one shared copy)
  uint64_t* bars = (uint64_t*)(tabs + Cfg::NTAB * Cfg::TAB_FLOATS);
  uint64_t *qk_full = bars, *qk_empty = bars + 1, *v_full = bars + 2, *v_empty = bars + 3;
  uint64_t *s_full = bars + 4, *p_full = bars + 6, *o_full = bars + 8, *o_empty = bars + 10;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 11);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
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
      mbar_init(&o_full[t], 1);  // one per tile parity: a warpgroup must never see the other parity's completion
    }
    mbar_init(o_empty, 4);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // item -> (head, sample, first query row).  Key-blocked: the CTA's head is fixed, items = (sample, tile pair) of that head.
  const int h_cta = BLOCKED ? (int)blockIdx.x / a.ctas_per_head : 0;
  const int n_items = BLOCKED ? a.B * Cfg::NTP : a.B * a.H;
  const int item0 = (BLOCKED ? (int)blockIdx.x % a.ctas_per_head : (int)blockIdx.x) * a.items_per_cta;
  const int item1 = min(n_items, item0 + a.items_per_cta);
  const int n_tiles = (item1 - item0) * NT;
  auto decode = [&](int it, int& h, int& b, int& q0) {
    if (BLOCKED) { h = h_cta; b = it / Cfg::NTP; q0 = (it % Cfg::NTP) * (NT * 128); }
    else { h = it / a.B; b = it % a.B; q0 = 0; }
  };
  if (BLOCKED) {   // the head never changes: one table copy, loaded here by every thread (log2 domain)
    for (int i = threadIdx.x; i < Cfg::T; i += blockDim.x)
      tabs[Cfg::OFFMAX + 1 + i] = a.table ? __ldg(a.table + (int64_t)i * a.H + h_cta) * 1.4426950408889634f : 0.f;
    const float row0 = a.table ? __ldg(a.table + (int64_t)(Cfg::T - 3) * a.H + h_cta) * 1.4426950408889634f : 0.f;
    for (int i = threadIdx.x; i <= Cfg::OFFMAX; i += blockDim.x) tabs[i] = row0;
    __syncthreads();
  }

  if (warp == 0) {
    if (lane == 0) {
      for (int it = item0; it < item1; ++it) {
        const uint32_t ph = (uint32_t)(it - item0) & 1u;
        int h, b, q0;
        decode(it, h, b, q0);
        mbar_wait_relaxed(qk_empty, ph ^ 1);
        mbar_arrive_expect_tx(qk_full, Cfg::Q_BYTES + Cfg::KV_BYTES);
        tma_load_2d(sQ, &map_q, qk_full, h * TC_HD, b * L + q0);
        tma_load_2d(sK, &map_k, qk_full, h * TC_HD, b * L + K0);
        mbar_wait_relaxed(v_empty, ph ^ 1);
        mbar_arrive_expect_tx(v_full, Cfg::KV_BYTES);
        tma_load_2d(sV, &map_v, v_full, h * TC_HD, b * L + K0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, LPAD, 0, 0);
      constexpr uint32_t idesc_o = make_idesc_bf16(128, TC_HD, 0, 1);
      const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV), aP = smem_u32(sP);
      auto issue_s = [&](int tau) {
        const int item = tau / NT, t = tau % NT;
        if (t == 0) {
          mbar_wait(qk_full, (uint32_t)item & 1u);
          tc_fence_after();
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base + (tau & 1) * LPAD, make_smem_desc(aQ + t * 16384 + k * 32, 16, 1024),
                    make_smem_desc(aK + k * 32, 16, 1024), idesc_s, k > 0 ? 1u : 0u);
        umma_commit(&s_full[tau & 1]);
        if (t == NT - 1) umma_commit(qk_empty);
      };
      for (int tau = 0; tau < 2 && tau < n_tiles; ++tau) issue_s(tau);
      for (int tau = 0; tau < n_tiles; ++tau) {
        const int item = tau / NT, t = tau % NT;
        mbar_wait(&p_full[tau & 1], (uint32_t)(tau >> 1) & 1u);   // P written, S[tau&1] drained
        if (t == 0) mbar_wait(v_full, (uint32_t)item & 1u);
        mbar_wait(o_empty, ((uint32_t)tau & 1u) ^ 1u);             // previous tile's O has been read out
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < LPAD / 16; ++k)
          umma_bf16(tmem_base + Cfg::TMEM_O, make_smem_desc(aP + (tau & 1) * Cfg::P_BYTES + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                    make_smem_desc(aV + k * 2048, 8192, 1024), idesc_o, k > 0 ? 1u : 0u);
        umma_commit(&o_full[tau & 1]);
        if (t == NT - 1) umma_commit(v_empty);
        if (tau + 2 < n_tiles) issue_s(tau + 2);
      }
    }
    __syncwarp();
  } else {
    const int wg = (warp - 2) >> 2;            // softmax warpgroup = tile parity
    const int quad = warp & 3;                 // TMEM lane quadrant
    const int r = quad * 32 + lane;            // row inside the tile
    const int wgt = (threadIdx.x - 64) & 127;  // 0..127 inside the warpgroup
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint32_t t_s = lane_base + (uint32_t)(wg * LPAD), t_o = lane_base + (uint32_t)Cfg::TMEM_O;
    float* tab = tabs + (BLOCKED ? 0 : wg) * Cfg::TAB_FLOATS;  // this warpgroup's copy: [0, OFFMAX] = table[T-3], then the table
    const float scale2 = a.scale * 1.4426950408889634f;
    uint8_t* myP = sP + wg * Cfg::P_BYTES + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    int cur_h = BLOCKED ? h_cta : -1;
    float bias_c0 = 0.f;
    long long pc[6] = {0, 0, 0, 0, 0, 0}, pt = clock64();
    auto tick = [&](int i) { if (a.prof) { const long long n = clock64(); pc[i] += n - pt; pt = n; } };
    for (int tau = wg; tau < n_tiles; tau += 2) {
      const int item = item0 + tau / NT, t = tau % NT;
      int h, b, q0;
      decode(item, h, b, q0);
      const int qi = q0 + t * 128 + r;         // query index inside the sample
      if (h != cur_h) {                         // (re)load this head's table column (log2 domain)
        named_bar_sync(1 + wg, 128);
        for (int i = wgt; i < Cfg::T; i += 128)
          tab[Cfg::OFFMAX + 1 + i] = a.table ? __ldg(a.table + (int64_t)i * a.H + h) * 1.4426950408889634f : 0.f;
        const float row0 = a.table ? __ldg(a.table + (int64_t)(Cfg::T - 3) * a.H + h) * 1.4426950408889634f : 0.f;
        for (int i = wgt; i <= Cfg::OFFMAX; i += 128) tab[i] = row0;
        named_bar_sync(1 + wg, 128);
        cur_h = h;
      }
      // closed form of beit2.py:104-114: idx(i, j) = base_i - off_j for i, j >= 1; row 0 reads the replicated
      // table[T-3] block through the same address arithmetic; column 0 is a per-row constant
      const int qc = qi < L ? qi : L - 1;
      const float* rb;
      if (qc >= 1) {
        const int pi = qc - 1;
        rb = tab + Cfg::OFFMAX + 1 + ((pi / W) + W - 1) * (2 * W - 1) + (pi % W) + W - 1;
      } else {
        rb = tab + Cfg::OFFMAX;
      }
      bias_c0 = tab[Cfg::OFFMAX + 1 + (qc >= 1 ? Cfg::T - 2 : Cfg::T - 1)];
      tick(0);
      mbar_wait(&s_full[wg], (uint32_t)(tau >> 1) & 1u);
      tc_fence_after();
      tick(1);
      // a warp whose 32 rows all lie beyond the sample's last query (rows 224..255 of the second tile at L = 197) has nothing
      // to compute: its P rows only feed output rows that are never stored.  It still takes part in every barrier.
      const bool warp_live = q0 + t * 128 + quad * 32 < L;
      float m = 0.f, sum = 1.f;
      if (warp_live) {
      // ---- pass 1: row maximum (with the bias: logits written back to TMEM)
      float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int c0 = 0; c0 < LPAD; c0 += 32) {
        uint32_t v[32];
        const bool full = c0 + 32 <= LPAD;
        if (full) tmem_ld_32x32(t_s + c0, v);
        else tmem_ld_32x32_16(t_s + c0, v);
        tmem_ld_wait();
        if constexpr (HAS_TAB) {   // logits (log2 domain) back into TMEM, exact row maximum
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int j = c0 + e;
            if (j < LPAD) {
              float l;                               // j: key inside the block, K0 + j inside the sample
              if (j >= KLEN) l = -INFINITY;
              else if (K0 + j == 0) l = fmaf(__uint_as_float(v[e]), scale2, bias_c0);
              else l = fmaf(__uint_as_float(v[e]), scale2, *(rb - rel_off<W>(K0 + j)));
              m4[e & 3] = fmaxf(m4[e & 3], l);
              v[e] = __float_as_uint(l);
            }
          }
          if (full) tmem_st_32x32(t_s + c0, v);
          else tmem_st_32x32_16(t_s + c0, v);
        } else {                   // no bias: the maximum of the raw scores is the row maximum up to the scale
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (c0 + e < KLEN) m4[e & 3] = fmaxf(m4[e & 3], __uint_as_float(v[e]));
        }
      }
      // The maximum must be the EXACT row maximum: the dominant probability is then exactly 1 and survives the bf16 rounding
      // of P unchanged, which the fp32 normaliser assumes.  (An upper bound — raw maximum + the head's largest bias — would
      // save the gather and the write-back of this pass, 59 -> 55 us, but shifts the dominant term off a power of two: its
      // rounding error, up to 2^-9, then goes straight into the output; measured as 3.5x the ITM-loss deviation.)
      m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      if constexpr (HAS_TAB) tmem_st_wait();
      else m *= scale2;                            // scale2 > 0: the maximum commutes with the scaling
      tick(2);
      // ---- pass 2: p = 2^(l - m), row sum, bf16 P -> shared memory (K-major, SWIZZLE_128B)
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c0 = 0; c0 < LPAD; c0 += 32) {
        uint32_t v[32];
        const bool full = c0 + 32 <= LPAD;
        if (full) tmem_ld_32x32(t_s + c0, v);
        else tmem_ld_32x32_16(t_s + c0, v);
        tmem_ld_wait();
        uint8_t* blk = myP + (c0 >> 6) * 16384;
        const int ch0 = (c0 & 63) >> 3;  // first 16-byte chunk of this 32-column group inside the 64-key block
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          if (c0 + g8 * 8 < LPAD) {
            float p[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              if constexpr (HAS_TAB) p[e] = ex2_approx(__uint_as_float(v[g8 * 8 + e]) - m);
              else p[e] = c0 + g8 * 8 + e < KLEN ? ex2_approx(fmaf(__uint_as_float(v[g8 * 8 + e]), scale2, -m)) : 0.f;
              s4[e & 3] += p[e];
            }
            uint4 u;
            __nv_bfloat162 t0 = __floats2bfloat162_rn(p[0], p[1]), t1 = __floats2bfloat162_rn(p[2], p[3]);
            __nv_bfloat162 t2 = __floats2bfloat162_rn(p[4], p[5]), t3 = __floats2bfloat162_rn(p[6], p[7]);
            u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
            *(uint4*)(blk + (((ch0 + g8) ^ sw) << 4)) = u;
          }
        }
      }
      sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      }
      fence_proxy_async();  // generic-proxy writes of P -> visible to the tensor core's async-proxy reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[wg]);
      tick(3);
      // ---- epilogue: O / rowsum -> global, lse
      mbar_wait(&o_full[wg], (uint32_t)(tau >> 1) & 1u);
      tc_fence_after();
      tick(4);
      uint32_t o[2][32];
      if (warp_live) {
        tmem_ld_32x32(t_o, o[0]);
        tmem_ld_32x32(t_o + 32, o[1]);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);  // the O accumulator is free for the next tile while we store
      if (warp_live) {
        // thread = row would store 16-byte pieces of 32 different rows per instruction.  The row goes through this thread's
        // own (now consumed: o_full) P row of key block 0 instead — same swizzle — and is read back four whole 128-byte rows
        // per instruction, so every global store instruction writes complete lines.
        const float inv = 1.0f / sum;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            uint4 u;
            __nv_bfloat162 t0 = __floats2bfloat162_rn(__uint_as_float(o[hh][e]) * inv, __uint_as_float(o[hh][e + 1]) * inv);
            __nv_bfloat162 t1 = __floats2bfloat162_rn(__uint_as_float(o[hh][e + 2]) * inv, __uint_as_float(o[hh][e + 3]) * inv);
            __nv_bfloat162 t2 = __floats2bfloat162_rn(__uint_as_float(o[hh][e + 4]) * inv, __uint_as_float(o[hh][e + 5]) * inv);
            __nv_bfloat162 t3 = __floats2bfloat162_rn(__uint_as_float(o[hh][e + 6]) * inv, __uint_as_float(o[hh][e + 7]) * inv);
            u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
            *(uint4*)(myP + (((hh * 4 + (e >> 3)) ^ sw) << 4)) = u;
          }
        if (qi < L && a.lse) a.lse[((int64_t)b * a.H + h) * L + qi] = (m + log2f(sum)) * 0.6931471805599453f;
        __syncwarp();
        const int ch = lane & 7;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int r2 = quad * 32 + it * 4 + (lane >> 3);
          const int q2 = q0 + t * 128 + r2;
          const uint4 u = *(const uint4*)(sP + wg * Cfg::P_BYTES + (r2 >> 3) * 1024 + (r2 & 7) * 128 + ((ch ^ (r2 & 7)) << 4));
          if (q2 < L) *(uint4*)(a.out + ((int64_t)b * L + q2) * a.o_stride + h * TC_HD + ch * 8) = u;
        }
        __syncwarp();  // the staging rows are overwritten by the next tile's probabilities
      }
      tick(5);
    }
    if (a.prof && blockIdx.x == 0 && lane == 0 && (warp == 2 || warp == 9))
      for (int i = 0; i < 6; ++i) a.prof[(warp == 2 ? 0 : 6) + i] = pc[i];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


// ================================================================================================ backward
// One kernel for dQ, dK and dV.  Per query tile S = Q K^T and dP = dO V^T are computed once into TMEM, the element-wise stage
// (P = 2^(S*scale2 + bias2 - lse2), dS = P o (dP - delta); the forward saved lse, delta = rowsum(dO o O) comes from
// attn_delta_kernel) writes P and dS to shared memory once, and three products are issued from those buffers — dQ = dS K (dS
// read K-major), dK = dS^T Q and dV = P^T dO (the same buffers read MN-major: keys become the M dimension, 64-key blocks are
// 16 KB apart).  The outputs re-use the TMEM columns of S / dP.  The gradient of the relative-position table is not formed
// here: dS goes to the optional bf16 dump, which the caller reduces (batch_sum_bf16, relpos_bias_bwd).
// Samples with more than 208 keys (384 px: W = 24, L = 577; 480 px: W = 30, L = 901) are processed one KEY BLOCK per launch
// (KeyBlocks: 192 / 192 / 193 keys at 577, 4 x 192 + 133 at 901; scores beyond a block's keys are masked): the backward needs no online softmax — P = 2^(S - lse) with the forward's lse — so a
// key block is just a narrower K / V operand, an offset into the relative-position index, per-block dK / dV rows, and dQ
// accumulated across the launches (block 0 stores, later blocks TMA-reduce-add; launches of one stream run in order).
struct VitBwdArgs {
  const float* lse;      // [B, H, L]
  const float* delta;    // [B, H, L]
  const float* table;    // [T, H] or null
  bf16* ds_dump;         // [B, H, L, ds_ld] bf16 dS (natural-logit gradient) or null
  int64_t ds_ld;
  bf16 *dq, *dk, *dv;
  int64_t dq_stride, dk_stride, dv_stride;
  int B, H;
  float scale;
  int items_per_cta;
  long long* prof;       // XFM_ATTN_PROF=1: per-phase clock64 totals of CTA 0, warps 2 and 15
};

template <int W>
struct VitFusedCfg {
  static constexpr int L = W * W + 1;
  static constexpr int NB = KeyBlocks::nb(L);                      // key blocks = launches
  static constexpr bool BLOCKED = NB > 1;
  static constexpr int KBS = KeyBlocks::kbs(L);                    // keys per block
  static constexpr int LAST = KeyBlocks::last(L);                  // keys of the last block
  static constexpr int LPAD = KeyBlocks::lpad(L);                  // score columns in TMEM / operand rows in shared memory
  static constexpr int NT = (L + 127) / 128;
  static constexpr int T = (2 * W - 1) * (2 * W - 1) + 3;
  static constexpr int OFFMAX = (W - 1) * (2 * W - 1) + (W - 1);
  static constexpr int KV_BYTES = LPAD * 128;
  static constexpr int NM = (LPAD + 127) / 128;                    // 128-key M tiles of dK / dV
  static constexpr int PD_BYTES = 2 * NM * 16384;                  // P / dS operand: whole 64-key blocks for every M tile
  static constexpr int SMEM_NO_TAB = 2 * 16384 + 2 * KV_BYTES + 2 * PD_BYTES + 128;
  // The bias table is staged as [OFFMAX+1 copies of table[T-3]] ++ [table], so that the CLS query row reads its constant
  // through the same address arithmetic as every other row.  Where that prefix does not fit (W = 30: 6 964 bytes over the
  // limit with it) only the table is staged and row 0 selects its constant instead; the values stay the exact fp32 entries.
  static constexpr bool ROW0_PREFIX = SMEM_NO_TAB + ((OFFMAX + 1 + T + 7) & ~7) * 4 <= 232448;
  static constexpr int PREFIX = ROW0_PREFIX ? OFFMAX + 1 : 0;      // table[i] is tab[PREFIX + i]
  static constexpr int TAB_FLOATS = (PREFIX + T + 7) & ~7;
  static constexpr int SMEM = SMEM_NO_TAB + TAB_FLOATS * 4;
  static constexpr int TM_DQ = 0, TM_DK = 64, TM_DV = 64 + 64 * NM, TM_END = 64 + 128 * NM;
  static constexpr int UNITS = TM_END / 32;                        // 32-column drain units, split between the warpgroups
  static_assert(LAST <= LPAD && 2 * LPAD <= 512 && TM_END <= 512, "TMEM");
  static_assert(SMEM <= 232448, "shared memory");
};
static_assert(VitFusedCfg<24>::NB == 3 && VitFusedCfg<24>::LAST == 193 && VitFusedCfg<24>::LPAD == 208 &&
              VitFusedCfg<24>::ROW0_PREFIX && VitFusedCfg<14>::ROW0_PREFIX, "384 / 224 px backward: unchanged geometry");
static_assert(VitFusedCfg<30>::NB == 5 && VitFusedCfg<30>::LAST == 133 && VitFusedCfg<30>::LPAD == 192 &&
              !VitFusedCfg<30>::ROW0_PREFIX, "480 px backward");

template <int W, int KB, bool PROF>
__global__ void __launch_bounds__(TCF_THREADS, 1)
vit_attn_bwd_fused_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                             const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                             const __grid_constant__ CUtensorMap map_dq, const __grid_constant__ CUtensorMap map_dk,
                             const __grid_constant__ CUtensorMap map_dv, const __grid_constant__ CUtensorMap map_ds,
                             const VitBwdArgs a) {
  using Cfg = VitFusedCfg<W>;
  constexpr int L = Cfg::L, LPAD = Cfg::LPAD, NT = Cfg::NT, NM = Cfg::NM;
  constexpr int K0 = KB * Cfg::KBS;                                   // first key of this launch's block
  constexpr int KLEN = KB == Cfg::NB - 1 ? Cfg::LAST : Cfg::KBS;      // its keys
  static_assert(KB < Cfg::NB, "key block");
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* sQ = smem;                       // one 128-row query tile
  uint8_t* sdO = sQ + 16384;
  uint8_t* sK = sdO + 16384;                // LPAD keys
  uint8_t* sV = sK + Cfg::KV_BYTES;
  uint8_t* sdS = sV + Cfg::KV_BYTES;
  uint8_t* sP = sdS + Cfg::PD_BYTES;
  float* tab = (float*)(sP + Cfg::PD_BYTES);    // [PREFIX copies of table[T-3]] ++ [table], log2 domain
  uint64_t* bars = (uint64_t*)(tab + Cfg::TAB_FLOATS);
  uint64_t *kv_full = bars, *kv_empty = bars + 1, *qdo_full = bars + 2, *qdo_empty = bars + 3, *sd_full = bars + 4,
           *ds_full = bars + 5, *out_full = bars + 6, *out_empty = bars + 7;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_do);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    tma_prefetch_desc(&map_dq);
    tma_prefetch_desc(&map_dk);
    tma_prefetch_desc(&map_dv);
    if (a.ds_dump) tma_prefetch_desc(&map_ds);
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
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  constexpr uint32_t TM_S = 0, TM_DP = LPAD;

  const int n_items = a.B * a.H;
  const int item0 = blockIdx.x * a.items_per_cta;
  const int item1 = min(n_items, item0 + a.items_per_cta);
  const int n_tiles = (item1 - item0) * NT;

  if (warp == 0) {
    if (lane == 0) {
      for (int tau = 0; tau < n_tiles; ++tau) {
        const int item = item0 + tau / NT, t = tau % NT;
        const int h = item / a.B, b = item % a.B;
        if (t == 0) {
          mbar_wait_relaxed(kv_empty, ((uint32_t)(tau / NT) & 1u) ^ 1u);
          mbar_arrive_expect_tx(kv_full, 2 * Cfg::KV_BYTES);
          tma_load_2d(sK, &map_k, kv_full, h * TC_HD, b * L + K0);
          tma_load_2d(sV, &map_v, kv_full, h * TC_HD, b * L + K0);
        }
        mbar_wait_relaxed(qdo_empty, ((uint32_t)tau & 1u) ^ 1u);
        mbar_arrive_expect_tx(qdo_full, 2 * 16384);
        tma_load_2d(sQ, &map_q, qdo_full, h * TC_HD, b * L + t * 128);
        tma_load_2d(sdO, &map_do, qdo_full, h * TC_HD, b * L + t * 128);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, LPAD, 0, 0);
      constexpr uint32_t idesc_dq = make_idesc_bf16(128, TC_HD, 0, 1);
      constexpr uint32_t idesc_dkv = make_idesc_bf16(128, TC_HD, 1, 1);
      const uint32_t aQ = smem_u32(sQ), adO = smem_u32(sdO), aK = smem_u32(sK), aV = smem_u32(sV), adS = smem_u32(sdS),
                     aP = smem_u32(sP);
      for (int tau = 0; tau < n_tiles; ++tau) {
        const int t = tau % NT;
        const uint32_t par = (uint32_t)tau & 1u;
        if (t == 0) mbar_wait(kv_full, (uint32_t)(tau / NT) & 1u);
        mbar_wait(qdo_full, par);
        mbar_wait(out_empty, par ^ 1u);        // the previous tile's outputs (which alias S / dP) are drained
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
        mbar_wait(ds_full, par);                // P / dS in shared memory, S / dP read out
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < LPAD / 16; ++k)     // dQ = dS K
          umma_bf16(tmem_base + Cfg::TM_DQ, make_smem_desc(adS + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                    make_smem_desc(aK + k * 2048, 8192, 1024), idesc_dq, k > 0 ? 1u : 0u);
        const int rows = min(128, L - t * 128);
        const int nk = (rows + 15) / 16;        // query k-steps: rows beyond the tile's live queries hold zeros in P / dS
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          for (int k = 0; k < nk; ++k)          // dK = dS^T Q
            umma_bf16(tmem_base + Cfg::TM_DK + m * 64, make_smem_desc(adS + m * 32768 + k * 2048, 16384, 1024),
                      make_smem_desc(aQ + k * 2048, 8192, 1024), idesc_dkv, k > 0 ? 1u : 0u);
          for (int k = 0; k < nk; ++k)          // dV = P^T dO
            umma_bf16(tmem_base + Cfg::TM_DV + m * 64, make_smem_desc(aP + m * 32768 + k * 2048, 16384, 1024),
                      make_smem_desc(adO + k * 2048, 8192, 1024), idesc_dkv, k > 0 ? 1u : 0u);
        }
        umma_commit(out_full);
        umma_commit(qdo_empty);
        if (t == NT - 1) umma_commit(kv_empty);
      }
    }
    __syncwarp();
  } else {
    const int wg = (warp - 2) >> 2;            // 0..3: column quarter in the element-wise stage, unit list in the drain
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const int wgt = threadIdx.x - 64;          // 0..511
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const float scale2 = a.scale * 1.4426950408889634f;
    uint8_t* myS = sdS + (r >> 3) * 1024 + (r & 7) * 128;
    uint8_t* myP = sP + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    constexpr int N16 = LPAD / 16;             // 16-column chunks of a score row, split in four runs
    const int ch_lo = (wg * N16) / 4, ch_hi = ((wg + 1) * N16) / 4;
    const bool elected = threadIdx.x == 64;   // issues every TMA store of this CTA (bulk groups are per thread)
    int cur_h = -1;
    long long pc[5] = {0, 0, 0, 0, 0}, pt = clock64();
    auto tick = [&](int i) { if (PROF) { const long long n = clock64(); pc[i] += n - pt; pt = n; } };
    for (int tau = 0; tau < n_tiles; ++tau) {
      const int item = item0 + tau / NT, t = tau % NT;
      const int h = item / a.B, b = item % a.B;
      const uint32_t par = (uint32_t)tau & 1u;
      const int qi = t * 128 + r;
      if (h != cur_h) {
        named_bar_sync(1, 512);
        for (int i = wgt; i < Cfg::T; i += 512)
          tab[Cfg::PREFIX + i] = a.table ? __ldg(a.table + (int64_t)i * a.H + h) * 1.4426950408889634f : 0.f;
        const float row0 = a.table ? __ldg(a.table + (int64_t)(Cfg::T - 3) * a.H + h) * 1.4426950408889634f : 0.f;
        for (int i = wgt; i < Cfg::PREFIX; i += 512) tab[i] = row0;
        named_bar_sync(1, 512);
        cur_h = h;
      }
      const int qc = qi < L ? qi : L - 1;
      const bool row_ok = qi < L;
      const bool wv = __any_sync(0xffffffffu, row_ok);
      // row 0 without the prefix: any base keeps the (discarded) gather inside the table
      const int rb_off = qc >= 1 ? Cfg::PREFIX + (((qc - 1) / W) + W - 1) * (2 * W - 1) + ((qc - 1) % W) + W - 1
                                 : (Cfg::ROW0_PREFIX ? Cfg::OFFMAX : Cfg::PREFIX + Cfg::OFFMAX);
      const float* rb = tab + rb_off;
      const int c0_idx = Cfg::PREFIX + (qc >= 1 ? Cfg::T - 2 : Cfg::T - 1);
      const float bias_c0 = tab[c0_idx];
      const bool cls_row = !Cfg::ROW0_PREFIX && qc == 0;
      const float bias_r0 = tab[Cfg::PREFIX + Cfg::T - 3];
      const int64_t st_row = ((int64_t)b * a.H + h) * L + qc;
      const float lse2 = __ldg(a.lse + st_row) * 1.4426950408889634f;
      const float dl = __ldg(a.delta + st_row);
      tick(0);
      mbar_wait(sd_full, par);
      tc_fence_after();
      // the previous tile's output / dS stores still read the P / dS buffers this tile is about to overwrite
      if (elected) tma_store_wait_read<0>();
      named_bar_sync(1, 512);
      tick(1);
      // ---- element-wise stage: 16-column chunks (four warps per scheduler hide the TMEM load latency; a second register
      // buffer for the next chunk does not fit the 96 registers 18 warps leave per thread)
      uint32_t vs[32], vp[32];                   // only [0..15] are used
#pragma unroll
      for (int ch = 0; ch < N16; ++ch) {
        if (ch < ch_lo || ch >= ch_hi) continue;   // warp-uniform
        if (!wv) {   // every row of this warp lies beyond the last query (second tile): only clear its operand rows
#pragma unroll
          for (int g8 = 0; g8 < 2; ++g8) {
            const int col8 = ch * 16 + g8 * 8;
            const int off8 = (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4);
            *(uint4*)(myS + off8) = make_uint4(0u, 0u, 0u, 0u);
            *(uint4*)(myP + off8) = make_uint4(0u, 0u, 0u, 0u);
          }
          continue;
        }
        tmem_ld_32x32_16(lane_base + TM_S + ch * 16, vs);
        tmem_ld_32x32_16(lane_base + TM_DP + ch * 16, vp);
        tmem_ld_wait();
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          const int col8 = ch * 16 + g8 * 8;
          const int off8 = (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4);
          float ds[8], pp[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int j = col8 + e;              // key inside the block; K0 + j inside the sample
            const float bias2 = K0 + j == 0 ? bias_c0 : (cls_row ? bias_r0 : *(rb - rel_off<W>(K0 + j)));
            float p = ex2_approx(fmaf(__uint_as_float(vs[g8 * 8 + e]), scale2, bias2) - lse2);
            if (j >= KLEN || !row_ok) p = 0.f;
            pp[e] = p;
            ds[e] = p * (__uint_as_float(vp[g8 * 8 + e]) - dl);
          }
          st_bf16x8(myS + off8, ds);
          st_bf16x8(myP + off8, pp);
        }
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
      tick(2);
      // ---- outputs: 32-column units [dQ | dK tiles | dV tiles].  thread = row would write (and, for the second query tile,
      // read-modify-write) 16-byte pieces of 32 different rows per instruction: 45 % of this kernel's time.  Instead every
      // 64-column output block is staged as bf16 in a SWIZZLE_128B [128 x 64] tile — the dK / dV blocks in the consumed P
      // buffer, dQ in block 0 of the consumed dS buffer — and one thread issues TMA stores through 3D maps [sample, row,
      // column] that clip at the sample's last row; the second query tile's dK / dV go out as TMA reduce-adds onto the first
      // tile's.  dS itself (the table gradient's input) is stored by TMA from the dS operand buffer it already sits in.
      // Units per warpgroup: 0: {dK unit 2, then dQ = units 0, 1}, 1: {3, 4, 5}, 2: {6, 7}, 3: {8, 9} (UNITS = 10; 6: only 0 and 1).
      mbar_wait(out_full, par);
      tc_fence_after();
      tick(3);
      if (elected) {
        if (a.ds_dump) {   // this block's columns; the last block also covers the zero padding up to ds_ld
          const int rem = (int)a.ds_ld - K0;
          const int ncols = KB == Cfg::NB - 1 ? (rem < LPAD ? rem : LPAD) : KLEN;
          for (int kb = 0; kb < (ncols + 63) >> 6; ++kb)
            tma_store_3d(&map_ds, sdS + kb * 16384, K0 + kb * 64, t * 128, b * a.H + h);
        }
        tma_store_commit();                      // (possibly empty) group: keeps the group count per tile fixed
      }
      static_assert(Cfg::UNITS == 10 || Cfg::UNITS == 6, "unit lists below");
      const int n_mine = wg < 2 ? 3 : (Cfg::UNITS == 10 ? 2 : 0);
      const int u_first = wg == 0 ? 2 : (wg == 1 ? 3 : 2 + 2 * wg);   // wg 0 continues with units 0, 1
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (i >= n_mine) continue;               // warp-uniform
        const int u = wg == 0 ? (i == 0 ? 2 : i - 1) : u_first + i;
        uint32_t o[32];
        tmem_ld_32x32(lane_base + (uint32_t)(u * 32), o);
        tmem_ld_wait();
        if (wg == 0 && i == 1) {                 // dQ is staged where dS lies: its TMA store must have read the buffer
          if (elected) tma_store_wait_read<0>();
          named_bar_sync(2, 128);
        }
        uint8_t* blk;
        float mul = a.scale;
        int half = u & 1;
        if (u < 2) {
          blk = sdS;
        } else {
          const bool is_dv = u >= 2 + 2 * NM;
          const int uu = is_dv ? u - 2 - 2 * NM : u - 2;
          blk = sP + ((is_dv ? NM : 0) + (uu >> 1)) * 16384;
          half = uu & 1;
          if (is_dv) mul = 1.0f;
        }
        uint8_t* row = blk + (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
        for (int e = 0; e < 32; e += 8) {
          float v[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = __uint_as_float(o[e + k]) * mul;
          st_bf16x8(row + (((half * 4 + (e >> 3)) ^ sw) << 4), v);
        }
      }
      tc_fence_before();                         // every TMEM read of this warp is complete (tcgen05.wait::ld above)
      __syncwarp();
      if (lane == 0) mbar_arrive(out_empty);
      fence_proxy_async();
      named_bar_sync(1, 512);
      if (elected) {
        if (KB == 0) tma_store_3d(&map_dq, sdS, h * TC_HD, t * 128, b);
        else tma_reduce_add_3d(&map_dq, sdS, h * TC_HD, t * 128, b);   // onto the earlier key blocks' launches
        if (t == 0) {
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            tma_store_3d(&map_dk, sP + m * 16384, h * TC_HD, m * 128, b);
            tma_store_3d(&map_dv, sP + (NM + m) * 16384, h * TC_HD, m * 128, b);
          }
        } else {
          tma_store_wait_all<1>();               // the first tile's dK / dV stores have landed (only this tile's dS may be pending)
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            tma_reduce_add_3d(&map_dk, sP + m * 16384, h * TC_HD, m * 128, b);
            tma_reduce_add_3d(&map_dv, sP + (NM + m) * 16384, h * TC_HD, m * 128, b);
          }
        }
        tma_store_commit();
      }
      tick(4);
    }
    if (PROF && blockIdx.x == 0 && lane == 0 && (warp == 2 || warp == 15))
      for (int i = 0; i < 5; ++i) a.prof[(warp == 2 ? 0 : 6) + i] = pc[i];
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
int encode_rows(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_rows) {
  auto fn = get_tensor_map_encoder();
  if (!fn) return XFM_ERR_NO_DRIVER;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {TC_HD, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("attention: cuTensorMapEncodeTiled failed: %d", (int)r);
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

// [sample, row, 64-column block] view of a bf16 activation: boxes of 128 rows are clipped at the sample's last row
int encode_rows_3d(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows_per_sample, uint64_t samples,
                   uint64_t ld_elems, uint64_t sample_stride_rows) {
  auto fn = get_tensor_map_encoder();
  if (!fn) return XFM_ERR_NO_DRIVER;
  if (sample_stride_rows == 0) sample_stride_rows = rows_per_sample;   // > rows_per_sample: a row window of every sample
  cuuint64_t dims[3] = {cols, rows_per_sample, samples};
  cuuint64_t strides[2] = {ld_elems * 2, sample_stride_rows * ld_elems * 2};
  cuuint32_t box[3] = {TC_HD, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("attention: cuTensorMapEncodeTiled (3D store map) failed: %d", (int)r);
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

// window sides with an instantiated kernel: 14 (224 px / 16), 12 and 7 (test sizes), 4 (tiny parity model); the fused
// backward, and the forward given the key-block scratch, also 24 (384 px / 16: three key blocks per sample) and 30
// (480 px / 16: five key blocks)
static int window_for(int L, bool bwd = false) {
  const int ws[] = {14, 12, 7, 4, 24, 30};
  for (int i = 0; i < (bwd ? 6 : 4); ++i)
    if (ws[i] * ws[i] + 1 == L) return ws[i];
  return 0;
}

bool vit_attention_tc_supported(const xfm_attn_params* p, bool bwd) {
  const int w = window_for(p->Lk, bwd || (p->part_out && p->part_lse));   // forward at 24 / 30: needs the key-block scratch
  return p->head_dim == TC_HD && p->Lq == p->Lk && w > 0 && !p->kmask && !p->kv_index &&
         (!p->bias || p->rel_table) && !(p->dropout_p > 0.f) && (p->Bkv == 0 || p->Bkv == p->B) &&
         (p->rel_table == nullptr || p->rel_window == w) &&
         ((uintptr_t)p->q & 15) == 0 && ((uintptr_t)p->k & 15) == 0 && ((uintptr_t)p->v & 15) == 0 &&
         ((p->q_stride | p->k_stride | p->v_stride | p->o_stride) & 7) == 0;
}

// Merge of the key blocks' partial results: out = sum_k w_k O_k with w_k = exp(lse_k - lse), lse = log sum_k exp(lse_k).
// One CTA per token row, one thread per 8 output columns (a head is 8 threads).
template <int NB>
__global__ void merge_parts_kernel(const bf16* __restrict__ part_out, const float* __restrict__ part_lse, bf16* __restrict__ out,
                                   int64_t o_stride, float* __restrict__ lse, int B, int H, int L) {
  const int row = blockIdx.x, c = threadIdx.x, h = c >> 3;
  const int b = row / L, q = row % L;
  const int64_t rows = (int64_t)B * L, lrow = ((int64_t)b * H + h) * L + q, lse_n = (int64_t)B * H * L;
  float l[NB], m = -INFINITY;
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    l[k] = __ldg(part_lse + k * lse_n + lrow);
    m = fmaxf(m, l[k]);
  }
  float wsum = 0.f;
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    l[k] = __expf(l[k] - m);
    wsum += l[k];
  }
  const float inv = 1.0f / wsum;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const uint4 u = *(const uint4*)(part_out + (k * rows + row) * (int64_t)(H * TC_HD) + c * 8);
    const __nv_bfloat162* p2 = (const __nv_bfloat162*)&u;
    const float w = l[k] * inv;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(p2[e]);
      acc[2 * e] = fmaf(w, f.x, acc[2 * e]);
      acc[2 * e + 1] = fmaf(w, f.y, acc[2 * e + 1]);
    }
  }
  st_bf16x8((uint8_t*)(out + row * o_stride + c * 8), acc);
  if (lse && (c & 7) == 0) lse[lrow] = m + __logf(wsum);
}

int launch_merge_parts(int nb, const void* part_out, const float* part_lse, void* out, int64_t o_stride, float* lse, int B, int H,
                       int L, cudaStream_t s) {
  if ((nb != 3 && nb != 5) || H * 8 > 1024) {
    set_error("merge of key-block partials: %d blocks / %d heads not instantiated", nb, H);
    return XFM_ERR_BAD_ARG;
  }
  if (nb == 3) merge_parts_kernel<3><<<(unsigned)(B * L), H * 8, 0, s>>>((const bf16*)part_out, part_lse, (bf16*)out, o_stride, lse, B, H, L);
  else merge_parts_kernel<5><<<(unsigned)(B * L), H * 8, 0, s>>>((const bf16*)part_out, part_lse, (bf16*)out, o_stride, lse, B, H, L);
  count_launch();
  return (int)cudaGetLastError();
}

template <int W, int KB>
static int launch_vit_fwd_block(const xfm_attn_params* p, const VitAttnArgs& a0, const CUtensorMap& mq, const CUtensorMap& mk,
                                const CUtensorMap& mv, cudaStream_t s) {
  using Cfg = VitFwdCfg<W>;
  VitAttnArgs a = a0;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(vit_attn_fwd_tc_kernel<W, KB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(vit_attn_fwd_tc_kernel<W, KB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  int grid;
  if (Cfg::BLOCKED) {   // a CTA stays on one head; this block's partial output / lse
    const int64_t rows = (int64_t)a.B * Cfg::L;
    a.out = (bf16*)p->part_out + KB * rows * (int64_t)(a.H * TC_HD);
    a.o_stride = (int64_t)a.H * TC_HD;
    a.lse = p->part_lse + KB * (int64_t)a.B * a.H * Cfg::L;
    const int per_head = a.B * Cfg::NTP;
    int cph = num_sms() / a.H;
    cph = cph < 1 ? 1 : (cph > per_head ? per_head : cph);
    a.items_per_cta = (per_head + cph - 1) / cph;
    a.ctas_per_head = (per_head + a.items_per_cta - 1) / a.items_per_cta;
    grid = a.ctas_per_head * a.H;
  } else {
    const int n_items = a.B * a.H;
    const int ctas = n_items < num_sms() ? n_items : num_sms();
    a.items_per_cta = (n_items + ctas - 1) / ctas;
    a.ctas_per_head = 0;
    grid = (n_items + a.items_per_cta - 1) / a.items_per_cta;
  }
  static const bool prof_on = getenv("XFM_ATTN_PROF") != nullptr;
  static long long* prof_buf = nullptr;
  a.prof = nullptr;
  if (prof_on) {
    if (!prof_buf) cudaMalloc(&prof_buf, 12 * sizeof(long long));
    a.prof = prof_buf;
  }
  if (a.table) vit_attn_fwd_tc_kernel<W, KB, true><<<grid, TC_THREADS, Cfg::SMEM_BYTES, s>>>(mq, mk, mv, a);
  else vit_attn_fwd_tc_kernel<W, KB, false><<<grid, TC_THREADS, Cfg::SMEM_BYTES, s>>>(mq, mk, mv, a);
  count_launch();
  if (prof_on) {  // debugging aid: synchronous, prints the phase totals of CTA 0 (warp 2 = parity-0 rows 0..31, warp 9 = parity-1 rows 96..127)
    long long h[12];
    cudaStreamSynchronize(s);
    cudaMemcpy(h, prof_buf, sizeof(h), cudaMemcpyDeviceToHost);
    for (int w = 0; w < 2; ++w)
      fprintf(stderr, "vit_attn_fwd prof %s: setup %lld wait_s %lld pass1 %lld pass2 %lld wait_o %lld epilogue %lld cycles (%d items/CTA)\n",
              w ? "warp9" : "warp2", h[w * 6], h[w * 6 + 1], h[w * 6 + 2], h[w * 6 + 3], h[w * 6 + 4], h[w * 6 + 5], a.items_per_cta);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if constexpr (KB + 1 < Cfg::NB) return launch_vit_fwd_block<W, KB + 1>(p, a0, mq, mk, mv, s);
  return 0;
}

template <int W>
static int launch_vit_fwd(const xfm_attn_params* p, cudaStream_t s) {
  using Cfg = VitFwdCfg<W>;
  VitAttnArgs a;
  a.out = (bf16*)p->out; a.o_stride = p->o_stride; a.lse = p->lse; a.table = p->rel_table;
  a.B = p->B; a.H = p->H; a.scale = p->scale;
  if (Cfg::BLOCKED && (!p->part_out || !p->part_lse || a.H * 8 > 1024)) {
    set_error("vit attention fwd: %d tokens need the part_out / part_lse scratch buffers", Cfg::L);
    return XFM_ERR_BAD_ARG;
  }
  const uint64_t rows = (uint64_t)a.B * Cfg::L, cols = (uint64_t)a.H * TC_HD;
  CUtensorMap mq, mk, mv;
  int rc = encode_rows(&mq, p->q, cols, rows, p->q_stride, Cfg::NT * 128);
  if (!rc) rc = encode_rows(&mk, p->k, cols, rows, p->k_stride, Cfg::LPAD);
  if (!rc) rc = encode_rows(&mv, p->v, cols, rows, p->v_stride, Cfg::LPAD);
  if (rc) return rc;
  rc = launch_vit_fwd_block<W, 0>(p, a, mq, mk, mv, s);
  if (rc || !Cfg::BLOCKED) return rc;
  return launch_merge_parts(Cfg::NB, p->part_out, p->part_lse, p->out, p->o_stride, p->lse, a.B, a.H, Cfg::L, s);
}

// One launch per key block.
template <int W, int KB>
static int launch_vit_bwd_fused_block(const xfm_attn_params* p, const VitBwdArgs& a0, const CUtensorMap& mq1, const CUtensorMap& mdo1,
                                      const CUtensorMap& mk_l, const CUtensorMap& mv_l, const CUtensorMap& m_dq,
                                      const CUtensorMap& m_ds, cudaStream_t s) {
  using FCfg = VitFusedCfg<W>;
  constexpr int K0 = KB * FCfg::KBS, KLEN = KB == FCfg::NB - 1 ? FCfg::LAST : FCfg::KBS;
  VitBwdArgs a = a0;
  const uint64_t cols = (uint64_t)a.H * TC_HD;
  CUtensorMap m_dk, m_dv;   // this block's key rows of every sample
  int rc = encode_rows_3d(&m_dk, (const bf16*)p->dk + (int64_t)K0 * p->dk_stride, cols, KLEN, a.B, p->dk_stride, FCfg::L);
  if (!rc) rc = encode_rows_3d(&m_dv, (const bf16*)p->dv + (int64_t)K0 * p->dv_stride, cols, KLEN, a.B, p->dv_stride, FCfg::L);
  if (rc) return rc;
  static bool fattr = false;
  if (!fattr) {
    cudaError_t e = cudaFuncSetAttribute(vit_attn_bwd_fused_tc_kernel<W, KB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FCfg::SMEM);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(vit_attn_bwd_fused_tc_kernel<W, KB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FCfg::SMEM);
    if (e != cudaSuccess) return (int)e;
    fattr = true;
  }
  const int n_items_f = a.B * a.H;
  const int ctas = n_items_f < num_sms() ? n_items_f : num_sms();
  a.items_per_cta = (n_items_f + ctas - 1) / ctas;
  const int grid = (n_items_f + a.items_per_cta - 1) / a.items_per_cta;
  static const bool prof_on = getenv("XFM_ATTN_PROF") != nullptr;
  static long long* prof_buf = nullptr;
  a.prof = nullptr;
  if (prof_on) {
    if (!prof_buf) cudaMalloc(&prof_buf, 12 * sizeof(long long));
    a.prof = prof_buf;
  }
  if (prof_on) vit_attn_bwd_fused_tc_kernel<W, KB, true><<<grid, TCF_THREADS, FCfg::SMEM, s>>>(mq1, mdo1, mk_l, mv_l, m_dq, m_dk, m_dv, m_ds, a);
  else vit_attn_bwd_fused_tc_kernel<W, KB, false><<<grid, TCF_THREADS, FCfg::SMEM, s>>>(mq1, mdo1, mk_l, mv_l, m_dq, m_dk, m_dv, m_ds, a);
  count_launch();
  if (prof_on) {  // debugging aid (synchronous)
    long long h[12];
    cudaStreamSynchronize(s);
    cudaMemcpy(h, prof_buf, sizeof(h), cudaMemcpyDeviceToHost);
    for (int w = 0; w < 2; ++w)
      fprintf(stderr, "vit_attn_bwd_fused prof %s: setup %lld wait_sd %lld elementwise %lld wait_out %lld drain %lld cycles (%d items/CTA)\n",
              w ? "warp15" : "warp2", h[w * 6], h[w * 6 + 1], h[w * 6 + 2], h[w * 6 + 3], h[w * 6 + 4], a.items_per_cta);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if constexpr (KB + 1 < FCfg::NB) return launch_vit_bwd_fused_block<W, KB + 1>(p, a0, mq1, mdo1, mk_l, mv_l, m_dq, m_ds, s);
  return 0;
}

template <int W>
static int launch_vit_bwd_fused(const xfm_attn_params* p, cudaStream_t s) {
  using FCfg = VitFusedCfg<W>;
  VitBwdArgs a;
  a.prof = nullptr;
  a.lse = p->lse; a.delta = p->delta; a.table = p->rel_table;
  a.ds_dump = (bf16*)p->ds_dump; a.ds_ld = p->ds_ld;
  a.dq = (bf16*)p->dq; a.dk = (bf16*)p->dk; a.dv = (bf16*)p->dv;
  a.dq_stride = p->dq_stride; a.dk_stride = p->dk_stride; a.dv_stride = p->dv_stride;
  a.B = p->B; a.H = p->H; a.scale = p->scale;
  const uint64_t rows = (uint64_t)a.B * FCfg::L, cols = (uint64_t)a.H * TC_HD;
  CUtensorMap mq1, mdo1, mk_l, mv_l, m_dq, m_ds;
  int rc = encode_rows(&mq1, p->q, cols, rows, p->q_stride, 128);
  if (!rc) rc = encode_rows(&mdo1, p->dout, cols, rows, p->do_stride, 128);
  if (!rc) rc = encode_rows(&mk_l, p->k, cols, rows, p->k_stride, FCfg::LPAD);
  if (!rc) rc = encode_rows(&mv_l, p->v, cols, rows, p->v_stride, FCfg::LPAD);
  if (!rc) rc = encode_rows_3d(&m_dq, p->dq, cols, FCfg::L, a.B, p->dq_stride);
  m_ds = m_dq;
  if (!rc && a.ds_dump) rc = encode_rows_3d(&m_ds, a.ds_dump, (uint64_t)a.ds_ld, FCfg::L, (uint64_t)a.B * a.H, (uint64_t)a.ds_ld);
  if (rc) return rc;
  return launch_vit_bwd_fused_block<W, 0>(p, a, mq1, mdo1, mk_l, mv_l, m_dq, m_ds, s);
}

// delta must already be in p->delta (attn_delta_kernel); dq / dk / dv are written, and dS to ds_dump when it is given.
int vit_attention_bwd_tc(const xfm_attn_params* p, cudaStream_t s) {
  if ((((uintptr_t)p->dout) & 15) || (p->do_stride & 7) || ((p->dq_stride | p->dk_stride | p->dv_stride) & 7) ||
      (((uintptr_t)p->dq | (uintptr_t)p->dk | (uintptr_t)p->dv) & 15)) {
    set_error("vit attention bwd: operands must be 16-byte aligned with row strides that are multiples of 8");
    return XFM_ERR_BAD_ARG;
  }
  switch (window_for(p->Lk, true)) {
    case 30: return launch_vit_bwd_fused<30>(p, s);
    case 24: return launch_vit_bwd_fused<24>(p, s);
    case 14: return launch_vit_bwd_fused<14>(p, s);
    case 12: return launch_vit_bwd_fused<12>(p, s);
    case 7: return launch_vit_bwd_fused<7>(p, s);
    case 4: return launch_vit_bwd_fused<4>(p, s);
  }
  set_error("vit attention: no tcgen05 instantiation for %d tokens", p->Lk);
  return XFM_ERR_BAD_ARG;
}

int vit_attention_fwd_tc(const xfm_attn_params* p, cudaStream_t s) {
  switch (window_for(p->Lk, true)) {
    case 30: return launch_vit_fwd<30>(p, s);
    case 24: return launch_vit_fwd<24>(p, s);
    case 14: return launch_vit_fwd<14>(p, s);
    case 12: return launch_vit_fwd<12>(p, s);
    case 7: return launch_vit_fwd<7>(p, s);
    case 4: return launch_vit_fwd<4>(p, s);
  }
  set_error("vit attention: no tcgen05 instantiation for %d tokens", p->Lk);
  return XFM_ERR_BAD_ARG;
}

}  // namespace xfm
