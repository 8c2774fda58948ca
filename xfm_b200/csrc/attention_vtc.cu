// Packed variable-length self-attention (RoBERTa sequence classification, run_glue.py batches) on tcgen05 + TMEM + TMA.
//
// The generalisation of attention_stc.cu from three 40-token samples per tile to any lengths of 1 to 128 tokens packed back
// to back with no padding rows: sequence s occupies rows [cu_seqlens[s], cu_seqlens[s+1]) of the Q / K / V column slices.
// A tile is a maximal run of consecutive sequences of at most 128 rows in total (xfm_attention_varlen_plan states the rule),
// so every operand of a tile is ONE TMA box of 128 rows starting at the tile's first row; rows past the tile end belong to the
// next tile (or are zero-filled past T), get zero probabilities and are never stored.  S = Q K^T is computed for the whole
// 128 x 128 tile and only the block diagonal is kept: each query row sees exactly the keys of its own sequence, whose bounds
// come from a per-tile table in shared memory.  Probabilities outside the segment are written as zeros, so O = P V and the
// three backward products come out per sequence from single MMA chains, and every key row belongs to exactly one tile: dK and
// dV are plain stores (deterministic, no atomics).
//
// The dropout element of (sequence s, head h, query i, key j) is numbered as in the padded [n, Lpad] layout the batch arrived
// in, ((s H + h) Lpad + i) ((Lpad + 1) & ~1) + j, so the mask equals the one the mma.sync kernels draw on that padded layout.
// lse and delta are f32 [H, T].
#include "common.cuh"
#include "internal.h"

namespace xfm {

constexpr int VT_HD = 64;
constexpr int VT_ROWS = 128;                 // rows of a tile
constexpr int VT_THREADS = 64 + 256;
constexpr int VT_OPB = VT_ROWS * 128;        // bytes one TMA box delivers (128 rows x 64 bf16)
constexpr int VT_TAB = 132;                  // ints of one segment table: bounds of up to 128 sequences (129 entries)
constexpr float VT_LOG2E = 1.4426950408889634f;

struct VAttnArgs {
  bf16* out;
  int64_t o_stride;
  float* lse;              // [H, T]
  const int32_t* cu;       // [n + 1]
  const int32_t* tiles;    // [n_tiles + 1]: first sequence of every tile, then n
  int n_tiles, H, Lpad, T;
  float scale, dropout_p;
  uint64_t seed;
  const uint64_t* salt;
  const float* delta;      // [H, T]
  bf16 *dq, *dk, *dv;
  int64_t dq_stride, dk_stride, dv_stride;
};

// Row r of a tile: its segment [lo, hi) in tile columns and its sequence index (lo = hi = 0 for rows past the tile end).
struct VRow {
  int lo, hi, seq;
};

// Writes the tile's segment table (bounds relative to the tile's first row) with the threads of a group of nthr threads
// (thread index r).  Returns the tile's first row.  Called before the group's barrier; vt_row reads the table after it.
XFM_DEVINL int vt_table(const VAttnArgs& a, int tile, int r, int nthr, int* tab, int& s0, int& nseq) {
  s0 = __ldg(a.tiles + tile);
  nseq = __ldg(a.tiles + tile + 1) - s0;
  const int row0 = __ldg(a.cu + s0);
  for (int j = r; j <= nseq; j += nthr) tab[j] = __ldg(a.cu + s0 + j) - row0;
  return row0;
}
XFM_DEVINL VRow vt_row(const int* tab, int s0, int nseq, int r) {
  VRow v{0, 0, 0};
  if (r >= tab[nseq]) return v;
  int lo = 0, hi = nseq;   // last j with tab[j] <= r
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (tab[mid] <= r) lo = mid; else hi = mid;
  }
  v.lo = tab[lo];
  v.hi = tab[lo + 1];
  v.seq = s0 + lo;
  return v;
}
// 16-column chunks [klo, khi) that hold the segments of a warp's 32 rows (empty when none of them is a tile row).
XFM_DEVINL void vt_union(const VRow& v, int& klo, int& khi) {
  const bool live = v.hi > v.lo;
  const int lo = __reduce_min_sync(0xffffffffu, live ? (unsigned)v.lo : 128u);
  const int hi = __reduce_max_sync(0xffffffffu, live ? (unsigned)v.hi : 0u);
  klo = lo >= hi ? 0 : lo >> 4;
  khi = lo >= hi ? 0 : (hi + 15) >> 4;
}
// Keep bits (bit 0: key j, bit 1: key j + 1) of the dropout mask of a row whose element index of key 0 is 2 * pair_row.
XFM_DEVINL uint32_t vt_keep2(uint64_t pair_row, int j, uint32_t seed_mix, uint32_t thr) {
  const uint64_t p0 = pair_row + (uint64_t)(j >> 1);
  const uint32_t k0 = drop_keep_pair(seed_mix, (uint32_t)p0, (uint32_t)(p0 >> 32), thr);
  if (!(j & 1)) return k0;
  const uint64_t p1 = p0 + 1;
  const uint32_t k1 = drop_keep_pair(seed_mix, (uint32_t)p1, (uint32_t)(p1 >> 32), thr);
  return ((k0 >> 1) & 1u) | ((k1 & 1u) << 1);
}
XFM_DEVINL uint64_t vt_pair_row(const VAttnArgs& a, int seq, int h, int q) {
  return ((((uint64_t)seq * a.H + h) * a.Lpad + q) * (uint64_t)((a.Lpad + 1) & ~1)) >> 1;
}

// ================================================================================================ forward
constexpr int VF_TAB = 2 * 3 * 16384 + 2 * 32768;                  // [tile buffer][unit parity][VT_TAB] segment tables
constexpr int VF_BARS = VF_TAB + 4 * VT_TAB * 4;
constexpr int VF_STAGE = (VF_BARS + 256 + 127) / 128 * 128;        // per-warp output staging: 8 x [32 rows][128 B]
constexpr int VF_SMEM = VF_STAGE + 8 * 4096;

__global__ void __launch_bounds__(VT_THREADS, 1)
vattn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const VAttnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* sQ = smem;                 // [2][16384]
  uint8_t* sK = sQ + 2 * 16384;
  uint8_t* sV = sK + 2 * 16384;
  uint8_t* sP = sV + 2 * 16384;       // [2][32768]: two 64-key blocks of 128 rows
  int* stab = (int*)(smem + VF_TAB);
  uint64_t* bars = (uint64_t*)(smem + VF_BARS);
  uint64_t *in_full = bars, *in_empty = bars + 2, *v_full = bars + 4, *v_empty = bars + 6, *s_full = bars + 8,
           *p_full = bars + 10, *o_full = bars + 12, *o_empty = bars + 14;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    for (int t = 0; t < 2; ++t) {
      mbar_init(&in_full[t], 1);
      mbar_init(&in_empty[t], 1);
      mbar_init(&v_full[t], 1);
      mbar_init(&v_empty[t], 1);
      mbar_init(&s_full[t], 1);
      mbar_init(&p_full[t], 4);
      mbar_init(&o_full[t], 1);
      mbar_init(&o_empty[t], 4);
    }
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
  constexpr uint32_t TM_O = 256;

  const int n_work = a.n_tiles * a.H;
  const int t0 = (int)((int64_t)blockIdx.x * n_work / gridDim.x);
  const int t1 = (int)((int64_t)(blockIdx.x + 1) * n_work / gridDim.x);
  const int n_units = (t1 - t0 + 1) / 2;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t ph = 0;
      for (int j = 0; j < n_units; ++j) {
        for (int t = 0; t < 2; ++t) {
          const int w = t0 + 2 * j + t;
          if (w >= t1) break;
          const int h = w / a.n_tiles, tile = w % a.n_tiles;
          const int row0 = __ldg(a.cu + __ldg(a.tiles + tile));
          mbar_wait_relaxed(&in_empty[t], ph ^ 1);
          mbar_arrive_expect_tx(&in_full[t], 2 * VT_OPB);
          tma_load_2d(sQ + t * 16384, &map_q, &in_full[t], h * VT_HD, row0);
          tma_load_2d(sK + t * 16384, &map_k, &in_full[t], h * VT_HD, row0);
          mbar_wait_relaxed(&v_empty[t], ph ^ 1);
          mbar_arrive_expect_tx(&v_full[t], VT_OPB);
          tma_load_2d(sV + t * 16384, &map_v, &v_full[t], h * VT_HD, row0);
        }
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idesc_o = make_idesc_bf16(128, VT_HD, 0, 1);
      const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV), aP = smem_u32(sP);
      uint32_t ph = 0;
      for (int j = 0; j < n_units; ++j) {
        for (int t = 0; t < 2; ++t) {   // S buffer t is free: the previous unit's p_full[t] was consumed below
          if (t0 + 2 * j + t >= t1) break;
          mbar_wait(&in_full[t], ph);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + t * 128, make_smem_desc(aQ + t * 16384 + k * 32, 16, 1024),
                      make_smem_desc(aK + t * 16384 + k * 32, 16, 1024), idesc_s, k > 0 ? 1u : 0u);
          umma_commit(&s_full[t]);
          umma_commit(&in_empty[t]);
        }
        for (int t = 0; t < 2; ++t) {
          if (t0 + 2 * j + t >= t1) break;
          mbar_wait(&v_full[t], ph);
          mbar_wait(&p_full[t], ph);
          mbar_wait(&o_empty[t], ph ^ 1);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16(tmem_base + TM_O + t * 64, make_smem_desc(aP + t * 32768 + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                      make_smem_desc(aV + t * 16384 + k * 2048, 8192, 1024), idesc_o, k > 0 ? 1u : 0u);
          umma_commit(&o_full[t]);
          umma_commit(&v_empty[t]);
        }
        ph ^= 1;
      }
    }
    __syncwarp();
  } else {
    const int t = (warp - 2) >> 2;             // tile buffer of this warpgroup
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint32_t t_s = lane_base + (uint32_t)(t * 128), t_o = lane_base + TM_O + (uint32_t)(t * 64);
    const float scale2 = a.scale * VT_LOG2E;
    const bool drop_on = a.dropout_p > 0.f;
    const float inv_keep = drop_on ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
    const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
    uint8_t* myP = sP + t * 32768 + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    uint32_t ph = 0;
    for (int j = 0; j < n_units; ++j) {
      const int w = t0 + 2 * j + t;
      if (w >= t1) break;
      const int h = w / a.n_tiles, tile = w % a.n_tiles;
      int* tab = stab + (t * 2 + (j & 1)) * VT_TAB;
      int s0, nseq;
      const int row0 = vt_table(a, tile, r, 128, tab, s0, nseq);
      named_bar_sync(1 + t, 128);
      const VRow rw = vt_row(tab, s0, nseq, r);
      const bool valid = rw.hi > rw.lo;
      const int len = rw.hi - rw.lo;
      int klo, khi;
      vt_union(rw, klo, khi);
      const uint64_t pair_row = vt_pair_row(a, rw.seq, h, r - rw.lo);
      mbar_wait(&s_full[t], ph);
      tc_fence_after();
      float m = -INFINITY;
      {
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll 1
        for (int k = klo; k < khi; ++k) {   // warp-uniform bounds
          uint32_t v[32];
          tmem_ld_32x32_16(t_s + k * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 16; ++e)
            if ((unsigned)(k * 16 + e - rw.lo) < (unsigned)len) m4[e & 3] = fmaxf(m4[e & 3], __uint_as_float(v[e]) * scale2);
        }
        m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      }
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
      for (int k = 0; k < 8; ++k) {
        uint32_t v[32];
        const bool in_union = k >= klo && k < khi;   // warp-uniform; other chunks of the row are zeros
        if (in_union) {
          tmem_ld_32x32_16(t_s + k * 16, v);
          tmem_ld_wait();
        }
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          const int col8 = k * 16 + g8 * 8;
          float p[8];
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            float p0 = 0.f, p1 = 0.f;
            const int jk = col8 + e - rw.lo;      // key position inside the sequence
            const bool in0 = in_union && (unsigned)jk < (unsigned)len, in1 = in_union && (unsigned)(jk + 1) < (unsigned)len;
            if (in0) {
              p0 = ex2_approx(fmaf(__uint_as_float(v[g8 * 8 + e]), scale2, -m));
              s4[e & 3] += p0;
            }
            if (in1) {
              p1 = ex2_approx(fmaf(__uint_as_float(v[g8 * 8 + e + 1]), scale2, -m));
              s4[(e + 1) & 3] += p1;
            }
            if (drop_on && (in0 || in1)) {
              const uint32_t keep = vt_keep2(pair_row, jk, seed_mix, thr);
              p0 = (keep & 1u) ? p0 * inv_keep : 0.f;
              p1 = (keep & 2u) ? p1 * inv_keep : 0.f;
            }
            p[e] = p0;
            p[e + 1] = p1;
          }
          st_bf16x8(myP + (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4), p);
        }
      }
      const float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[t]);
      mbar_wait(&o_full[t], ph);
      tc_fence_after();
      uint32_t o[2][32];
      tmem_ld_32x32(t_o, o[0]);
      tmem_ld_32x32(t_o + 32, o[1]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[t]);
      {
        // each warp stages its 32 rows and stores four whole 128-byte rows per instruction (tile rows are consecutive rows)
        uint8_t* stg = smem + VF_STAGE + (warp - 2) * 4096;
        const float inv = valid ? 1.0f / sum : 0.f;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            float vv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) vv[k] = __uint_as_float(o[hh][e + k]) * inv;
            st_bf16x8(stg + lane * 128 + (((hh * 4 + (e >> 3)) ^ (lane & 7)) << 4), vv);
          }
        if (valid && a.lse) a.lse[(int64_t)h * a.T + row0 + r] = (m + log2f(sum)) * 0.6931471805599453f;
        __syncwarp();
        const int ch = lane & 7;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int sl = it * 4 + (lane >> 3);
          const int v2 = __shfl_sync(0xffffffffu, (int)valid, sl);
          const uint4 v4 = *(const uint4*)(stg + sl * 128 + ((ch ^ (sl & 7)) << 4));
          if (v2) *(uint4*)(a.out + ((int64_t)row0 + quad * 32 + sl) * a.o_stride + h * VT_HD + ch * 8) = v4;
        }
        __syncwarp();
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

// ================================================================================================ backward (fused)
// Per tile: S = Q K^T and dP = dO V^T into TMEM stage i & 1; the two warpgroups split each warp's chunk union in halves (and
// zero the chunks outside it) and write P~ = keep * P / (1-p) and dS = P o (keep * dP / (1-p) - delta) to shared memory; then
// dQ = dS K, dK = dS^T Q and dV = P~^T dO accumulate into the TMEM columns S / dP occupied.  Operands and TMEM are
// double-buffered; P~ / dS are single-buffered (the next tile writes them after this tile's products completed: out_full).
constexpr int VB_TAB = 2 * 4 * 16384 + 2 * 32768;                 // [stage][VT_TAB] segment tables
constexpr int VB_BARS = VB_TAB + 2 * VT_TAB * 4;
constexpr int VB_STAGE = (VB_BARS + 256 + 127) / 128 * 128;       // per-warp output staging: 8 x [32 rows][64 B]
constexpr int VB_SMEM = VB_STAGE + 8 * 2048;

__global__ void __launch_bounds__(VT_THREADS, 1)
vattn_bwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                    const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v, const VAttnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* sQ = smem;                  // [2][16384] each
  uint8_t* sdO = sQ + 2 * 16384;
  uint8_t* sK = sdO + 2 * 16384;
  uint8_t* sV = sK + 2 * 16384;
  uint8_t* sP = sV + 2 * 16384;        // 32768
  uint8_t* sdS = sP + 32768;           // 32768
  int* stab = (int*)(smem + VB_TAB);
  uint64_t* bars = (uint64_t*)(smem + VB_BARS);
  uint64_t *in_full = bars, *in_empty = bars + 2, *sd_full = bars + 4, *tm_empty = bars + 6, *out_full = bars + 8,
           *ds_full = bars + 10;
  uint32_t* tmem_ptr = (uint32_t*)(bars + 11);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_do);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    for (int t = 0; t < 2; ++t) {
      mbar_init(&in_full[t], 1);
      mbar_init(&in_empty[t], 1);
      mbar_init(&sd_full[t], 1);
      mbar_init(&tm_empty[t], 8);
      mbar_init(&out_full[t], 1);
    }
    mbar_init(ds_full, 8);
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

  const int n_work = a.n_tiles * a.H;
  const int t0 = (int)((int64_t)blockIdx.x * n_work / gridDim.x);
  const int t1 = (int)((int64_t)(blockIdx.x + 1) * n_work / gridDim.x);
  const int n = t1 - t0;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < n; ++i) {
        const int st = i & 1;
        const uint32_t par = (uint32_t)(i >> 1) & 1u;
        const int w = t0 + i;
        const int h = w / a.n_tiles, tile = w % a.n_tiles;
        const int row0 = __ldg(a.cu + __ldg(a.tiles + tile));
        mbar_wait_relaxed(&in_empty[st], par ^ 1);
        mbar_arrive_expect_tx(&in_full[st], 4 * VT_OPB);
        tma_load_2d(sQ + st * 16384, &map_q, &in_full[st], h * VT_HD, row0);
        tma_load_2d(sK + st * 16384, &map_k, &in_full[st], h * VT_HD, row0);
        tma_load_2d(sdO + st * 16384, &map_do, &in_full[st], h * VT_HD, row0);
        tma_load_2d(sV + st * 16384, &map_v, &in_full[st], h * VT_HD, row0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idesc_dq = make_idesc_bf16(128, VT_HD, 0, 1);
      constexpr uint32_t idesc_dkv = make_idesc_bf16(128, VT_HD, 1, 1);
      const uint32_t aQ = smem_u32(sQ), adO = smem_u32(sdO), aK = smem_u32(sK), aV = smem_u32(sV), aP = smem_u32(sP),
                     adS = smem_u32(sdS);
      auto issue_sdp = [&](int i) {
        const int st = i & 1;
        const uint32_t par = (uint32_t)(i >> 1) & 1u;
        mbar_wait(&in_full[st], par);
        mbar_wait(&tm_empty[st], par ^ 1);
        tc_fence_after();
        const uint32_t tm = tmem_base + st * 256;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tm, make_smem_desc(aQ + st * 16384 + k * 32, 16, 1024), make_smem_desc(aK + st * 16384 + k * 32, 16, 1024),
                    idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tm + 128, make_smem_desc(adO + st * 16384 + k * 32, 16, 1024),
                    make_smem_desc(aV + st * 16384 + k * 32, 16, 1024), idesc_s, k > 0 ? 1u : 0u);
        umma_commit(&sd_full[st]);
      };
      if (n > 0) issue_sdp(0);
      for (int i = 0; i < n; ++i) {
        const int st = i & 1;
        if (i + 1 < n) issue_sdp(i + 1);
        mbar_wait(ds_full, (uint32_t)i & 1u);
        tc_fence_after();
        const uint32_t tm = tmem_base + st * 256;
#pragma unroll
        for (int k = 0; k < 8; ++k)   // dQ = dS K: dS K-major, K MN-major
          umma_bf16(tm, make_smem_desc(adS + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                    make_smem_desc(aK + st * 16384 + k * 2048, 8192, 1024), idesc_dq, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 8; ++k)   // dK = dS^T Q: the same dS buffer read MN-major (64-key blocks 16 KB apart)
          umma_bf16(tm + 64, make_smem_desc(adS + k * 2048, 16384, 1024), make_smem_desc(aQ + st * 16384 + k * 2048, 8192, 1024),
                    idesc_dkv, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 8; ++k)   // dV = P~^T dO
          umma_bf16(tm + 128, make_smem_desc(aP + k * 2048, 16384, 1024), make_smem_desc(adO + st * 16384 + k * 2048, 8192, 1024),
                    idesc_dkv, k > 0 ? 1u : 0u);
        umma_commit(&out_full[st]);
        umma_commit(&in_empty[st]);
      }
    }
    __syncwarp();
  } else {
    const int wg = (warp - 2) >> 2;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
    const float scale2 = a.scale * VT_LOG2E;
    const bool drop_on = a.dropout_p > 0.f;
    const float inv_keep = drop_on ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
    const uint32_t seed_mix = drop_seed_mix(a.seed + *a.salt), thr = drop_threshold(a.dropout_p);
    uint8_t* myP = sP + (r >> 3) * 1024 + (r & 7) * 128;
    uint8_t* myD = sdS + (r >> 3) * 1024 + (r & 7) * 128;
    const int sw = r & 7;
    for (int i = 0; i < n; ++i) {
      const int st = i & 1;
      const uint32_t par = (uint32_t)(i >> 1) & 1u;
      const int w = t0 + i;
      const int h = w / a.n_tiles, tile = w % a.n_tiles;
      int* tab = stab + st * VT_TAB;
      int s0, nseq;
      const int row0 = vt_table(a, tile, wg == 0 ? r : 1 << 20, 128, tab, s0, nseq);   // warpgroup 0 writes the table
      named_bar_sync(1, 256);
      const VRow rw = vt_row(tab, s0, nseq, r);
      const bool valid = rw.hi > rw.lo;
      const int len = rw.hi - rw.lo;
      int klo, khi;
      vt_union(rw, klo, khi);
      const int kmid = klo + (khi - klo + 1) / 2;
      const int kb = wg == 0 ? 0 : kmid, ke = wg == 0 ? kmid : 8;   // chunks of this warpgroup: its half of the union + zeros
      const int64_t st_row = (int64_t)h * a.T + row0 + r;
      const float lse2 = valid ? __ldg(a.lse + st_row) * VT_LOG2E : 0.f;
      const float dl = valid ? __ldg(a.delta + st_row) : 0.f;
      const uint64_t pair_row = vt_pair_row(a, rw.seq, h, r - rw.lo);
      const uint32_t tm = lane_base + (uint32_t)(st * 256);
      mbar_wait(&sd_full[st], par);
      tc_fence_after();
      for (int k = kb; k < ke; ++k) {
        uint32_t vs[32], vp[32];
        const bool in_union = k >= klo && k < khi;   // warp-uniform
        if (in_union) {
          tmem_ld_32x32_16(tm + k * 16, vs);
          tmem_ld_32x32_16(tm + 128 + k * 16, vp);
          tmem_ld_wait();
        }
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          const int col8 = k * 16 + g8 * 8;
          float pp[8], ds[8];
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            float p0 = 0.f, p1 = 0.f, d0 = 0.f, d1 = 0.f;
            const int jk = col8 + e - rw.lo;
            const bool in0 = in_union && (unsigned)jk < (unsigned)len, in1 = in_union && (unsigned)(jk + 1) < (unsigned)len;
            if (in0 || in1) {
              float k0 = 1.f, k1 = 1.f;
              if (drop_on) {
                const uint32_t keep = vt_keep2(pair_row, jk, seed_mix, thr);
                k0 = (keep & 1u) ? inv_keep : 0.f;
                k1 = (keep & 2u) ? inv_keep : 0.f;
              }
              if (in0) {
                p0 = ex2_approx(fmaf(__uint_as_float(vs[g8 * 8 + e]), scale2, -lse2));
                d0 = p0 * (__uint_as_float(vp[g8 * 8 + e]) * k0 - dl);
                p0 *= k0;
              }
              if (in1) {
                p1 = ex2_approx(fmaf(__uint_as_float(vs[g8 * 8 + e + 1]), scale2, -lse2));
                d1 = p1 * (__uint_as_float(vp[g8 * 8 + e + 1]) * k1 - dl);
                p1 *= k1;
              }
            }
            pp[e] = p0;
            pp[e + 1] = p1;
            ds[e] = d0;
            ds[e + 1] = d1;
          }
          const int off8 = (col8 >> 6) * 16384 + ((((col8 & 63) >> 3) ^ sw) << 4);
          st_bf16x8(myP + off8, pp);
          st_bf16x8(myD + off8, ds);
        }
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
      mbar_wait(&out_full[st], par);
      tc_fence_after();
      // TMEM columns of the stage: dQ [0,64)  dK [64,128)  dV [128,192).  Warpgroup 0 drains [0,96), warpgroup 1 [96,192).
      uint32_t o[3][32];
      const uint32_t src = tm + (uint32_t)(wg * 96);
      tmem_ld_32x32(src, o[0]);
      tmem_ld_32x32(src + 32, o[1]);
      tmem_ld_32x32(src + 64, o[2]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tm_empty[st]);
      {
        // wg 0: dQ[0:32) dQ[32:64) dK[0:32)     wg 1: dK[32:64) dV[0:32) dV[32:64).  Each 32-column part is staged per warp
        // ([32 rows][64 B], chunk index xor-ed with (row >> 1) & 3) and stored eight rows x 64 bytes per instruction.
        uint8_t* stg = smem + VB_STAGE + (warp - 2) * 2048;
        const int64_t rowq = (int64_t)row0 + quad * 32;
#pragma unroll
        for (int part = 0; part < 3; ++part) {
          bf16* dst;
          int64_t ld;
          float mul;
          if (wg == 0) {
            dst = part < 2 ? a.dq + part * 32 : a.dk;
            ld = part < 2 ? a.dq_stride : a.dk_stride;
            mul = a.scale;
          } else {
            dst = part == 0 ? a.dk + 32 : a.dv + (part - 1) * 32;
            ld = part == 0 ? a.dk_stride : a.dv_stride;
            mul = part == 0 ? a.scale : 1.0f;
          }
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            float vv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) vv[k] = __uint_as_float(o[part][e + k]) * mul;
            st_bf16x8(stg + lane * 64 + ((((e >> 3)) ^ ((lane >> 1) & 3)) << 4), vv);
          }
          __syncwarp();
          const int ch = lane & 3;
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int sl = it * 8 + (lane >> 2);
            const int v2 = __shfl_sync(0xffffffffu, (int)valid, sl);
            const uint4 v4 = *(const uint4*)(stg + sl * 64 + ((ch ^ ((sl >> 1) & 3)) << 4));
            if (v2) *(uint4*)(dst + (rowq + sl) * ld + h * VT_HD + ch * 8) = v4;
          }
          __syncwarp();
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------ host
// The tile rule: a tile is a maximal run of consecutive sequences of at most VT_ROWS rows in total.
int varlen_plan(const int32_t* lengths, int n, int32_t* cu_seqlens, int32_t* tiles, int32_t* n_tiles) {
  if (n <= 0 || !lengths || !cu_seqlens || !tiles || !n_tiles) {
    set_error("attention varlen plan: need n > 0 sequences and non-null pointers");
    return XFM_ERR_BAD_ARG;
  }
  int64_t total = 0;
  for (int s = 0; s < n; ++s) {
    if (lengths[s] < 1 || lengths[s] > VT_ROWS) {
      set_error("attention varlen plan: sequence %d has %d tokens (1 to %d are supported)", s, lengths[s], VT_ROWS);
      return XFM_ERR_BAD_ARG;
    }
    total += lengths[s];
  }
  if (total > INT32_MAX) {
    set_error("attention varlen plan: %lld rows do not fit int32", (long long)total);
    return XFM_ERR_BAD_ARG;
  }
  cu_seqlens[0] = 0;
  for (int s = 0; s < n; ++s) cu_seqlens[s + 1] = cu_seqlens[s] + lengths[s];
  int nt = 0;
  for (int s = 0; s < n;) {
    tiles[nt++] = s;
    int rows = 0;
    while (s < n && rows + lengths[s] <= VT_ROWS) rows += lengths[s++];
  }
  tiles[nt] = n;
  *n_tiles = nt;
  return 0;
}

static int vt_check(const xfm_varlen_params* p, bool bwd) {
  if (!p || !p->q || !p->k || !p->v || !p->out || !p->lse || !p->cu_seqlens || !p->tiles) {
    set_error("attention varlen: null pointer");
    return XFM_ERR_BAD_ARG;
  }
  if (p->n <= 0 || p->n_tiles <= 0 || p->n_tiles > p->n || p->H <= 0 || p->T <= 0 || p->Lpad <= 0) {
    set_error("attention varlen: bad shape (n %d, tiles %d, H %d, T %d, Lpad %d)", p->n, p->n_tiles, p->H, p->T, p->Lpad);
    return XFM_ERR_BAD_ARG;
  }
  if (!(p->dropout_p >= 0.f && p->dropout_p < 1.f)) {
    set_error("attention varlen: dropout p must be in [0, 1)");
    return XFM_ERR_BAD_ARG;
  }
  uintptr_t al = (uintptr_t)p->q | (uintptr_t)p->k | (uintptr_t)p->v | (uintptr_t)p->out;
  int64_t st = p->q_stride | p->k_stride | p->v_stride | p->o_stride;
  if (bwd) {
    if (!p->dout || !p->delta || !p->dq || !p->dk || !p->dv) {
      set_error("attention varlen bwd: null pointer");
      return XFM_ERR_BAD_ARG;
    }
    al |= (uintptr_t)p->dout | (uintptr_t)p->dq | (uintptr_t)p->dk | (uintptr_t)p->dv;
    st |= p->do_stride | p->dq_stride | p->dk_stride | p->dv_stride;
  }
  if ((al & 15) || (st & 7)) {
    set_error("attention varlen: operands must be 16-byte aligned with row strides that are multiples of 8");
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

static int vt_fill(const xfm_varlen_params* p, VAttnArgs& a) {
  a.out = (bf16*)p->out; a.o_stride = p->o_stride; a.lse = p->lse; a.cu = p->cu_seqlens; a.tiles = p->tiles;
  a.n_tiles = p->n_tiles; a.H = p->H; a.Lpad = p->Lpad; a.T = p->T;
  a.scale = p->scale; a.dropout_p = p->dropout_p; a.seed = p->dropout_seed; a.salt = seed_salt_ptr();
  a.delta = p->delta;
  a.dq = (bf16*)p->dq; a.dk = (bf16*)p->dk; a.dv = (bf16*)p->dv;
  a.dq_stride = p->dq_stride; a.dk_stride = p->dk_stride; a.dv_stride = p->dv_stride;
  const int n_work = a.n_tiles * a.H;
  return n_work < num_sms() ? n_work : num_sms();
}

static int vt_encode(CUtensorMap* map, const void* base, const xfm_varlen_params* p, int64_t ld) {
  return encode_rows(map, base, (uint64_t)p->H * VT_HD, (uint64_t)p->T, (uint64_t)ld, VT_ROWS);
}

int varlen_attention_fwd(const xfm_varlen_params* p, cudaStream_t s) {
  if (vt_check(p, false)) return XFM_ERR_BAD_ARG;
  VAttnArgs a;
  const int grid = vt_fill(p, a);
  CUtensorMap mq, mk, mv;
  int rc = vt_encode(&mq, p->q, p, p->q_stride);
  if (!rc) rc = vt_encode(&mk, p->k, p, p->k_stride);
  if (!rc) rc = vt_encode(&mv, p->v, p, p->v_stride);
  if (rc) return rc;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(vattn_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, VF_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  vattn_fwd_tc_kernel<<<grid, VT_THREADS, VF_SMEM, s>>>(mq, mk, mv, a);
  count_launch();
  return (int)cudaGetLastError();
}

int varlen_attention_bwd(const xfm_varlen_params* p, cudaStream_t s) {
  if (vt_check(p, true)) return XFM_ERR_BAD_ARG;
  VAttnArgs a;
  const int grid = vt_fill(p, a);
  int rc = launch_attn_delta((const bf16_t*)p->dout, p->do_stride, (const bf16_t*)p->out, p->o_stride, p->delta, 1, p->H, p->T, s);
  if (rc) return rc;
  CUtensorMap mq, mdo, mk, mv;
  rc = vt_encode(&mq, p->q, p, p->q_stride);
  if (!rc) rc = vt_encode(&mdo, p->dout, p, p->do_stride);
  if (!rc) rc = vt_encode(&mk, p->k, p, p->k_stride);
  if (!rc) rc = vt_encode(&mv, p->v, p, p->v_stride);
  if (rc) return rc;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(vattn_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, VB_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  vattn_bwd_tc_kernel<<<grid, VT_THREADS, VB_SMEM, s>>>(mq, mdo, mk, mv, a);
  count_launch();
  return (int)cudaGetLastError();
}

}  // namespace xfm
