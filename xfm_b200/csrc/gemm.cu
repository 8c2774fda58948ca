// K1 — persistent warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = epilogue(A[M,K] · B[N,K]^T), bf16 operands, fp32 accumulation in TMEM.
//
// CTA = 320 threads: warp 0 = TMA producer, warp 1 = TMEM owner + single-thread UMMA issuer,
// warps 2..9 = epilogue (two per TMEM lane quadrant, each taking half of the tile's columns).  Operands are staged by TMA into a
// multi-stage ring of SWIZZLE_128B tiles (128 x 64 for A, BLOCK_N x 64 for B); the accumulator
// is double-buffered in TMEM (2 x BLOCK_N columns) so the epilogue of tile i overlaps the MMAs
// of tile i+1.  Both operands may be K-major (torch Linear forward) or MN-major (the operand's
// transpose is what lives in memory: dgrad reads W as [K_red, N], wgrad reads dY / X as [tokens, *]).
// Split-K (wgrad: few output tiles, long reduction) accumulates with fp32 vector atomics.
#include "common.cuh"
#include "internal.h"

namespace xfm {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int GEMM_THREADS = 64 + 8 * 32;  // TMA warp, MMA warp, 8 epilogue warps

struct GemmArgs {
  int M, N, K;
  int num_m_tiles, num_n_tiles, split_k, kb_total;
  int c_dtype, accumulate, act, res_dtype, rows_per_group;
  int64_t ldc, ld_aux_in, ld_aux_out, ld_res;
  void* C;
  const float* bias;
  const bf16* aux_in;
  bf16* aux_out;
  const float* col_scale;
  const float* row_group_scale;
  const void* residual;
  float dropout_p;
  uint64_t dropout_seed;
  const uint64_t* seed_salt;  // device word added to every dropout seed (advanced once per step: CUDA-graph replays)
  int vec_ok;    // every epilogue pointer / leading dimension allows 2-element vector access at even columns
  int epi_mode;  // see epilogue_block
  int tma_epi;   // CTA-pair kernel: modes 0 / 1 store bf16 tiles with TMA (epilogue_tma_block); 2 = f32 TMA epilogue
  int epi_interleave;  // f32 / dGELU TMA epilogues: the two warps of a lane quadrant take alternate 32-column blocks
  int n_fastest; // CTA-pair kernel: consecutive tiles walk N first (all N tiles of an M tile run concurrently: A is read from
                 // HBM once even when it is far larger than L2; the weight operand B stays L2 resident either way)
};

template <int BLOCK_N>
struct GemmCfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BLOCK_N == 256) ? 4 : (BLOCK_N == 128 ? 6 : 8);
  static constexpr int TMEM_COLS = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;
  static constexpr int EPI_BYTES = 8 * 32 * 34 * 4;  // 8 epilogue warps x [32][EPI_LD] fp32 transposition blocks
  // 227 KB (232448 B) is the per-CTA limit; the BLOCK_N = 256 configuration uses all of it (768 B of alignment slack:
  // dynamic shared memory starts 1024-aligned when the kernel has no static shared memory, checked in the kernel).
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 768 + 256 /*barriers*/;
};

// ---------------------------------------------------------------------------------------------- epilogue
// Each epilogue warp owns 32 accumulator rows (one TMEM lane quadrant).  tcgen05.ld hands thread t the row t, i.e. a
// row-per-thread layout whose direct global stores touch 32 different rows per instruction (16 B each).  The tile is
// therefore transposed through a per-warp shared-memory block of 32 rows x 64 columns (fp32, leading dimension 66 words:
// 8-byte accesses are bank-conflict free in both directions) so that phase 2 runs with lane = column pair: every global
// load / store / reduction of the fused epilogue (output, saved pre-activation, residual, dGELU input) is one fully
// coalesced 128-byte (bf16) or 256-byte (fp32) row segment per warp instruction.
constexpr int EPI_WARPS = 8;   // two per TMEM lane quadrant, each taking half of the tile's columns
constexpr int EPI_COLS = 32;
constexpr int EPI_LD = 34;     // words; 136 B rows: float2 accesses are 8-byte aligned and conflict free per half warp
constexpr int EPI_WARP_FLOATS = 32 * EPI_LD;

XFM_DEVINL float2 ld2_bf16(const bf16* p, bool vec, bool c1) {
  if (vec) return __bfloat1622float2(*(const __nv_bfloat162*)p);
  return make_float2(__bfloat162float(p[0]), c1 ? __bfloat162float(p[1]) : 0.f);
}
XFM_DEVINL void st2_bf16(bf16* p, float2 v, bool vec, bool c1) {
  if (vec) {
    *(__nv_bfloat162*)p = __floats2bfloat162_rn(v.x, v.y);
  } else {
    p[0] = __float2bfloat16(v.x);
    if (c1) p[1] = __float2bfloat16(v.y);
  }
}

// Phase 2 for one 32 x 32 block: rows row_base .. +31, columns n .. n+31.  Lane l owns columns n + 2*(l%16), +1 of rows
// (l/16), (l/16)+2, ...: one warp instruction moves two 32-column row segments (64 B bf16 / 128 B fp32 each).
// The 16 row steps run as two batches of 8: all global loads of a batch (dGELU pre-activation, residual) are issued
// first, then the arithmetic, then the stores, so 8 loads per lane are in flight and no load waits behind a store
// that might alias it.
// MODE 0: C = bf16(act(acc + bias)), act in {none, GELU}, optional saved pre-activation  (forward Linear layers)
// MODE 1: C = bf16((acc + bias) * gelu'(aux_in))                                        (dgrad through GELU)
// MODE 2: everything (tanh, LayerScale / DropPath scales, dropout, residual, fp32 output, split-K reduction)
// FULL: the block lies inside the matrix and every pointer allows vector access, so all bounds predicates fold away.
template <int MODE, bool FULL>
XFM_DEVINL void epilogue_block(const GemmArgs& g, const float* stage, int row_base, int n, int lane) {
  const int col = n + 2 * (lane & 15);
  if (!FULL && col >= g.N) return;
  const bool c1 = FULL ? true : (col + 1 < g.N);
  const bool vec = FULL ? true : (g.vec_ok && c1);
  float2 bias = make_float2(0.f, 0.f), cs = make_float2(1.f, 1.f);
  if (g.bias) {
    bias.x = __ldg(g.bias + col);
    if (c1) bias.y = __ldg(g.bias + col + 1);
  }
  if (MODE == 2 && g.col_scale) {
    cs.x = __ldg(g.col_scale + col);
    if (c1) cs.y = __ldg(g.col_scale + col + 1);
  }
  const float inv_keep = (MODE == 2 && g.dropout_p > 0.f) ? 1.0f / (1.0f - g.dropout_p) : 1.0f;
  const int nrows = FULL ? 32 : min(32, g.M - row_base);
  // Per-sample (DropPath) scale: a 32-row block touches at most two row groups when a group has >= 32 rows, so the two
  // scales are fetched once per block instead of one divide + dependent load per row inside the arithmetic.
  float rgs_lo = 1.f, rgs_hi = 1.f;
  int rgs_split = 32;
  const bool rgs_fast = MODE == 2 && g.row_group_scale != nullptr && g.rows_per_group >= 32;
  if (rgs_fast) {
    const int g0 = row_base / g.rows_per_group;
    const int g1 = (row_base + nrows - 1) / g.rows_per_group;
    rgs_lo = __ldg(g.row_group_scale + g0);
    rgs_hi = __ldg(g.row_group_scale + g1);
    rgs_split = (g0 + 1) * g.rows_per_group - row_base;   // first row offset of the second group
  }
  const bool has_aux_out = MODE != 1 && g.aux_out != nullptr;
  const int act = g.act;
  const bool want_aux = MODE == 1 || (MODE == 2 && act == 2);
  const bool want_res = MODE == 2 && g.residual != nullptr;
  const int ldc = (int)g.ldc, ld_ai = (int)g.ld_aux_in, ld_ao = (int)g.ld_aux_out, ld_r = (int)g.ld_res;
  const int64_t rb = row_base;
  const bf16* aux_in0 = want_aux ? g.aux_in + rb * g.ld_aux_in + col : nullptr;
  bf16* aux_out0 = has_aux_out ? g.aux_out + rb * g.ld_aux_out + col : nullptr;
  const char* res0 = want_res ? (const char*)g.residual + (rb * g.ld_res + col) * (g.res_dtype == 0 ? 2 : 4) : nullptr;
  char* c0 = (char*)g.C + (rb * g.ldc + col) * (g.c_dtype == 0 ? 2 : 4);
  const float* st0 = stage + 2 * (lane & 15);
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    const int rr0 = (lane >> 4) + 16 * half;
    if (rr0 >= nrows) break;
    uint32_t aux[8];
    float2 res[8], v[8];
    if (want_aux) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = rr0 + 2 * i;
        aux[i] = 0u;
        if (rr < nrows) {
          const bf16* p = aux_in0 + rr * ld_ai;
          if (vec) aux[i] = *(const uint32_t*)p;
          else aux[i] = (uint32_t) * (const uint16_t*)p | (c1 ? ((uint32_t) * (const uint16_t*)(p + 1) << 16) : 0u);
        }
      }
    }
    if (want_res) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = rr0 + 2 * i;
        res[i] = make_float2(0.f, 0.f);
        if (rr < nrows) {
          if (g.res_dtype == 0) {
            const bf16* p = (const bf16*)res0 + rr * ld_r;
            res[i] = ld2_bf16(p, vec, c1);
          } else {
            const float* p = (const float*)res0 + rr * ld_r;
            res[i] = vec ? *(const float2*)p : make_float2(p[0], c1 ? p[1] : 0.f);
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i] = *(const float2*)(st0 + (rr0 + 2 * i) * EPI_LD);
      v[i].x += bias.x;
      v[i].y += bias.y;
    }
    if (has_aux_out) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (rr0 + 2 * i < nrows) st2_bf16(aux_out0 + (rr0 + 2 * i) * ld_ao, v[i], vec, c1);
    }
    if (MODE != 1 && act == 1) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        v[i].x = gelu_fast(v[i].x);
        v[i].y = gelu_fast(v[i].y);
      }
    }
    if (want_aux) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 a = __bfloat1622float2(*(const __nv_bfloat162*)&aux[i]);
        v[i].x *= gelu_grad_fast(a.x);
        v[i].y *= gelu_grad_fast(a.y);
      }
    }
    if (MODE == 2) {
      if (act == 3) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v[i].x = tanhf(v[i].x);
          v[i].y = tanhf(v[i].y);
        }
      }
      if (g.col_scale || g.row_group_scale) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float s = 1.f;
          if (rgs_fast) s = (rr0 + 2 * i < rgs_split) ? rgs_lo : rgs_hi;
          else if (g.row_group_scale) s = __ldg(g.row_group_scale + min(row_base + rr0 + 2 * i, g.M - 1) / g.rows_per_group);
          v[i].x *= cs.x * s;
          v[i].y *= cs.y * s;
        }
      }
      if (g.dropout_p > 0.f) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint64_t base = (uint64_t)(row_base + rr0 + 2 * i) * (uint64_t)g.N + (uint64_t)col;
          v[i].x = drop_keep_idx(g.dropout_seed + *g.seed_salt, base, g.dropout_p) ? v[i].x * inv_keep : 0.f;
          v[i].y = drop_keep_idx(g.dropout_seed + *g.seed_salt, base + 1, g.dropout_p) ? v[i].y * inv_keep : 0.f;
        }
      }
      if (want_res) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v[i].x += res[i].x;
          v[i].y += res[i].y;
        }
      }
    }
    if (MODE != 2 || g.c_dtype == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (rr0 + 2 * i < nrows) st2_bf16((bf16*)c0 + (rr0 + 2 * i) * ldc, v[i], vec, c1);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (rr0 + 2 * i >= nrows) continue;
        float* dst = (float*)c0 + (rr0 + 2 * i) * ldc;
        if (g.accumulate) {
          if (vec) {
            asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(dst), "f"(v[i].x), "f"(v[i].y) : "memory");
          } else {
            atomicAdd(dst, v[i].x);
            if (c1) atomicAdd(dst + 1, v[i].y);
          }
        } else if (vec) {
          *(float2*)dst = v[i];
        } else {
          dst[0] = v[i].x;
          if (c1) dst[1] = v[i].y;
        }
      }
    }
  }
}

template <int MODE>
XFM_DEVINL void epilogue_one(const GemmArgs& g, float* stage, uint32_t taddr, int row_base, int n, int lane, bool has_work) {
  uint32_t r[32];
  tmem_ld_32x32(taddr, r);
  tmem_ld_wait();
  if (!has_work) return;
  __syncwarp();  // phase 2 of the previous block has finished reading the staging block
#pragma unroll
  for (int j = 0; j < 32; j += 2)
    *(float2*)(stage + lane * EPI_LD + j) = make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1]));
  __syncwarp();
  if (g.vec_ok && row_base + 32 <= g.M && n + 32 <= g.N) epilogue_block<MODE, true>(g, stage, row_base, n, lane);
  else epilogue_block<MODE, false>(g, stage, row_base, n, lane);
}

// ---------------------------------------------------------------------------------------------- TMA-store epilogue
// Modes 0 and 1 of the CTA-pair kernel (bf16 outputs).  The accumulator block stays in its tcgen05.ld layout (lane = row,
// 32 consecutive columns): bias / GELU / dGELU are applied in registers, the bf16 row (64 bytes) goes to a dense 32 x 32
// staging tile in shared memory and ONE thread hands the tile to the TMA engine, which writes full 64-byte row segments and
// clips rows / columns beyond the matrix.  No transposition pass, no per-row address arithmetic, no bounds predicates: about
// 70 instructions per lane and block instead of ~500, which is what the fused epilogues are bound by.
// Four staging tiles per warp (8 KB): the saved pre-activation and the output of a block use two, so the copies of block i
// still read shared memory while block i + 1 is computed (cp.async.bulk.wait_group.read keeps at most one block in flight).
constexpr int TMA_EPI_TILE_BYTES = 32 * 32 * 2;
constexpr int TMA_EPI_WARP_BYTES = 4 * TMA_EPI_TILE_BYTES;

// `sw` = (row >> 1) & 3: SWIZZLE_64B position of the row's 16-byte chunks (tile base 512-byte aligned), which makes the
// lane = row stores of a quarter warp hit 8 different bank groups (dense 64-byte rows: 4-way conflicts, 6.0 M conflict
// cycles per fc1 GEMM in ncu, on the pipe the UMMA operand reads already keep ~60 % busy).
XFM_DEVINL void st_row_bf16x32(uint8_t* row, const float (&v)[32], int sw) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint4 u;
    __nv_bfloat162 t0 = __floats2bfloat162_rn(v[8 * c], v[8 * c + 1]), t1 = __floats2bfloat162_rn(v[8 * c + 2], v[8 * c + 3]);
    __nv_bfloat162 t2 = __floats2bfloat162_rn(v[8 * c + 4], v[8 * c + 5]), t3 = __floats2bfloat162_rn(v[8 * c + 6], v[8 * c + 7]);
    u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
    *(uint4*)(row + 16 * (c ^ sw)) = u;
  }
}

template <int MODE>
XFM_DEVINL void epilogue_tma_block(const GemmArgs& g, const CUtensorMap* map_c, const CUtensorMap* map_aux, uint8_t* tiles,
                                   int& slot, uint32_t taddr, int row_base, int n, int lane, bool has_work) {
  uint32_t r[32];
  tmem_ld_32x32(taddr, r);
  // dGELU operand: this lane's row, 64 contiguous bytes; issued before the TMEM wait so the two latencies overlap
  uint4 aux[4] = {};
  const int row = row_base + lane;
  if (MODE == 1 && has_work && row < g.M) {
    const bf16* ap = g.aux_in + (int64_t)row * g.ld_aux_in + n;
    if (n + 32 <= g.N) {
#pragma unroll
      for (int c = 0; c < 4; ++c) aux[c] = *(const uint4*)(ap + 8 * c);
    } else {
      bf16* a16 = (bf16*)aux;
      for (int j = 0; j < 32 && n + j < g.N; ++j) a16[j] = ap[j];
    }
  }
  tmem_ld_wait();
  if (!has_work) return;
  float v[32];
  if (g.bias) {
    if (n + 32 <= g.N) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 b4 = __ldg((const float4*)(g.bias + n) + c);
        v[4 * c] = __uint_as_float(r[4 * c]) + b4.x;
        v[4 * c + 1] = __uint_as_float(r[4 * c + 1]) + b4.y;
        v[4 * c + 2] = __uint_as_float(r[4 * c + 2]) + b4.z;
        v[4 * c + 3] = __uint_as_float(r[4 * c + 3]) + b4.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + (n + j < g.N ? __ldg(g.bias + n + j) : 0.f);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  }
  // the copies issued two blocks ago have finished reading their staging tiles
  if (lane == 0) tma_store_wait_read<1>();
  __syncwarp();
  const bool has_aux_out = MODE == 0 && g.aux_out != nullptr;
  uint8_t* t_aux = tiles + slot * TMA_EPI_TILE_BYTES;
  uint8_t* t_c = tiles + (slot ^ 1) * TMA_EPI_TILE_BYTES;
  const int sw = (lane >> 1) & 3;
  if (has_aux_out) st_row_bf16x32(t_aux + lane * 64, v, sw);
  if (MODE == 0 && g.act == 1) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = gelu_fast(v[j]);
  }
  if (MODE == 1) {
    const __nv_bfloat162* a2 = (const __nv_bfloat162*)aux;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float2 af = __bfloat1622float2(a2[j]);
      v[2 * j] *= gelu_grad_fast(af.x);
      v[2 * j + 1] *= gelu_grad_fast(af.y);
    }
  }
  st_row_bf16x32(t_c + lane * 64, v, sw);
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) {
    if (has_aux_out) tma_store_2d(map_aux, t_aux, n, row_base);
    tma_store_2d(map_c, t_c, n, row_base);
    tma_store_commit();
  }
  slot ^= 2;
}

template <int BLOCK_N, int A_MN, int B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const GemmArgs g) {
  using Cfg = GemmCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  if ((int)(smem - smem_raw) + STAGES * Cfg::STAGE_BYTES + Cfg::EPI_BYTES + 256 > Cfg::SMEM_BYTES) __trap();
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * Cfg::A_BYTES;
  float* epi_stage = (float*)(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* bars = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES + Cfg::EPI_BYTES);
  uint64_t* full_bar = bars;                    // [STAGES]
  uint64_t* empty_bar = bars + STAGES;          // [STAGES]
  uint64_t* tmem_full = bars + 2 * STAGES;      // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2; // [2]
  uint32_t* tmem_ptr = (uint32_t*)(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int num_tiles = g.num_m_tiles * g.num_n_tiles * g.split_k;
  const int kb_per_split = (g.kb_total + g.split_k - 1) / g.split_k;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int ks = t % g.split_k;
        const int rest = t / g.split_k;
        const int m0 = (rest % g.num_m_tiles) * BLOCK_M;
        const int n0 = (rest / g.num_m_tiles) * BLOCK_N;
        const int kb0 = ks * kb_per_split;
        const int kb1 = min(g.kb_total, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_relaxed(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
          uint8_t* sa = smem_a + stage * Cfg::A_BYTES;
          uint8_t* sb = smem_b + stage * Cfg::B_BYTES;
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < BLOCK_M / 64; ++j)
              tma_load_2d(sa + j * (64 * BLOCK_K * 2), &map_a, &full_bar[stage], m0 + 64 * j, kb * BLOCK_K);
          } else {
            tma_load_2d(sa, &map_a, &full_bar[stage], kb * BLOCK_K, m0);
          }
          if (B_MN) {
#pragma unroll
            for (int j = 0; j < BLOCK_N / 64; ++j)
              tma_load_2d(sb + j * (64 * BLOCK_K * 2), &map_b, &full_bar[stage], n0 + 64 * j, kb * BLOCK_K);
          } else {
            tma_load_2d(sb, &map_b, &full_bar[stage], kb * BLOCK_K, n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BLOCK_M, BLOCK_N, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int ks = t % g.split_k;
        const int kb0 = ks * kb_per_split;
        const int kb1 = min(g.kb_total, kb0 + kb_per_split);
        mbar_wait_relaxed(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BLOCK_N);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + stage * Cfg::A_BYTES);
          const uint32_t b_addr = smem_u32(smem_b + stage * Cfg::B_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // K-major: advance 16 elements = 32 B inside the 128 B swizzle row.
            // MN-major: advance 16 k-rows = two 8-row groups = 2048 B.
            const uint64_t a_desc = A_MN ? make_smem_desc(a_addr + k * 2048, 64 * BLOCK_K * 2, 1024)
                                         : make_smem_desc(a_addr + k * 32, 16, 1024);
            const uint64_t b_desc = B_MN ? make_smem_desc(b_addr + k * 2048, 64 * BLOCK_K * 2, 1024)
                                         : make_smem_desc(b_addr + k * 32, 16, 1024);
            umma_bf16(d_tmem, a_desc, b_desc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[as]);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3;          // TMEM lane quadrant this warp may access
    const int ew = warp - 2;         // 0..7
    const int c_begin = (ew >> 2) * (BLOCK_N / (2 * EPI_COLS));  // first 32-column block of this warp's column half
    constexpr int C_PER_WARP = BLOCK_N / (2 * EPI_COLS);
    float* stage = epi_stage + ew * EPI_WARP_FLOATS;
    int as = 0;
    uint32_t aphase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int rest = t / g.split_k;
      const int m0 = (rest % g.num_m_tiles) * BLOCK_M;
      const int n0 = (rest / g.num_m_tiles) * BLOCK_N;
      const int ks = t % g.split_k;
      const int kb0 = ks * kb_per_split;
      const int kb1 = min(g.kb_total, kb0 + kb_per_split);
      mbar_wait_relaxed(&tmem_full[as], aphase);
      tc_fence_after();
      const int row_base = m0 + q * 32;
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BLOCK_N);
      const bool has_work = kb1 > kb0 && row_base < g.M;  // empty split slices contribute nothing
#pragma unroll 1
      for (int c = c_begin; c < c_begin + C_PER_WARP; ++c) {
        const int n = n0 + c * EPI_COLS;
        if (n >= g.N) break;
        const uint32_t taddr = t_base + c * EPI_COLS;
        if (g.epi_mode == 0) epilogue_one<0>(g, stage, taddr, row_base, n, lane, has_work);
        else if (g.epi_mode == 1) epilogue_one<1>(g, stage, taddr, row_base, n, lane, has_work);
        else epilogue_one<2>(g, stage, taddr, row_base, n, lane, has_work);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ================================================================================================ CTA-pair GEMM
// Same pipeline with tcgen05 cta_group::2: a cluster of two CTAs (one TPC) computes one 256 x 256 tile.  Each CTA stages
// its own 128 rows of A and HALF of the B tile (128 of the 256 N rows), the leader's single thread issues M=256 MMAs that
// read both halves, and each CTA's TMEM receives its 128 x 256 accumulator.  Per CTA a k-block costs 32 KB of L2->SM
// traffic instead of 48 KB: the single-CTA kernel is capped by exactly that ingest rate (~47 B/clk/SM measured, tensor pipe
// 49 % busy), which is where cuBLAS's 1.5 PF on these shapes comes from.
constexpr int PAIR_STAGE_BYTES = 2 * 16384;  // A 128 x 64 + B 128 x 64 (bf16)
// Shared-memory plan of every variant: 5 operand stages + 64 KB of epilogue staging.  EPI = 0: bf16 TMA staging
// tiles (the fp32 transposition blocks of the generic mode 2 alias them).  EPI = 1 (fp32 residual in / fp32 out, see
// the f32 TMA epilogue below): a ring of two 4 KB fp32 tiles per epilogue warp.  (A three-tile ring with 4 operand stages
// was measured first: the K = 3072 GEMMs lost in the main loop what the epilogue gained.)
constexpr int F32_EPI_TILE_BYTES = 32 * 32 * 4;
// (Round 2: a four-tile ring with three operand stages for the short-K projections — two residual blocks in flight, no
// wait on the newest store — measured 54.1 us against 53.5 us for the 18912 x 768 x 768 projection, i.e. the residual
// latency is not what bounds this epilogue; removed again.  What did cost time: the per-lane row stores of the saved
// pre-scale value, see below.)
template <int EPI>   // 0: classic / bf16 TMA-store epilogues, 1: f32 TMA epilogue, 2: dGELU (bf16 in / bf16 out) TMA epilogue
struct PairCfg {
  static constexpr int STAGES = 5;
  static constexpr int RING = 2;
  static constexpr int EPI_BYTES = 8 * TMA_EPI_WARP_BYTES;   // >= the two-tile rings of the EPI = 1 / 2 variants
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM_BYTES = STAGES * PAIR_STAGE_BYTES + EPI_BYTES + BAR_BYTES;
  static_assert(EPI_BYTES >= 8 * 32 * 34 * 4 && EPI_BYTES >= 8 * RING * F32_EPI_TILE_BYTES, "staging must fit");
  static_assert((2 * STAGES + 5 + 8 * RING) * 8 <= BAR_BYTES, "barriers must fit");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
};

// Swizzle-128B position of 16-byte chunk `k` of row `r` in a TMA tile with 128-byte rows (tile base 1024-aligned), and the
// Swizzle-64B one for 64-byte rows (tile base 512-aligned).
XFM_DEVINL uint32_t swz128(int r, int k) { return (uint32_t)(r * 128 + ((k ^ (r & 7)) << 4)); }
XFM_DEVINL uint32_t swz64(int r, int k) { return (uint32_t)(r * 64 + ((k ^ ((r >> 1) & 3)) << 4)); }

template <int A_MN, int B_MN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                         const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_aux, const GemmArgs g) {
  using PC = PairCfg<EPI>;
  constexpr bool DG_EPI = EPI == 2;    // dGELU: bf16 pre-activation in / bf16 out (EPI == 1: f32 residual in / f32 out)
  constexpr int RING_TILE_BYTES = DG_EPI ? 32 * 32 * 2 : F32_EPI_TILE_BYTES;
  constexpr int STAGES = PC::STAGES;
  constexpr int F32_EPI_RING = PC::RING;
  constexpr int BLOCK_N = 256;
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023) __trap();
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * 16384;
  float* epi_stage = (float*)(smem + STAGES * PAIR_STAGE_BYTES);
  uint64_t* bars = (uint64_t*)(smem + STAGES * PAIR_STAGE_BYTES + PC::EPI_BYTES);
  uint64_t* full_bar = bars;                    // [STAGES]  used in the leader CTA only
  uint64_t* empty_bar = bars + STAGES;          // [STAGES]  one per CTA, arrived by the leader's multicast commit
  uint64_t* tmem_full = bars + 2 * STAGES;      // [2]       one per CTA, multicast commit
  uint64_t* tmem_empty = bars + 2 * STAGES + 2; // [2]       leader's copy: 2 x EPI_WARPS arrivals (peer arrives remotely)
  uint32_t* tmem_ptr = (uint32_t*)(bars + 2 * STAGES + 4);
  uint64_t* res_bar = bars + 2 * STAGES + 5;    // [EPI_WARPS][F32_EPI_RING]  residual tiles of the f32 TMA epilogue

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();     // 0 = leader
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 2 * EPI_WARPS);
    }
    if (EPI != 0) {
      tma_prefetch_desc(&map_c);
      tma_prefetch_desc(&map_aux);
      for (int s = 0; s < EPI_WARPS * F32_EPI_RING; ++s) mbar_init(&res_bar[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_2sm(tmem_ptr, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int num_m_pairs = (g.num_m_tiles + 1) / 2;
  const int num_tiles = num_m_pairs * g.num_n_tiles * g.split_k;
  const int kb_per_split = (g.kb_total + g.split_k - 1) / g.split_k;
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair_id; t < num_tiles; t += num_pairs) {
        const int ks = t % g.split_k;
        const int rest = t / g.split_k;
        const int mt = g.n_fastest ? rest / g.num_n_tiles : rest % num_m_pairs;
        const int nt = g.n_fastest ? rest % g.num_n_tiles : rest / num_m_pairs;
        const int m0 = (mt * 2 + (int)rank) * BLOCK_M;      // this CTA's 128 rows of the 256-row tile
        const int n0 = nt * BLOCK_N + (int)rank * 128;      // this CTA's half of the tile's N range
        const int kb0 = ks * kb_per_split;
        const int kb1 = min(g.kb_total, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_relaxed(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * PAIR_STAGE_BYTES);  // both CTAs' boxes land on this barrier
          uint8_t* sa = smem_a + stage * 16384;
          uint8_t* sb = smem_b + stage * 16384;
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < 2; ++j) tma_load_2d_2sm(sa + j * 8192, &map_a, &full_bar[stage], m0 + 64 * j, kb * BLOCK_K);
          } else {
            tma_load_2d_2sm(sa, &map_a, &full_bar[stage], kb * BLOCK_K, m0);
          }
          if (B_MN) {
#pragma unroll
            for (int j = 0; j < 2; ++j) tma_load_2d_2sm(sb + j * 8192, &map_b, &full_bar[stage], n0 + 64 * j, kb * BLOCK_K);
          } else {
            tma_load_2d_2sm(sb, &map_b, &full_bar[stage], kb * BLOCK_K, n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(256, BLOCK_N, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int t = pair_id; t < num_tiles; t += num_pairs) {
        const int ks = t % g.split_k;
        const int kb0 = ks * kb_per_split;
        const int kb1 = min(g.kb_total, kb0 + kb_per_split);
        mbar_wait_relaxed(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BLOCK_N);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + stage * 16384);
          const uint32_t b_addr = smem_u32(smem_b + stage * 16384);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t a_desc = A_MN ? make_smem_desc(a_addr + k * 2048, 64 * BLOCK_K * 2, 1024)
                                         : make_smem_desc(a_addr + k * 32, 16, 1024);
            const uint64_t b_desc = B_MN ? make_smem_desc(b_addr + k * 2048, 64 * BLOCK_K * 2, 1024)
                                         : make_smem_desc(b_addr + k * 32, 16, 1024);
            umma_bf16_2sm(d_tmem, a_desc, b_desc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit_2sm(&empty_bar[stage], 3);   // frees this stage in both CTAs
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[as], 3);        // accumulator ready in both CTAs
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
    __syncwarp();
  } else if (EPI != 0) {
    // ---- f32 TMA epilogue: C(f32) = dropout((acc + bias) * col_scale * row_group_scale) + residual(f32).
    // ---- dGELU TMA epilogue (EPI = 2): C(bf16) = (acc + bias) * gelu'(aux_in(bf16)); same ring with 2 KB SWIZZLE_64B tiles
    //      (the operand used to be fetched with lane = row 16-byte global loads: 32 L1 wavefronts per instruction).
    // The generic mode-2 path moves the residual and the output through a transposition block with 16 row steps of
    // dependent global accesses per 32 x 32 block and is latency bound (65 us for the 18912 x 768 x 768 ViT projection,
    // whose operands + residual + output take 22 us of HBM time).  Here every epilogue warp owns a ring of two
    // swizzled 4 KB tiles: the TMA engine prefetches the residual block one block ahead, the lane (= accumulator row)
    // reads its 128-byte row conflict-free, combines it with the accumulator in registers, writes the result IN PLACE and
    // one thread hands the tile back to the TMA engine for the store (edges are clipped / zero-filled by the tensor maps).
    const int q = warp & 3;
    const int ew = warp - 2;
    constexpr int C_PER_WARP = BLOCK_N / (2 * EPI_COLS);
    // The two warps of a TMEM lane quadrant take ALTERNATE 32-column blocks (c = half, half + 2, ...), so the pair
    // works on adjacent 128-byte row segments at the same time (256 contiguous bytes per row reach DRAM together).
    const int c_begin = g.epi_interleave ? (ew >> 2) : (ew >> 2) * C_PER_WARP;
    const int c_step = g.epi_interleave ? 2 : 1;
    const int c_end = c_begin + c_step * C_PER_WARP;
    uint8_t* ring = (uint8_t*)epi_stage + ew * F32_EPI_RING * RING_TILE_BYTES;
    uint64_t* rbar = res_bar + ew * F32_EPI_RING;
    const bool want_res = DG_EPI ? true : g.residual != nullptr;
    const bool has_scale = g.col_scale != nullptr || g.row_group_scale != nullptr;
    const bool has_drop = g.dropout_p > 0.f;
    const float inv_keep = has_drop ? 1.0f / (1.0f - g.dropout_p) : 1.0f;
    const uint32_t seed_mix = drop_seed_mix(g.dropout_seed + *g.seed_salt), thr = drop_threshold(g.dropout_p);
    // block sequence of this warp: tiles t = pair_id, pair_id + num_pairs, ...; blocks c_begin .. c_end-1 while inside N
    auto block_at = [&](int t, int c, int& rb, int& n) -> bool {
      if (t >= num_tiles) return false;
      const int mt = g.n_fastest ? t / g.num_n_tiles : t % num_m_pairs;
      const int nt = g.n_fastest ? t % g.num_n_tiles : t / num_m_pairs;
      rb = (mt * 2 + (int)rank) * BLOCK_M + q * 32;
      n = nt * BLOCK_N + c * EPI_COLS;
      return n < g.N;
    };
    int pf_t = pair_id, pf_c = c_begin, pf_k = 0;   // prefetch cursor (lane 0): next residual block to request
    auto prefetch = [&]() {
      int rb, n;
      if (!block_at(pf_t, pf_c, rb, n)) return;
      const int slot = pf_k % F32_EPI_RING;
      mbar_arrive_expect_tx(&rbar[slot], RING_TILE_BYTES);
      tma_load_2d(ring + slot * RING_TILE_BYTES, &map_aux, &rbar[slot], n, rb);
      ++pf_k;
      pf_c += c_step;
      if (pf_c >= c_end || !block_at(pf_t, pf_c, rb, n)) { pf_t += num_pairs; pf_c = c_begin; }
    };
    // residual blocks requested ahead of the one being combined: 1 with the two-tile ring, 2 with the four-tile ring
    constexpr int PF_AHEAD = F32_EPI_RING == 2 ? 1 : F32_EPI_RING - 2;
    if (want_res && lane == 0) {
#pragma unroll
      for (int k = 0; k < PF_AHEAD; ++k) prefetch();
    }
    int blk = 0;   // blocks consumed so far
    int as = 0;
    uint32_t aphase = 0;
    for (int t = pair_id; t < num_tiles; t += num_pairs) {
      mbar_wait_relaxed(&tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BLOCK_N);
#pragma unroll 1
      for (int c = c_begin; c < c_end; c += c_step) {
        int row_base, n;
        if (!block_at(t, c, row_base, n)) break;
        const int slot = blk % F32_EPI_RING;
        uint8_t* tile = ring + slot * RING_TILE_BYTES;
        uint32_t r[32];
        tmem_ld_32x32(t_base + c * EPI_COLS, r);
        float4 res[DG_EPI ? 4 : 8];   // f32: the residual row; dGELU: the bf16 pre-activation row (4 x 8 values)
        if (want_res) {
          mbar_wait(&rbar[slot], (uint32_t)(blk / F32_EPI_RING) & 1u);
          if (DG_EPI) {
#pragma unroll
            for (int k = 0; k < 4; ++k) res[k] = *(const float4*)(tile + swz64(lane, k));
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) res[k] = *(const float4*)(tile + swz128(lane, k));
          }
          if (lane == 0) {
            // the tile of block blk + PF_AHEAD was last read by the store of block blk + PF_AHEAD - RING: with two tiles
            // that is the newest store (wait for all), with four the one before it (the newest may still be reading)
            tma_store_wait_read<F32_EPI_RING - PF_AHEAD - 1>();
            prefetch();
          }
        }
        const int row = row_base + lane;
        float rs = 1.f;
        if (g.row_group_scale) rs = __ldg(g.row_group_scale + min(row, g.M - 1) / g.rows_per_group);
        float4 b4[8];   // requested before the TMEM wait so the latencies overlap
#pragma unroll
        for (int k = 0; k < 8; ++k) b4[k] = g.bias ? __ldg((const float4*)(g.bias + n) + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 cs4[DG_EPI ? 1 : 8];   // LayerScale gamma of the block's columns, likewise
        if (!DG_EPI && g.col_scale) {
#pragma unroll
          for (int k = 0; k < 8; ++k) cs4[k] = __ldg((const float4*)(g.col_scale + n) + k);
        }
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          v[4 * k] = __uint_as_float(r[4 * k]) + b4[k].x;
          v[4 * k + 1] = __uint_as_float(r[4 * k + 1]) + b4[k].y;
          v[4 * k + 2] = __uint_as_float(r[4 * k + 2]) + b4[k].z;
          v[4 * k + 3] = __uint_as_float(r[4 * k + 3]) + b4[k].w;
        }
        if (DG_EPI) {
          const __nv_bfloat162* a2 = (const __nv_bfloat162*)res;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float2 af = __bfloat1622float2(a2[j]);
            const float2 dg = gelu_grad_fast2(af.x, af.y);
            v[2 * j] *= dg.x;
            v[2 * j + 1] *= dg.y;
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {   // in place: the bf16 result replaces the pre-activation row this lane read
            uint4 u;
            __nv_bfloat162 t0 = __floats2bfloat162_rn(v[8 * k], v[8 * k + 1]), t1 = __floats2bfloat162_rn(v[8 * k + 2], v[8 * k + 3]);
            __nv_bfloat162 t2 = __floats2bfloat162_rn(v[8 * k + 4], v[8 * k + 5]), t3 = __floats2bfloat162_rn(v[8 * k + 6], v[8 * k + 7]);
            u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
            *(uint4*)(tile + swz64(lane, k)) = u;
          }
        } else {
        if (g.aux_out) {
          // saved pre-scale value z = acc + bias (bf16; LayerScale backward needs it).  Each lane holds the 64 bytes of
          // ITS row: storing them from there costs 32 L1 wavefronts per instruction (32 rows), 128 per block — 8 us of the
          // 50 us projection GEMM.  The block's tile is free between the residual read and the output write, so the rows
          // are transposed through it (SWIZZLE_64B positions, conflict free both ways): four lanes then store one row's
          // 64 bytes, 8 rows per instruction.
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint4 u;
            __nv_bfloat162 t0 = __floats2bfloat162_rn(v[8 * k], v[8 * k + 1]), t1 = __floats2bfloat162_rn(v[8 * k + 2], v[8 * k + 3]);
            __nv_bfloat162 t2 = __floats2bfloat162_rn(v[8 * k + 4], v[8 * k + 5]), t3 = __floats2bfloat162_rn(v[8 * k + 6], v[8 * k + 7]);
            u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
            *(uint4*)(tile + swz64(lane, k)) = u;
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int r = 8 * j + (lane >> 2), kk = lane & 3;
            const uint4 u = *(const uint4*)(tile + swz64(r, kk));
            if (row_base + r < g.M) *(uint4*)(g.aux_out + (int64_t)(row_base + r) * g.ld_aux_out + n + 8 * kk) = u;
          }
          __syncwarp();   // the output rows overwrite the tile next
        }
        if (has_scale) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float4 c4 = make_float4(1.f, 1.f, 1.f, 1.f);
            if (g.col_scale) c4 = cs4[k];
            v[4 * k] *= c4.x * rs;
            v[4 * k + 1] *= c4.y * rs;
            v[4 * k + 2] *= c4.z * rs;
            v[4 * k + 3] *= c4.w * rs;
          }
        }
        if (has_drop) {
          const uint64_t pair0 = ((uint64_t)row * (uint64_t)g.N + (uint64_t)n) >> 1;   // N and n are even
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const uint64_t pr = pair0 + j;
            const uint32_t keep = drop_keep_pair(seed_mix, (uint32_t)pr, (uint32_t)(pr >> 32), thr);
            v[2 * j] = (keep & 1u) ? v[2 * j] * inv_keep : 0.f;
            v[2 * j + 1] = (keep & 2u) ? v[2 * j + 1] * inv_keep : 0.f;
          }
        }
        if (want_res) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            v[4 * k] += res[k].x;
            v[4 * k + 1] += res[k].y;
            v[4 * k + 2] += res[k].z;
            v[4 * k + 3] += res[k].w;
          }
        }
        // in place: this lane overwrites exactly the chunks it read; without a residual the tile was last read by the
        // store of block blk - 2, which the wait_read<1> at the end of block blk - 1 has retired
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *(float4*)(tile + swz128(lane, k)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
        }   // !DG_EPI
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&map_c, tile, n, row_base);
          tma_store_commit();
          if (!want_res) tma_store_wait_read<1>();
        }
        __syncwarp();
        ++blk;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tmem_empty[as]);
        else mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty[as]), 0));
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) tma_store_wait_read<0>();   // shared memory must outlive the last copies
  } else {
    const int q = warp & 3;
    const int ew = warp - 2;
    constexpr int C_PER_WARP = BLOCK_N / (2 * EPI_COLS);
    const int c_begin = (ew >> 2) * C_PER_WARP;
    float* stage = epi_stage + ew * EPI_WARP_FLOATS;
    uint8_t* tma_tiles = (uint8_t*)epi_stage + ew * TMA_EPI_WARP_BYTES;
    int tma_slot = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int t = pair_id; t < num_tiles; t += num_pairs) {
      const int rest = t / g.split_k;
      const int mt = g.n_fastest ? rest / g.num_n_tiles : rest % num_m_pairs;
      const int nt = g.n_fastest ? rest % g.num_n_tiles : rest / num_m_pairs;
      const int m0 = (mt * 2 + (int)rank) * BLOCK_M;
      const int n0 = nt * BLOCK_N;
      const int ks = t % g.split_k;
      const int kb0 = ks * kb_per_split;
      const int kb1 = min(g.kb_total, kb0 + kb_per_split);
      mbar_wait_relaxed(&tmem_full[as], aphase);
      tc_fence_after();
      const int row_base = m0 + q * 32;
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BLOCK_N);
      const bool has_work = kb1 > kb0 && row_base < g.M;
#pragma unroll 1
      for (int c = c_begin; c < c_begin + C_PER_WARP; ++c) {
        const int n = n0 + c * EPI_COLS;
        if (n >= g.N) break;
        const uint32_t taddr = t_base + c * EPI_COLS;
        if (g.tma_epi) {
          if (g.epi_mode == 0) epilogue_tma_block<0>(g, &map_c, &map_aux, tma_tiles, tma_slot, taddr, row_base, n, lane, has_work);
          else epilogue_tma_block<1>(g, &map_c, &map_aux, tma_tiles, tma_slot, taddr, row_base, n, lane, has_work);
        } else if (g.epi_mode == 0) epilogue_one<0>(g, stage, taddr, row_base, n, lane, has_work);
        else if (g.epi_mode == 1) epilogue_one<1>(g, stage, taddr, row_base, n, lane, has_work);
        else epilogue_one<2>(g, stage, taddr, row_base, n, lane, has_work);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tmem_empty[as]);
        else mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty[as]), 0));
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (g.tma_epi && lane == 0) tma_store_wait_read<0>();   // shared memory must outlive the last copies
  }

  tc_fence_before();
  cluster_sync_all();   // neither CTA may exit (or free TMEM) while the other can still signal it or read its operands
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------ host
static int encode_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                     uint32_t box_inner, uint32_t box_outer) {
  auto fn = get_tensor_map_encoder();
  if (!fn) return XFM_ERR_NO_DRIVER;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: %d (inner=%llu outer=%llu ld=%llu box=%u,%u base=%p)", (int)r,
              (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld_elems, box_inner, box_outer,
              base);
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

// bf16 [outer, inner] tile map, SWIZZLE_64B (TMA-store epilogue: 64-byte rows in shared memory, see st_row_bf16x32)
static int encode_2d_plain(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                           uint32_t box_inner, uint32_t box_outer) {
  auto fn = get_tensor_map_encoder();
  if (!fn) return XFM_ERR_NO_DRIVER;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (output) failed: %d (inner=%llu outer=%llu ld=%llu base=%p)", (int)r,
              (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld_elems, base);
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

// f32 [outer, inner] tile map, 32 x 32 boxes with 128-byte rows, SWIZZLE_128B (f32 TMA epilogue: residual in, C out)
static int encode_2d_f32(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems) {
  auto fn = get_tensor_map_encoder();
  if (!fn) return XFM_ERR_NO_DRIVER;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (f32 epilogue) failed: %d (inner=%llu outer=%llu ld=%llu base=%p)", (int)r,
              (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld_elems, base);
    return XFM_ERR_BAD_ARG;
  }
  return 0;
}

template <int BLOCK_N, int A_MN, int B_MN>
static int launch_gemm(const xfm_gemm_params* p, const GemmArgs& g, cudaStream_t stream) {
  using Cfg = GemmCfg<BLOCK_N>;
  CUtensorMap map_a, map_b;
  int rc;
  if (A_MN) rc = encode_2d(&map_a, p->A, p->M, p->K, p->lda, 64, BLOCK_K);
  else rc = encode_2d(&map_a, p->A, p->K, p->M, p->lda, BLOCK_K, BLOCK_M);
  if (rc) return rc;
  if (B_MN) rc = encode_2d(&map_b, p->B, p->N, p->K, p->ldb, 64, BLOCK_K);
  else rc = encode_2d(&map_b, p->B, p->K, p->N, p->ldb, BLOCK_K, BLOCK_N);
  if (rc) return rc;
  auto kern = gemm_tcgen05_kernel<BLOCK_N, A_MN, B_MN>;
  static bool attr_set = false;  // per instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const int num_tiles = g.num_m_tiles * g.num_n_tiles * g.split_k;
  const int grid = num_tiles < num_sms() ? num_tiles : num_sms();
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(map_a, map_b, g);
  count_launch();
  return (int)cudaGetLastError();
}

template <int A_MN, int B_MN>
static int launch_gemm_pair(const xfm_gemm_params* p, const GemmArgs& g, cudaStream_t stream) {
  CUtensorMap map_a, map_b;
  int rc;
  if (A_MN) rc = encode_2d(&map_a, p->A, p->M, p->K, p->lda, 64, BLOCK_K);
  else rc = encode_2d(&map_a, p->A, p->K, p->M, p->lda, BLOCK_K, BLOCK_M);
  if (rc) return rc;
  if (B_MN) rc = encode_2d(&map_b, p->B, p->N, p->K, p->ldb, 64, BLOCK_K);
  else rc = encode_2d(&map_b, p->B, p->K, p->N, p->ldb, BLOCK_K, 128);   // half of the 256-wide tile per CTA
  if (rc) return rc;
  const int num_tiles = ((g.num_m_tiles + 1) / 2) * g.num_n_tiles * g.split_k;
  const int max_pairs = num_sms() / 2;
  const int pairs = num_tiles < max_pairs ? num_tiles : max_pairs;
  CUtensorMap map_c = map_a, map_aux = map_a;   // placeholders when the TMA-store epilogue is not used
  GemmArgs g2 = g;
  g2.tma_epi = 0;
  // Tile order.  M-fastest (default) keeps a B tile hot while the grid sweeps M; each wave then touches ALL of A, so an A
  // larger than L2 is re-read from HBM once per N tile (ncu: 407 MB read for the 18912 x 768 x 3072 fc2 GEMM whose
  // operands + residual are 174 MB).  N-fastest runs the N tiles of an M tile side by side instead.
  static const int raster_env = getenv("XFM_GEMM_RASTER") ? atoi(getenv("XFM_GEMM_RASTER")) : -1;
  const int64_t a_bytes = (int64_t)p->M * p->K * 2, b_bytes = (int64_t)p->N * p->K * 2;
  g2.n_fastest = (g.split_k == 1 && g.num_n_tiles > 1 && a_bytes > (40ll << 20) && b_bytes <= (16ll << 20)) ? 1 : 0;
  if (raster_env >= 0) g2.n_fastest = (raster_env != 0 && g.split_k == 1) ? 1 : 0;
  static const int il_env = getenv("XFM_GEMM_EPI_INTERLEAVE") ? atoi(getenv("XFM_GEMM_EPI_INTERLEAVE")) : 1;
  g2.epi_interleave = il_env;
  auto a16 = [](const void* q) { return ((uintptr_t)q & 15) == 0; };
  static const bool f32_epi_on = getenv("XFM_GEMM_F32_EPI") == nullptr || atoi(getenv("XFM_GEMM_F32_EPI")) != 0;
  static const bool dg_epi_on = getenv("XFM_GEMM_DG_EPI") == nullptr || atoi(getenv("XFM_GEMM_DG_EPI")) != 0;
  if (f32_epi_on && g.epi_mode == 2 && p->c_dtype == 1 && !p->accumulate && g.split_k == 1 && p->act == 0 &&
      (!p->aux_out || (a16(p->aux_out) && (p->ld_aux_out & 7) == 0)) && (p->N % 32) == 0 && a16(p->C) && (p->ldc & 3) == 0 &&
      (!p->residual || (p->res_dtype == 1 && a16(p->residual) && (p->ld_res & 3) == 0)) && (!p->bias || a16(p->bias)) &&
      (!p->col_scale || a16(p->col_scale))) {
    // f32 TMA epilogue variant (residual / output tiles through the TMA engine)
    rc = encode_2d_f32(&map_c, p->C, p->N, p->M, p->ldc);
    if (!rc && p->residual) rc = encode_2d_f32(&map_aux, p->residual, p->N, p->M, p->ld_res);
    if (rc) return rc;
    g2.tma_epi = 2;
    // the fp32 residual / output rows of an M tile are touched by all its N tiles at once: fuller DRAM pages
    // (18912 x 768 x 768 with residual: 39.5 -> 37.4 us)
    if (raster_env < 0 && g.split_k == 1 && g.num_n_tiles > 1 && b_bytes <= (16ll << 20)) g2.n_fastest = 1;
    auto kern32 = gemm_tcgen05_pair_kernel<A_MN, B_MN, 1>;
    static bool attr32_set = false;
    if (!attr32_set) {
      cudaError_t e = cudaFuncSetAttribute(kern32, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<1>::SMEM_BYTES);
      if (e != cudaSuccess) return (int)e;
      attr32_set = true;
    }
    kern32<<<2 * pairs, GEMM_THREADS, PairCfg<1>::SMEM_BYTES, stream>>>(map_a, map_b, map_c, map_aux, g2);
    count_launch();
    return (int)cudaGetLastError();
  }
  if (dg_epi_on && g.epi_mode == 1 && p->c_dtype == 0 && g.split_k == 1 && (p->N % 32) == 0 && a16(p->C) && (p->ldc & 7) == 0 &&
      p->aux_in && a16(p->aux_in) && (p->ld_aux_in & 7) == 0 && (!p->bias || a16(p->bias))) {
    // dGELU TMA epilogue variant (pre-activation tiles in, bf16 result out through the TMA engine)
    rc = encode_2d_plain(&map_c, p->C, p->N, p->M, p->ldc, 32, 32);
    if (!rc) rc = encode_2d_plain(&map_aux, p->aux_in, p->N, p->M, p->ld_aux_in, 32, 32);
    if (rc) return rc;
    g2.tma_epi = 3;
    auto kern_dg = gemm_tcgen05_pair_kernel<A_MN, B_MN, 2>;
    static bool attr_dg_set = false;
    if (!attr_dg_set) {
      cudaError_t e = cudaFuncSetAttribute(kern_dg, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<2>::SMEM_BYTES);
      if (e != cudaSuccess) return (int)e;
      attr_dg_set = true;
    }
    kern_dg<<<2 * pairs, GEMM_THREADS, PairCfg<2>::SMEM_BYTES, stream>>>(map_a, map_b, map_c, map_aux, g2);
    count_launch();
    return (int)cudaGetLastError();
  }
  auto kern = gemm_tcgen05_pair_kernel<A_MN, B_MN, 0>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<0>::SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  if ((g.epi_mode == 0 || g.epi_mode == 1) && g.split_k == 1 && ((uintptr_t)p->C & 15) == 0 && (p->ldc & 7) == 0 &&
      (!p->aux_out || (((uintptr_t)p->aux_out & 15) == 0 && (p->ld_aux_out & 7) == 0)) &&
      (!p->aux_in || (((uintptr_t)p->aux_in & 15) == 0 && (p->ld_aux_in & 7) == 0)) &&
      (!p->bias || ((uintptr_t)p->bias & 15) == 0)) {
    rc = encode_2d_plain(&map_c, p->C, p->N, p->M, p->ldc, 32, 32);
    if (!rc && g.epi_mode == 0 && p->aux_out) rc = encode_2d_plain(&map_aux, p->aux_out, p->N, p->M, p->ld_aux_out, 32, 32);
    if (rc) return rc;
    g2.tma_epi = 1;
  }
  kern<<<2 * pairs, GEMM_THREADS, PairCfg<0>::SMEM_BYTES, stream>>>(map_a, map_b, map_c, map_aux, g2);
  count_launch();
  return (int)cudaGetLastError();
}

static int dispatch_pair(const xfm_gemm_params* p, const GemmArgs& g, cudaStream_t s) {
  if (p->a_mn_major) {
    if (p->b_mn_major) return launch_gemm_pair<1, 1>(p, g, s);
    return launch_gemm_pair<1, 0>(p, g, s);
  }
  if (p->b_mn_major) return launch_gemm_pair<0, 1>(p, g, s);
  return launch_gemm_pair<0, 0>(p, g, s);
}

template <int BLOCK_N>
static int dispatch_major(const xfm_gemm_params* p, const GemmArgs& g, cudaStream_t s) {
  if (p->a_mn_major) {
    if (p->b_mn_major) return launch_gemm<BLOCK_N, 1, 1>(p, g, s);
    return launch_gemm<BLOCK_N, 1, 0>(p, g, s);
  }
  if (p->b_mn_major) return launch_gemm<BLOCK_N, 0, 1>(p, g, s);
  return launch_gemm<BLOCK_N, 0, 0>(p, g, s);
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

int gemm_bf16(const xfm_gemm_params* p, cudaStream_t stream) {
  if (!p || !p->A || !p->B || !p->C || p->M <= 0 || p->N <= 0 || p->K <= 0) {
    set_error("gemm: null pointer or non-positive shape");
    return XFM_ERR_BAD_ARG;
  }
  if ((p->lda & 7) || (p->ldb & 7) || !aligned16(p->A) || !aligned16(p->B)) {
    set_error("gemm: operands need 16-byte aligned bases and leading dimensions that are multiples of 8");
    return XFM_ERR_BAD_ARG;
  }
  const int split_k = p->split_k < 1 ? 1 : p->split_k;
  if ((split_k > 1 || p->accumulate) && p->c_dtype != 1) {
    set_error("gemm: split_k / accumulate need an f32 output");
    return XFM_ERR_BAD_ARG;
  }
  if (split_k > 1 && !p->accumulate) {
    set_error("gemm: split_k > 1 needs accumulate = 1 (caller zeroes or owns C)");
    return XFM_ERR_BAD_ARG;
  }
  // Every K slice runs the whole epilogue on its partial sum.  Only the steps linear in the accumulator with the same
  // factor in every slice (col_scale, row_group_scale, dropout) distribute over the slices; bias, residual, aux_out and
  // the activations would be applied once per slice.
  if (split_k > 1 && (p->bias || p->residual || p->aux_out || p->act != 0)) {
    set_error("gemm: split_k > 1 allows no bias, residual, aux_out or act (each K slice applies the epilogue)");
    return XFM_ERR_BAD_ARG;
  }
  if (p->act == 2 && !p->aux_in) {
    set_error("gemm: act=2 (dgelu) needs aux_in");
    return XFM_ERR_BAD_ARG;
  }
  int bn = p->block_n == 512 ? 256 : p->block_n;
  if (bn == 0) {
    // Largest tile that still yields >= ~1 wave of CTAs; small problems fall to narrower tiles.
    const int mt = (p->M + BLOCK_M - 1) / BLOCK_M;
    bn = 256;
    while (bn > 64 && (int64_t)mt * ((p->N + bn - 1) / bn) * split_k < num_sms()) bn >>= 1;
    if (p->N <= 64) bn = 64;
    else if (p->N <= 128 && bn > 128) bn = 128;
  }
  GemmArgs g;
  g.tma_epi = 0; g.n_fastest = 0; g.epi_interleave = 0;
  g.M = p->M; g.N = p->N; g.K = p->K;
  g.num_m_tiles = (p->M + BLOCK_M - 1) / BLOCK_M;
  g.num_n_tiles = (p->N + bn - 1) / bn;
  g.kb_total = (p->K + BLOCK_K - 1) / BLOCK_K;
  g.split_k = split_k > g.kb_total ? g.kb_total : split_k;
  g.c_dtype = p->c_dtype; g.accumulate = p->accumulate; g.act = p->act; g.res_dtype = p->res_dtype;
  g.rows_per_group = p->rows_per_group > 0 ? p->rows_per_group : 1;
  g.ldc = p->ldc; g.ld_aux_in = p->ld_aux_in; g.ld_aux_out = p->ld_aux_out; g.ld_res = p->ld_res;
  g.C = p->C; g.bias = p->bias; g.aux_in = (const bf16*)p->aux_in; g.aux_out = (bf16*)p->aux_out;
  g.col_scale = p->col_scale; g.row_group_scale = p->row_group_scale; g.residual = p->residual;
  g.dropout_p = p->dropout_p; g.dropout_seed = p->dropout_seed; g.seed_salt = seed_salt_ptr();
  auto al = [](const void* q, size_t bytes) { return ((uintptr_t)q & (bytes - 1)) == 0; };
  bool vec = al(p->C, p->c_dtype == 0 ? 4 : 8) && (p->ldc & 1) == 0;
  if (p->aux_in) vec = vec && al(p->aux_in, 4) && (p->ld_aux_in & 1) == 0;
  if (p->aux_out) vec = vec && al(p->aux_out, 4) && (p->ld_aux_out & 1) == 0;
  if (p->residual) vec = vec && al(p->residual, p->res_dtype == 0 ? 4 : 8) && (p->ld_res & 1) == 0;
  const bool plain = p->c_dtype == 0 && !p->col_scale && !p->row_group_scale && !p->residual && !(p->dropout_p > 0.f);
  g.epi_mode = (plain && p->act <= 1) ? 0 : ((plain && p->act == 2 && !p->aux_out) ? 1 : 2);
  g.vec_ok = vec ? 1 : 0;
  if (p->block_n == 512) {   // CTA-pair (cta_group::2) kernel: 256 x 256 tiles; num_n_tiles counted in 256-wide tiles
    g.num_n_tiles = (p->N + 255) / 256;
    return dispatch_pair(p, g, stream);
  }
  switch (bn) {
    case 64: return dispatch_major<64>(p, g, stream);
    case 128: return dispatch_major<128>(p, g, stream);
    case 256: return dispatch_major<256>(p, g, stream);
    default: set_error("gemm: block_n must be 0, 64, 128 or 256"); return XFM_ERR_BAD_ARG;
  }
}

}  // namespace xfm
