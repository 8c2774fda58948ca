// xfm_b200 — shared device helpers for sm_100a kernels.
// Raw PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA) and TMEM.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

namespace xfm {

typedef __nv_bfloat16 bf16;

#define XFM_DEVINL __device__ __forceinline__

XFM_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ----------------------------------------------------------------------------- mbarrier
XFM_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
XFM_DEVINL void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
XFM_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

XFM_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
XFM_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
XFM_DEVINL uint32_t mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok;
}
XFM_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  while (!mbar_try_wait(addr, parity)) {
  }
}
// Same, but sleeps between polls: for waits that are long by construction (a producer waiting for a free stage, the MMA
// issuer waiting for the epilogue to drain TMEM) so the polling warp does not steal issue slots from the epilogue
// warps on its scheduler (ncu: 14 % of all issued instructions were SYNCS/YIELD polls).
XFM_DEVINL void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  while (!mbar_try_wait(addr, parity)) __nanosleep(40);
}

// named barrier over a subset of the CTA's warps (id 0 is __syncthreads')
XFM_DEVINL void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ----------------------------------------------------------------------------- TMA
XFM_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// 2D tiled load: coordinates (c0 = inner/contiguous dim, c1 = outer dim)
XFM_DEVINL void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// TMA store (shared -> global, bulk-group completion).  The source tile must be written with generic-proxy stores followed
// by fence.proxy.async before the issuing thread executes the copy; out-of-range rows / columns of the box are clipped.
XFM_DEVINL void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
XFM_DEVINL void tma_reduce_add_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// 3D forms (c0 = contiguous dim, c1 = row inside a sample, c2 = sample): a box that starts inside a sample is clipped at the
// sample's last row, which a flat 2D [rows, cols] map cannot do.
XFM_DEVINL void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// element-wise add of the tile onto global memory (performed at L2; the tensor map's data type selects the arithmetic)
XFM_DEVINL void tma_reduce_add_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
XFM_DEVINL void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
XFM_DEVINL void tma_store_wait_all() {    // at most N of this thread's bulk groups may still be incomplete (writes included)
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
template <int N>
XFM_DEVINL void tma_store_wait_read() {   // at most N of this thread's bulk groups may still be READING shared memory
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
XFM_DEVINL void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
XFM_DEVINL void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
XFM_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
XFM_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
XFM_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16 inputs with fp32 accumulate.
XFM_DEVINL void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
XFM_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets row (lane base + t).
XFM_DEVINL void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
XFM_DEVINL void tmem_ld_32x32_16(uint32_t taddr, uint32_t (&r)[32]) {  // 16 columns into r[0..15]
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
XFM_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// eight fp32 values -> bf16 (round to nearest), one 16-byte store
XFM_DEVINL void st_bf16x8(uint8_t* dst, const float (&p)[8]) {
  uint4 u;
  __nv_bfloat162 t0 = __floats2bfloat162_rn(p[0], p[1]), t1 = __floats2bfloat162_rn(p[2], p[3]);
  __nv_bfloat162 t2 = __floats2bfloat162_rn(p[4], p[5]), t3 = __floats2bfloat162_rn(p[6], p[7]);
  u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
  *(uint4*)dst = u;
}

// Shared-memory matrix descriptor (sm_100 "version 1"), SWIZZLE_128B.
//  K-major  operand: rows of 128 B (64 bf16 along K); 8-row groups 1024 B apart  -> SBO = 1024, LBO unused.
//  MN-major operand: rows of 128 B (64 bf16 along MN), one row per k; 8-k groups 1024 B apart -> SBO = 1024;
//                    64-wide MN blocks LBO bytes apart.
XFM_DEVINL uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
XFM_DEVINL constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                      // c_format = F32
         | (1u << 7)                    // a_format = BF16
         | (1u << 10)                   // b_format = BF16
         | ((uint32_t)a_mn_major << 15) // a_major
         | ((uint32_t)b_mn_major << 16) // b_major
         | ((uint32_t)(N >> 3) << 17)   // n_dim
         | ((uint32_t)(M >> 4) << 24);  // m_dim
}

// ----------------------------------------------------------------------------- CTA pairs (cta_group::2)
XFM_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
XFM_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_addr` (a shared::cta address) in CTA `rank` of this cluster
XFM_DEVINL uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
XFM_DEVINL void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2-SM TMA load: data lands in THIS CTA's shared memory, completion bytes are signalled on the mbarrier at the same
// offset in the pair's leader CTA (address with the peer bit cleared).
XFM_DEVINL void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
XFM_DEVINL void tmem_alloc_2sm(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
XFM_DEVINL void tmem_relinquish_2sm() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
XFM_DEVINL void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem, 256 rows over the CTA pair] (+)= A * B, issued by one thread of the leader CTA; each CTA supplies its 128 rows of A
// and its half of B's N rows from the same shared-memory offsets.
XFM_DEVINL void umma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once all prior MMAs of this thread completed) on the mbarrier at this offset in every CTA of `mask`.
XFM_DEVINL void umma_commit_2sm(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ----------------------------------------------------------------------------- math
XFM_DEVINL float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
XFM_DEVINL float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// GELU(erf) for the GEMM epilogues, where every issue slot counts (a 128 x 256 x 768 tile leaves ~25 slots per element):
// erf by Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7, i.e. fp32 rounding level; measured 4.7e-7 on gelu, 3.0e-7 on
// its derivative over [-12, 12]) = 2 MUFU (ex2, rcp) + ~12 FMA-pipe ops, and the derivative reuses the same exponential.
XFM_DEVINL float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
XFM_DEVINL float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
XFM_DEVINL float erf_core(float x, float& E) {  // returns erf(|x| / sqrt 2); E = exp(-x^2 / 2)
  const float ax = fabsf(x);
  const float t = rcp_approx(fmaf(0.3275911f * 0.70710678118654752440f, ax, 1.0f));
  E = ex2_approx(ax * ax * (-0.5f * 1.4426950408889634f));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(t, p, 1.421413741f);
  p = fmaf(t, p, -0.284496736f);
  p = fmaf(t, p, 0.254829592f);
  p *= t;
  return fmaf(-p, E, 1.0f);
}
XFM_DEVINL float gelu_fast(float x) {
  float E;
  const float er = copysignf(erf_core(x, E), x);
  const float hx = 0.5f * x;
  return fmaf(hx, er, hx);
}
XFM_DEVINL float gelu_grad_fast(float x) {
  float E;
  const float er = copysignf(erf_core(x, E), x);
  return fmaf(0.5f, er, 0.5f) + x * E * 0.39894228040143267794f;
}

// The same two functions on a PAIR of values with Blackwell's packed fp32 pipe (FFMA2 / FMUL2: one issue slot per two
// elements); identical arithmetic per element, so results equal the scalar versions bit for bit.  Used by the dGELU TMA
// epilogue.  Measured: no change in GEMM time (dgelu 114.1 -> 112.8 us, gelu 104 -> 105.7 us where the paired registers
// added spills, so that path keeps the scalar form) — the fused epilogues are not bound by the polynomial's issue slots.
XFM_DEVINL uint64_t pk2(float lo, float hi) { return (uint64_t)__float_as_uint(lo) | ((uint64_t)__float_as_uint(hi) << 32); }
XFM_DEVINL float2 upk2(uint64_t v) { return make_float2(__uint_as_float((uint32_t)v), __uint_as_float((uint32_t)(v >> 32))); }
XFM_DEVINL uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
XFM_DEVINL uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// returns erf(|x| / sqrt 2) for both elements; E = exp(-x^2 / 2) (packed)
XFM_DEVINL uint64_t erf_core2(float x0, float x1, uint64_t& E) {
  const uint64_t ax = pk2(fabsf(x0), fabsf(x1));
  const float2 d = upk2(fma2(pk2(0.3275911f * 0.70710678118654752440f, 0.3275911f * 0.70710678118654752440f), ax, pk2(1.0f, 1.0f)));
  const uint64_t t = pk2(rcp_approx(d.x), rcp_approx(d.y));
  const float2 s = upk2(mul2(mul2(ax, ax), pk2(-0.5f * 1.4426950408889634f, -0.5f * 1.4426950408889634f)));
  E = pk2(ex2_approx(s.x), ex2_approx(s.y));
  uint64_t p = fma2(t, pk2(1.061405429f, 1.061405429f), pk2(-1.453152027f, -1.453152027f));
  p = fma2(t, p, pk2(1.421413741f, 1.421413741f));
  p = fma2(t, p, pk2(-0.284496736f, -0.284496736f));
  p = fma2(t, p, pk2(0.254829592f, 0.254829592f));
  p = mul2(p, t);
  const float2 pe = upk2(p);
  return fma2(pk2(-pe.x, -pe.y), E, pk2(1.0f, 1.0f));
}
XFM_DEVINL float2 gelu_fast2(float x0, float x1) {
  uint64_t E;
  const float2 er = upk2(erf_core2(x0, x1, E));
  const uint64_t hx = mul2(pk2(x0, x1), pk2(0.5f, 0.5f));
  return upk2(fma2(hx, pk2(copysignf(er.x, x0), copysignf(er.y, x1)), hx));
}
XFM_DEVINL float2 gelu_grad_fast2(float x0, float x1) {
  uint64_t E;
  const float2 er = upk2(erf_core2(x0, x1, E));
  const uint64_t cdf = fma2(pk2(0.5f, 0.5f), pk2(copysignf(er.x, x0), copysignf(er.y, x1)), pk2(0.5f, 0.5f));
  // scalar version: fmaf(0.5, er, 0.5) + x * E * 0.3989...: the sum is a separate rounding there too
  const uint64_t pdf = mul2(mul2(pk2(x0, x1), E), pk2(0.39894228040143267794f, 0.39894228040143267794f));
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(cdf), "l"(pdf));
  return upk2(r);
}

XFM_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
XFM_DEVINL float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Counter-based RNG (splitmix-style hash of (seed, index)) -> uniform in [0,1).
// Stateless so the backward pass regenerates the same dropout mask from (seed, index).
XFM_DEVINL uint32_t hash_u32(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + idx * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (uint32_t)(z >> 32);
}
// Dropout keep decision.  One 32-bit mix (lowbias32) per PAIR of consecutive element indices yields 16 random bits per
// element; every dropout site owns element pairs (2 keys per mma fragment register pair, 2 columns per epilogue lane), so
// this is ~5 integer instructions per element instead of the ~25 of the 64-bit hash above.  Stateless in (seed, index):
// the backward kernels regenerate the forward mask.  keep probability = 1 - round(p * 65536) / 65536.
XFM_DEVINL uint32_t mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352dU;
  x ^= x >> 15;
  x *= 0x846ca68bU;
  x ^= x >> 16;
  return x;
}
XFM_DEVINL bool drop_keep_idx(uint64_t seed, uint64_t idx, float p) {
  const uint32_t thr = (uint32_t)(p * 65536.0f + 0.5f);
  const uint64_t pair = idx >> 1;
  const uint32_t s = (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x85EBCA6Bu);
  const uint32_t x = mix32(((uint32_t)pair + (uint32_t)(pair >> 32) * 0x9E3779B1u) ^ s);
  const uint32_t bits = (idx & 1) ? (x >> 16) : (x & 0xFFFFu);
  return bits >= thr;
}
// The same decision for the two elements of pair index `pair` (= element index >> 1) at once: bit 0 = even element kept,
// bit 1 = odd element kept.  seed_mix = drop_seed_mix(seed), thr = drop_threshold(p).
XFM_DEVINL uint32_t drop_seed_mix(uint64_t seed) { return (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x85EBCA6Bu); }
XFM_DEVINL uint32_t drop_threshold(float p) { return (uint32_t)(p * 65536.0f + 0.5f); }
XFM_DEVINL uint32_t drop_keep_pair(uint32_t seed_mix, uint32_t pair_lo, uint32_t pair_hi, uint32_t thr) {
  const uint32_t x = mix32((pair_lo + pair_hi * 0x9E3779B1u) ^ seed_mix);
  return ((x & 0xFFFFu) >= thr ? 1u : 0u) | ((x >> 16) >= thr ? 2u : 0u);
}
XFM_DEVINL float hash_uniform(uint64_t seed, uint64_t idx) { return (float)(hash_u32(seed, idx) >> 8) * (1.0f / 16777216.0f); }

}  // namespace xfm
