// Device helpers shared by the library's sm_100a kernels (inline PTX): small math, the global timer, the 128-byte
// swizzle offset, mma.sync / ldmatrix, programmatic dependent launch, mbarrier, TMA and single-CTA tcgen05 / TMEM
// wrappers.  Only helpers that some library kernel calls live here; the microbenchmarks under tools/ keep their own
// extras.  Everything here is written for sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

#ifndef AVSEP_WATCHDOG_CYCLES
// Bounded spin on every mbarrier wait: a descriptor / byte-count bug traps instead of hanging the GPU.
#define AVSEP_WATCHDOG_CYCLES (4000000000ll)
#endif

namespace avsep {

// ------------------------------------------------------------------------------------------
// generic
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// sigmoid(z) = 1 / (1 + 2^(-z log2 e)) on the two MUFU approximations, nothing else: ex2 flushes to 0 below 2^-126
// (the mask is then exactly 1) and overflows to +inf for z < -88 (rcp(inf) = 0), so no range handling is needed.
__device__ __forceinline__ float sigmoid_fast(float z) {
  float t, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(z * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + t));
  return r;
}

// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, i.e. fp32-exact for our purposes), branch-free:
// erf(|z|) = 1 - (a1 t + a2 t^2 + a3 t^3 + a4 t^4 + a5 t^5) exp(-z^2), t = 1 / (1 + p |z|).
__device__ __forceinline__ float erf_as(float z) {
  const float az = fabsf(z);
  const float t = __fdividef(1.0f, fmaf(0.3275911f, az, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  const float e = exp2f(-az * az * 1.4426950408889634f);
  return copysignf(fmaf(-poly, e, 1.0f), z);
}
__device__ __forceinline__ float gelu_erf(float x) {          // nn.GELU() default (erf form)
  return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752440f));
}

// erf-GELU for results that are rounded to bf16 anyway: x clamped to [-4.5, 4.5], erf(x/sqrt2)/x as a degree-9
// polynomial in t = 2 x^2 / 4.5^2 - 1 (Chebyshev fit converted to monomials), 16 FMA-pipe instructions, no MUFU.
// |error| <= 3.5e-5 for |x| <= 4.5 and <= 1e-5 |x| beyond (bf16 rounding of the result is 4e-3 relative); the fp32-grade
// TF32 path keeps gelu_erf.  The GELU epilogues are issue-bound, so instruction count is what matters.
__device__ __forceinline__ float gelu_bf16_grade(float x) {
  const float xc = fminf(fmaxf(x, -4.5f), 4.5f);
  const float t = fmaf(xc * xc, 0.09876543209876543f, -1.0f);
  float p = -0.004680031910538673f;
  p = fmaf(p, t, 0.010336018167436123f);
  p = fmaf(p, t, -0.010503096505999565f);
  p = fmaf(p, t, 0.018587922677397728f);
  p = fmaf(p, t, -0.03804188221693039f);
  p = fmaf(p, t, 0.05810019373893738f);
  p = fmaf(p, t, -0.08021842688322067f);
  p = fmaf(p, t, 0.10921084135770798f);
  p = fmaf(p, t, -0.1543877273797989f);
  p = fmaf(p, t, 0.3138136863708496f);
  const float hx = 0.5f * x;
  return fmaf(hx, xc * p, hx);
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// fp32 -> TF32 with round-to-nearest (the tensor core would otherwise truncate the low 13 mantissa bits, which
// doubles the operand error and biases it towards zero).  Result is an fp32 bit pattern with a 10-bit mantissa.
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// Nanoseconds of the GPU's global timer (the debug trace stamps and the flag-wait timeout).
__device__ __forceinline__ unsigned long long globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)::"memory");
  return t;
}

// Byte offset of 16-byte chunk c of row r in a buffer of 128-byte rows with the 128-byte swizzle (the layout of TMA
// SWIZZLE_128B boxes and of the UMMA descriptors): the chunk sits at slot c ^ (r & 7).
__device__ __forceinline__ uint32_t sw128_off(int row, int c) {
  return static_cast<uint32_t>(row * 128 + ((c ^ (row & 7)) << 4));
}

// ------------------------------------------------------------------------------------------
// mma.sync (bf16 operands, fp32 accumulation) and its ldmatrix fragment loads
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
// c += A (16x16, row) * B (16x8, col)
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  mma_bf16_16816(c, a[0], a[1], a[2], a[3], b0, b1);
}

// ------------------------------------------------------------------------------------------
// programmatic dependent launch: a kernel launched with the programmatic-serialization attribute may start while
// its predecessor in the stream is still running; everything before griddep_wait() (barrier init, TMEM alloc,
// descriptor prefetch, constant loads) overlaps the predecessor's tail, nothing produced by it may be touched earlier.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// The watchdog's slow path is a real function call: inlined, its printf argument set-up added ~25 instructions to every
// wait, and the persistent multi-role kernels are instruction-cache bound (32 KB L1.5 per SM, three roles running
// different code at once).
static __device__ __noinline__ void mbar_timeout(uint64_t* bar, uint32_t parity) {
  // the barrier's shared-memory offset identifies the wait site (barriers sit in one block per kernel)
  printf("avsep: mbarrier watchdog fired (block %d,%d thread %d, barrier at smem +%u, parity %u)\n", blockIdx.x, blockIdx.y,
         threadIdx.x, static_cast<unsigned>(__cvta_generic_to_shared(bar)), parity);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > AVSEP_WATCHDOG_CYCLES) mbar_timeout(bar, parity);
  }
}

// Same, but each probe may suspend the thread in hardware for up to ~1 us (suspend-time hint) instead of spinning:
// for single-thread producer / MMA-issuer roles that share an SM sub-partition with compute warps, so that their
// polling does not take issue slots.  The watchdog is then checked about once per microsecond.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_hint(bar, parity, 1000u)) {
    if (clock64() - t0 > AVSEP_WATCHDOG_CYCLES) mbar_timeout(bar, parity);
  }
}

// ------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), completion on an mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// TMA store (shared -> global), bulk-group completion
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all bulk stores committed by this thread have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {        // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers fp16/bf16 operands with fp32 accumulation.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from tensor memory (128 lanes x K/2 32-bit columns, two consecutive K elements per column), B from smem.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all tcgen05 ops previously issued by this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets row (lane base + i), columns [col, col+32).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 16 consecutive 32-bit columns, registers -> tensor memory (thread i writes row lane base + i).
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (one swizzle atom = 8 rows x 128 B,
// rows 128 B apart, 8-row groups SBO bytes apart).  Bit layout (sm_100 UMMA descriptor):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (ignored for swizzled K-major; 1)
//   [32,46) stride byte offset >> 4 | [46,48) version = 1 | [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// MN-major operand, 128-byte swizzle: 64 contiguous elements (bf16) along MN per 128-B row, rows = K index,
// 8-row (8 x K) groups SBO bytes apart, 64-element MN atoms LBO bytes apart.
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                            uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// Instruction descriptor (32-bit) for kind::f16 / kind::tf32, fp32 accumulate, dense.
//   [4,6) D format (1 = f32) | [7,10) A format | [10,13) B format (0 = f16, 1 = bf16, 2 = tf32)
//   [15] A major (0 = K) | [16] B major (0 = K, 1 = MN) | [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t fmt, uint32_t M, uint32_t N, uint32_t a_mn = 0,
                                                  uint32_t b_mn = 0) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn << 15) | (b_mn << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace avsep
