// Microbenchmark: cycles per tcgen05.mma.cta_group::2 (M = 256 over a CTA pair, K = 16, kind::f16) issued back to back
// by the leader CTA, for N = 64 / 128 / 256, A from shared memory or tensor memory; 74 clusters (all SMs busy).
#include "common.cuh"
#include <cstdio>
using namespace avsep;

// ---- cta_group::2: one MMA spans a pair of CTAs (M = 256: 128 rows in each CTA's tensor memory, B split by N halves
// between the two CTAs' shared memories); issued by one thread of the even-ranked (leader) CTA ----
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_result, uint32_t ncols) {   // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_cg2(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_ts_cg2(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread are complete) on the barrier at this offset in every CTA of cta_mask
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {     // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__global__ void __launch_bounds__(64, 1) mma_rate_cg2_kernel(int N, int a_in_tmem, int reps, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  for (int i = threadIdx.x; i < (16384 + 32768) / 4; i += 64) reinterpret_cast<uint32_t*>(smem)[i] = 0;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_mbar_init(); }
  if (threadIdx.x < 32) tmem_alloc_cg2(&tmem_slot, 512);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tm = tmem_slot;
  if (threadIdx.x == 0 && cluster_ctarank() == 0) {
    const uint32_t idesc = umma_idesc(1u, 256, N);
    const uint64_t adesc = umma_desc_kmajor_sw128(smem_u32(smem), 1024);
    const uint64_t bdesc = umma_desc_kmajor_sw128(smem_u32(smem + 16384), 1024);
    for (int i = 0; i < 8; ++i) umma_f16_cg2(tm, adesc, bdesc, idesc, 1);
    umma_commit_cg2(&bar, 0x1);
    mbar_wait(&bar, 0);
    const long long t0 = clock64();
    if (a_in_tmem) {
      for (int i = 0; i < reps; ++i) umma_f16_ts_cg2(tm, tm + 256 + 8 * (i & 3), bdesc + 2 * (i & 3), idesc, 1);
    } else {
      for (int i = 0; i < reps; ++i) umma_f16_cg2(tm, adesc + 2 * (i & 3), bdesc + 2 * (i & 3), idesc, 1);
    }
    umma_commit_cg2(&bar, 0x1);
    mbar_wait(&bar, 1);
    const long long t2 = clock64();
    if (blockIdx.x == 0) out[0] = t2 - t0;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (threadIdx.x < 32) tmem_dealloc_cg2(tm, 512);
}

int main() {
  long long* out;
  cudaMallocManaged(&out, 16);
  cudaFuncSetAttribute(mma_rate_cg2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  const int reps = 2048;
  for (int a_in_tmem = 0; a_in_tmem < 2; ++a_in_tmem)
    for (int N : {64, 128, 256}) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(148); cfg.blockDim = dim3(64); cfg.dynamicSmemBytes = 64 * 1024;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      cudaLaunchKernelEx(&cfg, mma_rate_cg2_kernel, N, a_in_tmem, reps, out);
      if (cudaDeviceSynchronize() != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
      const double math = 128.0 * N * 16 * 2 / 8192.0;     // per-SM tensor time (each SM computes its 128 rows)
      printf("cta_group::2 M=256 N=%3d A=%s: %.1f clk/MMA (per-SM tensor time at 8192 FLOP/clk: %.0f)\n", N,
             a_in_tmem ? "tmem" : "smem", double(out[0]) / reps, math);
    }
  return 0;
}
