// Packed variable-length batches (avsep_forward_packed, include/avsep.h): utterances sit back to back, each as one
// contiguous block -- mixed (F, T_b), frames (N_b, H, W), separated / masks (S, F, T_b).  The unpack kernel expands
// the packed inputs into the padded (B, F, T) / (B, N, H, W) staging that the variable-length forward reads; the pack
// kernel gathers the padded (B, S, F, T) outputs into packed blocks.  Both are HBM-bound copies of the valid regions
// only: the forward never reads past the lengths, so the staging's padding is never written or cleared.
//
// Each CTA row (blockIdx.y) serves one utterance and finds its packed offset as the sum of the clamped lengths in front
// of it, read on the device: the launch parameters (base pointers, first utterance, B, T, N) do not depend on the
// length values, so a captured launch replays for any ragged batch held in the same buffers.  That sum costs each CTA
// O(b) L2-resident loads, a few hundred at the host path's chunk sizes.
#include "common.cuh"
#include "kernels.h"

#include <algorithm>

namespace avsep {

namespace {

constexpr int PK_THREADS = 256;
constexpr int PK_UNROLL = 4;                        // independent loads in flight per thread
constexpr int PK_SPAN = PK_THREADS * PK_UNROLL;     // elements per CTA per pass

// Sums of the clamped audio / lip lengths of utterances [0, n), in every thread of the CTA.
__device__ __forceinline__ void packed_prefix(const int* lens, int T, const int* flens, int N, int n, int& pt, int& pn) {
  __shared__ int red[2][PK_THREADS / 32];
  int st = 0, sn = 0;
  if (lens == nullptr) st = threadIdx.x == 0 ? n * T : 0;
  if (flens == nullptr) sn = threadIdx.x == 0 ? n * N : 0;
  for (int i = threadIdx.x; i < n; i += PK_THREADS) {
    if (lens != nullptr) st += utt_len(lens, i, T);
    if (flens != nullptr) sn += utt_len(flens, i, N);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    st += __shfl_xor_sync(0xffffffffu, st, o);
    sn += __shfl_xor_sync(0xffffffffu, sn, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = st;
    red[1][threadIdx.x >> 5] = sn;
  }
  __syncthreads();
  pt = 0;
  pn = 0;
#pragma unroll
  for (int w = 0; w < PK_THREADS / 32; ++w) {
    pt += red[0][w];
    pn += red[1][w];
  }
}

// One utterance's (rows, tb) block between its packed form (row pitch tb) and its padded form (row pitch T):
// PACK = false: padded[r * T + t] = packed[r * tb + t]; PACK = true: the reverse.  Element i of the packed block is
// row i / tb; every warp access is coalesced on the packed side and runs along t on the padded side.
template <bool PACK>
__device__ __forceinline__ void copy_rows(const float* __restrict__ src, float* __restrict__ dst, int n, int tb, int T) {
  for (int i0 = blockIdx.x * PK_SPAN + threadIdx.x; i0 < n; i0 += gridDim.x * PK_SPAN) {
    float v[PK_UNROLL];
#pragma unroll
    for (int k = 0; k < PK_UNROLL; ++k) {
      const int i = i0 + k * PK_THREADS;
      if (i < n) {
        const int r = i / tb;
        v[k] = __ldcs(src + (PACK ? r * T + (i - r * tb) : i));
      }
    }
#pragma unroll
    for (int k = 0; k < PK_UNROLL; ++k) {
      const int i = i0 + k * PK_THREADS;
      if (i < n) {
        const int r = i / tb;
        dst[PACK ? i : r * T + (i - r * tb)] = v[k];
      }
    }
  }
}

// A contiguous run of n elements (a lip-frame block is laid out the same in both forms).
template <typename V>
__device__ __forceinline__ void copy_run(const V* __restrict__ src, V* __restrict__ dst, int n) {
  for (int i0 = blockIdx.x * PK_SPAN + threadIdx.x; i0 < n; i0 += gridDim.x * PK_SPAN) {
    V v[PK_UNROLL];
#pragma unroll
    for (int k = 0; k < PK_UNROLL; ++k)
      if (i0 + k * PK_THREADS < n) v[k] = __ldcs(src + i0 + k * PK_THREADS);
#pragma unroll
    for (int k = 0; k < PK_UNROLL; ++k)
      if (i0 + k * PK_THREADS < n) dst[i0 + k * PK_THREADS] = v[k];
  }
}

// Utterance b = b0 + blockIdx.y; staging row blockIdx.y.  VEC: frames move as float4 (hw % 4 == 0, packed frames
// 16-byte aligned; the staging is workspace and always is).
template <bool VEC>
__global__ void __launch_bounds__(PK_THREADS)
unpack_kernel(const float* __restrict__ mixed_p, const float* __restrict__ frames_p, const int* __restrict__ lens,
              const int* __restrict__ flens, int b0, int F, int T, int N, int hw, float* __restrict__ mixed,
              float* __restrict__ frames) {
  griddep_launch_dependents();
  griddep_wait();
  const int j = blockIdx.y, b = b0 + j;
  int pt, pn;
  packed_prefix(lens, T, flens, N, b, pt, pn);
  const int tb = utt_len(lens, b, T), nb = utt_len(flens, b, N);
  copy_rows<false>(mixed_p + static_cast<size_t>(pt) * F, mixed + static_cast<size_t>(j) * F * T, F * tb, tb, T);
  const float* fs = frames_p + static_cast<size_t>(pn) * hw;
  float* fd = frames + static_cast<size_t>(j) * N * hw;
  if constexpr (VEC)
    copy_run(reinterpret_cast<const float4*>(fs), reinterpret_cast<float4*>(fd), nb * hw / 4);
  else
    copy_run(fs, fd, nb * hw);
}

// Utterance b = b0 + blockIdx.y: its (S, F, T_b) block of separated and masks from staging row blockIdx.y.
__global__ void __launch_bounds__(PK_THREADS)
pack_kernel(const float* __restrict__ sep, const float* __restrict__ masks, const int* __restrict__ lens, int b0,
            int SF, int T, float* __restrict__ sep_p, float* __restrict__ masks_p) {
  griddep_launch_dependents();
  griddep_wait();
  const int j = blockIdx.y, b = b0 + j;
  int pt, pn;
  packed_prefix(lens, T, nullptr, 0, b, pt, pn);
  const int tb = utt_len(lens, b, T);
  const size_t src = static_cast<size_t>(j) * SF * T, dst = static_cast<size_t>(pt) * SF;
  copy_rows<true>(sep + src, sep_p + dst, SF * tb, tb, T);
  copy_rows<true>(masks + src, masks_p + dst, SF * tb, tb, T);
}

unsigned ctas_for(long long elems) { return static_cast<unsigned>((elems + PK_SPAN - 1) / PK_SPAN); }

}  // namespace

const char* launch_unpack(LaunchCtx lc, const float* mixed_p, const float* frames_p, const int* lens,
                          const int* flens, int b0, int B, int F, int T, int N, int hw, float* mixed, float* frames) {
  if (B <= 0) return nullptr;
  if (static_cast<long long>(F) * T > 0x7fffffffLL || static_cast<long long>(N) * hw > 0x7fffffffLL)
    return "unpack: utterance too large";
  const bool vec = hw % 4 == 0 && (reinterpret_cast<uintptr_t>(frames_p) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(frames) & 15) == 0;
  const long long fr = static_cast<long long>(N) * hw / (vec ? 4 : 1);
  const dim3 grid(std::max(ctas_for(static_cast<long long>(F) * T), ctas_for(fr)), B);
  const cudaError_t e = launch_pdl(vec ? unpack_kernel<true> : unpack_kernel<false>, grid, dim3(PK_THREADS), 0, lc,
                                   mixed_p, frames_p, lens, flens, b0, F, T, N, hw, mixed, frames);
  return e == cudaSuccess ? nullptr : "unpack: launch failed";
}

const char* launch_pack(LaunchCtx lc, const float* sep, const float* masks, const int* lens, int b0, int B, int S,
                        int F, int T, float* sep_p, float* masks_p) {
  if (B <= 0) return nullptr;
  const long long SF = static_cast<long long>(S) * F;
  if (SF * T > 0x7fffffffLL) return "pack: utterance too large";
  const dim3 grid(ctas_for(SF * T), B);
  const cudaError_t e = launch_pdl(pack_kernel, grid, dim3(PK_THREADS), 0, lc, sep, masks, lens, b0,
                                   static_cast<int>(SF), T, sep_p, masks_p);
  return e == cudaSuccess ? nullptr : "pack: launch failed";
}

}  // namespace avsep
