// HBM-bound kernels of the path: fused residual-add + LayerNorm (warp per row, shuffle reductions, 128-bit
// accesses) and the mixed_spec transpose/pad/cast that feeds the Conv1d implicit GEMM.
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

constexpr int LN_WARPS = 8;
constexpr int LN_MAX_V4 = 8;   // float4 chunks cached per lane: d <= 8*32*4 = 1024

// x_out = x + y ; out = (x_out - mean) * rstd * gamma + beta      (nn.LayerNorm, eps 1e-5, biased variance;
// reference call sites model.py:149,168,172 and the encoder layers' norm1/norm2.)
// One warp owns one row: the row is read once with float4 loads, mean and centred variance are reduced with
// __shfl_xor, and every global access is a full 512-byte (fp32) or 256-byte (bf16) warp transaction.
template <bool TF32>
__global__ void __launch_bounds__(LN_WARPS * 32)
add_layernorm_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ gamma,
                     const float* __restrict__ beta, float* __restrict__ x_out, void* __restrict__ out_op, int M,
                     int d) {
  griddep_launch_dependents();
  griddep_wait();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * LN_WARPS + (threadIdx.x >> 5);
  if (row >= M) return;
  const int nv = d >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<size_t>(row) * d);
  const float4* yr = y ? reinterpret_cast<const float4*>(y + static_cast<size_t>(row) * d) : nullptr;
  float4 v[LN_MAX_V4];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAX_V4; ++i) {
    const int c = lane + 32 * i;
    if (c < nv) {
      float4 a = xr[c];
      if (yr) {
        const float4 b = yr[c];
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      v[i] = a;
      sum += (a.x + a.y) + (a.z + a.w);
    }
  }
  if (x_out != nullptr) {
    float4* xo = reinterpret_cast<float4*>(x_out + static_cast<size_t>(row) * d);
#pragma unroll
    for (int i = 0; i < LN_MAX_V4; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) xo[c] = v[i];
    }
  }
  if (out_op == nullptr) return;
  float mean = 0.f, rstd = 1.f;
  if (gamma != nullptr) {
    mean = warp_sum(sum) / static_cast<float>(d);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAX_V4; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        const float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, dd = v[i].w - mean;
        sq += (a * a + b * b) + (cc * cc + dd * dd);
      }
    }
    rstd = rsqrtf(warp_sum(sq) / static_cast<float>(d) + 1e-5f);
  }
#pragma unroll
  for (int i = 0; i < LN_MAX_V4; ++i) {
    const int c = lane + 32 * i;
    if (c < nv) {
      float4 o = v[i];
      if (gamma != nullptr) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c);
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + c);
        o.x = (o.x - mean) * rstd * g.x + b.x;
        o.y = (o.y - mean) * rstd * g.y + b.y;
        o.z = (o.z - mean) * rstd * g.z + b.z;
        o.w = (o.w - mean) * rstd * g.w + b.w;
      }
      if constexpr (TF32) {
        o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w);
        reinterpret_cast<float4*>(reinterpret_cast<float*>(out_op) + static_cast<size_t>(row) * d)[c] = o;
      } else {
        uint2 u;
        u.x = pack_bf16x2(o.x, o.y);
        u.y = pack_bf16x2(o.z, o.w);
        reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out_op) + static_cast<size_t>(row) * d)[c] = u;
      }
    }
  }
}

// mixed (B,F,T) fp32, T fastest  ->  xp (B, T+2, Fp), F fastest, rows 0 and T+1 zero (Conv1d padding=1,
// model.py:38), columns [F,Fp) zero.  32x32 smem-tile transpose: reads coalesced along T, writes along F.
// lens (variable-length batch, else null): rows t >= lens[b] are zero (the short clip's right-hand padding) and the
// mixture is not read there.
template <bool TF32>
__global__ void __launch_bounds__(256)
prep_audio_kernel(const float* __restrict__ mixed, void* __restrict__ xp, int F, int T, int Fp,
                  const int* __restrict__ lens) {
  __shared__ float tile[32][33];
  griddep_launch_dependents();
  griddep_wait();
  const int b = blockIdx.z;
  const int f0 = blockIdx.y * 32;
  const int t0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31;
  const int ty = threadIdx.x >> 5;   // 0..7
  const float* src = mixed + static_cast<size_t>(b) * F * T;
  const int Tb = utt_len(lens, b, T);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int f = f0 + ty + 8 * i;
    const int t = t0 + tx;
    tile[ty + 8 * i][tx] = (f < F && t < Tb) ? src[static_cast<size_t>(f) * T + t] : 0.f;
  }
  __syncthreads();
  const size_t base = static_cast<size_t>(b) * (T + 2) * Fp;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int t = t0 + ty + 8 * i;
    const int f = f0 + tx;
    if (t < T && f < Fp) {
      const float val = tile[tx][ty + 8 * i];
      const size_t o = base + static_cast<size_t>(t + 1) * Fp + f;
      if constexpr (TF32) reinterpret_cast<float*>(xp)[o] = round_tf32(val);
      else reinterpret_cast<__nv_bfloat16*>(xp)[o] = __float2bfloat16_rn(val);
    }
  }
  if (blockIdx.x == 0) {   // halo rows
    for (int i = threadIdx.x; i < 64; i += 256) {
      const int f = f0 + (i & 31);
      const int rowp = (i < 32) ? 0 : (T + 1);
      if (f < Fp) {
        const size_t o = base + static_cast<size_t>(rowp) * Fp + f;
        if constexpr (TF32) reinterpret_cast<float*>(xp)[o] = 0.f;
        else reinterpret_cast<__nv_bfloat16*>(xp)[o] = __float2bfloat16_rn(0.f);
      }
    }
  }
}

}  // namespace

const char* launch_add_layernorm(LaunchCtx lc, int prec, const float* x, const float* y, const float* gamma,
                                 const float* beta, float* x_out, void* out_op, int M, int d) {
  if ((d & 3) != 0 || d > LN_MAX_V4 * 128) return "layernorm: d_model must be a multiple of 4 and <= 1024";
  if (M <= 0) return "layernorm: empty";
  dim3 grid((M + LN_WARPS - 1) / LN_WARPS);
  if (prec == PREC_TF32)
    launch_pdl(add_layernorm_kernel<true>, dim3(grid), dim3(LN_WARPS * 32), 0, lc, x, y, gamma, beta, x_out, out_op, M, d);
  else
    launch_pdl(add_layernorm_kernel<false>, dim3(grid), dim3(LN_WARPS * 32), 0, lc, x, y, gamma, beta, x_out, out_op, M, d);
  return cudaGetLastError() == cudaSuccess ? nullptr : "layernorm: launch failed";
}

const char* launch_prep_audio(LaunchCtx lc, int prec, const float* mixed, void* xp, int B, int F, int T, int Fp,
                              const int* lens) {
  dim3 grid((T + 31) / 32, (Fp + 31) / 32, B);
  if (prec == PREC_TF32) launch_pdl(prep_audio_kernel<true>, grid, dim3(256), 0, lc, mixed, xp, F, T, Fp, lens);
  else launch_pdl(prep_audio_kernel<false>, grid, dim3(256), 0, lc, mixed, xp, F, T, Fp, lens);
  return cudaGetLastError() == cudaSuccess ? nullptr : "prep_audio: launch failed";
}

}  // namespace avsep
