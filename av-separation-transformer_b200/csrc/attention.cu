// Flash-style multi-head attention (no T x T materialisation, online softmax), forward only.
//
// Self-attention of the encoder stacks (reference: nn.TransformerEncoderLayer, model.py:48-52,97-101) and the
// audio-queries-visual cross-attention of CrossModalFusion (model.py:155,169).  For cross-attention the K/V rows
// are produced on load: the K/V projection is computed once on the N visual frames and the reference's
// F.interpolate(mode='linear', align_corners=False) (model.py:114-116) is applied to the projected rows while the
// tile is staged into shared memory (interp and projection commute: W(Ax)+b = A(Wx+b), rows of A sum to 1).
//
// One CTA = 64 query rows of one (utterance, head); 4 warps x 16 rows; K/V tiles of 64 rows; bf16 tensor-core
// contractions with fp32 accumulation, fp32 softmax statistics, exp2 with the 1/sqrt(hd)*log2(e) scale folded in.
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

struct AttnDev {
  const void* q;      // bf16 rows, or fp32 rows on the split (fp32-grade) path
  const void* k;
  const void* v;
  void* out;          // bf16, or fp32 on the split path
  int ldq, ldkv, ldo;
  int H, Lq, Lk, nsrc;
  float scale_log2;
  float lerp_scale;   // (float)nsrc / Lk, as ATen computes it
  // variable-length batch (null: all Lk / all nsrc): keys of utterance b, and its interpolation source rows.  Lk and
  // nsrc stay the row pitch of the K/V buffers.
  const int *k_lens, *src_lens;
};

// Keys of utterance b, its interpolation source rows and scale (ATen: (float)nsrc / (float)Lk).
struct UttKeys {
  int lk, nsrc;
  float scale;
};
template <bool LERP>
__device__ __forceinline__ UttKeys utt_keys(const AttnDev& p, int b) {
  UttKeys u;
  u.lk = utt_len(p.k_lens, b, p.Lk);
  u.nsrc = LERP ? utt_len(p.src_lens, b, p.nsrc) : 0;
  u.scale = (p.k_lens == nullptr && p.src_lens == nullptr) ? p.lerp_scale
                                                           : static_cast<float>(u.nsrc) / static_cast<float>(u.lk);
  return u;
}

constexpr int QT = 64;   // query rows per CTA
constexpr int KT = 64;   // key/value rows per tile

// Stage ROWS x HD bf16 rows into padded shared memory; rows >= nrows are zero.
template <int HD>
__device__ __forceinline__ void load_tile_bf16(__nv_bfloat16* dst, const __nv_bfloat16* src, int ld, int row0,
                                               int nrows) {
  constexpr int LDS = HD + 8;
  constexpr int CH = HD / 8;
  for (int i = threadIdx.x; i < 64 * CH; i += 128) {
    const int r = i / CH, c = i - r * CH;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (row0 + r < nrows) val = *reinterpret_cast<const uint4*>(src + static_cast<size_t>(row0 + r) * ld + c * 8);
    *reinterpret_cast<uint4*>(dst + r * LDS + c * 8) = val;
  }
}

// Same, but each output row t is the linear interpolation of two fp32 source rows (ATen upsample_linear1d,
// align_corners=False: src = max(scale*(t+0.5)-0.5, 0); i0 = floor(src); i1 = min(i0+1, n-1); lam = src-i0).
template <int HD>
__device__ __forceinline__ void load_tile_lerp(__nv_bfloat16* dst, const float* src, int ld, int row0, int nrows,
                                               int nsrc, float scale) {
  constexpr int LDS = HD + 8;
  constexpr int CH = HD / 8;
  for (int i = threadIdx.x; i < 64 * CH; i += 128) {
    const int r = i / CH, c = i - r * CH;
    const int t = row0 + r;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (t < nrows) {
      const float sp = fmaxf(scale * (static_cast<float>(t) + 0.5f) - 0.5f, 0.0f);
      int i0 = static_cast<int>(sp);
      if (i0 > nsrc - 1) i0 = nsrc - 1;
      const int i1 = min(i0 + 1, nsrc - 1);
      const float w1 = sp - static_cast<float>(i0);
      const float w0 = 1.0f - w1;
      const float4* p0 = reinterpret_cast<const float4*>(src + static_cast<size_t>(i0) * ld + c * 8);
      const float4* p1 = reinterpret_cast<const float4*>(src + static_cast<size_t>(i1) * ld + c * 8);
      const float4 a0 = __ldg(p0), a1 = __ldg(p0 + 1), b0 = __ldg(p1), b1 = __ldg(p1 + 1);
      val.x = pack_bf16x2(w0 * a0.x + w1 * b0.x, w0 * a0.y + w1 * b0.y);
      val.y = pack_bf16x2(w0 * a0.z + w1 * b0.z, w0 * a0.w + w1 * b0.w);
      val.z = pack_bf16x2(w0 * a1.x + w1 * b1.x, w0 * a1.y + w1 * b1.y);
      val.w = pack_bf16x2(w0 * a1.z + w1 * b1.z, w0 * a1.w + w1 * b1.w);
    }
    *reinterpret_cast<uint4*>(dst + r * LDS + c * 8) = val;
  }
}

// fp32 source rows -> bf16 hi and lo tiles (x = hi + lo to ~2^-17 relative): the split operands of the fp32-grade
// path.  nsrc > 0: rows are interpolated on load exactly as in load_tile_lerp.
template <int HD>
__device__ __forceinline__ void load_tile_split(__nv_bfloat16* dst_hi, __nv_bfloat16* dst_lo, const float* src, int ld,
                                                int row0, int nrows, int nsrc, float scale) {
  constexpr int LDS = HD + 8;
  constexpr int CH = HD / 8;
  for (int i = threadIdx.x; i < 64 * CH; i += 128) {
    const int r = i / CH, c = i - r * CH;
    const int t = row0 + r;
    float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (t < nrows) {
      if (nsrc > 0) {
        const float sp = fmaxf(scale * (static_cast<float>(t) + 0.5f) - 0.5f, 0.0f);
        int i0 = static_cast<int>(sp);
        if (i0 > nsrc - 1) i0 = nsrc - 1;
        const int i1 = min(i0 + 1, nsrc - 1);
        const float w1 = sp - static_cast<float>(i0), w0 = 1.0f - w1;
        const float4* p0 = reinterpret_cast<const float4*>(src + static_cast<size_t>(i0) * ld + c * 8);
        const float4* p1 = reinterpret_cast<const float4*>(src + static_cast<size_t>(i1) * ld + c * 8);
        const float4 a0 = __ldg(p0), a1 = __ldg(p0 + 1), b0 = __ldg(p1), b1 = __ldg(p1 + 1);
        x[0] = w0 * a0.x + w1 * b0.x; x[1] = w0 * a0.y + w1 * b0.y; x[2] = w0 * a0.z + w1 * b0.z; x[3] = w0 * a0.w + w1 * b0.w;
        x[4] = w0 * a1.x + w1 * b1.x; x[5] = w0 * a1.y + w1 * b1.y; x[6] = w0 * a1.z + w1 * b1.z; x[7] = w0 * a1.w + w1 * b1.w;
      } else {
        const float4* p0 = reinterpret_cast<const float4*>(src + static_cast<size_t>(t) * ld + c * 8);
        const float4 a0 = __ldg(p0), a1 = __ldg(p0 + 1);
        x[0] = a0.x; x[1] = a0.y; x[2] = a0.z; x[3] = a0.w; x[4] = a1.x; x[5] = a1.y; x[6] = a1.z; x[7] = a1.w;
      }
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * j]), h1 = __float2bfloat16_rn(x[2 * j + 1]);
      hi[j] = pack_bf16x2(__bfloat162float(h0), __bfloat162float(h1));
      lo[j] = pack_bf16x2(x[2 * j] - __bfloat162float(h0), x[2 * j + 1] - __bfloat162float(h1));
    }
    *reinterpret_cast<uint4*>(dst_hi + r * LDS + c * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst_lo + r * LDS + c * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// SPLIT = fp32-grade path: Q/K/V are fp32 in global memory and are staged as bf16 hi + lo tiles; every contraction is
// three tensor-core products (hi*hi + hi*lo + lo*hi); P is split the same way; the output is fp32.
// The minimum-blocks bound keeps the bf16 head-dim 64 / 128 variants at 128 / 168 registers, i.e. 4 / 3 resident
// CTAs per SM, which ptxas gives them without spills.
template <int HD, bool LERP, bool SPLIT>
__global__ void __launch_bounds__(128, SPLIT ? 0 : HD == 64 ? 4 : HD == 128 ? 3 : 0) attention_kernel(const AttnDev p) {
  constexpr int LDS = HD + 8;           // padded row (elements): 16-byte rows shifted by 4 banks -> conflict-free ldmatrix
  constexpr int KS = HD / 16;           // k-steps over the head dimension
  constexpr int NT_O = HD / 8;          // output n-tiles
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* sK = sQ + QT * LDS;
  __nv_bfloat16* sV = sK + KT * LDS;
  __nv_bfloat16* sQl = sV + KT * LDS;      // lo tiles (SPLIT only)
  __nv_bfloat16* sKl = sQl + QT * LDS;
  __nv_bfloat16* sVl = sKl + KT * LDS;

  griddep_launch_dependents();
  griddep_wait();
  const int q0 = blockIdx.x * QT;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int lk = utt_len(p.k_lens, b, p.Lk);

  auto load_kv = [&](int kv0) {
    const UttKeys uk = utt_keys<LERP>(p, b);       // re-derived per tile: fewer registers live across the sweep
    if constexpr (SPLIT) {
      const int src_rows = LERP ? p.nsrc : p.Lk;
      const float* ksrc = reinterpret_cast<const float*>(p.k) + static_cast<size_t>(b) * src_rows * p.ldkv + h * HD;
      const float* vsrc = reinterpret_cast<const float*>(p.v) + static_cast<size_t>(b) * src_rows * p.ldkv + h * HD;
      load_tile_split<HD>(sK, sKl, ksrc, p.ldkv, kv0, uk.lk, uk.nsrc, uk.scale);
      load_tile_split<HD>(sV, sVl, vsrc, p.ldkv, kv0, uk.lk, uk.nsrc, uk.scale);
    } else if constexpr (LERP) {
      const float* ksrc = reinterpret_cast<const float*>(p.k) + static_cast<size_t>(b) * p.nsrc * p.ldkv + h * HD;
      const float* vsrc = reinterpret_cast<const float*>(p.v) + static_cast<size_t>(b) * p.nsrc * p.ldkv + h * HD;
      load_tile_lerp<HD>(sK, ksrc, p.ldkv, kv0, uk.lk, uk.nsrc, uk.scale);
      load_tile_lerp<HD>(sV, vsrc, p.ldkv, kv0, uk.lk, uk.nsrc, uk.scale);
    } else {
      const __nv_bfloat16* ksrc =
          reinterpret_cast<const __nv_bfloat16*>(p.k) + static_cast<size_t>(b) * p.Lk * p.ldkv + h * HD;
      const __nv_bfloat16* vsrc =
          reinterpret_cast<const __nv_bfloat16*>(p.v) + static_cast<size_t>(b) * p.Lk * p.ldkv + h * HD;
      load_tile_bf16<HD>(sK, ksrc, p.ldkv, kv0, uk.lk);
      load_tile_bf16<HD>(sV, vsrc, p.ldkv, kv0, uk.lk);
    }
  };
  // Q and the first K/V tile are staged together: one exposed global-load latency instead of two (at T <= 64 the
  // whole problem is this one tile).
  if constexpr (SPLIT) {
    const float* qsrc = reinterpret_cast<const float*>(p.q) + static_cast<size_t>(b) * p.Lq * p.ldq + h * HD;
    load_tile_split<HD>(sQ, sQl, qsrc, p.ldq, q0, p.Lq, 0, 0.f);
  } else {
    const __nv_bfloat16* qsrc = reinterpret_cast<const __nv_bfloat16*>(p.q) + static_cast<size_t>(b) * p.Lq * p.ldq + h * HD;
    load_tile_bf16<HD>(sQ, qsrc, p.ldq, q0, p.Lq);
  }
  load_kv(0);
  __syncthreads();

  // Q fragments stay in registers for the whole K/V sweep.
  uint32_t qf[KS][4];
  uint32_t qfl[SPLIT ? KS : 1][4];
  {
    const int row = warp * 16 + (lane & 15);
    const int col = (lane >> 4) * 8;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      ldmatrix_x4(qf[ks], smem_u32(sQ + row * LDS + ks * 16 + col));
      if constexpr (SPLIT) ldmatrix_x4(qfl[ks], smem_u32(sQl + row * LDS + ks * 16 + col));
    }
  }

  float o[NT_O][4];
#pragma unroll
  for (int i = 0; i < NT_O; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY};
  float l_run[2] = {0.f, 0.f};

  const int num_kv_tiles = (lk + KT - 1) / KT;       // key tiles wholly past the utterance's keys are skipped
  for (int jt = 0; jt < num_kv_tiles; ++jt) {
    const int kv0 = jt * KT;
    if (jt > 0) {
      __syncthreads();   // previous tile fully consumed
      load_kv(kv0);
      __syncthreads();
    }

    // ---- S = Q K^T (16 x 64 per warp) ----
    float s[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
      for (int np = 0; np < 4; ++np) {   // pairs of 8-wide kv n-tiles
        uint32_t bf[4];
        const int row = np * 16 + ((lane >> 4) << 3) + (lane & 7);
        const int col = ks * 16 + ((lane >> 3) & 1) * 8;
        ldmatrix_x4(bf, smem_u32(sK + row * LDS + col));
        mma_bf16_16816(s[2 * np], qf[ks], bf[0], bf[1]);
        mma_bf16_16816(s[2 * np + 1], qf[ks], bf[2], bf[3]);
        if constexpr (SPLIT) {
          mma_bf16_16816(s[2 * np], qfl[ks], bf[0], bf[1]);          // lo * hi
          mma_bf16_16816(s[2 * np + 1], qfl[ks], bf[2], bf[3]);
          uint32_t bl[4];
          ldmatrix_x4(bl, smem_u32(sKl + row * LDS + col));
          mma_bf16_16816(s[2 * np], qf[ks], bl[0], bl[1]);           // hi * lo
          mma_bf16_16816(s[2 * np + 1], qf[ks], bl[2], bl[3]);
        }
      }
    }

    // ---- online softmax (rows lane/4 and lane/4 + 8; columns 2*(lane%4)+{0,1} of each n-tile) ----
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int c = kv0 + nt * 8 + 2 * (lane & 3);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool ok = (c + (e & 1)) < lk;
        const float val = ok ? s[nt][e] * p.scale_log2 : -INFINITY;
        s[nt][e] = val;
        mx[e >> 1] = fmaxf(mx[e >> 1], val);
      }
    }
    float alpha[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m_run[r], mx[r]);     // finite: every tile has at least one valid column
      alpha[r] = exp2f(m_run[r] - m_new);
      m_run[r] = m_new;
      l_run[r] *= alpha[r];
    }
    uint32_t pf[4][4];   // P as A fragments for the 4 k-steps over this kv tile
    uint32_t pfl[SPLIT ? 4 : 1][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float p0 = exp2f(s[nt][0] - m_run[0]);
      const float p1 = exp2f(s[nt][1] - m_run[0]);
      const float p2 = exp2f(s[nt][2] - m_run[1]);
      const float p3 = exp2f(s[nt][3] - m_run[1]);
      l_run[0] += p0 + p1;
      l_run[1] += p2 + p3;
      pf[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16x2(p0, p1);
      pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p2, p3);
      if constexpr (SPLIT) {
        const float h0 = __bfloat162float(__float2bfloat16_rn(p0)), h1 = __bfloat162float(__float2bfloat16_rn(p1));
        const float h2 = __bfloat162float(__float2bfloat16_rn(p2)), h3 = __bfloat162float(__float2bfloat16_rn(p3));
        pfl[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16x2(p0 - h0, p1 - h1);
        pfl[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p2 - h2, p3 - h3);
      }
    }
#pragma unroll
    for (int i = 0; i < NT_O; ++i) {
      o[i][0] *= alpha[0]; o[i][1] *= alpha[0];
      o[i][2] *= alpha[1]; o[i][3] *= alpha[1];
    }

    // ---- O += P V ----
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {          // 16 kv rows per step
#pragma unroll
      for (int np = 0; np < NT_O / 2; ++np) { // pairs of 8-wide hd n-tiles
        uint32_t bf[4];
        const int row = ks * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
        const int col = np * 16 + (lane >> 4) * 8;
        ldmatrix_x4_trans(bf, smem_u32(sV + row * LDS + col));
        mma_bf16_16816(o[2 * np], pf[ks], bf[0], bf[1]);
        mma_bf16_16816(o[2 * np + 1], pf[ks], bf[2], bf[3]);
        if constexpr (SPLIT) {
          mma_bf16_16816(o[2 * np], pfl[ks], bf[0], bf[1]);
          mma_bf16_16816(o[2 * np + 1], pfl[ks], bf[2], bf[3]);
          uint32_t bl[4];
          ldmatrix_x4_trans(bl, smem_u32(sVl + row * LDS + col));
          mma_bf16_16816(o[2 * np], pf[ks], bl[0], bl[1]);
          mma_bf16_16816(o[2 * np + 1], pf[ks], bl[2], bl[3]);
        }
      }
    }
  }

  // ---- normalise and store ----
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  const float inv0 = 1.0f / l_run[0];
  const float inv1 = 1.0f / l_run[1];
  const int r0 = q0 + warp * 16 + (lane >> 2);
  const int r1 = r0 + 8;
  if constexpr (SPLIT) {
    float* ob = reinterpret_cast<float*>(p.out) + static_cast<size_t>(b) * p.Lq * p.ldo + h * HD + 2 * (lane & 3);
#pragma unroll
    for (int nt = 0; nt < NT_O; ++nt) {
      if (r0 < p.Lq)
        *reinterpret_cast<float2*>(ob + static_cast<size_t>(r0) * p.ldo + nt * 8) = make_float2(round_tf32(o[nt][0] * inv0), round_tf32(o[nt][1] * inv0));
      if (r1 < p.Lq)
        *reinterpret_cast<float2*>(ob + static_cast<size_t>(r1) * p.ldo + nt * 8) = make_float2(round_tf32(o[nt][2] * inv1), round_tf32(o[nt][3] * inv1));
    }
    return;
  }
  __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<size_t>(b) * p.Lq * p.ldo + h * HD + 2 * (lane & 3);
#pragma unroll
  for (int nt = 0; nt < NT_O; ++nt) {
    if (r0 < p.Lq)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(r0) * p.ldo + nt * 8) =
          pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
    if (r1 < p.Lq)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(r1) * p.ldo + nt * 8) =
          pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
  }
}

// Single-tile specialisation for Lq, Lk <= 64 (the 1-second clips: T = 63, N = 50), bf16, head dim 64: no online-softmax
// state, Q fragments re-read from shared memory per k-step, so the kernel fits 72 registers and seven CTAs per SM -
// the B*H = 1024 CTAs of a B = 256 launch then run as one wave instead of two (the generic kernel needs 128 registers).
template <bool LERP>
__global__ void __launch_bounds__(128, 7) attention_small_kernel(const AttnDev p) {
  constexpr int HD = 64, LDS = HD + 8, KS = HD / 16, NT_O = HD / 8;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* sK = sQ + QT * LDS;
  __nv_bfloat16* sV = sK + KT * LDS;
  griddep_launch_dependents();
  griddep_wait();
  const int h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const UttKeys uk = utt_keys<LERP>(p, b);
  {
    const __nv_bfloat16* qsrc = reinterpret_cast<const __nv_bfloat16*>(p.q) + static_cast<size_t>(b) * p.Lq * p.ldq + h * HD;
    load_tile_bf16<HD>(sQ, qsrc, p.ldq, 0, p.Lq);
    if constexpr (LERP) {
      const float* ksrc = reinterpret_cast<const float*>(p.k) + static_cast<size_t>(b) * p.nsrc * p.ldkv + h * HD;
      const float* vsrc = reinterpret_cast<const float*>(p.v) + static_cast<size_t>(b) * p.nsrc * p.ldkv + h * HD;
      load_tile_lerp<HD>(sK, ksrc, p.ldkv, 0, uk.lk, uk.nsrc, uk.scale);
      load_tile_lerp<HD>(sV, vsrc, p.ldkv, 0, uk.lk, uk.nsrc, uk.scale);
    } else {
      const __nv_bfloat16* ksrc = reinterpret_cast<const __nv_bfloat16*>(p.k) + static_cast<size_t>(b) * p.Lk * p.ldkv + h * HD;
      const __nv_bfloat16* vsrc = reinterpret_cast<const __nv_bfloat16*>(p.v) + static_cast<size_t>(b) * p.Lk * p.ldkv + h * HD;
      load_tile_bf16<HD>(sK, ksrc, p.ldkv, 0, uk.lk);
      load_tile_bf16<HD>(sV, vsrc, p.ldkv, 0, uk.lk);
    }
  }
  __syncthreads();
  // ---- S = Q K^T (16 x 64 per warp) ----
  float s[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    uint32_t qf[4];
    ldmatrix_x4(qf, smem_u32(sQ + (warp * 16 + (lane & 15)) * LDS + ks * 16 + (lane >> 4) * 8));
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bf[4];
      ldmatrix_x4(bf, smem_u32(sK + (np * 16 + ((lane >> 4) << 3) + (lane & 7)) * LDS + ks * 16 + ((lane >> 3) & 1) * 8));
      mma_bf16_16816(s[2 * np], qf, bf[0], bf[1]);
      mma_bf16_16816(s[2 * np + 1], qf, bf[2], bf[3]);
    }
  }
  // ---- softmax over the (single) tile ----
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int c = nt * 8 + 2 * (lane & 3);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float val = (c + (e & 1)) < uk.lk ? s[nt][e] * p.scale_log2 : -INFINITY;
      s[nt][e] = val;
      if (e < 2) mx0 = fmaxf(mx0, val); else mx1 = fmaxf(mx1, val);
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float l0 = 0.f, l1 = 0.f;
  uint32_t pf[4][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const float p0 = exp2f(s[nt][0] - mx0), p1 = exp2f(s[nt][1] - mx0);
    const float p2 = exp2f(s[nt][2] - mx1), p3 = exp2f(s[nt][3] - mx1);
    l0 += p0 + p1; l1 += p2 + p3;
    pf[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16x2(p0, p1);
    pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p2, p3);
  }
  // ---- O = P V ----
  float o[NT_O][4];
#pragma unroll
  for (int i = 0; i < NT_O; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int np = 0; np < NT_O / 2; ++np) {
      uint32_t bf[4];
      ldmatrix_x4_trans(bf, smem_u32(sV + (ks * 16 + ((lane >> 3) & 1) * 8 + (lane & 7)) * LDS + np * 16 + (lane >> 4) * 8));
      mma_bf16_16816(o[2 * np], pf[ks], bf[0], bf[1]);
      mma_bf16_16816(o[2 * np + 1], pf[ks], bf[2], bf[3]);
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
  const int r0 = warp * 16 + (lane >> 2), r1 = r0 + 8;
  __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<size_t>(b) * p.Lq * p.ldo + h * HD + 2 * (lane & 3);
#pragma unroll
  for (int nt = 0; nt < NT_O; ++nt) {
    if (r0 < p.Lq)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(r0) * p.ldo + nt * 8) = pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
    if (r1 < p.Lq)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(r1) * p.ldo + nt * 8) = pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
  }
}

template <bool LERP>
const char* launch_small(cudaStream_t s, const AttnDev& d, int B, int H) {
  constexpr int SMEM = 3 * 64 * (64 + 8) * 2;
  dim3 grid(1, H, B);
  if (launch_pdl(attention_small_kernel<LERP>, grid, dim3(128), SMEM, s, d) != cudaSuccess) {
    cudaGetLastError();
    return "attention: launch failed";
  }
  return nullptr;
}

template <int HD, bool LERP, bool SPLIT>
const char* launch_t(cudaStream_t s, const AttnDev& d, int B, int H, int Lq) {
  constexpr int SMEM = (SPLIT ? 6 : 3) * 64 * (HD + 8) * 2;
  auto kern = attention_kernel<HD, LERP, SPLIT>;
  if (!smem_opt_in(kern, SMEM)) return "attention: cudaFuncSetAttribute failed";
  dim3 grid((Lq + QT - 1) / QT, H, B);
  if (launch_pdl(kern, grid, dim3(128), SMEM, s, d) != cudaSuccess) {
    cudaGetLastError();
    return "attention: launch failed";
  }
  return nullptr;
}

}  // namespace

// tc_mode 1: the tcgen05 kernel takes sequences this long or longer on both sides; shorter ones stay on mma.sync.
constexpr int ATTN_TC_MIN_LEN = 96;

bool attention_tc_wanted(int prec, const AttnProblem& p) {
  if (p.tc_mode == 0 || !attention_tc_usable(prec, p)) return false;
  return p.tc_mode == 2 || (p.Lq < p.Lk ? p.Lq : p.Lk) >= ATTN_TC_MIN_LEN;
}

const char* launch_attention(cudaStream_t s, int prec, const AttnProblem& p) {
  if (p.B <= 0 || p.Lq <= 0 || p.Lk <= 0) return "attention: empty problem";
  if (attention_tc_wanted(prec, p)) return launch_attention_tc(s, p);
  const bool split = (prec == PREC_TF32);     // fp32 operands, bf16 hi/lo split contractions, fp32 output
  AttnDev d;
  d.q = p.q;
  d.k = p.k; d.v = p.v;
  d.out = p.out;
  d.ldq = p.ldq; d.ldkv = p.ldkv; d.ldo = p.ldo;
  d.H = p.H; d.Lq = p.Lq; d.Lk = p.Lk; d.nsrc = p.lerp_src;
  d.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(p.hd));
  d.lerp_scale = p.lerp_src > 0 ? static_cast<float>(p.lerp_src) / static_cast<float>(p.Lk) : 0.f;
  d.k_lens = p.k_lens; d.src_lens = p.lerp_src > 0 ? p.src_lens : nullptr;
  const bool lerp = p.lerp_src > 0;
  if (split) {
    if ((p.ldq & 3) || (p.ldo & 1) || (p.ldkv & 3)) return "attention: misaligned leading dimension";
  } else {
    if (p.hd == 64 && p.Lq <= QT && p.Lk <= KT && !(p.ldq & 7) && !(p.ldo & 1) && !(lerp ? (p.ldkv & 3) : (p.ldkv & 7)))
      return lerp ? launch_small<true>(s, d, p.B, p.H) : launch_small<false>(s, d, p.B, p.H);
  }
  if (!split) {
    if ((p.ldq & 7) || (p.ldo & 1) || (lerp ? (p.ldkv & 3) : (p.ldkv & 7))) return "attention: misaligned leading dimension";
  }
#define AVSEP_ATTN_CASE(HDV)                                                                              \
  case HDV:                                                                                               \
    if (split) return lerp ? launch_t<HDV, true, true>(s, d, p.B, p.H, p.Lq) : launch_t<HDV, false, true>(s, d, p.B, p.H, p.Lq); \
    return lerp ? launch_t<HDV, true, false>(s, d, p.B, p.H, p.Lq) : launch_t<HDV, false, false>(s, d, p.B, p.H, p.Lq);
  switch (p.hd) {
    AVSEP_ATTN_CASE(16)
    AVSEP_ATTN_CASE(32)
    AVSEP_ATTN_CASE(64)
    AVSEP_ATTN_CASE(128)
    default: return "attention: head dim must be 16, 32, 64 or 128";
  }
#undef AVSEP_ATTN_CASE
}

}  // namespace avsep
