// VisualEncoder.conv (model.py:81-92,106-107) as ONE fused kernel per group of frames:
//   Conv2d(1->32,k3,s2,p1)+BN+ReLU -> Conv2d(32->64,...)+BN+ReLU -> Conv2d(64->128,...)+BN+ReLU -> global mean.
// BatchNorm (eval: running statistics, eps 1e-5) is folded into the conv weights/bias on the host at weight
// finalisation.  Each conv is an implicit GEMM on tensor cores (bf16 operands, fp32 accumulation):
//   rows = output pixels of the frames in the group, cols = output channels, K = 3*3*Cin (tap-major),
// the A operand is gathered straight from the previous stage's activations in shared memory (no im2col buffer),
// the B operand (weights) is pre-packed on the host in mma-fragment order so that every load is one conflict-free
// 8-byte access per lane.  Intermediate activations never leave the SM; HBM traffic is the 4 KB frame in and the
// 256 B pooled feature row out.
#include "common.cuh"
#include "kernels.h"

#include <math.h>
#include <string.h>

#include <vector>

namespace avsep {

namespace {

constexpr int CNN_THREADS = 256;
constexpr int C1 = 32, C2 = 64, C3 = 128;
constexpr int A1_PIX_WORDS = 18;   // 32 ch bf16 = 16 words + 2 pad: stride-2 pixel gathers hit distinct banks
constexpr int A2_PIX_WORDS = 34;   // 64 ch bf16 = 32 words + 2 pad
constexpr int W2_WORDS = 18 * 8 * 64;    // [k-step 18][n-tile 8][lane 32][2]
constexpr int W3_WORDS = 36 * 16 * 64;   // [k-step 36][n-tile 16][lane 32][2]
constexpr int W1_WORDS = 4 * 64;         // [n-tile 4][lane 32][2]

struct CnnDev {
  const float* frames;
  void* pooled;
  const uint32_t* w1; const float* b1;
  const uint32_t* w2; const float* b2;
  const uint32_t* w3; const float* b3;
  const uint32_t *w1l, *w2l, *w3l;   // lo parts (w - bf16(w)) for the fp32-grade split path
  int M, H, W, H1, W1, H2, W2, H3, W3, G, num_groups;
  const int* frame_lens;             // variable-length batch: frames past an utterance's length are staged as zeros
  int N;                             // frames per utterance (pitch of frame_lens)
};

// Gather state for one accumulator row of a stride-2 / pad-1 3x3 conv: top-left input coordinate and frame base.
struct RowRef {
  int base;   // word offset of the frame's activation block (or -1 when the row does not exist)
  int y0, x0; // input coordinate of tap (0,0)
};

__device__ __forceinline__ RowRef make_rowref(int r, int rows_total, int Ho, int Wo, int frame_words) {
  RowRef rr;
  if (r >= rows_total) { rr.base = -1; rr.y0 = 0; rr.x0 = 0; return rr; }
  const int per = Ho * Wo;
  const int g = r / per;
  const int rem = r - g * per;
  const int y = rem / Wo;
  const int x = rem - y * Wo;
  rr.base = g * frame_words;
  rr.y0 = 2 * y - 1;
  rr.x0 = 2 * x - 1;
  return rr;
}

__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// SPLIT = fp32-grade path: activations and weights are carried as bf16 hi + lo pairs and every contraction is three
// tensor-core products (hi*hi + lo*hi + hi*lo); the pooled output is fp32.
template <bool SPLIT>
__global__ void __launch_bounds__(CNN_THREADS, 1) visual_cnn_kernel(const CnnDev p) {
  extern __shared__ __align__(16) uint8_t smem_cnn[];
  const int Hp = p.H + 2, Wp = p.W + 2;
  const int in_words = Hp * Wp;
  const int a1_words = p.H1 * p.W1 * A1_PIX_WORDS;
  const int a2_words = p.H2 * p.W2 * A2_PIX_WORDS;
  uint32_t* sW2 = reinterpret_cast<uint32_t*>(smem_cnn);
  uint32_t* sW1 = sW2 + W2_WORDS;
  float* sB1 = reinterpret_cast<float*>(sW1 + W1_WORDS);
  float* sB2 = sB1 + C1;
  float* sB3 = sB2 + C2;
  float* sPool = sB3 + C3;                                   // [G][128]
  float* sIn = sPool + p.G * C3;                              // [G][Hp][Wp] fp32, zero border
  uint32_t* sA1 = reinterpret_cast<uint32_t*>(sIn + p.G * in_words);   // [G][H1][W1][18 words]
  uint32_t* sA2 = sA1 + p.G * a1_words;                        // [G][H2][W2][34 words]
  // lo halves (SPLIT only)
  uint32_t* sA1l = sA2 + p.G * a2_words;
  uint32_t* sA2l = sA1l + p.G * a1_words;
  uint32_t* sW2l = sA2l + p.G * a2_words;
  uint32_t* sW1l = sW2l + W2_WORDS;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int gid = lane >> 2, tig = lane & 3;

  for (int i = tid; i < W2_WORDS; i += CNN_THREADS) sW2[i] = p.w2[i];
  for (int i = tid; i < W1_WORDS; i += CNN_THREADS) sW1[i] = p.w1[i];
  if constexpr (SPLIT) {
    for (int i = tid; i < W2_WORDS; i += CNN_THREADS) sW2l[i] = p.w2l[i];
    for (int i = tid; i < W1_WORDS; i += CNN_THREADS) sW1l[i] = p.w1l[i];
  }
  for (int i = tid; i < C1; i += CNN_THREADS) sB1[i] = p.b1[i];
  for (int i = tid; i < C2; i += CNN_THREADS) sB2[i] = p.b2[i];
  for (int i = tid; i < C3; i += CNN_THREADS) sB3[i] = p.b3[i];
  for (int i = tid; i < p.G * C3; i += CNN_THREADS) sPool[i] = 0.f;
  for (int i = tid; i < p.G * in_words; i += CNN_THREADS) sIn[i] = 0.f;
  __syncthreads();

  const int R1 = p.G * p.H1 * p.W1, R2 = p.G * p.H2 * p.W2, R3 = p.G * p.H3 * p.W3;
  const float inv_pool = 1.0f / static_cast<float>(p.H3 * p.W3);

  for (int grp = blockIdx.x; grp < p.num_groups; grp += gridDim.x) {
    const int frame0 = grp * p.G;
    // ---- stage input frames (interior of the zero-bordered tiles) ----
    {
      const int per = p.H * p.W;
      for (int i = tid; i < p.G * per; i += CNN_THREADS) {
        const int g = i / per;
        const int rem = i - g * per;
        const int y = rem / p.W, x = rem - y * p.W;
        const int fr = frame0 + g;
        const float val = fr < p.M && frame_live(p.frame_lens, p.N, fr) ? __ldg(p.frames + static_cast<size_t>(fr) * per + rem) : 0.f;
        sIn[g * in_words + (y + 1) * Wp + (x + 1)] = val;
      }
    }
    __syncthreads();

    // ---- conv1: K = 9 taps padded to 16, N = 32 ----
    {
      uint32_t bw[4][2], bwl[4][2];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        bw[nt][0] = sW1[nt * 64 + lane * 2];
        bw[nt][1] = sW1[nt * 64 + lane * 2 + 1];
        bwl[nt][0] = SPLIT ? sW1l[nt * 64 + lane * 2] : 0u;
        bwl[nt][1] = SPLIT ? sW1l[nt * 64 + lane * 2 + 1] : 0u;
      }
      const int k0 = 2 * tig, k1 = 2 * tig + 1;           // taps handled by this lane (k < 8)
      const int off0 = (k0 / 3) * Wp + (k0 % 3);
      const int off1 = (k1 / 3) * Wp + (k1 % 3);
      const int off8 = 2 * Wp + 2;                         // tap 8
      const int tiles = (R1 + 15) / 16;
      for (int t = warp; t < tiles; t += CNN_THREADS / 32) {
        uint32_t a[4] = {0, 0, 0, 0}, al[4] = {0, 0, 0, 0};
        int pix[2];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const int r = t * 16 + gid + 8 * hf;
          pix[hf] = -1;
          if (r < R1) {
            const int per = p.H1 * p.W1;
            const int g = r / per;
            const int rem = r - g * per;
            const int y = rem / p.W1, x = rem - y * p.W1;
            pix[hf] = r;
            const float* base = sIn + g * in_words + (2 * y) * Wp + 2 * x;
            const float v0 = base[off0], v1 = base[off1];
            a[hf] = pack_bf16x2(v0, v1);
            if constexpr (SPLIT) al[hf] = pack_bf16x2(v0 - bf16_round(v0), v1 - bf16_round(v1));
            if (tig == 0) {
              const float v8 = base[off8];
              a[2 + hf] = pack_bf16x2(v8, 0.f);
              if constexpr (SPLIT) al[2 + hf] = pack_bf16x2(v8 - bf16_round(v8), 0.f);
            }
          }
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          float c[4] = {0.f, 0.f, 0.f, 0.f};
          mma_bf16_16816(c, a[0], a[1], a[2], a[3], bw[nt][0], bw[nt][1]);
          if constexpr (SPLIT) {
            mma_bf16_16816(c, al[0], al[1], al[2], al[3], bw[nt][0], bw[nt][1]);
            mma_bf16_16816(c, a[0], a[1], a[2], a[3], bwl[nt][0], bwl[nt][1]);
          }
          const int ch = nt * 8 + 2 * tig;
          const float bb0 = sB1[ch], bb1 = sB1[ch + 1];
          const float o0 = fmaxf(c[0] + bb0, 0.f), o1 = fmaxf(c[1] + bb1, 0.f);
          const float o2 = fmaxf(c[2] + bb0, 0.f), o3 = fmaxf(c[3] + bb1, 0.f);
          if (pix[0] >= 0) {
            sA1[pix[0] * A1_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o0, o1);
            if constexpr (SPLIT) sA1l[pix[0] * A1_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o0 - bf16_round(o0), o1 - bf16_round(o1));
          }
          if (pix[1] >= 0) {
            sA1[pix[1] * A1_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o2, o3);
            if constexpr (SPLIT) sA1l[pix[1] * A1_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o2 - bf16_round(o2), o3 - bf16_round(o3));
          }
        }
      }
    }
    __syncthreads();

    // ---- conv2: K = 9 taps x 32 ch (18 k-steps), N = 64; work item = 2 m-tiles x 4 n-tiles ----
    {
      const int mpairs = (R2 + 31) / 32;
      const int items = mpairs * 2;
      for (int it = warp; it < items; it += CNN_THREADS / 32) {
        const int mp = it >> 1, ng = it & 1;
        RowRef rr[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          rr[j] = make_rowref(mp * 32 + (j >> 1) * 16 + gid + 8 * (j & 1), R2, p.H2, p.W2, a1_words);
        float acc[2][4][4];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = acc[a][b][2] = acc[a][b][3] = 0.f;
        for (int tap = 0; tap < 9; ++tap) {
          const int ky = tap / 3, kx = tap - ky * 3;
          int off[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int yy = rr[j].y0 + ky, xx = rr[j].x0 + kx;
            const bool ok = rr[j].base >= 0 && yy >= 0 && yy < p.H1 && xx >= 0 && xx < p.W1;
            off[j] = ok ? rr[j].base + (yy * p.W1 + xx) * A1_PIX_WORDS + tig : -1;
          }
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int ks = tap * 2 + half;
            uint32_t af[2][4], afl[2][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
              const int o0 = off[mt * 2], o1 = off[mt * 2 + 1];
              af[mt][0] = o0 >= 0 ? sA1[o0 + half * 8] : 0u;
              af[mt][1] = o1 >= 0 ? sA1[o1 + half * 8] : 0u;
              af[mt][2] = o0 >= 0 ? sA1[o0 + half * 8 + 4] : 0u;
              af[mt][3] = o1 >= 0 ? sA1[o1 + half * 8 + 4] : 0u;
              if constexpr (SPLIT) {
                afl[mt][0] = o0 >= 0 ? sA1l[o0 + half * 8] : 0u;
                afl[mt][1] = o1 >= 0 ? sA1l[o1 + half * 8] : 0u;
                afl[mt][2] = o0 >= 0 ? sA1l[o0 + half * 8 + 4] : 0u;
                afl[mt][3] = o1 >= 0 ? sA1l[o1 + half * 8 + 4] : 0u;
              }
            }
#pragma unroll
            for (int n = 0; n < 4; ++n) {
              const uint2 bw = *reinterpret_cast<const uint2*>(sW2 + (ks * 8 + ng * 4 + n) * 64 + lane * 2);
              mma_bf16_16816(acc[0][n], af[0][0], af[0][1], af[0][2], af[0][3], bw.x, bw.y);
              mma_bf16_16816(acc[1][n], af[1][0], af[1][1], af[1][2], af[1][3], bw.x, bw.y);
              if constexpr (SPLIT) {
                const uint2 bl = *reinterpret_cast<const uint2*>(sW2l + (ks * 8 + ng * 4 + n) * 64 + lane * 2);
                mma_bf16_16816(acc[0][n], afl[0][0], afl[0][1], afl[0][2], afl[0][3], bw.x, bw.y);
                mma_bf16_16816(acc[1][n], afl[1][0], afl[1][1], afl[1][2], afl[1][3], bw.x, bw.y);
                mma_bf16_16816(acc[0][n], af[0][0], af[0][1], af[0][2], af[0][3], bl.x, bl.y);
                mma_bf16_16816(acc[1][n], af[1][0], af[1][1], af[1][2], af[1][3], bl.x, bl.y);
              }
            }
          }
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
          for (int n = 0; n < 4; ++n) {
            const int ch = (ng * 4 + n) * 8 + 2 * tig;
            const float bb0 = sB2[ch], bb1 = sB2[ch + 1];
            const int r0 = mp * 32 + mt * 16 + gid, r1 = r0 + 8;
            const float o0 = fmaxf(acc[mt][n][0] + bb0, 0.f), o1 = fmaxf(acc[mt][n][1] + bb1, 0.f);
            const float o2 = fmaxf(acc[mt][n][2] + bb0, 0.f), o3 = fmaxf(acc[mt][n][3] + bb1, 0.f);
            if (r0 < R2) {
              sA2[r0 * A2_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o0, o1);
              if constexpr (SPLIT) sA2l[r0 * A2_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o0 - bf16_round(o0), o1 - bf16_round(o1));
            }
            if (r1 < R2) {
              sA2[r1 * A2_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o2, o3);
              if constexpr (SPLIT) sA2l[r1 * A2_PIX_WORDS + (ch >> 1)] = pack_bf16x2(o2 - bf16_round(o2), o3 - bf16_round(o3));
            }
          }
        }
      }
    }
    __syncthreads();

    // ---- conv3: K = 9 taps x 64 ch (36 k-steps), N = 128; work item = 4 m-tiles x 2 n-tiles; mean pool ----
    {
      const int mquads = (R3 + 63) / 64;
      const int items = mquads * 8;
      const int per3 = p.H3 * p.W3;
      for (int it = warp; it < items; it += CNN_THREADS / 32) {
        const int mq = it >> 3, np = it & 7;
        RowRef rr[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          rr[j] = make_rowref(mq * 64 + (j >> 1) * 16 + gid + 8 * (j & 1), R3, p.H3, p.W3, a2_words);
        float acc[4][2][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 2; ++b) acc[a][b][0] = acc[a][b][1] = acc[a][b][2] = acc[a][b][3] = 0.f;
        const uint2* wbase = reinterpret_cast<const uint2*>(p.w3) + lane;
        const uint2* wbase_l = reinterpret_cast<const uint2*>(SPLIT ? p.w3l : p.w3) + lane;
        for (int tap = 0; tap < 9; ++tap) {
          const int ky = tap / 3, kx = tap - ky * 3;
          int off[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int yy = rr[j].y0 + ky, xx = rr[j].x0 + kx;
            const bool ok = rr[j].base >= 0 && yy >= 0 && yy < p.H2 && xx >= 0 && xx < p.W2;
            off[j] = ok ? rr[j].base + (yy * p.W2 + xx) * A2_PIX_WORDS + tig : -1;
          }
          uint2 bw[4][2];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int ks = tap * 4 + q;
            bw[q][0] = __ldg(wbase + (ks * 16 + np * 2) * 32);
            bw[q][1] = __ldg(wbase + (ks * 16 + np * 2 + 1) * 32);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) {
              const int o0 = off[mt * 2], o1 = off[mt * 2 + 1];
              const uint32_t a0 = o0 >= 0 ? sA2[o0 + q * 8] : 0u;
              const uint32_t a1 = o1 >= 0 ? sA2[o1 + q * 8] : 0u;
              const uint32_t a2 = o0 >= 0 ? sA2[o0 + q * 8 + 4] : 0u;
              const uint32_t a3 = o1 >= 0 ? sA2[o1 + q * 8 + 4] : 0u;
              mma_bf16_16816(acc[mt][0], a0, a1, a2, a3, bw[q][0].x, bw[q][0].y);
              mma_bf16_16816(acc[mt][1], a0, a1, a2, a3, bw[q][1].x, bw[q][1].y);
              if constexpr (SPLIT) {
                const uint32_t l0 = o0 >= 0 ? sA2l[o0 + q * 8] : 0u;
                const uint32_t l1 = o1 >= 0 ? sA2l[o1 + q * 8] : 0u;
                const uint32_t l2 = o0 >= 0 ? sA2l[o0 + q * 8 + 4] : 0u;
                const uint32_t l3 = o1 >= 0 ? sA2l[o1 + q * 8 + 4] : 0u;
                mma_bf16_16816(acc[mt][0], l0, l1, l2, l3, bw[q][0].x, bw[q][0].y);
                mma_bf16_16816(acc[mt][1], l0, l1, l2, l3, bw[q][1].x, bw[q][1].y);
                const int ksl = tap * 4 + q;
                const uint2 wl0 = __ldg(wbase_l + (ksl * 16 + np * 2) * 32);
                const uint2 wl1 = __ldg(wbase_l + (ksl * 16 + np * 2 + 1) * 32);
                mma_bf16_16816(acc[mt][0], a0, a1, a2, a3, wl0.x, wl0.y);
                mma_bf16_16816(acc[mt][1], a0, a1, a2, a3, wl1.x, wl1.y);
              }
            }
          }
        }
        // bias + ReLU + mean over the frame's H3 x W3 pixels
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          const int rbase = mq * 64 + mt * 16;
          const bool uniform = (per3 % 16 == 0) && (rbase + 16 <= R3);   // all 16 rows belong to one frame
#pragma unroll
          for (int n = 0; n < 2; ++n) {
            const int ch = (np * 2 + n) * 8 + 2 * tig;
            const float bb0 = sB3[ch], bb1 = sB3[ch + 1];
            float v0 = fmaxf(acc[mt][n][0] + bb0, 0.f), v1 = fmaxf(acc[mt][n][1] + bb1, 0.f);
            float v2 = fmaxf(acc[mt][n][2] + bb0, 0.f), v3 = fmaxf(acc[mt][n][3] + bb1, 0.f);
            if (uniform) {
              float s0 = v0 + v2, s1 = v1 + v3;
#pragma unroll
              for (int o = 4; o < 32; o <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
              }
              if (gid == 0) {
                const int g = rbase / per3;
                atomicAdd(&sPool[g * C3 + ch], s0);
                atomicAdd(&sPool[g * C3 + ch + 1], s1);
              }
            } else {
              const int r0 = rbase + gid, r1 = r0 + 8;
              if (r0 < R3) {
                atomicAdd(&sPool[(r0 / per3) * C3 + ch], v0);
                atomicAdd(&sPool[(r0 / per3) * C3 + ch + 1], v1);
              }
              if (r1 < R3) {
                atomicAdd(&sPool[(r1 / per3) * C3 + ch], v2);
                atomicAdd(&sPool[(r1 / per3) * C3 + ch + 1], v3);
              }
            }
          }
        }
      }
    }
    __syncthreads();

    // ---- pooled features out (operand precision), reset the pool accumulators ----
    for (int i = tid; i < p.G * C3; i += CNN_THREADS) {
      const int g = i / C3;
      const int fr = frame0 + g;
      const float val = sPool[i] * inv_pool;
      sPool[i] = 0.f;
      if (fr < p.M) {
        if constexpr (SPLIT) reinterpret_cast<float*>(p.pooled)[static_cast<size_t>(fr) * C3 + (i - g * C3)] = round_tf32(val);
        else reinterpret_cast<__nv_bfloat16*>(p.pooled)[static_cast<size_t>(fr) * C3 + (i - g * C3)] =
            __float2bfloat16_rn(val);
      }
    }
    // sIn interior is overwritten and sA1/sA2 fully rewritten next round; the barrier after staging orders it.
  }
}

// Pack a [N][K] fp32 matrix into mma.m16n8k16 B-fragment order: [k-step][n-tile][lane][2 words].
void pack_frag(const float* w_in, int N, int K, int Kpad, uint32_t* out, bool lo_part) {
  std::vector<float> tmp;
  const float* w = w_in;
  if (lo_part) {      // residual after bf16 rounding
    tmp.resize(static_cast<size_t>(N) * K);
    for (size_t i = 0; i < tmp.size(); ++i) {
      const uint32_t hb = static_cast<uint32_t>(f2bf(w_in[i])) << 16;
      float hf;
      memcpy(&hf, &hb, 4);
      tmp[i] = w_in[i] - hf;
    }
    w = tmp.data();
  }
  const int ksteps = Kpad / 16, ntiles = N / 8;
  for (int ks = 0; ks < ksteps; ++ks)
    for (int nt = 0; nt < ntiles; ++nt)
      for (int lane = 0; lane < 32; ++lane) {
        const int n = nt * 8 + lane / 4;
        const int k0 = ks * 16 + 2 * (lane % 4);
        auto at = [&](int k) { return k < K ? w[static_cast<size_t>(n) * K + k] : 0.f; };
        uint32_t* o = out + ((static_cast<size_t>(ks) * ntiles + nt) * 32 + lane) * 2;
        o[0] = static_cast<uint32_t>(f2bf(at(k0))) | (static_cast<uint32_t>(f2bf(at(k0 + 1))) << 16);
        o[1] = static_cast<uint32_t>(f2bf(at(k0 + 8))) | (static_cast<uint32_t>(f2bf(at(k0 + 9))) << 16);
      }
}

}  // namespace

size_t visual_cnn_pack_sizes(int which) { return which == 1 ? W1_WORDS : which == 2 ? W2_WORDS : W3_WORDS; }

// w1 [32][9], w2 [64][9*32], w3 [128][9*64] fp32, already BN-folded, K index = tap*Cin + c.
void visual_cnn_pack(const float* w1, const float* w2, const float* w3, uint32_t* p1, uint32_t* p2, uint32_t* p3,
                     bool lo_part) {
  pack_frag(w1, C1, 9, 16, p1, lo_part);
  pack_frag(w2, C2, 9 * C1, 9 * C1, p2, lo_part);
  pack_frag(w3, C3, 9 * C2, 9 * C2, p3, lo_part);
}

const char* launch_visual_cnn(cudaStream_t s, int prec, const float* frames, int M, int H, int W, const CnnWeights& w,
                              void* pooled, int num_sms, const int* frame_lens, int N) {
  if (M <= 0 || H <= 0 || W <= 0) return "visual_cnn: empty problem";
  CnnDev d;
  d.frames = frames; d.pooled = pooled;
  d.frame_lens = frame_lens; d.N = N;
  d.w1 = w.w1; d.b1 = w.b1; d.w2 = w.w2; d.b2 = w.b2; d.w3 = w.w3; d.b3 = w.b3;
  d.w1l = w.w1l; d.w2l = w.w2l; d.w3l = w.w3l;
  const bool split = (prec == PREC_TF32);
  const size_t mul = split ? 2 : 1;
  d.M = M; d.H = H; d.W = W;
  d.H1 = (H + 1) / 2; d.W1 = (W + 1) / 2;
  d.H2 = (d.H1 + 1) / 2; d.W2 = (d.W1 + 1) / 2;
  d.H3 = (d.H2 + 1) / 2; d.W3 = (d.W2 + 1) / 2;
  const size_t fixed = (mul * (W2_WORDS + W1_WORDS) + C1 + C2 + C3) * 4;
  const size_t per_frame = static_cast<size_t>((H + 2) * (W + 2) + mul * (d.H1 * d.W1 * A1_PIX_WORDS +
                                               d.H2 * d.W2 * A2_PIX_WORDS) + C3) * 4;
  const size_t cap = 227 * 1024;
  if (fixed + per_frame > cap) return "visual_cnn: frame too large for the fused kernel (shared memory)";
  int G = static_cast<int>((cap - fixed) / per_frame);
  if (G > 4) G = 4;
  d.G = G;
  d.num_groups = (M + G - 1) / G;
  const size_t smem = fixed + per_frame * G;
  auto kern = split ? visual_cnn_kernel<true> : visual_cnn_kernel<false>;
  if (!smem_opt_in(kern, static_cast<int>(cap))) return "visual_cnn: cannot raise the shared-memory limit";
  const int grid = d.num_groups < num_sms ? d.num_groups : num_sms;
  kern<<<grid, CNN_THREADS, smem, s>>>(d);
  return cudaGetLastError() == cudaSuccess ? nullptr : "visual_cnn: launch failed";
}

}  // namespace avsep
