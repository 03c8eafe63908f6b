// Fused feed-forward sub-layer for d_model = 256 (hidden = 1024), bf16 operands:
//
//   x' = x + W2 * act(W1 * a + b1) + b2 ;   out = LayerNorm_{gamma,beta}(x')        (a = LayerNorm output, bf16)
//
// i.e. TransformerEncoderLayer's linear1 -> ReLU -> linear2 -> +residual (torch transformer.py:946-950) and
// CrossAttentionLayer.ff (Linear -> GELU -> Linear, model.py:156-161,172) together with the LayerNorm that follows.
// The 4d hidden activation never leaves the SM.
//
// One CTA per 128-row tile (persistent over tiles), 576 threads:
//   warp 0 / lane 0 : TMA producer - A tile (4 k-slabs, loaded once per tile) and an 8-slot ring of 16 KB weight slabs
//   warp 1 / lane 0 : MMA issuer   - per hidden chunk j (128 columns):
//                        GEMM1_j : acc1[j&1] (TMEM, 128 cols)  = A (K=256) x W1[j]            (4 k-slabs, N=128)
//                        GEMM2_j : acc2 (TMEM, 256 cols)      += H_j (K=128, A operand read from TMEM) x W2[:, j]
//                                                                                             (2 k-slabs, N=256)
//                     software-pipelined (G1_0, G1_1, G2_0, G1_2, G2_1, ...) so the tensor pipe stays busy while
//                     the epilogue warps convert chunk j
//   warps 2..17     : epilogue-1  - tcgen05.ld acc1 -> +b1 -> ReLU / erf-GELU -> bf16 pairs -> tcgen05.st back into
//                                   the first 64 columns of the same accumulator stage (H never touches shared
//                                   memory: the kernel is bound by shared-memory bandwidth - UMMA operand reads plus
//                                   TMA fills - so GEMM2 reads only its weights from smem),
//                     epilogue-2  - acc2 + b2 + residual (TMA slab) -> x' (TMA store) -> LayerNorm -> bf16 (TMA store)
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

constexpr int D = 256, HID = 1024, CHUNK = 128, NCHUNK = HID / CHUNK;
constexpr int SLAB = 128 * 128;                       // 128 rows x 128 B
constexpr int WSLOTS = 8;                             // even: the two 128-row halves of a W2 k-slab sit in adjacent slots
constexpr int OFF_A = 0;                              // 4 slabs  (A tile, K = 256)
constexpr int OFF_W = OFF_A + 4 * SLAB;               // 8 slabs (weight ring)
constexpr int OFF_BAR = OFF_W + WSLOTS * SLAB;        // barriers
constexpr int OFF_RED = OFF_BAR + 512;                // LN partial statistics [128 rows][4 parts] float2
constexpr int OFF_VEC = OFF_RED + 128 * 4 * 8;        // b1 [1024], b2 [256], gamma [256], beta [256]
constexpr int FFN_SMEM = OFF_VEC + (HID + 3 * D) * 4;
static_assert(FFN_SMEM <= 227 * 1024, "ffn_fused: shared memory budget exceeded");
constexpr int FFN_THREADS = 32 * 18;

struct FfnDev {
  const float *b1, *b2, *gamma, *beta;
  const float* resid;     // == x_out (in place) or null
  int M, act;
  int has_xout, has_op;
  unsigned long long* trace;   // optional [grid][64] globaltimer stamps of the CTA's first tile (debug), else null
};

#define FTRACE(slot) do { if (p.trace != nullptr && lt == 0) p.trace[blockIdx.x * 64 + (slot)] = globaltimer(); } while (0)

__global__ void __launch_bounds__(FFN_THREADS, 1)
ffn_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW1,
                 const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmX,
                 const __grid_constant__ CUtensorMap tmOp, const FfnDev p) {
  extern __shared__ __align__(1024) uint8_t smem_ffn[];
  uint8_t* const smem = smem_ffn;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* a_full = bars;                 // A tile landed
  uint64_t* a_empty = bars + 1;            // epilogue-2 (which stages in the A region) of the tile is done
  uint64_t* w_full = bars + 2;             // [5]
  uint64_t* w_empty = w_full + WSLOTS;     // [5]
  uint64_t* acc1_full = w_empty + WSLOTS;  // [2]
  uint64_t* h_full = acc1_full + 2;        // [2] H_j written into accumulator stage j&1 (16 warp arrivals); the stage is
                                           //     reused by GEMM1_{j+2}, which the in-order tensor pipe runs after GEMM2_j
  uint64_t* acc2_full = h_full + 2;        // 1
  uint64_t* acc2_empty = acc2_full + 1;    // 1 (16 warp arrivals)
  uint64_t* resid_bar = acc2_empty + 1;    // [4]
  uint64_t* resid_bar2 = resid_bar + 4;    // [4] second residual chunk, prefetched into the idle weight ring (last tile)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resid_bar2 + 4);
  float2* red = reinterpret_cast<float2*>(smem + OFF_RED);
  float* sb1 = reinterpret_cast<float*>(smem + OFF_VEC);
  float* sb2 = sb1 + HID;
  float* sgamma = sb2 + D;
  float* sbeta = sgamma + D;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (p.M + 127) / 128;
  if (threadIdx.x == 0 && p.trace != nullptr) p.trace[blockIdx.x * 64] = globaltimer();

  for (int i = threadIdx.x; i < HID; i += FFN_THREADS) sb1[i] = __ldg(p.b1 + i);
  for (int i = threadIdx.x; i < D; i += FFN_THREADS) {
    sb2[i] = __ldg(p.b2 + i);
    sgamma[i] = p.gamma ? __ldg(p.gamma + i) : 1.f;
    sbeta[i] = p.beta ? __ldg(p.beta + i) : 0.f;
  }
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmW1); tma_prefetch_desc(&tmW2);
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int i = 0; i < WSLOTS; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc1_full[i], 1);
      mbar_init(&h_full[i], 16);
    }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, 16);
    for (int i = 0; i < 4; ++i) { mbar_init(&resid_bar[i], 1); mbar_init(&resid_bar2[i], 1); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tm_acc2 = tmem_base;            // columns [0,256)
  const uint32_t tm_acc1 = tmem_base + 256;      // two stages of 128 columns
  griddep_launch_dependents();
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer ----------------
      uint32_t wn = 0;      // weight slabs issued so far
      auto load_w = [&](const CUtensorMap* tm, int c0, int c1) {
        const uint32_t slot = wn % WSLOTS, use = wn / WSLOTS;
        mbar_wait(&w_empty[slot], (use & 1) ^ 1);
        mbar_arrive_expect_tx(&w_full[slot], SLAB);
        tma_load_2d(smem + OFF_W + slot * SLAB, tm, &w_full[slot], c0, c1);
        ++wn;
      };
      int lt = 0;
      for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++lt) {
        mbar_wait(a_empty, (lt & 1) ^ 1);
        mbar_arrive_expect_tx(a_full, 4 * SLAB);
        for (int k = 0; k < 4; ++k) tma_load_2d(smem + OFF_A + k * SLAB, &tmA, a_full, k * 64, tile * 128);
        for (int j = 0; j <= NCHUNK; ++j) {
          if (j < NCHUNK)                       // W1 rows [j*128, +128), k-slab k
            for (int k = 0; k < 4; ++k) load_w(&tmW1, k * 64, j * CHUNK);
          if (j >= 1)                           // W2 rows half*128.., columns (hidden) (j-1)*128 + k*64
            for (int k = 0; k < 2; ++k)
              for (int hf = 0; hf < 2; ++hf) load_w(&tmW2, (j - 1) * CHUNK + k * 64, hf * 128);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ---------------- MMA issuer ----------------
      const uint32_t idesc = umma_idesc(1u, 128, 128);
      const uint32_t idesc2 = umma_idesc(1u, 128, 256);
      uint32_t wn = 0;
      uint32_t c1n = 0;      // GEMM1 chunks issued so far (acc1 stage = c1n & 1)
      uint32_t c2n = 0;      // GEMM2 chunks issued so far (H buffer = c2n & 1)
      auto next_w = [&]() -> uint32_t {
        const uint32_t slot = wn % WSLOTS, use = wn / WSLOTS;
        mbar_wait(&w_full[slot], use & 1);
        tc_fence_after();
        ++wn;
        return slot;
      };
      int lt = 0;
      for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++lt) {
        mbar_wait(a_full, lt & 1);
        mbar_wait(acc2_empty, (lt & 1) ^ 1);          // epilogue-2 of the previous tile has drained acc2
        tc_fence_after();
        FTRACE(1);                                     // A tile landed
        for (int j = 0; j <= NCHUNK; ++j) {
          if (j < NCHUNK) {
            // GEMM1_j -> acc1[c1n & 1]
            const uint32_t st = c1n & 1;
            const uint32_t d_tmem = tm_acc1 + st * CHUNK;
            for (int k = 0; k < 4; ++k) {
              const uint32_t slot = next_w();
              const uint64_t adesc = umma_desc_kmajor_sw128(smem_u32(smem + OFF_A + k * SLAB), 1024);
              const uint64_t bdesc = umma_desc_kmajor_sw128(smem_u32(smem + OFF_W + slot * SLAB), 1024);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16(d_tmem, adesc + 2 * kk, bdesc + 2 * kk, idesc, (k | kk) != 0 ? 1u : 0u);
              umma_commit(&w_empty[slot]);
            }
            umma_commit(&acc1_full[st]);
            FTRACE(8 + 4 * j);                               // GEMM1_j issued
            ++c1n;
          }
          if (j >= 1) {
            // GEMM2_{j-1}: acc2 += H x W2 chunk, H read from TMEM (accumulator stage of chunk j-1)
            const uint32_t st2 = c2n & 1;
            mbar_wait(&h_full[st2], (c2n >> 1) & 1);
            tc_fence_after();
            for (int k = 0; k < 2; ++k) {
              const uint32_t slot0 = next_w();
              const uint32_t slot1 = next_w();            // rows 128..255: the adjacent slot (slot0 is even)
              const uint64_t bdesc = umma_desc_kmajor_sw128(smem_u32(smem + OFF_W + slot0 * SLAB), 1024);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16_ts(tm_acc2, tm_acc1 + st2 * CHUNK + (k * 4 + kk) * 8, bdesc + 2 * kk, idesc2,
                            ((j - 1) | k | kk) != 0 ? 1u : 0u);
              umma_commit(&w_empty[slot0]);
              umma_commit(&w_empty[slot1]);
            }
            FTRACE(8 + 4 * (j - 1) + 1);                     // GEMM2_{j-1} issued
            ++c2n;
          }
        }
        umma_commit(acc2_full);
      }
    }
  } else {
    // ---------------- epilogue warps: lane quarter q = warp % 4, column part = (warp - 2) / 4 ----------------
    const int q = warp & 3, part = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const bool elected = (warp == 2 + 4 * part) && (lane == 0);
    const int part_bar = 6 + part;
    uint8_t* const slab = smem + OFF_A + part * SLAB;         // epilogue-2 staging: the A tile is dead once acc2 is complete
    uint8_t* const slab_q = slab + q * 4096;
    uint32_t c1n = 0;
    uint32_t rph = 0;
    int lt = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++lt) {
      const int m0 = tile * 128;
      // ---- epilogue-1: 8 hidden chunks ----
      for (int j = 0; j < NCHUNK; ++j, ++c1n) {
        const uint32_t st = c1n & 1, use = c1n >> 1;
        mbar_wait(&acc1_full[st], use & 1);
        tc_fence_after();
        if (threadIdx.x == 64) FTRACE(8 + 4 * j + 2);        // acc1_j ready (epilogue-1 starts)
        uint32_t v[32];
        tmem_ld_32x32b_x32(tm_acc1 + st * CHUNK + (static_cast<uint32_t>(q * 32) << 16) + part * 32, v);
        tmem_ld_wait();
        float h[32];
        const float* bj = sb1 + j * CHUNK + part * 32;
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(bj + i);
          h[i] = __uint_as_float(v[i]) + b4.x; h[i + 1] = __uint_as_float(v[i + 1]) + b4.y;
          h[i + 2] = __uint_as_float(v[i + 2]) + b4.z; h[i + 3] = __uint_as_float(v[i + 3]) + b4.w;
        }
        if (p.act == ACT_RELU) {
#pragma unroll
          for (int i = 0; i < 32; ++i) h[i] = fmaxf(h[i], 0.f);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) h[i] = gelu_bf16_grade(h[i]);   // H is rounded to bf16 next
        }
        // bf16 pairs back into the same accumulator stage: columns [16*part, +16) of the stage hold this warp's 32
        // hidden columns.  They alias fp32 columns other parts are still reading, hence the quarter-wide barrier.
        uint32_t hp[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) hp[i] = pack_bf16x2(h[2 * i], h[2 * i + 1]);
        tc_fence_before();
        named_bar_sync(10 + q, 128);
        tc_fence_after();
        tmem_st_32x32b_x16(tm_acc1 + st * CHUNK + (static_cast<uint32_t>(q * 32) << 16) + part * 16, hp);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_full[st]);
        if (threadIdx.x == 64) FTRACE(8 + 4 * j + 3);        // H_j published
      }
      // ---- epilogue-2: acc2 + b2 + residual -> x' ; LayerNorm -> operand ----
      mbar_wait(acc2_full, lt & 1);
      tc_fence_after();
      if (threadIdx.x == 64) FTRACE(2);                      // acc2 complete
      const bool row_ok = (m0 + r) < p.M;
      (void)row_ok;
      // On the CTA's last tile the weight ring is idle (every slab has been consumed): the second residual chunk is
      // fetched into ring slot `part` together with the first one instead of after the first chunk's x' store.
      const bool last_tile = tile + static_cast<int>(gridDim.x) >= m_tiles;
      uint8_t* const slab1_q = last_tile ? smem + OFF_W + part * SLAB + q * 4096 : slab_q;
      if (p.resid != nullptr && elected) {
        bulk_wait_read0();
        mbar_arrive_expect_tx(&resid_bar[part], SLAB);
        tma_load_2d(slab, &tmX, &resid_bar[part], part * 64, m0);
        if (last_tile) {
          mbar_arrive_expect_tx(&resid_bar2[part], SLAB);
          tma_load_2d(smem + OFF_W + part * SLAB, &tmX, &resid_bar2[part], part * 64 + 32, m0);
        }
      }
      float val[2][32];
      float sum = 0.f, sq = 0.f;
#pragma unroll
      for (int ci = 0; ci < 2; ++ci) {
        const int c0 = part * 64 + ci * 32;
        uint32_t v[32];
        tmem_ld_32x32b_x32(tm_acc2 + (static_cast<uint32_t>(q * 32) << 16) + c0, v);
        uint8_t* const sl_q = ci == 0 ? slab_q : slab1_q;
        if (p.resid != nullptr) {
          if (ci == 1 && last_tile) {
            mbar_wait(&resid_bar2[part], 0);
          } else {
            mbar_wait(&resid_bar[part], rph);
            rph ^= 1;
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(sb2 + c0 + i);
          val[ci][i] = __uint_as_float(v[i]) + b4.x; val[ci][i + 1] = __uint_as_float(v[i + 1]) + b4.y;
          val[ci][i + 2] = __uint_as_float(v[i + 2]) + b4.z; val[ci][i + 3] = __uint_as_float(v[i + 3]) + b4.w;
        }
        if (p.resid != nullptr) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 x4 = *reinterpret_cast<const float4*>(sl_q + sw128_off(lane, c));
            val[ci][4 * c] += x4.x; val[ci][4 * c + 1] += x4.y; val[ci][4 * c + 2] += x4.z; val[ci][4 * c + 3] += x4.w;
          }
        }
        if (p.has_xout) {
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<float4*>(sl_q + sw128_off(lane, c)) =
                make_float4(val[ci][4 * c], val[ci][4 * c + 1], val[ci][4 * c + 2], val[ci][4 * c + 3]);
          fence_proxy_async_smem();
        }
        if (p.has_xout || (p.resid != nullptr && ci == 0)) named_bar_sync(part_bar, 128);
        if (elected) {
          if (p.has_xout) {
            tma_store_2d(&tmX, sl_q - q * 4096, c0, m0);
            bulk_commit();
          }
          if (ci == 0 && p.resid != nullptr && !last_tile) {
            bulk_wait_read0();
            mbar_arrive_expect_tx(&resid_bar[part], SLAB);
            tma_load_2d(slab, &tmX, &resid_bar[part], c0 + 32, m0);
          }
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          sum += val[ci][i];
          sq = fmaf(val[ci][i], val[ci][i], sq);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc2_empty);
      if (p.gamma != nullptr) {
        const float mean_h = sum * (1.0f / 64.0f);
        const float m2 = fmaxf(sq - sum * mean_h, 0.f);
        float2* slot = red + r * 4;
        named_bar_sync(1 + q, 128);                 // previous tile's readers are done with `red`
        slot[part] = make_float2(mean_h, m2);
        named_bar_sync(1 + q, 128);
        const float2 s0 = slot[0], s1 = slot[1], s2 = slot[2], s3 = slot[3];
        const float mean = 0.25f * ((s0.x + s1.x) + (s2.x + s3.x));
        const float d0 = s0.x - mean, d1 = s1.x - mean, d2 = s2.x - mean, d3 = s3.x - mean;
        const float m2_all = (s0.y + s1.y) + (s2.y + s3.y) + 64.0f * ((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3));
        const float rstd = rsqrtf(m2_all * (1.0f / 256.0f) + 1e-5f);
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int c0 = part * 64 + ci * 32;
#pragma unroll
          for (int i = 0; i < 32; ++i) val[ci][i] = (val[ci][i] - mean) * rstd * sgamma[c0 + i] + sbeta[c0 + i];
        }
      }
      if (p.has_op) {
        if (elected) bulk_wait_read0();
        named_bar_sync(part_bar, 128);
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4 u;
            u.x = pack_bf16x2(val[ci][8 * c], val[ci][8 * c + 1]);
            u.y = pack_bf16x2(val[ci][8 * c + 2], val[ci][8 * c + 3]);
            u.z = pack_bf16x2(val[ci][8 * c + 4], val[ci][8 * c + 5]);
            u.w = pack_bf16x2(val[ci][8 * c + 6], val[ci][8 * c + 7]);
            *reinterpret_cast<uint4*>(slab_q + sw128_off(lane, ci * 4 + c)) = u;
          }
        }
        fence_proxy_async_smem();
        named_bar_sync(part_bar, 128);
        if (elected) {
          tma_store_2d(&tmOp, slab, part * 64, m0);
          bulk_commit();
          bulk_wait_read0();          // the slab (A region) is refilled by the producer for the next tile
        }
      } else {
        if (elected) bulk_wait_read0();
      }
      // all four staging slabs (= the A region) are drained: let the producer load the next tile's A
      named_bar_sync(5, 512);
      if (threadIdx.x == 64) mbar_arrive(a_empty);
      if (threadIdx.x == 64) FTRACE(3);                      // epilogue-2 done
    }
    if (elected) bulk_wait_read0();     // shared memory may be released; the stores complete with the grid
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

bool ffn_fusable(int prec, int d_model) { return prec == PREC_BF16 && d_model == D; }

// a [M,256] bf16; w1 [1024,256] bf16; w2 [256,1024] bf16; x [M,256] fp32 (residual in, x' out, in place) or null
// residual with x_out; out_op [M,256] bf16 (LayerNorm(x') or cast when gamma == null).
const char* launch_ffn_fused(cudaStream_t s, const void* a, const void* w1, const float* b1, const void* w2,
                             const float* b2, int act, const float* resid, float* x_out, const float* gamma,
                             const float* beta, void* out_op, int M, int num_sms, unsigned long long* trace) {
  if (M <= 0) return "ffn_fused: empty problem";
  if (resid != nullptr && resid != x_out) return "ffn_fused: residual must be updated in place";
  CUtensorMap ta, tw1, tw2, tx, top;
  if (const char* e = tma_encode_2d(&ta, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a, D, M, D, 64, 128)) return e;
  if (const char* e = tma_encode_2d(&tw1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w1, D, HID, D, 64, 128)) return e;
  if (const char* e = tma_encode_2d(&tw2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w2, HID, D, HID, 64, 128)) return e;
  tx = ta; top = ta;
  if (x_out != nullptr)
    if (const char* e = tma_encode_2d(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, x_out, D, M, D, 32, 128)) return e;
  if (out_op != nullptr)
    if (const char* e = tma_encode_2d(&top, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, out_op, D, M, D, 64, 128)) return e;
  if (!smem_opt_in(ffn_fused_kernel, FFN_SMEM)) return "ffn_fused: cudaFuncSetAttribute failed";
  FfnDev d;
  d.b1 = b1; d.b2 = b2; d.gamma = gamma; d.beta = beta; d.resid = resid;
  d.M = M; d.act = act; d.has_xout = x_out != nullptr; d.has_op = out_op != nullptr;
  d.trace = trace;
  const int m_tiles = (M + 127) / 128;
  const int grid = m_tiles < num_sms ? m_tiles : num_sms;
  if (launch_pdl(ffn_fused_kernel, dim3(grid), dim3(FFN_THREADS), FFN_SMEM, s, ta, tw1, tw2, tx, top, d) != cudaSuccess) {
    cudaGetLastError();
    return "ffn_fused: launch failed";
  }
  return nullptr;
}

}  // namespace avsep
