// Flash attention on the 5th-generation tensor cores (tcgen05 + TMEM), forward only, head dim 64, bf16 operands.
//
// Same contraction as attention.cu (reference: nn.MultiheadAttention inside nn.TransformerEncoderLayer,
// model.py:48-52,97-101, and CrossModalFusion, model.py:155,169) for the long-sequence configurations, where the
// mma.sync kernel tops out near 100 TFLOP/s.  For cross-attention the interpolated K/V rows are materialised once
// by lerp_rows_kernel (bf16, [B*T, 2d]) so that TMA can stage them.
//
// One CTA = 128 query rows of one (utterance, head); two CTAs are co-resident per SM (113 KB smem, 256 TMEM columns
// each), so one CTA's softmax overlaps the other's MMAs.
//   warp 0      TMA producer: Q once, then K and V tiles (128 rows x 64) through two 2-slot rings
//   warp 1      MMA issuer:   S = Q K^T   (M128 N128 K64, both operands K-major SW128)        -> TMEM cols [0,128)
//                             O_j = P V   (M128 N64 K128, P K-major from smem, V MN-major)    -> TMEM cols 128 + 64*(j&1)
//   warps 2..5  softmax: thread = query row (TMEM lane).  Pass 1 row max, pass 2 exp2 / row sum / bf16 P into
//               swizzled smem; the running output lives in registers and takes O_j from TMEM one tile late
//               (O = O * alpha_j + O_j), so no TMEM read-modify-write and no correction warp.
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

constexpr int QT = 128;
constexpr int KT = 128;
constexpr int HD = 64;
constexpr int TILE_BYTES = 128 * HD * 2;                 // 16 KB: 128 rows x 128 B
constexpr int OFF_Q = 0;
constexpr int OFF_K = OFF_Q + TILE_BYTES;                // 2 slots
constexpr int OFF_V = OFF_K + 2 * TILE_BYTES;            // 2 slots
constexpr int OFF_P = OFF_V + 2 * TILE_BYTES;            // 2 slabs of [128 rows x 64 kv] bf16
constexpr int OFF_BAR = OFF_P + 2 * TILE_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 256;
constexpr int NTHREADS = 192;
constexpr uint32_t TMEM_COLS = 256;

struct AttnTcDev {
  int Lq, Lk;
  float scale_log2;
  const int* k_lens;    // variable-length batch: keys of utterance b (null: all Lk)
};

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

__global__ void __launch_bounds__(NTHREADS, 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                    const AttnTcDev p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* sQ = smem + OFF_Q;
  uint8_t* sK = smem + OFF_K;
  uint8_t* sV = smem + OFF_V;
  uint8_t* sP = smem + OFF_P;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;    // [2]
  uint64_t* k_empty = bars + 3;   // [2]
  uint64_t* v_full = bars + 5;    // [2]
  uint64_t* v_empty = bars + 7;   // [2]
  uint64_t* s_full = bars + 9;
  uint64_t* p_full = bars + 10;
  uint64_t* o_full = bars + 11;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * QT;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int lk = utt_len(p.k_lens, b, p.Lk);
  const int nkv = (lk + KT - 1) / KT;                 // key tiles wholly past the utterance's keys are skipped

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(k_full + i, 1); mbar_init(k_empty + i, 1);
      mbar_init(v_full + i, 1); mbar_init(v_empty + i, 1);
      mbar_init(o_full + i, 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 128);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmO);
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch_dependents();
  griddep_wait();

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, TILE_BYTES);
      tma_load_3d(sQ, &tmQ, q_full, h * HD, q0, b);
      for (int j = 0; j < nkv; ++j) {
        const int st = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        mbar_wait_sleep(k_empty + st, ph ^ 1);
        mbar_arrive_expect_tx(k_full + st, TILE_BYTES);
        tma_load_3d(sK + st * TILE_BYTES, &tmK, k_full + st, h * HD, j * KT, b);
        mbar_wait_sleep(v_empty + st, ph ^ 1);
        mbar_arrive_expect_tx(v_full + st, TILE_BYTES);
        tma_load_3d(sV + st * TILE_BYTES, &tmV, v_full + st, h * HD, j * KT, b);
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    if (lane == 0) {
      constexpr uint32_t IDESC_S = umma_idesc(1, 128, 128);
      constexpr uint32_t IDESC_O = umma_idesc(1, 128, 64, 0, 1);      // B (= V) is MN-major
      const uint64_t dq = umma_desc_kmajor_sw128(smem_u32(sQ), 1024);
      auto issue_s = [&](int j) {
        const int st = j & 1;
        mbar_wait_sleep(k_full + st, (j >> 1) & 1);
        tc_fence_after();
        const uint64_t dk = umma_desc_kmajor_sw128(smem_u32(sK + st * TILE_BYTES), 1024);
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) umma_f16(tmem_base, dq + 2 * ks, dk + 2 * ks, IDESC_S, ks > 0);
        umma_commit(s_full);
        umma_commit(k_empty + st);
      };
      mbar_wait_sleep(q_full, 0);
      issue_s(0);
      for (int j = 0; j < nkv; ++j) {
        const int st = j & 1;
        mbar_wait_sleep(p_full, j & 1);          // softmax(j) has read S and written P(j)
        tc_fence_after();
        if (j + 1 < nkv) issue_s(j + 1);
        mbar_wait_sleep(v_full + st, (j >> 1) & 1);
        tc_fence_after();
        const uint32_t d_o = tmem_base + 128 + 64 * st;
#pragma unroll
        for (int ks = 0; ks < KT / 16; ++ks) {
          const uint64_t dp = umma_desc_kmajor_sw128(smem_u32(sP + (ks >> 2) * TILE_BYTES), 1024) + 2 * (ks & 3);
          const uint64_t dv = umma_desc_mnmajor_sw128(smem_u32(sV + st * TILE_BYTES + ks * 2048), 1024, 1024);
          umma_f16(d_o, dp, dv, IDESC_O, ks > 0);
        }
        umma_commit(o_full + st);
        umma_commit(v_empty + st);
      }
    }
  } else {
    // ---------------- softmax / output: thread = query row ----------------
    const int quarter = warp & 3;                       // TMEM lane quarter this warp may read
    const int row = quarter * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    float o_acc[HD];
#pragma unroll
    for (int i = 0; i < HD; ++i) o_acc[i] = 0.f;
    float m_run = -INFINITY, l_run = 0.f, alpha_prev = 0.f;
    const uint32_t p_row = smem_u32(sP) + row * 128;
    const int sw = row & 7;

    auto update_o = [&](int j, float alpha) {           // o_acc = o_acc * alpha + O_j
      const uint32_t t_o = t_lane + 128 + 64 * (j & 1);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_o + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) o_acc[c * 32 + i] = fmaf(o_acc[c * 32 + i], alpha, __uint_as_float(r[i]));
      }
    };

    for (int j = 0; j < nkv; ++j) {
      const int valid = lk - j * KT;                    // columns of this tile that exist
      mbar_wait_sleep(s_full, j & 1);
      tc_fence_after();
      // pass 1: row max (four independent chains; the chunk that straddles Lk takes the masked branch)
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      {
        uint32_t ra[32], rb[32];
        auto chunk_max = [&](const uint32_t (&r)[32], int c) {
          const int vc = valid - c * 32;
          if (vc >= 32) {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(r[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx4[i & 3] = (i < vc) ? fmaxf(mx4[i & 3], __uint_as_float(r[i])) : mx4[i & 3];
          }
        };
        tmem_ld_32x32b_x32(t_lane, ra);
        tmem_ld_32x32b_x32(t_lane + 32, rb);
        tmem_ld_wait();
        chunk_max(ra, 0);
        tmem_ld_32x32b_x32(t_lane + 64, ra);
        chunk_max(rb, 1);
        tmem_ld_wait();
        tmem_ld_32x32b_x32(t_lane + 96, rb);
        chunk_max(ra, 2);
        tmem_ld_wait();
        chunk_max(rb, 3);
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_new = fmaxf(m_run, mx * p.scale_log2);     // finite: every tile has a valid column
      const float alpha = ex2_approx(m_run - m_new);
      m_run = m_new;
      if (j > 0) mbar_wait_sleep(o_full + ((j - 1) & 1), ((j - 1) >> 1) & 1);   // PV(j-1) done: P is free, O_{j-1} ready
      // pass 2: P = exp2(S * scale - m), row sum, bf16 into the swizzled K-major slabs
      float l4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_lane + c * 32, r);
        tmem_ld_wait();
        const int vc = valid - c * 32;
        const uint32_t slab = p_row + (c >> 1) * TILE_BYTES;
        if (vc >= 32) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              e[i] = ex2_approx(fmaf(__uint_as_float(r[g * 8 + i]), p.scale_log2, -m_new));
              l4[i & 3] += e[i];
            }
            const uint32_t addr = slab + ((((c & 1) * 4 + g) ^ sw) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_bf16x2(e[0], e[1])),
                         "r"(pack_bf16x2(e[2], e[3])), "r"(pack_bf16x2(e[4], e[5])), "r"(pack_bf16x2(e[6], e[7]))
                         : "memory");
          }
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float x = ex2_approx(fmaf(__uint_as_float(r[g * 8 + i]), p.scale_log2, -m_new));
              e[i] = (g * 8 + i < vc) ? x : 0.f;
              l4[i & 3] += e[i];
            }
            const uint32_t addr = slab + ((((c & 1) * 4 + g) ^ sw) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_bf16x2(e[0], e[1])),
                         "r"(pack_bf16x2(e[2], e[3])), "r"(pack_bf16x2(e[4], e[5])), "r"(pack_bf16x2(e[6], e[7]))
                         : "memory");
          }
        }
      }
      const float l_tile = (l4[0] + l4[1]) + (l4[2] + l4[3]);
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive(p_full);
      l_run = fmaf(l_run, alpha, l_tile);
      if (j > 0) {
        tc_fence_after();
        update_o(j - 1, alpha_prev);
      }
      alpha_prev = alpha;
    }
    mbar_wait_sleep(o_full + ((nkv - 1) & 1), ((nkv - 1) >> 1) & 1);
    tc_fence_after();
    update_o(nkv - 1, alpha_prev);

    // normalise, bf16, stage in the (now dead) Q tile, TMA store (rows >= Lq are clipped by the tensor map)
    const float inv = 1.0f / l_run;
    const uint32_t o_row = smem_u32(sQ) + row * 128;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const uint32_t addr = o_row + ((g ^ sw) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr),
                   "r"(pack_bf16x2(o_acc[g * 8 + 0] * inv, o_acc[g * 8 + 1] * inv)),
                   "r"(pack_bf16x2(o_acc[g * 8 + 2] * inv, o_acc[g * 8 + 3] * inv)),
                   "r"(pack_bf16x2(o_acc[g * 8 + 4] * inv, o_acc[g * 8 + 5] * inv)),
                   "r"(pack_bf16x2(o_acc[g * 8 + 6] * inv, o_acc[g * 8 + 7] * inv))
                   : "memory");
    }
    fence_proxy_async_smem();
    named_bar_sync(1, 128);
    if (threadIdx.x == 64) {
      tma_store_3d(&tmO, sQ, h * HD, q0, b);
      bulk_commit();
      bulk_wait_read0();     // the staging tile may be released; the stores themselves complete with the grid
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// out[b*L + t, :] = lerp of two fp32 source rows (ATen upsample_linear1d, align_corners=False; model.py:114-116).
// src_lens / dst_lens (variable-length batch, else null): utterance b interpolates its first src_lens[b] source rows
// to dst_lens[b] rows; the rows past dst_lens[b] take the same formula (finite filler for masked keys).
__global__ void lerp_rows_kernel(const float* __restrict__ src, int ld_src, int nsrc, int L, int chunks, float scale,
                                 __nv_bfloat16* __restrict__ dst, int ld_dst, long long total,
                                 const int* __restrict__ src_lens, const int* __restrict__ dst_lens) {
  griddep_launch_dependents();
  griddep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = static_cast<int>(i % chunks);
  const long long rt = i / chunks;
  const int t = static_cast<int>(rt % L);
  const long long bb = rt / L;
  int ns = nsrc;
  if (src_lens != nullptr || dst_lens != nullptr) {
    ns = utt_len(src_lens, static_cast<int>(bb), nsrc);
    scale = static_cast<float>(ns) / static_cast<float>(utt_len(dst_lens, static_cast<int>(bb), L));
  }
  const float sp = fmaxf(scale * (static_cast<float>(t) + 0.5f) - 0.5f, 0.0f);
  int i0 = static_cast<int>(sp);
  if (i0 > ns - 1) i0 = ns - 1;
  const int i1 = min(i0 + 1, ns - 1);
  const float w1 = sp - static_cast<float>(i0), w0 = 1.0f - w1;
  const float4* p0 = reinterpret_cast<const float4*>(src + (bb * nsrc + i0) * ld_src + c * 8);
  const float4* p1 = reinterpret_cast<const float4*>(src + (bb * nsrc + i1) * ld_src + c * 8);
  const float4 a0 = __ldg(p0), a1 = __ldg(p0 + 1), b0 = __ldg(p1), b1 = __ldg(p1 + 1);
  uint4 val;
  val.x = pack_bf16x2(w0 * a0.x + w1 * b0.x, w0 * a0.y + w1 * b0.y);
  val.y = pack_bf16x2(w0 * a0.z + w1 * b0.z, w0 * a0.w + w1 * b0.w);
  val.z = pack_bf16x2(w0 * a1.x + w1 * b1.x, w0 * a1.y + w1 * b1.y);
  val.w = pack_bf16x2(w0 * a1.z + w1 * b1.z, w0 * a1.w + w1 * b1.w);
  *reinterpret_cast<uint4*>(dst + rt * ld_dst + c * 8) = val;
}

}  // namespace

bool attention_tc_usable(int prec, const AttnProblem& p) {
  return prec == PREC_BF16 && p.hd == HD && p.lerp_src == 0 && (p.ldq & 7) == 0 && (p.ldkv & 7) == 0 &&
         (p.ldo & 7) == 0;
}

const char* launch_attention_tc(cudaStream_t s, const AttnProblem& p) {
  if (p.B <= 0 || p.Lq <= 0 || p.Lk <= 0) return "attention_tc: empty problem";
  if (p.hd != HD || p.lerp_src != 0) return "attention_tc: needs head dim 64 and materialised K/V rows";
  if (!smem_opt_in(attention_tc_kernel, SMEM_BYTES)) return "attention_tc: cudaFuncSetAttribute failed";
  const int cols = p.H * HD;
  // rows [B, L] x cols, bf16, box = 64 cols x 128 rows of one utterance; rows past L are zero-filled / clipped
  CUtensorMap tq, tk, tv, to;
  if (const char* e = tma_encode_3d(&tq, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p.q, cols, p.Lq, p.B, p.ldq, 64, 128)) return e;
  if (const char* e = tma_encode_3d(&tk, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p.k, cols, p.Lk, p.B, p.ldkv, 64, 128)) return e;
  if (const char* e = tma_encode_3d(&tv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p.v, cols, p.Lk, p.B, p.ldkv, 64, 128)) return e;
  if (const char* e = tma_encode_3d(&to, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p.out, cols, p.Lq, p.B, p.ldo, 64, 128)) return e;
  AttnTcDev d;
  d.Lq = p.Lq; d.Lk = p.Lk;
  d.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(HD));
  d.k_lens = p.k_lens;
  dim3 grid((p.Lq + QT - 1) / QT, p.H, p.B);
  if (launch_pdl(attention_tc_kernel, grid, dim3(NTHREADS), SMEM_BYTES, s, tq, tk, tv, to, d) != cudaSuccess) {
    cudaGetLastError();
    return "attention_tc: launch failed";
  }
  return nullptr;
}

const char* launch_lerp_rows(cudaStream_t s, const float* src, int ld_src, int B, int nsrc, int L, int cols,
                             void* dst_bf16, int ld_dst, const int* src_lens, const int* dst_lens) {
  if ((cols & 7) || (ld_src & 3) || (ld_dst & 7)) return "lerp_rows: misaligned";
  const int chunks = cols / 8;
  const long long total = static_cast<long long>(B) * L * chunks;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  launch_pdl(lerp_rows_kernel, dim3(static_cast<unsigned>(blocks)), dim3(threads), 0, s, src, ld_src, nsrc, L, chunks,
             static_cast<float>(nsrc) / static_cast<float>(L), reinterpret_cast<__nv_bfloat16*>(dst_bf16), ld_dst, total,
             src_lens, dst_lens);
  return cudaGetLastError() == cudaSuccess ? nullptr : "lerp_rows: launch failed";
}

}  // namespace avsep
