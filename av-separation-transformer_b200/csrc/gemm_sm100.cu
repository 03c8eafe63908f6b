// Persistent TMA-fed tcgen05 GEMM for sm_100a with fused epilogues.
//
//   acc[m, n] = sum_{tap < taps} sum_{k < K} A[m + row_shift + tap, k] * W[n, tap*tap_stride + k]
//
// taps = 1 is every nn.Linear of the path (QKV / out-proj / FFN / frame_proj / decoder);
// taps = 3 is nn.Conv1d(k=3, padding=1) as an implicit GEMM: three row-shifted TMA views of the
// zero-haloed activation accumulate into the same TMEM tile (reference: model.py:37-42,56).
//
// One persistent CTA per SM (320 threads) walks 128 x n_tile output tiles (m fastest, so CTAs that run together
// share the weight tile in L2):
//   warp 0 / lane 0 : TMA producer  - cp.async.bulk.tensor A/W tiles (128B swizzle) into a 4-deep smem ring that
//                                     runs ahead across tile boundaries
//   warp 1 / lane 0 : MMA issuer    - tcgen05.mma (M=128, N=n_tile<=256, K=16 bf16 | 8 tf32) into one of TWO TMEM
//                                     accumulator stages; tcgen05.commit frees smem stages / publishes the tile
//   warps 2..9      : epilogue      - two warps per TMEM lane quarter (interleaved 32-column chunks), so tile i's
//                                     epilogue overlaps tile i+1's main loop.  Thread = accumulator row.
// Epilogues (template EPI):
//   EPI_STD  bias / ReLU / exact GELU / positional-encoding add / Conv1d halo handling, fp32 and/or bf16 stores
//   EPI_TAIL SeparationDecoder head: sigmoid, x mixed_spec, (B,S,F,T) stores coalesced along T (model.py:204-220)
//   EPI_LN   EPI_STD value + residual add, write the fp32 residual stream, then LayerNorm of the full row
//            (n_tile == N == d_model <= 256, row held in registers, exact two-pass statistics merged across the
//            two column halves) and write the normalised bf16 operand of the next GEMM -- the fused
//            residual+LayerNorm of every encoder / fusion sub-layer (model.py:149,168-172).
#include "common.cuh"
#include "kernels.h"

#include <stdio.h>

namespace avsep {

namespace {

constexpr int BM = 128;
constexpr int BN_MAX = 256;
constexpr int STAGES = 3;
constexpr int TILE_K_BYTES = 128;            // one 128-byte swizzle span per row per stage
constexpr int A_STAGE_BYTES = BM * TILE_K_BYTES;
constexpr int B_STAGE_BYTES = BN_MAX * TILE_K_BYTES;
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int NUM_EPI_WARPS = 16;
constexpr int NUM_THREADS = 32 * (2 + NUM_EPI_WARPS);
constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
constexpr int RED_OFFSET = BAR_OFFSET + 256;                 // LN partial statistics: [2 parity][128 rows][4 parts] float2
constexpr int VEC_OFFSET = RED_OFFSET + 2 * 128 * 4 * 8;   // bias [2][256], gamma [256], beta [256] fp32
constexpr int STG_OFFSET = (VEC_OFFSET + 4 * BN_MAX * 4 + 1023) / 1024 * 1024;   // 16 x 4 KB = four 128-row x 128-B slabs (one per column part)
constexpr int SMEM_TOTAL = STG_OFFSET + NUM_EPI_WARPS * 4096 + 1024;
static_assert(SMEM_TOTAL <= 227 * 1024, "gemm: shared memory budget exceeded");
constexpr int TMEM_COLS = 2 * BN_MAX;                        // two accumulator stages

struct GemmDev {
  int M, N, K, taps, tap_stride, row_shift, n_tile;
  GemmEpilogue e;
  int use_tma;                 // epilogue I/O through TMA slabs (ROW_IDENT, 64-column aligned)
  unsigned long long* trace;   // optional [grid][64] globaltimer stamps (debug hook), else null:
                               //   [0] entry [1] setup done [7] CTA done; per local tile lt < 12 at 8 + 4*lt:
                               //   +0 first operands of the tile landed, +1 tile's MMAs issued, +2 accumulator ready
                               //   (epilogue), +3 epilogue done
};

#define TRACE(slot) do { if (p.trace != nullptr) p.trace[blockIdx.x * 64 + (slot)] = globaltimer(); } while (0)
#define TRACE_TILE(lt, k) do { if (p.trace != nullptr && (lt) < 12) p.trace[blockIdx.x * 64 + 8 + 4 * (lt) + (k)] = globaltimer(); } while (0)

// 32-byte (full-sector) global store: one request per thread writes a whole sector of its row.
__device__ __forceinline__ void st_global_v8(void* ptr, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t e,
                                             uint32_t f, uint32_t g, uint32_t h) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(a), "r"(b), "r"(c), "r"(d),
               "r"(e), "r"(f), "r"(g), "r"(h)
               : "memory");
}
__device__ __forceinline__ void store_f32_chunk(float* o, const float (&val)[32]) {   // 32 fp32, 32-byte aligned
#pragma unroll
  for (int j = 0; j < 32; j += 8)
    st_global_v8(o + j, __float_as_uint(val[j]), __float_as_uint(val[j + 1]), __float_as_uint(val[j + 2]),
                 __float_as_uint(val[j + 3]), __float_as_uint(val[j + 4]), __float_as_uint(val[j + 5]),
                 __float_as_uint(val[j + 6]), __float_as_uint(val[j + 7]));
}

template <bool TF32>
__device__ __forceinline__ void store_op_chunk(void* out_op, size_t off, const float (&val)[32], int ncols, bool vec) {
  if constexpr (TF32) {
    float* o = reinterpret_cast<float*>(out_op) + off;
    float rv[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) rv[j] = round_tf32(val[j]);
    if (vec) {
      store_f32_chunk(o, rv);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) o[j] = rv[j];
    }
  } else {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out_op) + off;
    if (vec) {
#pragma unroll
      for (int j = 0; j < 32; j += 16)
        st_global_v8(o + j, pack_bf16x2(val[j], val[j + 1]), pack_bf16x2(val[j + 2], val[j + 3]),
                     pack_bf16x2(val[j + 4], val[j + 5]), pack_bf16x2(val[j + 6], val[j + 7]),
                     pack_bf16x2(val[j + 8], val[j + 9]), pack_bf16x2(val[j + 10], val[j + 11]),
                     pack_bf16x2(val[j + 12], val[j + 13]), pack_bf16x2(val[j + 14], val[j + 15]));
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) o[j] = __float2bfloat16_rn(val[j]);
    }
  }
}

// ---- per-warp transpose buffer: 32 rows x 128 B; 16-byte chunk c of row r lives at slot (c ^ (r & 7)) ----------
// Thread-per-row accesses (lane = row) and row-contiguous cooperative accesses (8 lanes = one 128-byte row) are both
// bank-conflict free, so the epilogue can read TMEM with thread = row and still move whole 128-byte lines to and
// from global memory (4 rows per instruction instead of 32 partial lines).

// global [32 rows x 128 B] -> buffer.  row_ptr = this lane's row base (already offset to the tile's first column) or 0.
__device__ __forceinline__ void stg_load_rows(uint8_t* buf, unsigned long long row_ptr, int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = i * 4 + (lane >> 3), c = lane & 7;
    const unsigned long long rp = __shfl_sync(0xffffffffu, row_ptr, row);
    uint4 x = make_uint4(0, 0, 0, 0);
    if (rp != 0) x = *reinterpret_cast<const uint4*>(rp + c * 16);
    *reinterpret_cast<uint4*>(buf + sw128_off(row, c)) = x;
  }
}
// buffer -> global [32 rows x 128 B]
__device__ __forceinline__ void stg_store_rows(const uint8_t* buf, unsigned long long row_ptr, int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = i * 4 + (lane >> 3), c = lane & 7;
    const unsigned long long rp = __shfl_sync(0xffffffffu, row_ptr, row);
    if (rp != 0) *reinterpret_cast<uint4*>(rp + c * 16) = *reinterpret_cast<const uint4*>(buf + sw128_off(row, c));
  }
}
// own row (lane) += 32 fp32 values of the slab
__device__ __forceinline__ void stg_add_own_f32(const uint8_t* buf, int lane, float (&x)[32]) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float4 v4 = *reinterpret_cast<const float4*>(buf + sw128_off(lane, c));
    x[4 * c] += v4.x; x[4 * c + 1] += v4.y; x[4 * c + 2] += v4.z; x[4 * c + 3] += v4.w;
  }
}
__device__ __forceinline__ void stg_write_own_f32(uint8_t* buf, int lane, const float (&x)[32]) {
#pragma unroll
  for (int c = 0; c < 8; ++c)
    *reinterpret_cast<float4*>(buf + sw128_off(lane, c)) = make_float4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
}
__device__ __forceinline__ void stg_write_own_tf32(uint8_t* buf, int lane, const float (&x)[32]) {
#pragma unroll
  for (int c = 0; c < 8; ++c)
    *reinterpret_cast<float4*>(buf + sw128_off(lane, c)) =
        make_float4(round_tf32(x[4 * c]), round_tf32(x[4 * c + 1]), round_tf32(x[4 * c + 2]), round_tf32(x[4 * c + 3]));
}
// own row: 32 values as bf16 into chunk slots [slot0, slot0+4) (two calls fill one 128-byte row of 64 bf16)
__device__ __forceinline__ void stg_write_own_bf16(uint8_t* buf, int lane, int slot0, const float (&x)[32]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint4 u;
    u.x = pack_bf16x2(x[8 * c], x[8 * c + 1]);
    u.y = pack_bf16x2(x[8 * c + 2], x[8 * c + 3]);
    u.z = pack_bf16x2(x[8 * c + 4], x[8 * c + 5]);
    u.w = pack_bf16x2(x[8 * c + 6], x[8 * c + 7]);
    *reinterpret_cast<uint4*>(buf + sw128_off(lane, slot0 + c)) = u;
  }
}

// Row bookkeeping shared by the epilogues: where accumulator row m goes and which PE row it takes.
struct RowInfo {
  bool valid, zero_row;
  long long orow;
  int pos;
};
__device__ __forceinline__ RowInfo row_info(const GemmEpilogue& e, int m, int M) {
  RowInfo r;
  r.valid = m < M;
  r.zero_row = false;
  r.orow = m;
  r.pos = 0;
  if (e.rowmap == ROW_IDENT) {
    if (e.pe_period > 0) r.pos = m % e.pe_period;
  } else {
    const int b = m / e.Lp;
    const int tp = m - b * e.Lp;
    const bool halo = (tp == 0) || (tp == e.Lp - 1);
    r.pos = tp - 1;
    if (e.rowmap == ROW_PAD2PAD) {
      // rows past a short utterance's length are its right-hand Conv1d padding (rows m >= M of the last tile have
      // no utterance: lens is not read for them)
      r.zero_row = halo || (r.valid && e.lens != nullptr && tp - 1 >= utt_len(e.lens, b, e.Lp - 2));
    } else {
      r.valid = r.valid && !halo;
      r.orow = static_cast<long long>(b) * (e.Lp - 2) + (tp - 1);
    }
  }
  return r;
}

// acc chunk -> value chunk: (+ prior contents when ACCUM) + bias (shared memory), activation, + PE, halo zeroing.
template <bool ACCUM, bool SKIP_PE = false>
__device__ __forceinline__ void value_chunk(const GemmEpilogue& e, const RowInfo& ri, const uint32_t (&v)[32],
                                            float (&val)[32], const float* sbias_c0, int col0, int ncols, int N) {
  const bool full = (ncols == 32);
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const float4 b4 = *reinterpret_cast<const float4*>(sbias_c0 + j);     // zero beyond N
    if constexpr (ACCUM) {
      val[j] += __uint_as_float(v[j]) + b4.x;
      val[j + 1] += __uint_as_float(v[j + 1]) + b4.y;
      val[j + 2] += __uint_as_float(v[j + 2]) + b4.z;
      val[j + 3] += __uint_as_float(v[j + 3]) + b4.w;
    } else {
      val[j] = __uint_as_float(v[j]) + b4.x;
      val[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
      val[j + 2] = __uint_as_float(v[j + 2]) + b4.z;
      val[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
    }
  }
  if (e.act == ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) val[j] = fmaxf(val[j], 0.0f);
  } else if (e.act == ACT_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) val[j] = gelu_erf(val[j]);
  } else if (e.act == ACT_GELU_BF16) {
#pragma unroll
    for (int j = 0; j < 32; ++j) val[j] = gelu_bf16_grade(val[j]);
  }
  if (!SKIP_PE && e.pe != nullptr && ri.valid) {
    const float* pr = e.pe + static_cast<size_t>(ri.pos) * N + col0;
    if (full && (N & 3) == 0) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 p4 = __ldg(reinterpret_cast<const float4*>(pr + j));
        val[j] += p4.x; val[j + 1] += p4.y; val[j + 2] += p4.z; val[j + 3] += p4.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) val[j] += __ldg(pr + j);
    }
  }
  if (ri.zero_row) {
#pragma unroll
    for (int j = 0; j < 32; ++j) val[j] = 0.0f;
  }
}

// Decoder-head epilogue (EPI_TAIL) for 16 columns of one accumulator row, split in two so that the mixed_spec loads
// of the next chunk are issued before the stores of the current one (and the first chunk's before the accumulator is
// even complete): column c = s*F + f sits c*T floats further in masks / separated and f*T further in mixed_spec.
// Whole chunks that do not cross a speaker boundary take branch-free bodies - the per-element guards and the frequency
// wrap cost more instructions than the sigmoid.  All tests except `valid` are warp-uniform.
// live == false: the row lies past its utterance's length; mixed_spec is not read there and both outputs are 0.
__device__ __forceinline__ void tail_load16(const GemmEpilogue& e, int N, int col0, const float* mixed_row, bool valid,
                                            bool live, float (&mx)[16]) {
  const int ncols = min(16, N - col0);
  if (!valid || ncols <= 0) return;
  if (!live) {
#pragma unroll
    for (int j = 0; j < 16; ++j) mx[j] = 0.f;
    return;
  }
  int f = col0 % e.F;
  if (ncols == 16 && f + 16 <= e.F) {
    const float* mp = mixed_row + static_cast<size_t>(f) * e.T;
#pragma unroll
    for (int j = 0; j < 16; ++j) mx[j] = __ldg(mp + static_cast<size_t>(j) * e.T);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      mx[j] = (j < ncols) ? __ldg(mixed_row + static_cast<size_t>(f) * e.T) : 0.f;
      if (++f == e.F) f = 0;
    }
  }
}

__device__ __forceinline__ void tail_store16(const GemmEpilogue& e, int N, int col0, size_t out_base, bool valid,
                                             bool live, const uint32_t (&v)[16], const float* sb, const float (&mx)[16]) {
  const int ncols = min(16, N - col0);
  if (!valid || ncols <= 0) return;
  float* mo = e.masks + out_base + static_cast<size_t>(col0) * e.T;
  float* so = e.separated + out_base + static_cast<size_t>(col0) * e.T;
  if (ncols == 16) {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float mk = live ? sigmoid_fast(__uint_as_float(v[j]) + sb[j]) : 0.f;
      __stcs(mo + static_cast<size_t>(j) * e.T, mk);
      __stcs(so + static_cast<size_t>(j) * e.T, mk * mx[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (j < ncols) {
        const float mk = live ? sigmoid_fast(__uint_as_float(v[j]) + sb[j]) : 0.f;
        __stcs(mo + static_cast<size_t>(j) * e.T, mk);
        __stcs(so + static_cast<size_t>(j) * e.T, mk * mx[j]);
      }
    }
  }
}

template <int EPI, bool TF32>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                    const __grid_constant__ CUtensorMap tmOp, const __grid_constant__ CUtensorMap tmF32, const GemmDev p) {
  // Dynamic shared memory is declared 1024-byte aligned (128B-swizzle atoms) and used directly: deriving the base
  // through an integer round trip would make the compiler fall back to generic LD/ST for every access.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* const smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + BAR_OFFSET);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;     // [2] accumulator stage complete
  uint64_t* tempty_bar = tfull_bar + 2;         // [2] accumulator stage drained by the epilogue
  uint64_t* resid_bar = tempty_bar + 2;         // [4] residual slab of column part p landed (TMA)
  uint64_t* resid_bar2 = resid_bar + 4;         // [4] second residual chunk, fetched into the idle pipeline stages (last tile)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resid_bar2 + 4);
  float2* red = reinterpret_cast<float2*>(smem + RED_OFFSET);
  float* sbias = reinterpret_cast<float*>(smem + VEC_OFFSET);       // [2][BN_MAX], double-buffered per tile
  float* sgamma = sbias + 2 * BN_MAX;
  float* sbeta = sgamma + BN_MAX;
  uint8_t* stg_all = smem + STG_OFFSET;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int ELEMS_PER_TILE = TF32 ? 32 : 64;                 // elements per 128-byte K span
  const int kt_per_tap = (p.K + ELEMS_PER_TILE - 1) / ELEMS_PER_TILE;
  const int num_kt = kt_per_tap * p.taps;
  const int m_tiles = (p.M + BM - 1) / BM;
  const int n_tiles = (p.N + p.n_tile - 1) / p.n_tile;
  const int total_tiles = m_tiles * n_tiles;

  if (threadIdx.x == 0) {
    TRACE(0);                                  // kernel entry
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], NUM_EPI_WARPS);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) { mbar_init(&resid_bar[a], 1); mbar_init(&resid_bar2[a], 1); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  if constexpr (EPI == EPI_LN || EPI == EPI_LN_TMA) {
    if (p.e.ln_gamma != nullptr) {
      for (int i = threadIdx.x; i < p.n_tile; i += NUM_THREADS) {
        sgamma[i] = __ldg(p.e.ln_gamma + i);
        sbeta[i] = __ldg(p.e.ln_beta + i);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // the setup above overlapped the previous kernel's tail; its results are needed from here on
  griddep_launch_dependents();
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      TRACE(1);                                // setup done (barriers, TMEM alloc)
      // ---------------- TMA producer ----------------
      const uint32_t stage_bytes = A_STAGE_BYTES + static_cast<uint32_t>(p.n_tile) * TILE_K_BYTES;
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile % m_tiles) * BM;
        const int n0 = (tile / m_tiles) * p.n_tile;
        for (int kt = 0; kt < num_kt; ++kt, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          const int tap = kt / kt_per_tap;
          const int kk = (kt - tap * kt_per_tap) * ELEMS_PER_TILE;
          uint8_t* a_dst = smem + s * STAGE_BYTES;
          uint8_t* b_dst = a_dst + A_STAGE_BYTES;
          mbar_arrive_expect_tx(&full_bar[s], stage_bytes);
          tma_load_2d(a_dst, &tmA, &full_bar[s], kk, m0 + p.row_shift + tap);
          tma_load_2d(b_dst, &tmW, &full_bar[s], tap * p.tap_stride + kk, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ---------------- MMA issuer ----------------
      const uint32_t idesc = umma_idesc(TF32 ? 2u : 1u, BM, static_cast<uint32_t>(p.n_tile));
      int it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
        const int acc = lt & 1;
        const uint32_t aph = (lt >> 1) & 1;
        mbar_wait(&tempty_bar[acc], aph ^ 1);        // epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN_MAX);
        for (int kt = 0; kt < num_kt; ++kt, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (kt == 0) TRACE_TILE(lt, 0);      // first operands of this tile landed
          const uint32_t a_addr = smem_u32(smem + s * STAGE_BYTES);
          const uint32_t b_addr = a_addr + A_STAGE_BYTES;
          const uint64_t adesc = umma_desc_kmajor_sw128(a_addr, 1024);
          const uint64_t bdesc = umma_desc_kmajor_sw128(b_addr, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) {   // 4 x 32 bytes of K per stage: advance the start address by 32 B (>>4 = 2)
            const uint32_t accum = (kt | k) != 0 ? 1u : 0u;
            if constexpr (TF32) umma_tf32(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, accum);
            else                umma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, accum);
          }
          umma_commit(&empty_bar[s]);      // smem stage reusable once these MMAs have read it
        }
        umma_commit(&tfull_bar[acc]);      // accumulator stage complete
        TRACE_TILE(lt, 1);                   // all MMAs of this tile issued
      }
    }
  } else {
    // ---------------- epilogue: warps 2..17; TMEM lane quarter = warp % 4, column part = (warp - 2) / 4 ----------------
    const int q = warp & 3;
    const int part = (warp - 2) >> 2;            // 0..3
    const int r = q * 32 + lane;
    const GemmEpilogue& e = p.e;
    uint8_t* const slab = stg_all + part * 16384;            // this column part's 128-row x 128-B slab (TMA box)
    uint8_t* const slab_q = slab + q * 4096;                 // this warp's 32 rows of it
    const bool elected = (warp == 2 + 4 * part) && (lane == 0);   // issues this part's TMA loads / stores
    const int part_bar = 6 + part;                            // named barrier of the part's 4 warps (128 threads)
    uint32_t rph = 0;                                         // parity of resid_bar[part]
    int lt = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
      const int acc = lt & 1;
      const uint32_t aph = (lt >> 1) & 1;
      const int m0 = (tile % m_tiles) * BM;
      const int n0 = (tile / m_tiles) * p.n_tile;
      const int m = m0 + r;
      // stage this tile's bias slice in shared memory while the main loop is still running
      float* sb = sbias + (lt & 1) * BN_MAX;
      if constexpr (EPI != EPI_TAIL) {
        const int i = threadIdx.x - 64;                       // 0..511 over the 16 epilogue warps
        if (i < BN_MAX) sb[i] = (e.bias != nullptr && i < p.n_tile && n0 + i < p.N) ? __ldg(e.bias + n0 + i) : 0.f;
      }
      if constexpr (EPI == EPI_LN_TMA) {
        // TMA epilogue: fetch the residual slab of this part's first chunk while the main loop runs
        if (e.resid != nullptr && elected) {
          bulk_wait_read0();                                    // previous tile's stores have left the slab
          mbar_arrive_expect_tx(&resid_bar[part], 16384);
          tma_load_2d(slab, &tmF32, &resid_bar[part], part * 64, m0);
        }
      }
      // EPI_TAIL: this thread's row of the (B,S,F,T) outputs, its share of the tile's columns, and the mixed_spec
      // values of its first 16 columns - requested now, while the tile's MMAs are still running
      bool t_valid = false, t_live = true;
      const float* t_mixed_row = nullptr;
      size_t t_out_base = 0;
      int t_cbeg = 0, t_cend = 0;
      float mxa[16], mxb[16];
      if constexpr (EPI == EPI_TAIL) {
        // SeparationDecoder head (model.py:204-207,220): column c = s*F + f, so masks[b,s,f,t] sits at
        // ((b*S*F + c)*T + t); lanes are consecutive t, so the (B,S,F,T) stores and the mixed_spec (B,F,T) loads are
        // both contiguous across the warp.
        t_valid = m < p.M;
        const int tb = m / e.T;
        const int tt = m - tb * e.T;
        t_live = e.lens == nullptr || (t_valid && tt < utt_len(e.lens, tb, e.T));
        t_mixed_row = e.mixed + static_cast<size_t>(tb) * e.F * e.T + tt;
        t_out_base = static_cast<size_t>(tb) * e.S * e.F * e.T + tt;
        // Each column part takes a contiguous, balanced share of the tile in units of 16 columns (176 columns ->
        // 48/48/48/32); handing out whole 32-column chunks round-robin left two parts with twice the work of the
        // others and the tile waiting on them at the next barrier.
        const int units = p.n_tile >> 4, ubase = units >> 2, urem = units & 3;
        t_cbeg = (part * ubase + min(part, urem)) << 4;
        t_cend = t_cbeg + ((ubase + (part < urem ? 1 : 0)) << 4);
        if (t_cbeg < t_cend) tail_load16(e, p.N, n0 + t_cbeg, t_mixed_row, t_valid, t_live, mxa);
        // each column part stages its own bias slice and synchronises only its 4 warps (same columns, same amount
        // of work): with one 512-thread barrier per tile every part waited ~1.2 us for the slowest of the 16 warps
        const int c = t_cbeg + r;
        if (c < t_cend) sb[c] = (e.bias != nullptr && n0 + c < p.N) ? __ldg(e.bias + n0 + c) : 0.f;
      }
      if (lt == 1 && threadIdx.x == 64) TRACE(2);               // [2] tile-1 epilogue entered (bias load issued)
      if constexpr (EPI == EPI_TAIL) named_bar_sync(part_bar, 128);
      else asm volatile("bar.sync 5, 512;" ::: "memory");       // bias slice visible to all epilogue warps
      if (lt == 1 && threadIdx.x == 64) TRACE(3);               // [3] bias barrier passed
      mbar_wait(&tfull_bar[acc], aph);
      tc_fence_after();
      if (threadIdx.x == 64) TRACE_TILE(lt, 2);     // accumulator ready
      const uint32_t taddr_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BN_MAX);

      if constexpr (EPI == EPI_TAIL) {
        // 16 columns at a time (16 accumulator values + two 16-value mixed_spec buffers stay within the 96 registers
        // this 640-thread CTA allows), two chunks per iteration so that the buffers alternate statically.
        for (int c0 = t_cbeg; c0 < t_cend; c0 += 32) {
          if (n0 + c0 >= p.N) break;                   // warp-uniform
          uint32_t v[16];
          tmem_ld_32x32b_x16(taddr_row + static_cast<uint32_t>(c0), v);
          const bool second = c0 + 16 < t_cend;
          if (second) tail_load16(e, p.N, n0 + c0 + 16, t_mixed_row, t_valid, t_live, mxb);
          tmem_ld_wait();
          tail_store16(e, p.N, n0 + c0, t_out_base, t_valid, t_live, v, sb + c0, mxa);
          if (second && n0 + c0 + 16 < p.N) {
            tmem_ld_32x32b_x16(taddr_row + static_cast<uint32_t>(c0 + 16), v);
            if (c0 + 32 < t_cend) tail_load16(e, p.N, n0 + c0 + 32, t_mixed_row, t_valid, t_live, mxa);
            tmem_ld_wait();
            tail_store16(e, p.N, n0 + c0 + 16, t_out_base, t_valid, t_live, v, sb + c0 + 16, mxb);
          }
        }
      } else if constexpr (EPI == EPI_LN_TMA) {
        // ---- LN epilogue with TMA I/O (n_tile == 256, ROW_IDENT): each column part owns 64 columns = 2 chunks.
        // residual chunk: TMA-loaded slab -> own-row LDS; x' chunk: own-row STS into the same slab -> one TMA store;
        // normalised bf16 row (64 columns = 128 B): own-row STS -> one TMA store.  No per-element address math.
        const RowInfo ri = row_info(e, m, p.M);
        // On the CTA's last tile every pipeline stage has been consumed (this tile's accumulator is complete and
        // nothing more will be loaded): the second residual chunk is fetched into stage memory right away instead of
        // after the first chunk's x' store has left the slab.
        const bool last_tile = tile + static_cast<int>(gridDim.x) >= total_tiles;
        uint8_t* const slab1 = last_tile ? smem + part * 16384 : slab;
        if (last_tile && e.resid != nullptr && elected) {
          mbar_arrive_expect_tx(&resid_bar2[part], 16384);
          tma_load_2d(slab1, &tmF32, &resid_bar2[part], part * 64 + 32, m0);
        }
        float val[2][32];
        float sum = 0.f, sq = 0.f;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int c0 = part * 64 + ci * 32;
          uint8_t* const sl = ci == 0 ? slab : slab1;
          uint8_t* const sl_q = sl + q * 4096;
          uint32_t v[32];
          tmem_ld_32x32b_x32(taddr_row + static_cast<uint32_t>(c0), v);
          if (e.resid != nullptr) {
            if (ci == 1 && last_tile) {
              mbar_wait(&resid_bar2[part], 0);
            } else {
              mbar_wait(&resid_bar[part], rph);
              rph ^= 1;
            }
          }
          tmem_ld_wait();
          value_chunk<false>(e, ri, v, val[ci], sb + c0, c0, 32, p.N);
          if (e.resid != nullptr) stg_add_own_f32(sl_q, lane, val[ci]);
          if (e.out_f32 != nullptr) {
            stg_write_own_f32(sl_q, lane, val[ci]);
            fence_proxy_async_smem();
          }
          if (e.out_f32 != nullptr || (e.resid != nullptr && ci == 0)) named_bar_sync(part_bar, 128);
          if (elected) {
            if (e.out_f32 != nullptr) {
              tma_store_2d(&tmF32, sl, c0, m0);
              bulk_commit();
            }
            if (ci == 0 && e.resid != nullptr && !last_tile) {
              bulk_wait_read0();                              // the store has read the slab: refill it
              mbar_arrive_expect_tx(&resid_bar[part], 16384);
              tma_load_2d(slab, &tmF32, &resid_bar[part], c0 + 32, m0);
            }
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            sum += val[ci][j];
            sq = fmaf(val[ci][j], val[ci][j], sq);
          }
        }
        // accumulator fully read: hand the TMEM stage back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        if (e.ln_gamma != nullptr) {
          // row statistics: this part's (sum, sum of squares about the part mean) merged over the 4 parts
          const float mean_h = sum * (1.0f / 64.0f);
          const float m2 = fmaxf(sq - sum * mean_h, 0.f);
          float2* slot = red + ((lt & 1) * 128 + r) * 4;
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
            for (int j = 0; j < 32; j += 4) {
              const float4 g4 = *reinterpret_cast<const float4*>(sgamma + c0 + j);
              const float4 b4 = *reinterpret_cast<const float4*>(sbeta + c0 + j);
              val[ci][j] = (val[ci][j] - mean) * rstd * g4.x + b4.x;
              val[ci][j + 1] = (val[ci][j + 1] - mean) * rstd * g4.y + b4.y;
              val[ci][j + 2] = (val[ci][j + 2] - mean) * rstd * g4.z + b4.z;
              val[ci][j + 3] = (val[ci][j + 3] - mean) * rstd * g4.w + b4.w;
            }
          }
        }
        if (e.out_op != nullptr) {
          if (elected) bulk_wait_read0();                     // last x' store has read the slab
          named_bar_sync(part_bar, 128);
          if constexpr (TF32) {
#pragma unroll
            for (int ci = 0; ci < 2; ++ci) {
              stg_write_own_tf32(slab_q, lane, val[ci]);
              fence_proxy_async_smem();
              named_bar_sync(part_bar, 128);
              if (elected) {
                tma_store_2d(&tmOp, slab, part * 64 + ci * 32, m0);
                bulk_commit();
                bulk_wait_read0();
              }
              named_bar_sync(part_bar, 128);
            }
          } else {
            stg_write_own_bf16(slab_q, lane, 0, val[0]);
            stg_write_own_bf16(slab_q, lane, 4, val[1]);
            fence_proxy_async_smem();
            named_bar_sync(part_bar, 128);
            if (elected) {
              tma_store_2d(&tmOp, slab, part * 64, m0);
              bulk_commit();
            }
          }
        }
        if (threadIdx.x == 64) TRACE_TILE(lt, 3);     // LN: epilogue done
        continue;   // tempty already signalled
      } else if constexpr (EPI == EPI_LN) {
        // value = acc + bias (+act, +PE) + residual; fp32 residual-stream store; LayerNorm over the whole row;
        // operand store.  Each warp owns 32 rows x (n_tile/2) contiguous columns; all global traffic goes through
        // the warp's transpose buffer as whole 128-byte lines.
        const RowInfo ri = row_info(e, m, p.M);
        uint8_t* stg = stg_all + (warp - 2) * 4096;
        const int nch = p.n_tile >> 5;                       // 32-column chunks in the row (<= 8)
        const int per = (nch + 3) >> 2;                      // chunks per column part (<= 2)
        const int ch_first = part * per;
        const int ch_count = max(0, min(per, nch - ch_first));
        const unsigned long long resid_row =
            (ri.valid && e.resid != nullptr) ? reinterpret_cast<unsigned long long>(e.resid + static_cast<size_t>(ri.orow) * p.N) : 0ull;
        const unsigned long long xout_row =
            (ri.valid && e.out_f32 != nullptr) ? reinterpret_cast<unsigned long long>(e.out_f32 + static_cast<size_t>(ri.orow) * e.ld_f32) : 0ull;
        const unsigned long long op_row =
            (ri.valid && e.out_op != nullptr)
                ? reinterpret_cast<unsigned long long>(e.out_op) + static_cast<size_t>(ri.orow) * e.ld_op * (TF32 ? 4 : 2) : 0ull;
        // positional-encoding rows are fetched like the residual: whole 128-byte lines, 4 rows per warp instruction,
        // through the warp's transpose buffer (a thread-per-row read touches 32 lines per instruction)
        const unsigned long long pe_row =
            (ri.valid && !ri.zero_row && e.pe != nullptr) ? reinterpret_cast<unsigned long long>(e.pe + static_cast<size_t>(ri.pos) * p.N) : 0ull;
        float val[2][32];
        float sum = 0.f;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          if (ci < ch_count) {                          // warp-uniform
            const int c0 = (ch_first + ci) * 32;
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr_row + static_cast<uint32_t>(c0), v);
            if (e.pe != nullptr) stg_load_rows(stg, pe_row ? pe_row + c0 * 4 : 0ull, lane);
            tmem_ld_wait();
            value_chunk<false, true>(e, ri, v, val[ci], sb + c0, c0, 32, p.N);
            __syncwarp();
            if (e.pe != nullptr) {
              stg_add_own_f32(stg, lane, val[ci]);
              __syncwarp();
            }
            if (e.resid != nullptr) {
              stg_load_rows(stg, resid_row ? resid_row + c0 * 4 : 0ull, lane);
              __syncwarp();
              stg_add_own_f32(stg, lane, val[ci]);
            }
            if (e.out_f32 != nullptr) {
              stg_write_own_f32(stg, lane, val[ci]);
              __syncwarp();
              stg_store_rows(stg, xout_row ? xout_row + c0 * 4 : 0ull, lane);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 32; ++j) sum += val[ci][j];
          }
        }
        // accumulator fully read: hand the TMEM stage back before the statistics / stores
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        const int cnt = ch_count * 32;
        if (e.ln_gamma != nullptr) {
          // exact two-pass statistics of this column part, merged across the four parts (Chan's parallel formula)
          const float n_h = static_cast<float>(cnt);
          const float mean_h = cnt > 0 ? sum / n_h : 0.f;
          float m2 = 0.f;
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            if (ci < ch_count) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float dlt = val[ci][j] - mean_h;
                m2 += dlt * dlt;
              }
            }
          }
          float2* slot = red + ((lt & 1) * 128 + r) * 4;
          slot[part] = make_float2(mean_h, m2);
          asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
          float n_acc = 0.f, mean = 0.f, m2_all = 0.f;
#pragma unroll
          for (int pp = 0; pp < 4; ++pp) {
            const float n_p = static_cast<float>(max(0, min(per, nch - pp * per)) * 32);
            if (n_p > 0.f) {
              const float2 st = slot[pp];
              const float n_new = n_acc + n_p;
              const float dm = st.x - mean;
              mean += dm * (n_p / n_new);
              m2_all += st.y + dm * dm * (n_acc * n_p / n_new);
              n_acc = n_new;
            }
          }
          const float rstd = rsqrtf(m2_all / n_acc + 1e-5f);
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            if (ci < ch_count) {
              const int c0 = (ch_first + ci) * 32;
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 g4 = *reinterpret_cast<const float4*>(sgamma + c0 + j);
                const float4 b4 = *reinterpret_cast<const float4*>(sbeta + c0 + j);
                val[ci][j] = (val[ci][j] - mean) * rstd * g4.x + b4.x;
                val[ci][j + 1] = (val[ci][j + 1] - mean) * rstd * g4.y + b4.y;
                val[ci][j + 2] = (val[ci][j + 2] - mean) * rstd * g4.z + b4.z;
                val[ci][j + 3] = (val[ci][j + 3] - mean) * rstd * g4.w + b4.w;
              }
            }
          }
        }
        if (e.out_op != nullptr) {
          if constexpr (TF32) {
#pragma unroll
            for (int ci = 0; ci < 2; ++ci) {
              if (ci < ch_count) {
                stg_write_own_tf32(stg, lane, val[ci]);
                __syncwarp();
                stg_store_rows(stg, op_row ? op_row + (ch_first + ci) * 128 : 0ull, lane);
                __syncwarp();
              }
            }
          } else {
            // bf16: two chunks (64 columns) make one 128-byte row
#pragma unroll
            for (int cp = 0; cp < 1; ++cp) {
              if (2 * cp + 1 < ch_count) {
                stg_write_own_bf16(stg, lane, 0, val[2 * cp]);
                stg_write_own_bf16(stg, lane, 4, val[2 * cp + 1]);
                __syncwarp();
                stg_store_rows(stg, op_row ? op_row + (ch_first + 2 * cp) * 64 : 0ull, lane);
                __syncwarp();
              } else if (2 * cp < ch_count) {          // odd trailing chunk: thread-per-row 32-byte stores
                if (ri.valid)
                  store_op_chunk<TF32>(e.out_op, static_cast<size_t>(ri.orow) * e.ld_op + (ch_first + 2 * cp) * 32,
                                       val[2 * cp], 32, true);
              }
            }
          }
        }
        if (threadIdx.x == 64) TRACE_TILE(lt, 3);     // LN: epilogue done
        continue;   // tempty already signalled
      } else {
        const RowInfo ri = row_info(e, m, p.M);
        uint8_t* stg = stg_all + (warp - 2) * 4096;
        // Coalesced path: each warp owns a contiguous half of the tile's 64-column units, stages two chunks as one
        // 128-byte bf16 row (or one chunk as a 128-byte fp32 row) and stores whole lines.
        const bool coalesced = (p.N % 64 == 0) && (p.n_tile % 64 == 0) && (e.out_op == nullptr || (e.ld_op & 63) == 0) &&
                               (e.out_f32 == nullptr || (e.ld_f32 & 31) == 0);
        if (p.use_tma) {
          // ---- TMA-store epilogue: each part stages one 64-column unit (128-B bf16 rows, or two 32-column fp32
          // slabs) in its swizzled slab with thread-per-row STS; one elected thread stores the whole 128-row box.
          const int npair = p.n_tile >> 6;
          for (int pi = part; pi < npair; pi += 4) {
#pragma unroll
            for (int hc = 0; hc < 2; ++hc) {
              const int c0 = pi * 64 + hc * 32;
              uint32_t v[32];
              tmem_ld_32x32b_x32(taddr_row + static_cast<uint32_t>(c0), v);
              tmem_ld_wait();
              float a[32];
              value_chunk<false>(e, ri, v, a, sb + c0, n0 + c0, 32, p.N);
              if (e.out_f32 != nullptr) {                      // exact fp32 output: one 32-column slab per chunk
                if (elected) bulk_wait_read0();
                named_bar_sync(part_bar, 128);
                stg_write_own_f32(slab_q, lane, a);
                fence_proxy_async_smem();
                named_bar_sync(part_bar, 128);
                if (elected) {
                  tma_store_2d(&tmF32, slab, n0 + c0, m0);
                  bulk_commit();
                }
              }
              if (TF32 && e.out_op != nullptr) {               // tf32 operand output (rounded to nearest)
                if (elected) bulk_wait_read0();
                named_bar_sync(part_bar, 128);
                stg_write_own_tf32(slab_q, lane, a);
                fence_proxy_async_smem();
                named_bar_sync(part_bar, 128);
                if (elected) {
                  tma_store_2d(&tmOp, slab, n0 + c0, m0);
                  bulk_commit();
                }
              }
              if (!TF32 && e.out_op != nullptr) {
                if (hc == 0) {
                  if (elected) bulk_wait_read0();
                  named_bar_sync(part_bar, 128);
                }
                stg_write_own_bf16(slab_q, lane, hc * 4, a);
                if (hc == 1) {
                  fence_proxy_async_smem();
                  named_bar_sync(part_bar, 128);
                  if (elected) {
                    tma_store_2d(&tmOp, slab, n0 + pi * 64, m0);
                    bulk_commit();
                  }
                }
              }
            }
          }
        } else if (coalesced) {
          const int npair = p.n_tile >> 6;
          const unsigned long long f32_row =
              (ri.valid && e.out_f32 != nullptr) ? reinterpret_cast<unsigned long long>(e.out_f32 + static_cast<size_t>(ri.orow) * e.ld_f32 + n0) : 0ull;
          const unsigned long long op_row =
              (ri.valid && e.out_op != nullptr)
                  ? reinterpret_cast<unsigned long long>(e.out_op) + (static_cast<size_t>(ri.orow) * e.ld_op + n0) * (TF32 ? 4 : 2) : 0ull;
          for (int pi = part; pi < npair; pi += 4) {
#pragma unroll
            for (int hc = 0; hc < 2; ++hc) {             // the two 32-column chunks of this 64-column unit
              const int c0 = pi * 64 + hc * 32;
              uint32_t v[32];
              tmem_ld_32x32b_x32(taddr_row + static_cast<uint32_t>(c0), v);
              tmem_ld_wait();
              if (lt == 1 && threadIdx.x == 64 && hc == 0) TRACE(4);   // [4] first TMEM chunk in registers
              float a[32];
              value_chunk<false>(e, ri, v, a, sb + c0, n0 + c0, 32, p.N);
              if (lt == 1 && threadIdx.x == 64 && hc == 1) TRACE(5);   // [5] second chunk's values computed
              if (e.out_f32 != nullptr) {
                stg_write_own_f32(stg, lane, a);
                __syncwarp();
                stg_store_rows(stg, f32_row ? f32_row + c0 * 4 : 0ull, lane);
                __syncwarp();
              }
              if (e.out_op != nullptr) {
                if constexpr (TF32) {
                  stg_write_own_tf32(stg, lane, a);
                  __syncwarp();
                  stg_store_rows(stg, op_row ? op_row + c0 * 4 : 0ull, lane);
                  __syncwarp();
                } else {
                  stg_write_own_bf16(stg, lane, hc * 4, a);   // two chunks make one 128-byte bf16 row
                  if (hc == 1) {
                    __syncwarp();
                    stg_store_rows(stg, op_row ? op_row + (pi * 64) * 2 : 0ull, lane);
                    __syncwarp();
                    if (lt == 1 && threadIdx.x == 64) TRACE(6);        // [6] line stores issued
                  }
                }
              }
            }
          }
        } else {
          for (int c0 = part * 32; c0 < p.n_tile; c0 += 128) {
            const int col0 = n0 + c0;
            if (col0 >= p.N) break;                      // warp-uniform
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr_row + static_cast<uint32_t>(c0), v);
            tmem_ld_wait();
            const int ncols = min(32, min(p.N - col0, p.n_tile - c0));
            if (!ri.valid) continue;
            float val[32];
            value_chunk<false>(e, ri, v, val, sb + c0, col0, ncols, p.N);
            const bool full = (ncols == 32);
            if (e.out_f32 != nullptr) {
              float* o = e.out_f32 + static_cast<size_t>(ri.orow) * e.ld_f32 + col0;
              if (full && (e.ld_f32 & 7) == 0) {
                store_f32_chunk(o, val);
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (j < ncols) o[j] = val[j];
              }
            }
            if (e.out_op != nullptr) {
              const bool vec = full && ((e.ld_op & 15) == 0);
              store_op_chunk<TF32>(e.out_op, static_cast<size_t>(ri.orow) * e.ld_op + col0, val, ncols, vec);
            }
          }
        }
      }
      // release this accumulator stage
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (threadIdx.x == 64) TRACE_TILE(lt, 3);       // epilogue done
    }
  }

  if (p.use_tma && warp >= 2 && ((warp - 2) & 3) == 0 && lane == 0) bulk_wait_read0();   // outstanding TMA stores have read their slabs (they complete with the grid)
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) TRACE(7);              // all tiles of this CTA done
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
template <int EPI, bool TF32>
const char* launch_cfg(cudaStream_t s, const CUtensorMap& ta, const CUtensorMap& tw, const CUtensorMap& top,
                       const CUtensorMap& tf32m, const GemmDev& d, int num_sms) {
  auto kern = gemm_tcgen05_kernel<EPI, TF32>;
  if (!smem_opt_in(kern, SMEM_TOTAL)) return "gemm: cudaFuncSetAttribute(smem) failed";
  const int tiles = ((d.M + BM - 1) / BM) * ((d.N + d.n_tile - 1) / d.n_tile);
  const int grid = tiles < num_sms ? tiles : num_sms;
  if (launch_pdl(kern, dim3(grid), dim3(NUM_THREADS), SMEM_TOTAL, s, ta, tw, top, tf32m, d) != cudaSuccess) {
    cudaGetLastError();
    return "gemm: kernel launch failed";
  }
  return nullptr;
}

}  // namespace

bool gemm_ln_fusable(int N) { return N <= BN_MAX && N >= 32 && (N % 32) == 0; }

const char* launch_gemm(cudaStream_t s, int prec, const GemmProblem& p, const GemmEpilogue& e, int num_sms,
                        int force_bn, unsigned long long* trace) {
  if (p.M <= 0 || p.N <= 0 || p.K <= 0) return "gemm: empty problem";
  const bool tf32 = (prec == PREC_TF32);
  const int m_tiles = (p.M + BM - 1) / BM;
  int n_tile;
  if (e.kind == EPI_LN) {
    if (!gemm_ln_fusable(p.N)) return "gemm: LayerNorm epilogue needs N <= 256 and N % 32 == 0";
    if (e.ld_f32 != p.N && e.out_f32 != nullptr) return "gemm: LayerNorm epilogue expects dense fp32 rows";
    n_tile = p.N;
  } else if (force_bn > 0) {
    n_tile = force_bn;
  } else {
    // Tile width by a two-term cost model fitted to tools/gemm_bn_sweep.py: the kernel is paced by operand ingest
    // (A tile 128 rows + W tile n_tile rows per k-step) and by the epilogue (~ n_tile), and a CTA runs
    // ceil(tiles / SMs) tiles back to back.  N is split evenly and rounded to the UMMA N granularity (16).
    int best = BN_MAX;
    long best_cost = -1;
    for (int bn = BN_MAX; bn >= 64; bn -= 64) {
      const int ntiles = (p.N + bn - 1) / bn;
      const int width = ((p.N + ntiles - 1) / ntiles + 15) / 16 * 16;
      const long rounds = (static_cast<long>(m_tiles) * ntiles + num_sms - 1) / num_sms;
      const long cost = rounds * (128 + width);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = width; }
    }
    n_tile = best;
  }
  if (n_tile > BN_MAX || n_tile < 16 || (n_tile % 16) != 0) return "gemm: bad tile width";
  GemmDev d;
  d.M = p.M; d.N = p.N; d.K = p.K; d.taps = p.taps; d.tap_stride = p.tap_stride; d.row_shift = p.row_shift;
  d.n_tile = n_tile;
  d.e = e;
  d.trace = trace;
  CUtensorMap ta, tw;
  const CUtensorMapDataType op_dt = tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const int op_esz = tf32 ? 4 : 2;
  const uint32_t box_k = tf32 ? 32 : 64;
  if (const char* err = tma_encode_2d(&ta, op_dt, op_esz, p.A, p.K, p.rowsA, p.lda, box_k, BM)) return err;
  if (const char* err = tma_encode_2d(&tw, op_dt, op_esz, p.W, p.ldw, p.N, p.ldw, box_k, n_tile)) return err;
  // Epilogue I/O through TMA slabs: rows map one-to-one (no Conv1d halo remap), columns in 64-wide units.
  CUtensorMap top = ta, tf32m = ta;   // placeholders when unused
  bool use_tma = e.kind != EPI_TAIL && e.rowmap == ROW_IDENT && (p.N % 64 == 0) && (n_tile % 64 == 0);
  if (e.kind == EPI_STD && e.out_f32 != nullptr && e.out_op != nullptr && !tf32) use_tma = false;   // one slab, one output
  if (e.kind == EPI_LN) {
    use_tma = use_tma && n_tile == 256 && (e.resid == nullptr || e.resid == e.out_f32 || e.out_f32 == nullptr);
    if (use_tma && e.resid != nullptr && e.out_f32 == nullptr) use_tma = false;   // residual map is the out_f32 map
  }
  if (use_tma) {
    if (e.out_op != nullptr) {
      if (tma_encode_2d(&top, op_dt, op_esz, e.out_op, p.N, p.M, e.ld_op, box_k, BM)) use_tma = false;
    }
    if (use_tma && e.out_f32 != nullptr) {
      if (tma_encode_2d(&tf32m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, e.out_f32, p.N, p.M, e.ld_f32, 32, BM)) use_tma = false;
    }
  }
  d.use_tma = use_tma ? 1 : 0;
  switch (e.kind) {
    case EPI_STD: return tf32 ? launch_cfg<EPI_STD, true>(s, ta, tw, top, tf32m, d, num_sms) : launch_cfg<EPI_STD, false>(s, ta, tw, top, tf32m, d, num_sms);
    case EPI_TAIL: return tf32 ? launch_cfg<EPI_TAIL, true>(s, ta, tw, top, tf32m, d, num_sms) : launch_cfg<EPI_TAIL, false>(s, ta, tw, top, tf32m, d, num_sms);
    case EPI_LN:
      if (use_tma) return tf32 ? launch_cfg<EPI_LN_TMA, true>(s, ta, tw, top, tf32m, d, num_sms) : launch_cfg<EPI_LN_TMA, false>(s, ta, tw, top, tf32m, d, num_sms);
      return tf32 ? launch_cfg<EPI_LN, true>(s, ta, tw, top, tf32m, d, num_sms) : launch_cfg<EPI_LN, false>(s, ta, tw, top, tf32m, d, num_sms);
    default: return "gemm: unknown epilogue";
  }
}

}  // namespace avsep
