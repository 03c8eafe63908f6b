// A whole transformer stack in one persistent kernel (d_model = 256, 4 heads of 64, hidden 1024, bf16 operands):
//
//   self  : nn.TransformerEncoderLayer x L (pre-norm, ReLU FFN)        model.py:48-52,59,97-101,111;
//                                                                       torch/nn/modules/transformer.py:946-950
//   cross : CrossAttentionLayer x L (audio queries, visual keys/values, erf-GELU FFN)   model.py:152-173
//
// One CTA owns a tile of whole utterances (U = 2 for 33..64 rows each: two 63-frame audio clips or two 50-frame lip
// sequences; U is a power of two and utterance u sits at tile rows [u * 128/U, +len), so the attention blocks line up
// with 32-column parts) through EVERY layer of the stack.  The fp32 residual stream of the tile lives in
// tensor memory (256 of the 512 columns) for the whole kernel: out_proj and linear2 accumulate straight onto it
// (D += A B with D = the residual), so no residual ever goes through shared memory, L2 or HBM between sub-layers.
// The only traffic in the steady state is the weight stream: 1.5 MB per layer, prepacked as 32 KB shared-memory
// images in consumption order and pulled by 1-D bulk copies (tools/tma_rate.cu: 88 B/clk/SM with 32 KB copies against
// 41 B/clk/SM for the 16 KB tensor boxes the stand-alone GEMM kernels use).
//
// Roles (18 warps): warp 0 lane 0 streams weights (3-slot ring) and the x / K / V tiles; warp 1 lane 0 issues every
// tcgen05.mma; warps 2..17 are "row" warps: thread = (tile row r = TMEM lane, column part p of 4).
// 18 warps cap every thread at 96 registers, and with the shared-memory carve-out this kernel needs L1 has no room
// for spilled registers (every spill is an L2 round trip): hot loops are written to stay inside the cap.  (setmaxnreg
// with a 20-warp layout was tried: ptxas then spills several times more in the row-warp code.)
//
// Tensor memory map (columns): X [0,256) residual | W [256,512) work area:
//   attention, per head h:  W[0,128)  Q_h|K_h accumulator -> S = Q K^T -> P (bf16 pairs, first 64 columns)
//                           W[128,192) V_h accumulator -> O_h = P V accumulator
//                           W[192,224) Q_h as a bf16 A operand | W[224,256) O_h / rowsum as a bf16 A operand
//   FFN, per 128-wide hidden chunk j: W[(j&1)*128, +128) accumulator of linear1 -> H_j (bf16 pairs, first 64 columns),
//                           which linear2 reads as its A operand while accumulating onto X.
// Per head:  QKV_h = LN1(x) Wqkv_h^T (+bias) ; S = (Q scale) K^T ; block-diagonal softmax (an utterance attends only to
// itself) ; O = P V / rowsum ; X += O Wo[:, h]^T.  The bias of out_proj / linear2 is added when the next LayerNorm
// pass reads X (and written back), so X is always the true residual.
//
// Measured limits that shape the schedule (tools/tmem_rate.cu, tools/mma_rate.cu): tcgen05.ld drains tensor memory at
// ~57 B/clk/SM whatever the number of warps, tcgen05.st fills it at > 500 B/clk; M128 N128 K16 = 64 clk.
#include "common.cuh"
#include "kernels.h"

#include <stdlib.h>
#include <string.h>

#include <type_traits>
#include <vector>

namespace avsep {

namespace {

constexpr int D = 256, HID = 1024, NH = 4, HDIM = 64, NCHUNK = 8;
constexpr int SLAB = 16384;                       // 128 rows x 128 B
constexpr int ITEM = 32768;                       // one weight item of the stream
constexpr int NSLOT = 3;
constexpr int OFF_A = 0;                          // LayerNorm output (A operand, 4 k-slabs); x / output staging slabs 0..3
constexpr int OFF_RING = OFF_A + 4 * SLAB;        // weight ring; its first 64 KB double as staging slabs 4..7
constexpr int OFF_KT = OFF_RING + NSLOT * ITEM;   // K_h tile [keys x 64] K-major
constexpr int OFF_VT = OFF_KT + SLAB;             // V_h tile [keys x 64] (MN-major B operand of P V)
constexpr int OFF_RED = OFF_VT + SLAB;            // 2 x [128 rows][4 parts] float2
// per-layer vector block = first item of every layer in the weight stream
constexpr int VEC_BQKV = 0, VEC_BO = 768, VEC_B1 = 1024, VEC_B2 = 2048, VEC_N1G = 2304, VEC_N1B = 2560,
              VEC_N2G = 2816, VEC_N2B = 3072, VEC_B0 = 3328, VEC_FLOATS = 3584;   // VEC_B0: bias of the input projection (layer 0)
constexpr int OFF_VEC = OFF_RED + 2 * 4096;
constexpr int OFF_PEND = OFF_VEC + VEC_FLOATS * 4;   // [256] bias carried into the next LayerNorm | final gamma | beta
constexpr int OFF_BAR = OFF_PEND + 3 * 1024;
constexpr int STACK_SMEM = OFF_BAR + 512;
static_assert(STACK_SMEM <= 227 * 1024, "xformer_stack: shared memory budget exceeded");
constexpr int STACK_THREADS = 32 * 18;
constexpr int ITEMS_SELF = 49, ITEMS_CROSS = 41;   // vector block + weights

constexpr uint32_t TM_X = 0, TM_W = 256;          // tensor-memory column bases
constexpr uint32_t TW_S = 0, TW_V = 128, TW_QOP = 192, TW_OOP = 224;

struct StackDev {
  const uint8_t* wstream;       // n_layers x items x 32 KB, consumption order (see xformer_pack_*)
  const float *fin_gamma, *fin_beta;
  int n_layers, items_per_layer, cross;
  int L, U, stride, B, n_tiles; // rows per utterance, utterances per tile, tile rows per utterance slot (128 / U)
  int act;
  int out_x, out_op;
  int kv_ld_layer;              // cross: column offset between layers in the K|V matrix (2 * D)
  float qscale;
  // SeparationDecoder fused behind the last layer (model.py:201-220): Linear(256 -> 512) + GELU, Linear(512 -> S*F),
  // sigmoid, x mixed_spec, (B,S,F,T) stores.  decoder != 0: the stream holds 1 + 8 + 4 * nc3 more items per tile.
  int decoder, nc3, SF, F, S;
  const float* mixed;
  float *masks, *separated;
  // Input projection fused in front of layer 0 (self stacks): x = act(sum_tap A[row + tap] W_tap^T + b0) + PE[t], with
  // A = bf16 rows [*, pro_ks * 64] (pro_pitch rows per utterance; tap = row shift), W as pro_taps * pro_ks stream items
  // ahead of layer 0, PE = fp32 [*, 256].  pro_taps == 0: x comes from x_in instead.
  //   audio  (model.py:56-58): Conv1d(256 -> 256, k = 3, pad 1) + ReLU on the zero-haloed Conv1d #1 output, + PE
  //   visual (model.py:108-110): frame_proj Linear(128 -> 256) on the pooled CNN features, + PE
  int pro_taps, pro_ks, pro_pitch, pro_relu;
  const float* pe;
  // K | V projection of the fusion layers fused behind the last layer (visual stack; replaces out_x / out_op): the
  // stack output rows are interpolated to kvp_L rows per utterance (F.interpolate linear, align_corners=False;
  // model.py:114-116) and multiplied by the kvp_chunks * 128 stacked K | V weight rows of every fusion layer
  // (model.py:155,169; functional.py:5847-5865): out = bf16 [B * kvp_L, kvp_ld].  kvp_chunks == 0: off.
  int kvp_chunks, kvp_L, kvp_ld;
  float kvp_scale;              // lerp_scale(L, kvp_L), from the host so that the uniform kernel has no division
  __nv_bfloat16* kvp_out;
  // variable-length batch (null: all L / all kvp_L): rows of each utterance that are real, K | V interpolation targets
  const int *lens, *kvp_lens;
  long long* trace;             // optional [grid][256] clock64 stamps of the CTA's first tile (debug), else null:
                                //   row thread (warp 2 lane 0) in [0,128), MMA thread in [128,256); see tools/stack_trace.py
};

#define XTRACE(slot) do { if (p.trace != nullptr && lt == 0 && (slot) < 128) p.trace[blockIdx.x * 256 + trace_base + (slot)] = clock64(); } while (0)

// Weight items are read by every CTA of every launch: keep them in L2 (evict_last) against the step's streaming traffic
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void prefetch_l2_line(const void* g) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<uint64_t>(g)));
}

__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// VARLEN = false (no length arrays): every per-utterance length is p.L / p.kvp_L at compile time, so the uniform
// batch runs exactly the code it ran before variable-length batches existed.
template <bool VARLEN>
__global__ void __launch_bounds__(STACK_THREADS, 1)
xformer_stack_kernel(const __grid_constant__ CUtensorMap tmXin, const __grid_constant__ CUtensorMap tmXout,
                     const __grid_constant__ CUtensorMap tmOp, const __grid_constant__ CUtensorMap tmKV,
                     const StackDev p) {
  extern __shared__ __align__(1024) uint8_t smem_stack[];
  const int* const lens = VARLEN ? p.lens : nullptr;
  const int* const kvp_lens = VARLEN ? p.kvp_lens : nullptr;
  uint8_t* const smem = smem_stack;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* w_full = bars;                 // [3]
  uint64_t* w_empty = bars + 3;            // [3]
  uint64_t* x_full = bars + 6;             // x tile staged
  uint64_t* x_taken = bars + 7;            // (16) staging copied into tensor memory
  uint64_t* stage_free = bars + 8;         // (4) output stores have read the staging slabs
  uint64_t* a_ready = bars + 9;            // (16) LayerNorm output in smem, X updated
  uint64_t* qk_full = bars + 10;           // Q_h | K_h accumulators complete
  uint64_t* qop_ready = bars + 11;         // (16) Q operand in tensor memory, K tile in shared memory
  uint64_t* s_full = bars + 12;
  uint64_t* p_ready = bars + 13;           // (16)
  uint64_t* o_full = bars + 14;
  uint64_t* o_ready = bars + 15;           // (16)
  uint64_t* kv_full = bars + 16;           // cross: K_h / V_h tiles landed
  uint64_t* kv_empty = bars + 17;          // cross: P V of the head complete
  uint64_t* attn_done = bars + 18;
  uint64_t* acc1_full = bars + 19;         // [2]
  uint64_t* h_full = bars + 21;            // [2] (16)
  uint64_t* ffn_done = bars + 23;
  uint64_t* v_full = bars + 24;            // self: V_h accumulator complete
  uint64_t* v_ready = bars + 25;           // (16) self: V tile in shared memory
  uint64_t* pa_full = bars + 26;           // [4] input projection: A slab landed
  uint64_t* pa_free = bars + 30;           // [4] input projection: the MMAs have read the A slab
  uint64_t* x_ready = bars + 34;           // input projection complete (X holds the pre-activation rows)
  uint64_t* kv_stage_free = bars + 35;     // (16) K|V projection: the fp32 staging in the ring has been read
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);
  float2* red = reinterpret_cast<float2*>(smem + OFF_RED);
  float* vec = reinterpret_cast<float*>(smem + OFF_VEC);
  float* pend = reinterpret_cast<float*>(smem + OFF_PEND);
  float* fin_g = pend + 256;
  float* fin_b = pend + 512;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmXin);
    if (p.out_x) tma_prefetch_desc(&tmXout);
    if (p.out_op) tma_prefetch_desc(&tmOp);
    if (p.cross || p.pro_taps) tma_prefetch_desc(&tmKV);
    for (int i = 0; i < NSLOT; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    mbar_init(x_full, 1);
    mbar_init(x_taken, 16);
    mbar_init(stage_free, 4);
    mbar_init(a_ready, 16);
    mbar_init(qk_full, 1);
    mbar_init(qop_ready, 16);
    mbar_init(s_full, 1);
    mbar_init(p_ready, 16);
    mbar_init(o_full, 1);
    mbar_init(o_ready, 16);
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    mbar_init(attn_done, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc1_full[i], 1); mbar_init(&h_full[i], 16); }
    mbar_init(ffn_done, 1);
    mbar_init(v_full, 1);
    mbar_init(v_ready, 16);
    for (int i = 0; i < 4; ++i) { mbar_init(&pa_full[i], 1); mbar_init(&pa_free[i], 1); }
    mbar_init(x_ready, 1);
    mbar_init(kv_stage_free, 16);
    fence_mbar_init();
  }
  for (int i = threadIdx.x; i < D; i += STACK_THREADS) {
    fin_g[i] = p.fin_gamma ? __ldg(p.fin_gamma + i) : 1.f;
    fin_b[i] = p.fin_beta ? __ldg(p.fin_beta + i) : 0.f;
  }
  // K / V tiles: rows the TMA loads of the cross-attention path never write (past an utterance's length) must be
  // finite: P is 0 there, and 0 x NaN would poison real rows
  for (int i = threadIdx.x; i < 2 * SLAB / 16; i += STACK_THREADS)
    *reinterpret_cast<uint4*>(smem + OFF_KT + i * 16) = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async_smem();
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmX = tmem_base + TM_X, tmW = tmem_base + TM_W;
  const int n_pro = p.pro_taps * p.pro_ks;      // stream items of the input projection (ahead of layer 0)
  griddep_launch_dependents();
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- producer: x tile, weight stream (incl. the per-layer vector block), (cross) K / V tiles ------
      uint32_t wn = 0;          // stream items issued
      uint32_t an = 0;          // input-projection A slabs issued
      uint32_t hn = 0;          // heads whose K/V tiles were issued (cross)
      const uint32_t box_bytes = static_cast<uint32_t>(p.L) * 128u;
      const uint64_t pol = l2_policy_evict_last();
      auto load_item = [&](const uint8_t* src) {
        const uint32_t slot = wn % NSLOT, use = wn / NSLOT;
        mbar_wait(&w_empty[slot], (use & 1) ^ 1);
        mbar_arrive_expect_tx(&w_full[slot], ITEM);
        bulk_load_1d(smem + OFF_RING + slot * ITEM, src, ITEM, &w_full[slot], pol);
        ++wn;
      };
      int lt = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++lt) {
        const int utt0 = tile * p.U;
        auto load_kv = [&](int l, int h) {
          if (hn > 0) mbar_wait(kv_empty, (hn - 1) & 1);
          mbar_arrive_expect_tx(kv_full, 2u * p.U * box_bytes);
          for (int u = 0; u < p.U; ++u) {
            tma_load_2d(smem + OFF_KT + u * p.stride * 128, &tmKV, kv_full, l * p.kv_ld_layer + h * HDIM, (utt0 + u) * p.L);
            tma_load_2d(smem + OFF_VT + u * p.stride * 128, &tmKV, kv_full, l * p.kv_ld_layer + D + h * HDIM, (utt0 + u) * p.L);
          }
          ++hn;
        };
        if (lt > 0) mbar_wait(stage_free, (lt - 1) & 1);
        if (p.pro_taps) {
          // input projection: A slabs (tensor map tmKV: boxes of a whole utterance slot, so that every tile row holds
          // finite data) through a 4-slot ring in the operand area, one weight item per slab
          const uint8_t* src = p.wstream;
          int st = 0;
          for (int tap = 0; tap < p.pro_taps; ++tap)
            for (int ks = 0; ks < p.pro_ks; ++ks, ++st, ++an) {
              const uint32_t sa = an & 3;
              mbar_wait(&pa_free[sa], ((an >> 2) & 1) ^ 1);
              mbar_arrive_expect_tx(&pa_full[sa], static_cast<uint32_t>(p.U * p.stride) * 128u);
              for (int u = 0; u < p.U; ++u)
                tma_load_2d(smem + OFF_A + sa * SLAB + u * p.stride * 128, &tmKV, &pa_full[sa], ks * 64,
                            (utt0 + u) * p.pro_pitch + tap);
              load_item(src + static_cast<size_t>(st) * ITEM);
            }
        } else {
          mbar_arrive_expect_tx(x_full, 8u * p.U * box_bytes);
          for (int s = 0; s < 8; ++s)
            for (int u = 0; u < p.U; ++u)
              tma_load_2d(smem + OFF_A + s * SLAB + u * p.stride * 128, &tmXin, x_full, s * 32, (utt0 + u) * p.L);
          mbar_wait(x_taken, lt & 1);            // staging (a_op + first two ring slots) is free again
        }
        for (int l = 0; l < p.n_layers; ++l) {
          const uint8_t* src = p.wstream + static_cast<size_t>(n_pro + l * p.items_per_layer) * ITEM;
          load_item(src);                      // vector block
          src += ITEM;
          if (!p.cross) {
            for (int i = 0; i < 16; ++i) load_item(src + static_cast<size_t>(i) * ITEM);
            src += 16 * ITEM;
          } else {
            // consumption order: Q_0 | per head h: Q_{h+1}, Wo_h ; K/V tiles of head h+1 once P V of head h is done
            load_item(src);
            load_kv(l, 0);
            int it = 1;
            for (int h = 0; h < NH; ++h) {
              if (h + 1 < NH) {
                load_item(src + static_cast<size_t>(it++) * ITEM);
                load_kv(l, h + 1);
              }
              load_item(src + static_cast<size_t>(it++) * ITEM);
            }
            src += 8 * ITEM;
          }
          for (int i = 0; i < 32; ++i) load_item(src + static_cast<size_t>(i) * ITEM);
        }
        if (p.decoder) {
          const uint8_t* src = p.wstream + static_cast<size_t>(n_pro + p.n_layers * p.items_per_layer) * ITEM;
          const int n = 1 + 8 + 4 * p.nc3;
          for (int i = 0; i < n; ++i) load_item(src + static_cast<size_t>(i) * ITEM);
        }
        if (p.kvp_chunks) {
          const uint8_t* src = p.wstream + static_cast<size_t>(n_pro + p.n_layers * p.items_per_layer) * ITEM;
          mbar_wait(kv_stage_free, lt & 1);       // the ring doubled as the fp32 staging of the interpolation
          for (int i = 0; i < 1 + 2 * p.kvp_chunks; ++i) load_item(src + static_cast<size_t>(i) * ITEM);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ---------------- MMA issuer ----------------
      constexpr uint32_t ID128 = umma_idesc(1u, 128, 128);
      constexpr uint32_t ID64 = umma_idesc(1u, 128, 64);
      constexpr uint32_t ID64_MN = umma_idesc(1u, 128, 64, 0, 1);      // B (= V) MN-major
      uint32_t wn = 0, n_a = 0, n_h = 0, c1n = 0, c2n = 0;
      uint32_t cur_slot = 0;
      auto next_item = [&]() -> uint32_t {
        cur_slot = wn % NSLOT;
        mbar_wait(&w_full[cur_slot], (wn / NSLOT) & 1);
        tc_fence_after();
        ++wn;
        return smem_u32(smem + OFF_RING + cur_slot * ITEM);
      };
      const uint32_t a_base = smem_u32(smem + OFF_A);
      // Q_h | K_h (self: N = 128 into W[0,128), two items) or Q_h (cross: N = 64 into W[0,64), one item)
      auto issue_qk = [&]() {
        if (!p.cross) {
          for (int it = 0; it < 2; ++it) {
            const uint32_t base = next_item();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              const int ks = 2 * it + half;
              const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
              const uint64_t bdesc = umma_desc_kmajor_sw128(base + half * SLAB, 1024);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16(tmW + TW_S, adesc + 2 * kk, bdesc + 2 * kk, ID128, (ks | kk) != 0 ? 1u : 0u);
            }
            umma_commit(&w_empty[cur_slot]);
          }
        } else {
          const uint32_t base = next_item();
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
            const uint64_t bdesc = umma_desc_kmajor_sw128(base + ks * 8192, 1024);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_f16(tmW + TW_S, adesc + 2 * kk, bdesc + 2 * kk, ID64, (ks | kk) != 0 ? 1u : 0u);
          }
          umma_commit(&w_empty[cur_slot]);
        }
        umma_commit(qk_full);
      };
      // V_h : N = 64 into W[128,192) (self-attention); its epilogue runs under the S = Q K^T round trip
      auto issue_v = [&]() {
        const uint32_t base = next_item();
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
          const uint64_t bdesc = umma_desc_kmajor_sw128(base + ks * 8192, 1024);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16(tmW + TW_V, adesc + 2 * kk, bdesc + 2 * kk, ID64, (ks | kk) != 0 ? 1u : 0u);
        }
        umma_commit(&w_empty[cur_slot]);
        umma_commit(v_full);
      };
      constexpr int trace_base = 128;
      int lt = 0;
      XTRACE(0);
      uint32_t am = 0;                             // input-projection A slabs consumed
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++lt) {
        if (p.pro_taps) {
          // X = sum over (tap, k-slab) of A_slab W_item^T : two 128-column halves per item
          for (int st = 0; st < n_pro; ++st, ++am) {
            const uint32_t sa = am & 3;
            mbar_wait(&pa_full[sa], (am >> 2) & 1);
            const uint32_t base = next_item();
            const uint64_t adesc = umma_desc_kmajor_sw128(a_base + sa * SLAB, 1024);
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const uint64_t bdesc = umma_desc_kmajor_sw128(base + hf * SLAB, 1024);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16(tmX + hf * 128, adesc + 2 * kk, bdesc + 2 * kk, ID128, (st | kk) != 0 ? 1u : 0u);
            }
            umma_commit(&w_empty[cur_slot]);
            umma_commit(&pa_free[sa]);
          }
          umma_commit(x_ready);
        }
        for (int l = 0; l < p.n_layers; ++l) {
          const int tb = 1 + l * 60;               // MMA-thread stamps of layer l: tb + 0 LN1 seen; per head 6; FFN per chunk 3
          ++wn;                                    // the layer's vector block is consumed by the row warps
          // ======== attention sub-layer ========
          mbar_wait(a_ready, n_a & 1); ++n_a;
          tc_fence_after();
          XTRACE(tb);
          issue_qk();
          if (!p.cross) issue_v();
          for (int h = 0; h < NH; ++h, ++n_h) {
            const int th = tb + 1 + h * 6;
            // S = Q K^T : A = Q_h from tensor memory, B = K tile
            mbar_wait(qop_ready, n_h & 1);
            if (p.cross) mbar_wait(kv_full, n_h & 1);
            tc_fence_after();
            XTRACE(th);                                     // Q operand / K tile seen
            {
              const uint64_t kdesc = umma_desc_kmajor_sw128(smem_u32(smem + OFF_KT), 1024);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16_ts(tmW + TW_S, tmW + TW_QOP + kk * 8, kdesc + 2 * kk, ID128, kk != 0 ? 1u : 0u);
            }
            umma_commit(s_full);
            XTRACE(th + 1);                                 // S_h issued
            // O = P V : A = P from tensor memory (K = 128 keys), B = V tile (MN-major)
            mbar_wait(p_ready, n_h & 1);
            if (!p.cross) mbar_wait(v_ready, n_h & 1);
            tc_fence_after();
            XTRACE(th + 2);                                 // P and V seen
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
              const uint64_t vdesc = umma_desc_mnmajor_sw128(smem_u32(smem + OFF_VT + ks * 2048), 1024, 1024);
              umma_f16_ts(tmW + TW_V, tmW + TW_S + ks * 8, vdesc, ID64_MN, ks != 0 ? 1u : 0u);
            }
            umma_commit(o_full);
            if (p.cross) umma_commit(kv_empty);
            // the next head's Q | K projection runs under this head's output epilogue (W[0,128) is free once P V has
            // read P: the tensor pipe executes in issue order)
            if (h + 1 < NH) issue_qk();
            // X += O_h Wo[:, h*64 : (h+1)*64]^T : A = O_h from tensor memory, two 128-row halves of Wo
            mbar_wait(o_ready, n_h & 1);
            tc_fence_after();
            XTRACE(th + 3);                                 // o_ready seen
            {
              const uint32_t base = next_item();
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const uint64_t bdesc = umma_desc_kmajor_sw128(base + hf * SLAB, 1024);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  umma_f16_ts(tmX + hf * 128, tmW + TW_OOP + kk * 8, bdesc + 2 * kk, ID128, 1u);
              }
              umma_commit(&w_empty[cur_slot]);
            }
            // W[128,192) is free again (the output epilogue has drained O_h): the next head's V projection
            if (!p.cross && h + 1 < NH) issue_v();
          }
          umma_commit(attn_done);
          XTRACE(tb + 25);                                  // attention issued
          // ======== feed-forward sub-layer ========
          mbar_wait(a_ready, n_a & 1); ++n_a;
          tc_fence_after();
          XTRACE(tb + 26);                                  // LN2 seen
          for (int j = 0; j <= NCHUNK; ++j) {
            if (j < NCHUNK) {
              const uint32_t st = c1n & 1;
              for (int it = 0; it < 2; ++it) {
                const uint32_t base = next_item();
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                  const int ks = 2 * it + half;
                  const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
                  const uint64_t bdesc = umma_desc_kmajor_sw128(base + half * SLAB, 1024);
#pragma unroll
                  for (int kk = 0; kk < 4; ++kk)
                    umma_f16(tmW + st * 128, adesc + 2 * kk, bdesc + 2 * kk, ID128, (ks | kk) != 0 ? 1u : 0u);
                }
                umma_commit(&w_empty[cur_slot]);
              }
              umma_commit(&acc1_full[st]);
              XTRACE(tb + 27 + 3 * j);                      // G1_j issued
              ++c1n;
            }
            if (j >= 1) {
              const uint32_t st2 = c2n & 1;
              mbar_wait(&h_full[st2], (c2n >> 1) & 1);
              tc_fence_after();
              XTRACE(tb + 28 + 3 * (j - 1));                // H_{j-1} seen
              for (int ks = 0; ks < 2; ++ks) {
                const uint32_t base = next_item();
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  const uint64_t bdesc = umma_desc_kmajor_sw128(base + hf * SLAB, 1024);
#pragma unroll
                  for (int kk = 0; kk < 4; ++kk)
                    umma_f16_ts(tmX + hf * 128, tmW + st2 * 128 + (ks * 4 + kk) * 8, bdesc + 2 * kk, ID128, 1u);
                }
                umma_commit(&w_empty[cur_slot]);
              }
              XTRACE(tb + 29 + 3 * (j - 1));                // G2_{j-1} issued
              ++c2n;
            }
          }
          umma_commit(ffn_done);
        }
        if (p.decoder) {
          auto wait_h = [&]() {                    // hidden / output chunk c2n has left its accumulator stage
            const uint32_t st2 = c2n & 1;
            mbar_wait(&h_full[st2], (c2n >> 1) & 1);
            tc_fence_after();
            ++c2n;
          };
          mbar_wait(&w_full[wn % NSLOT], (wn / NSLOT) & 1);   // decoder vector block (row warps): see it land (as below)
          ++wn;
          mbar_wait(a_ready, n_a & 1); ++n_a;       // a = fusion.norm(x) in shared memory
          tc_fence_after();
          XTRACE(112);                              // decoder: a seen
          // Linear(256 -> 512): four 128-wide chunks, A = a (smem); GELU'd H goes to tensor memory over X (dead now)
          for (int j = 0; j < 4; ++j, ++c1n) {
            const uint32_t st = c1n & 1;
            if (j >= 2) wait_h();
            for (int it = 0; it < 2; ++it) {
              const uint32_t base = next_item();
#pragma unroll
              for (int half = 0; half < 2; ++half) {
                const int ks = 2 * it + half;
                const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
                const uint64_t bdesc = umma_desc_kmajor_sw128(base + half * SLAB, 1024);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  umma_f16(tmW + st * 128, adesc + 2 * kk, bdesc + 2 * kk, ID128, (ks | kk) != 0 ? 1u : 0u);
              }
              umma_commit(&w_empty[cur_slot]);
            }
            umma_commit(&acc1_full[st]);
          }
          XTRACE(113);                              // decoder: hidden GEMMs issued
          wait_h();
          wait_h();
          XTRACE(114);                              // decoder: H complete in tensor memory
          // Linear(512 -> S*F): chunks of 128 output columns, A = H from tensor memory (K = 512), B streamed
          for (int c = 0; c < p.nc3; ++c, ++c1n) {
            const uint32_t st = c1n & 1;
            if (c >= 2) wait_h();
            for (int it = 0; it < 4; ++it) {
              const uint32_t base = next_item();
#pragma unroll
              for (int half = 0; half < 2; ++half) {
                const uint64_t bdesc = umma_desc_kmajor_sw128(base + half * SLAB, 1024);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  umma_f16_ts(tmW + st * 128, tmX + ((2 * it + half) * 4 + kk) * 8, bdesc + 2 * kk, ID128,
                              (it | half | kk) != 0 ? 1u : 0u);
              }
              umma_commit(&w_empty[cur_slot]);
            }
            umma_commit(&acc1_full[st]);
            XTRACE(115 + c);                        // decoder: output chunk c issued
          }
          for (int c = p.nc3 < 2 ? 0 : p.nc3 - 2; c < p.nc3; ++c) wait_h();
        }
        if (p.kvp_chunks) {
          auto wait_h = [&]() {
            const uint32_t st2 = c2n & 1;
            mbar_wait(&h_full[st2], (c2n >> 1) & 1);
            tc_fence_after();
            ++c2n;
          };
          // K | V bias block: consumed by the row warps, but this thread must see it land before it moves on -- three
          // items later it waits on the same ring slot, and a parity wait is only unambiguous one phase behind (the
          // producer issues the block when the staging is released, i.e. at the same moment this thread starts; the
          // next two items can overtake it)
          mbar_wait(&w_full[wn % NSLOT], (wn / NSLOT) & 1);
          ++wn;
          mbar_wait(a_ready, n_a & 1); ++n_a;       // interpolated rows in shared memory
          tc_fence_after();
          for (int c = 0; c < p.kvp_chunks; ++c, ++c1n) {
            const uint32_t st = c1n & 1;
            if (c >= 2) wait_h();
            for (int it = 0; it < 2; ++it) {
              const uint32_t base = next_item();
#pragma unroll
              for (int half = 0; half < 2; ++half) {
                const int ks = 2 * it + half;
                const uint64_t adesc = umma_desc_kmajor_sw128(a_base + ks * SLAB, 1024);
                const uint64_t bdesc = umma_desc_kmajor_sw128(base + half * SLAB, 1024);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  umma_f16(tmW + st * 128, adesc + 2 * kk, bdesc + 2 * kk, ID128, (ks | kk) != 0 ? 1u : 0u);
              }
              umma_commit(&w_empty[cur_slot]);
            }
            umma_commit(&acc1_full[st]);
          }
          for (int c = p.kvp_chunks < 2 ? 0 : p.kvp_chunks - 2; c < p.kvp_chunks; ++c) wait_h();
        }
      }
    }
  } else {
    // ---------------- row warps: lane quarter q = warp % 4 (TMEM lanes 32q..32q+31), column part = (warp - 2) / 4 ----
    const int q = warp & 3, part = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const int etid = threadIdx.x - 64;                       // 0..511
    const uint32_t lane_sel = static_cast<uint32_t>(q * 32) << 16;
    const bool elected = (warp == 2 + 4 * part) && (lane == 0);
    // block-diagonal attention: row r attends the keys [klo, klo + lk) of its own utterance slot (lk: per tile below)
    const int klo = (r / p.stride) * p.stride;
    const bool row_valid = (r - klo) < p.L;                  // tile rows past the slot pitch are padding
    // this row's valid score columns within the part start at lo_i
    const int lo_i = klo - part * 32;
    // stream items per tile: input projection | layers | decoder block or K|V projection block
    const uint32_t per_tile = static_cast<uint32_t>(n_pro + p.n_layers * p.items_per_layer + (p.decoder ? 1 + 8 + 4 * p.nc3 : 0) +
                                                    (p.kvp_chunks ? 1 + 2 * p.kvp_chunks : 0));
    uint32_t nx = 0;                                         // exchanges through `red` so far (double buffered)
    uint32_t n_h = 0, n_attn = 0, n_ffn = 0, c1n = 0;
    const int trace_base = (threadIdx.x == 64) ? 0 : 1024;   // only the first row thread stamps

    auto exchange = [&](float2 mine, float2 (&all)[4]) {
      float2* buf = red + (nx & 1) * 512 + r * 4;
      ++nx;
      buf[part] = mine;
      named_bar_sync(1 + q, 128);
      all[0] = buf[0]; all[1] = buf[1]; all[2] = buf[2]; all[3] = buf[3];
    };
    // vu[0..63] = X[r, 64 part .. +64) (+ bias, written back so that X stays the true residual); returns sum, sum of squares
    auto read_x = [&](uint32_t (&vu)[64], const float* bias, bool write_back, float& sum, float& sq) {
      tmem_ld_32x32b_x32(tmX + lane_sel + part * 64, reinterpret_cast<uint32_t(&)[32]>(vu[0]));
      tmem_ld_32x32b_x32(tmX + lane_sel + part * 64 + 32, reinterpret_cast<uint32_t(&)[32]>(vu[32]));
      tmem_ld_wait();
      if (bias != nullptr) {
#pragma unroll
        for (int i = 0; i < 64; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(bias + part * 64 + i);
          vu[i] = __float_as_uint(__uint_as_float(vu[i]) + b4.x);
          vu[i + 1] = __float_as_uint(__uint_as_float(vu[i + 1]) + b4.y);
          vu[i + 2] = __float_as_uint(__uint_as_float(vu[i + 2]) + b4.z);
          vu[i + 3] = __float_as_uint(__uint_as_float(vu[i + 3]) + b4.w);
        }
        if (write_back) {
          tmem_st_32x32b_x32(tmX + lane_sel + part * 64, reinterpret_cast<const uint32_t(&)[32]>(vu[0]));
          tmem_st_32x32b_x32(tmX + lane_sel + part * 64 + 32, reinterpret_cast<const uint32_t(&)[32]>(vu[32]));
        }
      }
      sum = 0.f; sq = 0.f;
#pragma unroll
      for (int i = 0; i < 64; ++i) {
        const float x = __uint_as_float(vu[i]);
        sum += x;
        sq = fmaf(x, x, sq);
      }
    };
    // LayerNorm statistics of the full row from the part's (sum, sum of squares): merged over the 4 column parts
    auto row_stats = [&](float sum, float sq, float& mean, float& rstd) {
      const float mean_p = sum * (1.0f / 64.0f);
      float2 all[4];
      exchange(make_float2(mean_p, fmaxf(sq - sum * mean_p, 0.f)), all);
      mean = 0.25f * ((all[0].x + all[1].x) + (all[2].x + all[3].x));
      const float d0 = all[0].x - mean, d1 = all[1].x - mean, d2 = all[2].x - mean, d3 = all[3].x - mean;
      const float m2 = (all[0].y + all[1].y) + (all[2].y + all[3].y) + 64.0f * ((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3));
      rstd = rsqrtf(m2 * (1.0f / 256.0f) + 1e-5f);
    };
    // (v - mean) * rstd * g + b as bf16 -> k-slab `part` of the 128-row x 256-column operand image at `base`
    // (128B-swizzled, K-major); eight columns at a time so that the row slice dies as it is stored
    auto store_op_row = [&](const uint32_t (&vu)[64], float mean, float rstd, const float* g, const float* b,
                            uint8_t* base) {
      uint8_t* slab = base + part * SLAB;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; i += 4) {
          const float4 g4 = *reinterpret_cast<const float4*>(g + part * 64 + c * 8 + i);
          const float4 b4 = *reinterpret_cast<const float4*>(b + part * 64 + c * 8 + i);
          y[i] = fmaf((__uint_as_float(vu[c * 8 + i]) - mean) * rstd, g4.x, b4.x);
          y[i + 1] = fmaf((__uint_as_float(vu[c * 8 + i + 1]) - mean) * rstd, g4.y, b4.y);
          y[i + 2] = fmaf((__uint_as_float(vu[c * 8 + i + 2]) - mean) * rstd, g4.z, b4.z);
          y[i + 3] = fmaf((__uint_as_float(vu[c * 8 + i + 3]) - mean) * rstd, g4.w, b4.w);
        }
        uint4 w;
        w.x = pack_bf16x2(y[0], y[1]); w.y = pack_bf16x2(y[2], y[3]);
        w.z = pack_bf16x2(y[4], y[5]); w.w = pack_bf16x2(y[6], y[7]);
        *reinterpret_cast<uint4*>(slab + sw128_off(r, c)) = w;
      }
    };
    auto ln_to_a = [&](const float* bias, const float* g, const float* b) {
      uint32_t vu[64];
      float sum, sq, mean, rstd;
      read_x(vu, bias, true, sum, sq);
      row_stats(sum, sq, mean, rstd);
      store_op_row(vu, mean, rstd, g, b, smem + OFF_A);
      tmem_st_wait();
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready);
    };

    int lt = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++lt) {
      const int utt0 = tile * p.U;
      // keys of this row's utterance (p.L unless the batch has per-utterance lengths); the rows of the slot in
      // [lk, L) are computed like any other row but no row attends to them
      const int lk = VARLEN ? utt_len(lens, min(utt0 + r / p.stride, p.B - 1), p.L) : p.L;
      // ---- residual tile: staging slabs (fp32, 32 columns each) -> tensor memory ----
      XTRACE(0);
      if (!p.pro_taps) {
      mbar_wait(x_full, lt & 1);
      XTRACE(1);                                             // x staged
      {
        uint32_t u[32];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint8_t* slab = smem + OFF_A + (part * 2 + c) * SLAB;
          if (row_valid) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint4 w = *reinterpret_cast<const uint4*>(slab + sw128_off(r, i));
              u[4 * i] = w.x; u[4 * i + 1] = w.y; u[4 * i + 2] = w.z; u[4 * i + 3] = w.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) u[i] = 0u;
          }
          tmem_st_32x32b_x32(tmX + lane_sel + part * 64 + c * 32, u);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(x_taken);
      }
      }
      if (p.decoder) {
        // the tile's mixture planes (contiguous: utterances utt0 .. utt0 + U - 1) are wanted in L2 by the decoder phase
        const int n_utt = p.B - utt0 < p.U ? p.B - utt0 : p.U;
        const size_t bytes = static_cast<size_t>(n_utt) * p.F * p.L * sizeof(float);
        const uint8_t* base = reinterpret_cast<const uint8_t*>(p.mixed + static_cast<size_t>(utt0) * p.F * p.L);
        for (size_t off = static_cast<size_t>(etid) * 128; off < bytes; off += 512 * 128) prefetch_l2_line(base + off);
      }
      for (int l = 0; l < p.n_layers; ++l) {
        // ---- per-layer vectors: first item of the layer in the weight stream (it was prefetched under the previous
        // layer's FFN); the previous layer's linear2 bias is carried into this layer's first LayerNorm ----
        const uint32_t vn = static_cast<uint32_t>(lt) * per_tile + static_cast<uint32_t>(n_pro + l * p.items_per_layer);
        const uint32_t vslot = vn % NSLOT;
        if (l == 0 && p.pro_taps) {
          // the projection items went through the same ring slots: only once they are all consumed does a wait on the
          // slot's parity mean "the vector block has landed" (a waiter may be at most one phase behind)
          mbar_wait(x_ready, lt & 1);
          tc_fence_after();
          XTRACE(1);                                         // projection complete
        }
        named_bar_sync(5, 512);                              // every row warp is done with the previous vectors
        if (l > 0 && etid < D) pend[etid] = vec[VEC_B2 + etid];
        mbar_wait(&w_full[vslot], (vn / NSLOT) & 1);
        named_bar_sync(5, 512);
        {
          const float4* src = reinterpret_cast<const float4*>(smem + OFF_RING + vslot * ITEM);
          float4* dst = reinterpret_cast<float4*>(vec);
          for (int i = etid; i < VEC_FLOATS / 4; i += 512) dst[i] = src[i];
        }
        named_bar_sync(5, 512);
        if (etid == 0) mbar_arrive(&w_empty[vslot]);
        tc_fence_after();
        const int tb = 2 + l * 60;     // row-thread stamps of layer l: +0 LN1 start, +1 LN1 done; per head 6; +26.. FFN
        XTRACE(tb);
        if (l == 0 && p.pro_taps) {
          // input projection epilogue, in place: X = act(X + b0) + PE[t] (32 columns at a time)
          const float* per = p.pe + static_cast<size_t>(row_valid ? r - klo : 0) * D + part * 64;
          const float* b0 = vec + VEC_B0 + part * 64;
#pragma unroll
          for (int hc = 0; hc < 2; ++hc) {
            float4 pv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) pv[i] = __ldg(reinterpret_cast<const float4*>(per + hc * 32) + i);
            uint32_t v[32];
            tmem_ld_32x32b_x32(tmX + lane_sel + part * 64 + hc * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b4 = *reinterpret_cast<const float4*>(b0 + hc * 32 + 4 * i);
              float x0 = __uint_as_float(v[4 * i]) + b4.x, x1 = __uint_as_float(v[4 * i + 1]) + b4.y;
              float x2 = __uint_as_float(v[4 * i + 2]) + b4.z, x3 = __uint_as_float(v[4 * i + 3]) + b4.w;
              if (p.pro_relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); x2 = fmaxf(x2, 0.f); x3 = fmaxf(x3, 0.f); }
              v[4 * i] = __float_as_uint(x0 + pv[i].x); v[4 * i + 1] = __float_as_uint(x1 + pv[i].y);
              v[4 * i + 2] = __float_as_uint(x2 + pv[i].z); v[4 * i + 3] = __float_as_uint(x3 + pv[i].w);
            }
            tmem_st_32x32b_x32(tmX + lane_sel + part * 64 + hc * 32, v);
          }
          tmem_st_wait();
        }
        ln_to_a(l > 0 ? pend : nullptr, vec + VEC_N1G, vec + VEC_N1B);
        XTRACE(tb + 1);

        // ======== attention ========
        for (int h = 0; h < NH; ++h, ++n_h) {
          const int th = tb + 2 + h * 6;
          // ---- Q (scaled, bf16, back into tensor memory as an A operand); K (bf16) into its shared-memory tile ----
          mbar_wait(qk_full, n_h & 1);
          tc_fence_after();
          XTRACE(th);                                        // Q_h | K_h accumulators complete
          {
            uint32_t a[16];
            tmem_ld_32x32b_x16(tmW + lane_sel + TW_S + part * 16, a);
            tmem_ld_wait();
            uint32_t qp[8];
            const float* bq = vec + VEC_BQKV + h * HDIM + part * 16;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              qp[i] = pack_bf16x2((__uint_as_float(a[2 * i]) + bq[2 * i]) * p.qscale,
                                  (__uint_as_float(a[2 * i + 1]) + bq[2 * i + 1]) * p.qscale);
            tmem_st_32x32b_x8(tmW + lane_sel + TW_QOP + part * 8, qp);
            if (!p.cross) {
              tmem_ld_32x32b_x16(tmW + lane_sel + TW_S + 64 + part * 16, a);
              tmem_ld_wait();
              const float* bk = vec + VEC_BQKV + D + h * HDIM + part * 16;
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                uint4 w;
                w.x = pack_bf16x2(__uint_as_float(a[8 * c]) + bk[8 * c], __uint_as_float(a[8 * c + 1]) + bk[8 * c + 1]);
                w.y = pack_bf16x2(__uint_as_float(a[8 * c + 2]) + bk[8 * c + 2], __uint_as_float(a[8 * c + 3]) + bk[8 * c + 3]);
                w.z = pack_bf16x2(__uint_as_float(a[8 * c + 4]) + bk[8 * c + 4], __uint_as_float(a[8 * c + 5]) + bk[8 * c + 5]);
                w.w = pack_bf16x2(__uint_as_float(a[8 * c + 6]) + bk[8 * c + 6], __uint_as_float(a[8 * c + 7]) + bk[8 * c + 7]);
                *reinterpret_cast<uint4*>(smem + OFF_KT + sw128_off(r, part * 2 + c)) = w;
              }
              fence_proxy_async_smem();
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(qop_ready);
          }
          XTRACE(th + 1);                                    // Q operand / K tile written
          // ---- V_h (bf16) into its shared-memory tile (self-attention; cross-attention gets it by TMA) ----
          if (!p.cross) {
            mbar_wait(v_full, n_h & 1);
            tc_fence_after();
            uint32_t a[16];
            tmem_ld_32x32b_x16(tmW + lane_sel + TW_V + part * 16, a);
            tmem_ld_wait();
            const float* bv = vec + VEC_BQKV + 2 * D + h * HDIM + part * 16;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              uint4 w;
              w.x = pack_bf16x2(__uint_as_float(a[8 * c]) + bv[8 * c], __uint_as_float(a[8 * c + 1]) + bv[8 * c + 1]);
              w.y = pack_bf16x2(__uint_as_float(a[8 * c + 2]) + bv[8 * c + 2], __uint_as_float(a[8 * c + 3]) + bv[8 * c + 3]);
              w.z = pack_bf16x2(__uint_as_float(a[8 * c + 4]) + bv[8 * c + 4], __uint_as_float(a[8 * c + 5]) + bv[8 * c + 5]);
              w.w = pack_bf16x2(__uint_as_float(a[8 * c + 6]) + bv[8 * c + 6], __uint_as_float(a[8 * c + 7]) + bv[8 * c + 7]);
              *reinterpret_cast<uint4*>(smem + OFF_VT + sw128_off(r, part * 2 + c)) = w;
            }
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(v_ready);
          }
          // ---- softmax over the row's own utterance; P (bf16 pairs) over the first 64 columns of S.  Every part
          // normalises by its own maximum first; one exchange of (max, sum) then gives the row maximum, the row sum
          // and the factor 2^(own max - row max) that rescales the part's probabilities ----
          float inv_l;
          mbar_wait(s_full, n_h & 1);
          tc_fence_after();
          XTRACE(th + 2);                                    // S complete
          if (p.stride == 64) {
            // two utterance slots of 64 rows: the row's 64 candidate keys split into four 16-column parts, so that all
            // 16 row warps work (columns klo + 16 part .. +16; valid while < klo + lk)
            const int nval = lk - part * 16;                 // valid columns of this part: [0, nval)
            uint32_t s[16];
            tmem_ld_32x32b_x16(tmW + lane_sel + TW_S + klo + part * 16, s);
            tmem_ld_wait();
            float e[16];
            float mx = -INFINITY, sum = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              e[i] = (i < nval) ? __uint_as_float(s[i]) : -INFINITY;
              mx = fmaxf(mx, e[i]);
            }
            const float mref = (mx == -INFINITY) ? 0.f : mx;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              e[i] = ex2_approx(e[i] - mref);
              sum += e[i];
            }
            float2 all[4];
            exchange(make_float2(mx, sum), all);             // every part has read its S columns before this barrier
            const float m = fmaxf(fmaxf(all[0].x, all[1].x), fmaxf(all[2].x, all[3].x));
            const float l_row = (all[0].y * ex2_approx(all[0].x - m) + all[1].y * ex2_approx(all[1].x - m)) +
                                (all[2].y * ex2_approx(all[2].x - m) + all[3].y * ex2_approx(all[3].x - m));
            inv_l = 1.0f / l_row;
            const float f = ex2_approx(mx - m);
            uint32_t pp[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) pp[i] = pack_bf16x2(e[2 * i] * f, e[2 * i + 1] * f);
            // P of the OTHER utterance slot's keys is zero for this row: each part clears its share of those 32 packed
            // columns as well (the P V contraction runs over all 128 keys)
            const uint32_t zz[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            tmem_st_32x32b_x8(tmW + lane_sel + TW_S + (klo >> 1) + part * 8, pp);
            tmem_st_32x32b_x8(tmW + lane_sel + TW_S + ((klo ^ 64) >> 1) + part * 8, zz);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_ready);
          } else {
            const int hi_i = lo_i + lk;                      // valid score columns within the part: [lo_i, hi_i)
            const bool any = __any_sync(0xffffffffu, (lo_i < 32) && (hi_i > 0));
            float e[32];
            float mx = -INFINITY, sum = 0.f;
            if (any) {
              uint32_t s[32];
              tmem_ld_32x32b_x32(tmW + lane_sel + TW_S + part * 32, s);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) {                 // masked scores become -inf: exp2 gives exactly 0 below
                e[i] = (i >= lo_i && i < hi_i) ? __uint_as_float(s[i]) : -INFINITY;
                mx = fmaxf(mx, e[i]);
              }
              const float mref = (mx == -INFINITY) ? 0.f : mx;       // a row with no valid column in this part
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                e[i] = ex2_approx(e[i] - mref);
                sum += e[i];
              }
            }
            float2 all[4];
            exchange(make_float2(mx, sum), all);             // every part has read its S columns before this barrier
            const float m = fmaxf(fmaxf(all[0].x, all[1].x), fmaxf(all[2].x, all[3].x));   // finite: the row has valid keys
            const float l_row = (all[0].y * ex2_approx(all[0].x - m) + all[1].y * ex2_approx(all[1].x - m)) +
                                (all[2].y * ex2_approx(all[2].x - m) + all[3].y * ex2_approx(all[3].x - m));
            inv_l = 1.0f / l_row;
            uint32_t pp[16];
            if (any) {
              const float f = ex2_approx(mx - m);            // 0 when this part holds no valid column of the row
#pragma unroll
              for (int i = 0; i < 16; ++i) pp[i] = pack_bf16x2(e[2 * i] * f, e[2 * i + 1] * f);
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) pp[i] = 0u;
            }
            tmem_st_32x32b_x16(tmW + lane_sel + TW_S + part * 16, pp);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_ready);
          }
          XTRACE(th + 3);                                    // P written
          // ---- O_h / rowsum -> bf16 A operand of the out_proj slice ----
          mbar_wait(o_full, n_h & 1);
          tc_fence_after();
          XTRACE(th + 4);                                    // O complete
          {
            uint32_t o[16], op[8];
            tmem_ld_32x32b_x16(tmW + lane_sel + TW_V + part * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i)
              op[i] = pack_bf16x2(__uint_as_float(o[2 * i]) * inv_l, __uint_as_float(o[2 * i + 1]) * inv_l);
            tmem_st_32x32b_x8(tmW + lane_sel + TW_OOP + part * 8, op);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(o_ready);
          }
          XTRACE(th + 5);                                    // O operand written
        }
        // ======== x += out_proj bias; LayerNorm 2 ========
        mbar_wait(attn_done, n_attn & 1); ++n_attn;
        tc_fence_after();
        XTRACE(tb + 26);                                     // attention complete
        ln_to_a(vec + VEC_BO, vec + VEC_N2G, vec + VEC_N2B);
        XTRACE(tb + 27);                                     // LN2 done

        // ======== feed-forward: bias + activation on each 128-wide hidden chunk, back into tensor memory as bf16 ====
        for (int j = 0; j < NCHUNK; ++j, ++c1n) {
          const uint32_t st = c1n & 1;
          mbar_wait(&acc1_full[st], (c1n >> 1) & 1);
          tc_fence_after();
          XTRACE(tb + 28 + 2 * j);                           // acc1_j complete
          uint32_t v[32];
          tmem_ld_32x32b_x32(tmW + lane_sel + st * 128 + part * 32, v);
          tmem_ld_wait();
          float hv[32];
          const float* bj = vec + VEC_B1 + j * 128 + part * 32;
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bj + i);
            hv[i] = __uint_as_float(v[i]) + b4.x; hv[i + 1] = __uint_as_float(v[i + 1]) + b4.y;
            hv[i + 2] = __uint_as_float(v[i + 2]) + b4.z; hv[i + 3] = __uint_as_float(v[i + 3]) + b4.w;
          }
          if (p.act == ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) hv[i] = fmaxf(hv[i], 0.f);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) hv[i] = gelu_bf16_grade(hv[i]);
          }
          uint32_t hp[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) hp[i] = pack_bf16x2(hv[2 * i], hv[2 * i + 1]);
          tc_fence_before();
          named_bar_sync(1 + q, 128);          // the bf16 pairs alias fp32 columns the other parts of this quarter read
          tc_fence_after();
          tmem_st_32x32b_x16(tmW + lane_sel + st * 128 + part * 16, hp);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&h_full[st]);
          XTRACE(tb + 29 + 2 * j);                           // H_j written
        }
        mbar_wait(ffn_done, n_ffn & 1); ++n_ffn;
        tc_fence_after();
        XTRACE(tb + 44);                                     // FFN complete
      }
      if (p.decoder) {
        // ---- SeparationDecoder on the tile (model.py:201-220): a = fusion.norm(x) -> H = GELU(a W0^T + b0) kept in tensor
        // memory over X -> masks = sigmoid(H W3^T + b3), separated = masks * mixed_spec, stored along T ----
        ln_to_a(vec + VEC_B2, fin_g, fin_b);
        XTRACE(107);                                         // decoder: final LayerNorm done
        // decoder vector block (b0 [512] | b3 [nc3 * 128]): next item of the weight stream
        {
          const uint32_t vn = static_cast<uint32_t>(lt) * per_tile + static_cast<uint32_t>(n_pro + p.n_layers * p.items_per_layer);
          const uint32_t vslot = vn % NSLOT;
          named_bar_sync(5, 512);                            // every row warp has read the last layer's vectors
          mbar_wait(&w_full[vslot], (vn / NSLOT) & 1);
          const float4* src = reinterpret_cast<const float4*>(smem + OFF_RING + vslot * ITEM);
          float4* dst = reinterpret_cast<float4*>(vec);
          for (int i = etid; i < (512 + p.nc3 * 128) / 4; i += 512) dst[i] = src[i];
          named_bar_sync(5, 512);
          if (etid == 0) mbar_arrive(&w_empty[vslot]);
        }
        XTRACE(108);                                         // decoder: vectors loaded
        // hidden chunks: bias + GELU -> bf16 pairs into X[64 j + 16 part, +16)
        for (int j = 0; j < 4; ++j, ++c1n) {
          const uint32_t st = c1n & 1;
          mbar_wait(&acc1_full[st], (c1n >> 1) & 1);
          tc_fence_after();
          uint32_t v[32];
          tmem_ld_32x32b_x32(tmW + lane_sel + st * 128 + part * 32, v);
          tmem_ld_wait();
          uint32_t hp[16];
          const float* bj = vec + j * 128 + part * 32;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            hp[i] = pack_bf16x2(gelu_bf16_grade(__uint_as_float(v[2 * i]) + bj[2 * i]),
                                gelu_bf16_grade(__uint_as_float(v[2 * i + 1]) + bj[2 * i + 1]));
          tmem_st_32x32b_x16(tmX + lane_sel + j * 64 + part * 16, hp);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&h_full[st]);
          XTRACE(109 + j);                                   // decoder: H_j written
        }
        // output chunks of 128 columns; the packer orders the columns of a chunk as (frequency bin, speaker) pairs -
        // column i of chunk c is bin c * 128/S + i / S of speaker i % S - so that one mixture value serves the S masks
        // computed next to it.  This thread: row = (utterance, t), 32 columns as two halves of 16 (16 / S bins each).
        // An (s, f) column of (B, S, F, T) is a plane of L floats: a warp (32 consecutive t) writes 128 contiguous
        // bytes per column.  The mixture values of the next half are in flight while the current one is stored; the
        // live set (two mixture buffers, 16 accumulator values, S + S running pointers) stays inside the 96 registers.
        const int utt = utt0 + r / p.stride, t = r - klo;
        const bool out_ok = row_valid && utt < p.B;
        const bool live = !VARLEN || t < lk;               // past the utterance's length: masks = separated = 0
        const int Lp = p.L;
        const size_t obase = static_cast<size_t>(out_ok ? utt : 0) * p.SF * Lp + t;
        float* const mo_u = p.masks + obase;
        float* const so_u = p.separated + obase;
        const float* const mx_u = p.mixed + static_cast<size_t>(out_ok ? utt : 0) * p.F * Lp + t;
        auto dec_out = [&](auto S_) {
          constexpr int S = decltype(S_)::value;
          constexpr int G = 16 / S;                            // frequency bins per half
          constexpr int FPC = 128 / S;                         // frequency bins per chunk
          const size_t FL = static_cast<size_t>(p.F) * Lp;     // floats between the planes of consecutive speakers
          auto load_mx = [&](float (&mx)[G], int f0) {         // mixture values of bins [f0, f0 + G)
            const float* q = mx_u + f0 * Lp;
#pragma unroll
            for (int j = 0; j < G; ++j, q += Lp) mx[j] = (out_ok && live && f0 + j < p.F) ? __ldg(q) : 0.f;
          };
          auto store_half = [&](const uint32_t (&v)[16], const float (&mx)[G], int f0, int col) {
            if (!out_ok || f0 >= p.F) return;
            const float* b3 = vec + 512 + col;                 // biases in the packed column order
            float* mo = mo_u + static_cast<size_t>(f0) * Lp;
            float* so = so_u + static_cast<size_t>(f0) * Lp;
            if (f0 + G <= p.F) {
#pragma unroll
              for (int j = 0; j < G; ++j, mo += Lp, so += Lp) {
#pragma unroll
                for (int sp = 0; sp < S; ++sp) {
                  const float mk = live ? sigmoid_fast(__uint_as_float(v[j * S + sp]) + b3[j * S + sp]) : 0.f;
                  __stcs(mo + sp * FL, mk);
                  __stcs(so + sp * FL, mk * mx[j]);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < G; ++j, mo += Lp, so += Lp) {
                if (f0 + j < p.F) {
#pragma unroll
                  for (int sp = 0; sp < S; ++sp) {
                    const float mk = live ? sigmoid_fast(__uint_as_float(v[j * S + sp]) + b3[j * S + sp]) : 0.f;
                    __stcs(mo + sp * FL, mk);
                    __stcs(so + sp * FL, mk * mx[j]);
                  }
                }
              }
            }
          };
          float mxa[G], mxb[G];
          load_mx(mxa, part * (32 / S));
          for (int c = 0; c < p.nc3; ++c, ++c1n) {
            const uint32_t st = c1n & 1;
            const int f0 = c * FPC + part * (32 / S);
            load_mx(mxb, f0 + G);
            XTRACE(113 + 2 * c);                               // decoder: mixture loads of chunk c issued
            mbar_wait(&acc1_full[st], (c1n >> 1) & 1);
            tc_fence_after();
            XTRACE(114 + 2 * c);                               // decoder: output chunk c complete
            uint32_t v[16];
            tmem_ld_32x32b_x16(tmW + lane_sel + st * 128 + part * 32, v);
            tmem_ld_wait();
            store_half(v, mxa, f0, c * 128 + part * 32);
            tmem_ld_32x32b_x16(tmW + lane_sel + st * 128 + part * 32 + 16, v);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&h_full[st]);           // the accumulator stage is drained (values in registers)
            if (c + 1 < p.nc3) load_mx(mxa, f0 + FPC);
            store_half(v, mxb, f0 + G, c * 128 + part * 32 + 16);
          }
        };
        if (p.S == 2) dec_out(std::integral_constant<int, 2>());
        else if (p.S == 1) dec_out(std::integral_constant<int, 1>());
        else dec_out(std::integral_constant<int, 4>());
        named_bar_sync(5, 512);
        XTRACE(127);                                         // tile done
        if (elected) mbar_arrive(stage_free);
      } else if (p.kvp_chunks) {
        // ---- K | V rows of the fusion layers from this tile's output (model.py:114-116 then 155,169) ----
        // 1. x = X + last linear2 bias -> fp32 staging rows in the (idle) weight ring + K/V tile area: 1 KB per row,
        //    16-byte chunks XOR-swizzled by the row so that thread-per-row accesses are conflict-free
        uint8_t* const stg = smem + OFF_RING;
        {
          uint32_t vu[64];
          float sum, sq;
          read_x(vu, vec + VEC_B2, false, sum, sq);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            *reinterpret_cast<uint4*>(stg + r * 1024 + (((part * 16 + i) ^ (r & 7)) << 4)) =
                make_uint4(vu[4 * i], vu[4 * i + 1], vu[4 * i + 2], vu[4 * i + 3]);
        }
        named_bar_sync(5, 512);
        // 2. linear interpolation along time (ATen upsample_linear1d, align_corners = False) -> bf16 A operand
        {
          const int t = r - klo;
          const bool live = t < p.kvp_L;
          // a short utterance: lk source rows interpolated to its own target length (the rows past that target are
          // finite and masked as keys by the fusion stack)
          const float scale =
              VARLEN ? lerp_scale(lk, utt_len(kvp_lens, min(utt0 + r / p.stride, p.B - 1), p.kvp_L)) : p.kvp_scale;
          const LerpTap k = lerp_tap(t, lk, scale);
          const int r0 = klo + k.i0, r1 = klo + k.i1;
          uint8_t* slab = smem + OFF_A + part * SLAB;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint4 w = make_uint4(0u, 0u, 0u, 0u);
            if (live) {
              const float4 a0 = *reinterpret_cast<const float4*>(stg + r0 * 1024 + (((part * 16 + 2 * c) ^ (r0 & 7)) << 4));
              const float4 a1 = *reinterpret_cast<const float4*>(stg + r0 * 1024 + (((part * 16 + 2 * c + 1) ^ (r0 & 7)) << 4));
              const float4 b0 = *reinterpret_cast<const float4*>(stg + r1 * 1024 + (((part * 16 + 2 * c) ^ (r1 & 7)) << 4));
              const float4 b1 = *reinterpret_cast<const float4*>(stg + r1 * 1024 + (((part * 16 + 2 * c + 1) ^ (r1 & 7)) << 4));
              w = pack_bf16x8(lerp4(a0, b0, k.w0, k.w1), lerp4(a1, b1, k.w0, k.w1));
            }
            *reinterpret_cast<uint4*>(slab + sw128_off(r, c)) = w;
          }
          fence_proxy_async_smem();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { mbar_arrive(kv_stage_free); mbar_arrive(a_ready); }
        }
        // 3. bias block: next item of the weight stream
        {
          const uint32_t vn = static_cast<uint32_t>(lt) * per_tile + static_cast<uint32_t>(n_pro + p.n_layers * p.items_per_layer);
          const uint32_t vslot = vn % NSLOT;
          named_bar_sync(5, 512);                            // every row warp has read the last layer's vectors
          mbar_wait(&w_full[vslot], (vn / NSLOT) & 1);
          const float4* src = reinterpret_cast<const float4*>(smem + OFF_RING + vslot * ITEM);
          float4* dst = reinterpret_cast<float4*>(vec);
          for (int i = etid; i < p.kvp_chunks * 128 / 4; i += 512) dst[i] = src[i];
          named_bar_sync(5, 512);
          if (etid == 0) mbar_arrive(&w_empty[vslot]);
        }
        // 4. per 128-column chunk: accumulator + bias -> bf16 -> 64 contiguous bytes of the row in global memory
        {
          const int utt = utt0 + r / p.stride, t = r - klo;
          const bool out_ok = t < p.kvp_L && utt < p.B;
          __nv_bfloat16* orow = p.kvp_out + (static_cast<size_t>(out_ok ? utt : 0) * p.kvp_L + (out_ok ? t : 0)) * p.kvp_ld + part * 32;
          for (int c = 0; c < p.kvp_chunks; ++c, ++c1n) {
            const uint32_t st = c1n & 1;
            mbar_wait(&acc1_full[st], (c1n >> 1) & 1);
            tc_fence_after();
            uint32_t v[32];
            tmem_ld_32x32b_x32(tmW + lane_sel + st * 128 + part * 32, v);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&h_full[st]);
            if (out_ok) {
              const float* bj = vec + c * 128 + part * 32;
              uint4* o = reinterpret_cast<uint4*>(orow + c * 128);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 ba = *reinterpret_cast<const float4*>(bj + 8 * i), bb = *reinterpret_cast<const float4*>(bj + 8 * i + 4);
                uint4 w;
                w.x = pack_bf16x2(__uint_as_float(v[8 * i]) + ba.x, __uint_as_float(v[8 * i + 1]) + ba.y);
                w.y = pack_bf16x2(__uint_as_float(v[8 * i + 2]) + ba.z, __uint_as_float(v[8 * i + 3]) + ba.w);
                w.z = pack_bf16x2(__uint_as_float(v[8 * i + 4]) + bb.x, __uint_as_float(v[8 * i + 5]) + bb.y);
                w.w = pack_bf16x2(__uint_as_float(v[8 * i + 6]) + bb.z, __uint_as_float(v[8 * i + 7]) + bb.w);
                o[i] = w;
              }
            }
          }
        }
        named_bar_sync(5, 512);
        XTRACE(127);                                         // tile done
        if (elected) mbar_arrive(stage_free);
      } else
      // ---- stack output: x + last linear2 bias -> fp32 residual rows and / or (final LayerNorm | cast) bf16 rows ----
      {
        uint32_t vu[64];
        float sum, sq, mean = 0.f, rstd = 1.f;
        read_x(vu, vec + VEC_B2, false, sum, sq);
        tc_fence_before();
        if (p.out_x) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint8_t* slab = smem + OFF_A + (part * 2 + c) * SLAB;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              *reinterpret_cast<uint4*>(slab + sw128_off(r, i)) =
                  make_uint4(vu[c * 32 + 4 * i], vu[c * 32 + 4 * i + 1], vu[c * 32 + 4 * i + 2], vu[c * 32 + 4 * i + 3]);
          }
          fence_proxy_async_smem();
          named_bar_sync(6 + part, 128);
          if (elected) {
            for (int u = 0; u < p.U; ++u) {
              tma_store_2d(&tmXout, smem + OFF_A + (part * 2) * SLAB + u * p.stride * 128, part * 64, (utt0 + u) * p.L);
              tma_store_2d(&tmXout, smem + OFF_A + (part * 2 + 1) * SLAB + u * p.stride * 128, part * 64 + 32, (utt0 + u) * p.L);
            }
            bulk_commit();
          }
        }
        if (p.out_op) {
          if (p.fin_gamma != nullptr) row_stats(sum, sq, mean, rstd);
          if (p.out_x) {                        // the bf16 image reuses staging slabs 0..3: wait for every part's x stores
            if (elected) bulk_wait_read0();
            named_bar_sync(5, 512);
          }
          store_op_row(vu, mean, rstd, fin_g, fin_b, smem + OFF_A);      // cast only: mean 0, rstd 1, gamma 1, beta 0
          fence_proxy_async_smem();
          named_bar_sync(6 + part, 128);
          if (elected) {
            for (int u = 0; u < p.U; ++u)
              tma_store_2d(&tmOp, smem + OFF_A + part * SLAB + u * p.stride * 128, part * 64, (utt0 + u) * p.L);
            bulk_commit();
          }
        }
        if (elected) {
          bulk_wait_read0();
          mbar_arrive(stage_free);
        }
        XTRACE(127);                                         // tile done
      }
    }
    if (elected) bulk_wait_read0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// [nrows x 64] bf16 tile of W (row-major, leading dimension ld) starting at (row0, col0), written as the 128B-swizzled
// K-major shared-memory image the UMMA descriptors expect (row r at r * 128 B, 16-byte chunk c at (c ^ (r & 7))).
void put_tile(uint8_t* dst, const float* W, int ld, int row0, int nrows, int col0) {
  for (int r = 0; r < nrows; ++r)
    for (int k = 0; k < 64; ++k) {
      const uint16_t b = f2bf(W[static_cast<size_t>(row0 + r) * ld + col0 + k]);
      memcpy(dst + r * 128 + (((k >> 3) ^ (r & 7)) << 4) + (k & 7) * 2, &b, 2);
    }
}

void pack_ffn_items(uint8_t* dst, const float* w1, const float* w2) {
  // issue order of the MMA thread: G1_0, G1_1, G2_0, G1_2, G2_1, ..., G1_7, G2_6, G2_7
  auto g1 = [&](int j) {
    for (int it = 0; it < 2; ++it, dst += ITEM)
      for (int half = 0; half < 2; ++half) put_tile(dst + half * SLAB, w1, D, j * 128, 128, (2 * it + half) * 64);
  };
  auto g2 = [&](int j) {
    for (int ks = 0; ks < 2; ++ks, dst += ITEM)
      for (int hf = 0; hf < 2; ++hf) put_tile(dst + hf * SLAB, w2, HID, hf * 128, 128, j * 128 + ks * 64);
  };
  for (int j = 0; j <= NCHUNK; ++j) {
    if (j < NCHUNK) g1(j);
    if (j >= 1) g2(j - 1);
  }
}

}  // namespace

size_t xformer_stream_bytes(bool cross) { return static_cast<size_t>(cross ? ITEMS_CROSS : ITEMS_SELF) * ITEM; }
int xformer_vec_floats() { return VEC_FLOATS; }

// Stream of one self-attention layer, in the order the kernel consumes it: vector block | Q_0|K_0 (2 items), V_0 | per
// head h: Q_{h+1}|K_{h+1} (2 items, h < 3), Wo_h, V_{h+1} (h < 3) | FFN items.
// in_proj_weight [768, 256] (q | k | v rows), out_proj [256, 256], linear1 [1024, 256], linear2 [256, 1024]
void xformer_pack_self(const float* wqkv, const float* wo, const float* w1, const float* w2, const float* vecs,
                       uint8_t* dst) {
  memset(dst, 0, xformer_stream_bytes(false));
  memcpy(dst, vecs, sizeof(float) * VEC_FLOATS);
  dst += ITEM;
  auto qk = [&](int h) {
    for (int it = 0; it < 2; ++it, dst += ITEM)
      for (int half = 0; half < 2; ++half) {
        const int col0 = (2 * it + half) * 64;
        put_tile(dst + half * SLAB, wqkv, D, h * HDIM, 64, col0);                    // Q_h rows
        put_tile(dst + half * SLAB + 64 * 128, wqkv, D, D + h * HDIM, 64, col0);     // K_h rows
      }
  };
  auto vh = [&](int h) {
    for (int ks = 0; ks < 4; ++ks) put_tile(dst + ks * 8192, wqkv, D, 2 * D + h * HDIM, 64, ks * 64);
    dst += ITEM;
  };
  qk(0);
  vh(0);
  for (int h = 0; h < NH; ++h) {
    if (h + 1 < NH) qk(h + 1);
    for (int hf = 0; hf < 2; ++hf) put_tile(dst + hf * SLAB, wo, D, hf * 128, 128, h * HDIM);
    dst += ITEM;
    if (h + 1 < NH) vh(h + 1);
  }
  pack_ffn_items(dst, w1, w2);
}

// Cross-attention layer: vector block | Q_0 | per head h: Q_{h+1} (h < 3), Wo_h | FFN items.
// wq = rows [0, 256) of the packed in_proj_weight of nn.MultiheadAttention (model.py:155; functional.py:5847-5865)
void xformer_pack_cross(const float* wq, const float* wo, const float* w1, const float* w2, const float* vecs,
                        uint8_t* dst) {
  memset(dst, 0, xformer_stream_bytes(true));
  memcpy(dst, vecs, sizeof(float) * VEC_FLOATS);
  dst += ITEM;
  auto qh = [&](int h) {
    for (int ks = 0; ks < 4; ++ks) put_tile(dst + ks * 8192, wq, D, h * HDIM, 64, ks * 64);
    dst += ITEM;
  };
  qh(0);
  for (int h = 0; h < NH; ++h) {
    if (h + 1 < NH) qh(h + 1);
    for (int hf = 0; hf < 2; ++hf) put_tile(dst + hf * SLAB, wo, D, hf * 128, 128, h * HDIM);
    dst += ITEM;
  }
  pack_ffn_items(dst, w1, w2);
}

void xformer_pack_vecs(const float* bqkv, int n_bqkv, const float* bo, const float* b1, const float* b2, const float* n1g,
                       const float* n1b, const float* n2g, const float* n2b, float* dst, const float* b0) {
  memset(dst, 0, sizeof(float) * VEC_FLOATS);
  memcpy(dst + VEC_BQKV, bqkv, sizeof(float) * n_bqkv);
  memcpy(dst + VEC_BO, bo, sizeof(float) * D);
  memcpy(dst + VEC_B1, b1, sizeof(float) * HID);
  memcpy(dst + VEC_B2, b2, sizeof(float) * D);
  memcpy(dst + VEC_N1G, n1g, sizeof(float) * D);
  memcpy(dst + VEC_N1B, n1b, sizeof(float) * D);
  memcpy(dst + VEC_N2G, n2g, sizeof(float) * D);
  memcpy(dst + VEC_N2B, n2b, sizeof(float) * D);
  if (b0 != nullptr) memcpy(dst + VEC_B0, b0, sizeof(float) * D);
}

// Input projection items (ahead of layer 0): item (tap, k-slab) = W_tap[:, 64 ks .. +64) as two 128-row slabs
size_t xformer_pro_bytes(int taps, int K) { return static_cast<size_t>(taps) * (K / 64) * ITEM; }
void xformer_pack_pro(const float* W, int ld, int col_stride, int taps, int K, uint8_t* dst) {
  std::vector<float> tile(static_cast<size_t>(D) * 64);
  for (int tap = 0; tap < taps; ++tap)
    for (int ks = 0; ks < K / 64; ++ks, dst += ITEM) {
      for (int n = 0; n < D; ++n)
        for (int k = 0; k < 64; ++k) tile[n * 64 + k] = W[static_cast<size_t>(n) * ld + static_cast<size_t>(ks * 64 + k) * col_stride + tap];
      for (int hf = 0; hf < 2; ++hf) put_tile(dst + hf * SLAB, tile.data(), 64, hf * 128, 128, 0);
    }
}

// K | V projection block behind the last layer of a self stack: bias block | per 128-row chunk of wkv two items
// (k-slab pairs), as linear1 chunks are packed
size_t xformer_kvp_bytes(int n) { return static_cast<size_t>(1 + 2 * (n / 128)) * ITEM; }
bool xformer_kvp_usable(int n, int L_src, int L_out) {
  if (n < 128 || n % 128 != 0 || n > VEC_FLOATS || L_src < 1 || L_src > 128 || L_out < 1) return false;
  int U = 1;
  while (U < 16 && 2 * U * L_src <= 128) U *= 2;
  return L_out <= 128 / U;                       // the interpolated rows of an utterance stay inside its tile slot
}
void xformer_pack_kvp(const float* wkv, const float* bkv, int n, uint8_t* dst) {
  memset(dst, 0, xformer_kvp_bytes(n));
  memcpy(dst, bkv, sizeof(float) * n);
  dst += ITEM;
  for (int c = 0; c < n / 128; ++c)
    for (int it = 0; it < 2; ++it, dst += ITEM)
      for (int half = 0; half < 2; ++half) put_tile(dst + half * SLAB, wkv, D, c * 128, 128, (2 * it + half) * 64);
}

// SeparationDecoder block of the fusion stream (after the last layer): vector block (b0 [512] | b3 in packed column
// order), Linear(256 -> 512) as 8 items (chunk j, k-slab pair), Linear(512 -> S*F) as 4 items per 128-column chunk.
// Packed column order: column i of chunk c is frequency bin c * 128/S + i / S of speaker i % S (zero rows past F).
int xformer_decoder_chunks(int S, int F) { return (F + 128 / S - 1) / (128 / S); }
bool xformer_decoder_usable(int S, int F) {
  return (S == 1 || S == 2 || S == 4) && F >= 1 && 512 + xformer_decoder_chunks(S, F) * 128 <= VEC_FLOATS;
}
size_t xformer_decoder_bytes(int S, int F) { return static_cast<size_t>(1 + 8 + 4 * xformer_decoder_chunks(S, F)) * ITEM; }
void xformer_pack_decoder(const float* w0, const float* b0, const float* w3, const float* b3, int S, int F, uint8_t* dst) {
  const int nc3 = xformer_decoder_chunks(S, F), fpc = 128 / S;
  memset(dst, 0, xformer_decoder_bytes(S, F));
  std::vector<float> wp(static_cast<size_t>(nc3) * 128 * 2 * D, 0.f);
  float* v = reinterpret_cast<float*>(dst);
  memcpy(v, b0, sizeof(float) * 512);
  for (int c = 0; c < nc3; ++c)
    for (int i = 0; i < 128; ++i) {
      const int f = c * fpc + i / S, sp = i % S;
      if (f >= F) continue;
      v[512 + c * 128 + i] = b3[sp * F + f];
      memcpy(&wp[static_cast<size_t>(c * 128 + i) * 2 * D], w3 + static_cast<size_t>(sp * F + f) * 2 * D, sizeof(float) * 2 * D);
    }
  dst += ITEM;
  for (int j = 0; j < 4; ++j)
    for (int it = 0; it < 2; ++it, dst += ITEM)
      for (int half = 0; half < 2; ++half) put_tile(dst + half * SLAB, w0, D, j * 128, 128, (2 * it + half) * 64);
  for (int c = 0; c < nc3; ++c)
    for (int it = 0; it < 4; ++it, dst += ITEM)
      for (int half = 0; half < 2; ++half) put_tile(dst + half * SLAB, wp.data(), 2 * D, c * 128, 128, (2 * it + half) * 64);
}

bool xformer_stack_usable(int prec, int d_model, int nhead, int len) {
  return prec == PREC_BF16 && d_model == D && nhead == NH && len >= 1 && len <= 128;
}

const char* launch_xformer_stack(LaunchCtx lc, const StackProblem& sp, int num_sms) {
  if (sp.B <= 0 || sp.L <= 0 || sp.L > 128 || sp.n_layers <= 0) return "xformer_stack: bad problem";
  const bool decoder = sp.masks != nullptr;
  const bool pro = sp.pro_a != nullptr;
  const bool kvp = sp.kvp_out != nullptr;
  if (!sp.out_x && !sp.out_op && !decoder && !kvp) return "xformer_stack: no output requested";
  if (kvp && (sp.cross || sp.out_x || sp.out_op || !xformer_kvp_usable(sp.kvp_n, sp.L, sp.kvp_L) || sp.kvp_ld < sp.kvp_n ||
              sp.kvp_ld % 8 != 0 || (reinterpret_cast<uintptr_t>(sp.kvp_out) & 15) != 0))
    return "xformer_stack: bad K|V projection";
  if (pro && (sp.cross || (sp.pro_taps != 1 && sp.pro_taps != 3) || sp.pro_k < 64 || sp.pro_k % 64 != 0 || sp.pe == nullptr ||
              sp.pro_pitch < sp.L + sp.pro_taps - 1 || sp.pro_rows < 1))
    return "xformer_stack: bad input projection";
  if (!pro && sp.x_in == nullptr) return "xformer_stack: no input";
  if (decoder) {
    if (!sp.cross || sp.out_x || sp.out_op || !sp.mixed || !sp.separated || sp.F < 1 || sp.S < 1)
      return "xformer_stack: the fused decoder follows the fusion stack and replaces its outputs";
    if (!xformer_decoder_usable(sp.S, sp.F)) return "xformer_stack: speaker count / freq_bins not supported by the fused decoder";
  }
  int U = 1;                                   // utterances per tile: the largest power of two with U * L <= 128
  while (U < 16 && 2 * U * sp.L <= 128) U *= 2;
  const int stride = 128 / U;
  const int M = sp.B * sp.L;
  const int n_tiles = (sp.B + U - 1) / U;
  CUtensorMap tin, tout, top, tkv;
  if (pro) {
    if (const char* e = tma_encode_2d(&tkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, sp.pro_a, sp.pro_k, sp.pro_rows, sp.pro_k, 64, stride)) return e;
    tin = tkv;
  } else {
    if (const char* e = tma_encode_2d(&tin, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, sp.x_in, D, M, D, 32, sp.L)) return e;
    tkv = tin;
  }
  tout = tin; top = tin;
  if (sp.out_x)
    if (const char* e = tma_encode_2d(&tout, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, sp.out_x, D, M, D, 32, sp.L)) return e;
  if (sp.out_op)
    if (const char* e = tma_encode_2d(&top, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, sp.out_op, D, M, D, 64, sp.L)) return e;
  if (sp.cross) {
    if (sp.kv == nullptr || sp.kv_ld < sp.n_layers * 2 * D) return "xformer_stack: cross-attention needs the K|V rows";
    if (const char* e = tma_encode_2d(&tkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, sp.kv, sp.kv_ld, M, sp.kv_ld, 64, sp.L)) return e;
  }
  StackDev d{};
  d.wstream = sp.wstream; d.fin_gamma = sp.fin_gamma; d.fin_beta = sp.fin_beta;
  d.n_layers = sp.n_layers; d.items_per_layer = sp.cross ? ITEMS_CROSS : ITEMS_SELF; d.cross = sp.cross ? 1 : 0;
  d.L = sp.L; d.U = U; d.stride = stride; d.B = sp.B; d.n_tiles = n_tiles;
  d.act = sp.act; d.out_x = sp.out_x != nullptr; d.out_op = sp.out_op != nullptr;
  d.kv_ld_layer = 2 * D;
  d.qscale = 1.4426950408889634f / 8.0f;       // log2(e) / sqrt(head dim 64)
  d.trace = sp.trace;
  d.pro_taps = pro ? sp.pro_taps : 0; d.pro_ks = sp.pro_k / 64; d.pro_pitch = sp.pro_pitch; d.pro_relu = sp.pro_relu; d.pe = sp.pe;
  d.kvp_chunks = kvp ? sp.kvp_n / 128 : 0; d.kvp_L = sp.kvp_L; d.kvp_ld = sp.kvp_ld;
  d.kvp_scale = kvp ? lerp_scale(sp.L, sp.kvp_L) : 0.f;
  d.kvp_out = static_cast<__nv_bfloat16*>(sp.kvp_out);
  d.lens = sp.lens; d.kvp_lens = kvp ? sp.kvp_lens : nullptr;
  d.decoder = decoder ? 1 : 0;
  d.SF = sp.S * sp.F; d.F = sp.F; d.S = sp.S; d.nc3 = decoder ? xformer_decoder_chunks(sp.S, sp.F) : 0;
  d.mixed = sp.mixed; d.masks = sp.masks; d.separated = sp.separated;
  const int grid = n_tiles < num_sms ? n_tiles : num_sms;
  auto kern = (d.lens != nullptr || d.kvp_lens != nullptr) ? xformer_stack_kernel<true> : xformer_stack_kernel<false>;
  if (!smem_opt_in(kern, STACK_SMEM)) return "xformer_stack: cannot raise the shared-memory limit";
  if (launch_pdl(kern, dim3(grid), dim3(STACK_THREADS), STACK_SMEM, lc, tin, tout, top, tkv, d) !=
      cudaSuccess) {
    cudaGetLastError();
    return "xformer_stack: launch failed";
  }
  return nullptr;
}

}  // namespace avsep
