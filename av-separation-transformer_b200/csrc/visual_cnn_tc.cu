// VisualEncoder.conv (model.py:81-92,106-107) for 32x32 frames on the 5th-gen tensor cores.
//
// One persistent CTA per SM walks groups of 8 frames.  Per group:
//   for each pair of frames:
//     conv1 (K = 9 taps, tensor cores via mma.sync, 3 % of the FLOPs)        -> act1 (bf16, smem, 16x16x32 / frame)
//     conv2 as an implicit GEMM  M = 128 (2 frames x 64 px), N = 64, K = 9x32:
//       im2col slabs [128 rows x 64 k] (two taps each) are gathered from act1 straight into TENSOR MEMORY (an 8-slot
//       ring of 32 columns: thread = row, tcgen05.st) and fed to tcgen05.mma as the A operand from TMEM, so the slab
//       costs no shared-memory store and no shared-memory operand read (the kernel was bound by shared-memory
//       bandwidth and by the build -> MMA -> free round trip of a 2-slot smem ring); all 18 k-steps accumulate in
//       TMEM.  Epilogue: tcgen05.ld -> bias(BN-folded)+ReLU -> act2 (bf16, smem)
//   conv3 as an implicit GEMM  M = 128 (8 frames x 16 px), N = 128, K = 9x64: one slab per tap gathered from act2,
//       the matching 16 KB weight slab streamed by TMA (3-slot ring, L2-resident), 36 tcgen05.mma k-steps;
//       epilogue: tcgen05.ld -> bias+ReLU -> 16-pixel mean by warp shuffles -> pooled (M,128) bf16.
// BatchNorm (eval) is folded into weights/bias on the host.  Nothing but the 4 KB frame and the 256 B feature row
// touches HBM.
#include "common.cuh"
#include "kernels.h"

#include <string.h>

namespace avsep {

namespace {

constexpr int TC_BUILDERS = 256;          // 8 warps: gather im2col slabs, conv1, epilogues
constexpr int TC_THREADS = TC_BUILDERS + 64;   // + 1 MMA-issuer warp + 1 TMA-producer warp (conv3 weights)
constexpr int W3S = 4;                    // conv3 weight ring slots
constexpr int GROUP = 8;                 // frames per conv3 tile
constexpr int SLAB_BYTES = 128 * 128;    // 128 rows x 128 B
constexpr int W2_SLABS = 5, W2_SLAB_BYTES = 64 * 128;
// shared memory map (bytes, all tensor-core regions 1024-aligned)
constexpr int NSLOT = 6;                                  // im2col ring slots in tensor memory (32 columns each)
constexpr int OFF_W3 = 0;                                 // W3S x 16 KB  conv3 weight slabs (TMA)
constexpr int OFF_W2 = OFF_W3 + W3S * SLAB_BYTES;         // 5 x 8 KB   conv2 weight slabs (resident)
constexpr int OFF_ACT2 = OFF_W2 + W2_SLABS * W2_SLAB_BYTES;   // 8 frames x 64 px x 128 B
constexpr int OFF_ACT1 = OFF_ACT2 + GROUP * 64 * 128;     // 2 frames x 256 px x 64 B
constexpr int OFF_IN = OFF_ACT1 + 2 * 256 * 64;           // 2 frames x 34 x 34 fp32
constexpr int OFF_MISC = OFF_IN + 2 * 34 * 34 * 4;        // barriers, TMEM slot
constexpr int TC_SMEM = OFF_MISC + 256 + 1024;            // + alignment slack (<= 227 KB)
static_assert(TC_SMEM <= 227 * 1024, "visual_cnn_tc: shared memory budget exceeded");

struct CnnTcDev {
  const float* frames;
  __nv_bfloat16* pooled;
  const uint32_t* w1; const float* b1;
  const uint8_t* w2_slabs; const float* b2;
  const float* b3;
  int M, num_groups;
  const int* frame_lens;       // variable-length batch: frames past an utterance's length are staged as zeros
  int N;                       // frames per utterance (pitch of frame_lens)
  unsigned long long* trace;   // optional [grid][64] globaltimer stamps of the CTA's 2nd group (debug), else null
};

#define CTRACE(slot) do { if (p.trace != nullptr && tid == 0 && grp == static_cast<int>(blockIdx.x + gridDim.x)) \
    p.trace[blockIdx.x * 64 + (slot)] = globaltimer(); } while (0)

// act1: 2 pixels per 128-byte line, 16-byte chunk slot XOR-swizzled by the line index.
__device__ __forceinline__ int act1_chunk_off(int pixel, int c) {   // pixel = f*256 + y*16 + x, c = 8-channel chunk 0..3
  const int line = pixel >> 1;
  return line * 128 + ((((pixel & 1) << 2) | c) ^ (line & 7)) * 16;
}
// act2: one pixel (64 ch) per 128-byte line, chunk slot XOR-swizzled by the pixel index.
__device__ __forceinline__ int act2_chunk_off(int pixel, int c) {   // pixel = g*64 + y*8 + x, c = 0..7
  return pixel * 128 + ((c ^ (pixel & 7)) * 16);
}

__global__ void __launch_bounds__(TC_THREADS, 1)
visual_cnn_tc_kernel(const __grid_constant__ CUtensorMap tmW3, const CnnTcDev p) {
  // Dynamic shared memory is declared 1024-byte aligned (128B-swizzle atoms) and used directly: deriving the base
  // through an integer round trip would make the compiler fall back to generic LD/ST for every access.
  extern __shared__ __align__(1024) uint8_t smem_raw_cnn[];
  uint8_t* const smem = smem_raw_cnn;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* w3s = smem + OFF_W3;
  uint8_t* w2s = smem + OFF_W2;
  uint8_t* act2 = smem + OFF_ACT2;
  uint8_t* act1 = smem + OFF_ACT1;
  float* sIn = reinterpret_cast<float*>(smem + OFF_IN);
  uint64_t* ring_full = reinterpret_cast<uint64_t*>(smem + OFF_MISC);   // [NSLOT] slab written by all 8 builder warps
  uint64_t* ring_free = ring_full + NSLOT;                         // [NSLOT] MMAs that read the slab have completed
  uint64_t* bar_acc = ring_free + NSLOT;                           // accumulator complete
  uint64_t* bar_acc3 = bar_acc + 1;                                // [2] conv3 accumulator (double-buffered) complete
  uint64_t* bar_w3 = bar_acc3 + 2;                                 // [W3S] W3 slab landed
  uint64_t* w3_free = bar_w3 + W3S;                                // [W3S] the MMAs that read the slab have completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w3_free + W3S);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  for (int i = tid; i < W2_SLABS * W2_SLAB_BYTES / 16; i += TC_THREADS)
    reinterpret_cast<uint4*>(w2s)[i] = reinterpret_cast<const uint4*>(p.w2_slabs)[i];
  for (int i = tid; i < 2 * 34 * 34; i += TC_THREADS) sIn[i] = 0.f;
  if (tid == 0) {
    tma_prefetch_desc(&tmW3);
    for (int i = 0; i < NSLOT; ++i) {
      mbar_init(&ring_full[i], TC_BUILDERS / 32);
      mbar_init(&ring_free[i], 1);
    }
    mbar_init(bar_acc, 1);
    mbar_init(&bar_acc3[0], 1);
    mbar_init(&bar_acc3[1], 1);
    for (int i = 0; i < W3S; ++i) { mbar_init(&bar_w3[i], 1); mbar_init(&w3_free[i], 1); }
    fence_mbar_init();
  }
  if (warp == TC_BUILDERS / 32) tmem_alloc(tmem_slot, 512);
  fence_proxy_async_smem();     // W2 slabs were written with generic stores, read by the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_acc2 = tmem_base;          // 64 columns
  const uint32_t tmem_acc3 = tmem_base + 64;     // 2 x 128 columns: the conv3 epilogue of group g runs inside group g+1
  const uint32_t tmem_ring = tmem_base + 320;    // NSLOT x 32 columns: A operand slabs (128 rows x 64 bf16)
  griddep_launch_dependents();
  griddep_wait();

  if (warp == TC_BUILDERS / 32) {
    // =========================== MMA issuer (one lane) ===========================
    if (lane == 0) {
      const uint32_t idesc2 = umma_idesc(1u, 128, 64);
      const uint32_t idesc3 = umma_idesc(1u, 128, 128);
      uint32_t n_slab = 0, n_w3 = 0, lt = 0;
      for (int grp = blockIdx.x; grp < p.num_groups; grp += gridDim.x, ++lt) {
        for (int pair = 0; pair < GROUP / 2; ++pair) {
          for (int j = 0; j < W2_SLABS; ++j, ++n_slab) {
            const uint32_t slot = n_slab % NSLOT, use = n_slab / NSLOT;
            mbar_wait(&ring_full[slot], use & 1);
            tc_fence_after();
            const uint32_t a_t = tmem_ring + slot * 32;
            const uint64_t bdesc = umma_desc_kmajor_sw128(smem_u32(w2s + j * W2_SLAB_BYTES), 1024);
            const int ksteps = (j == W2_SLABS - 1) ? 2 : 4;     // the last slab holds tap 8 only
            for (int k = 0; k < ksteps; ++k)
              umma_f16_ts(tmem_acc2, a_t + 8 * k, bdesc + 2 * k, idesc2, (j | k) != 0 ? 1u : 0u);
            umma_commit(&ring_free[slot]);
            if (j == W2_SLABS - 1) umma_commit(bar_acc);
          }
        }
        for (int t = 0; t < 9; ++t, ++n_slab, ++n_w3) {
          const uint32_t slot = n_slab % NSLOT, use = n_slab / NSLOT;
          mbar_wait(&ring_full[slot], use & 1);
          const uint32_t ws = n_w3 % W3S;
          mbar_wait(&bar_w3[ws], (n_w3 / W3S) & 1);
          tc_fence_after();
          const uint32_t a_t = tmem_ring + slot * 32;
          const uint64_t bdesc = umma_desc_kmajor_sw128(smem_u32(w3s + ws * SLAB_BYTES), 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16_ts(tmem_acc3 + (lt & 1) * 128, a_t + 8 * k, bdesc + 2 * k, idesc3, (t | k) != 0 ? 1u : 0u);
          umma_commit(&ring_free[slot]);
          umma_commit(&w3_free[ws]);
          if (t == 8) umma_commit(&bar_acc3[lt & 1]);
        }
      }
    }
  } else if (warp == TC_BUILDERS / 32 + 1) {
    // =========================== TMA producer: conv3 weight slabs (one lane) ===========================
    if (lane == 0) {
      uint32_t n = 0;
      for (int grp = blockIdx.x; grp < p.num_groups; grp += gridDim.x) {
        for (int t = 0; t < 9; ++t, ++n) {
          const uint32_t ws = n % W3S, use = n / W3S;
          if (use > 0) mbar_wait(&w3_free[ws], (use - 1) & 1);
          mbar_arrive_expect_tx(&bar_w3[ws], SLAB_BYTES);
          tma_load_2d(w3s + ws * SLAB_BYTES, &tmW3, &bar_w3[ws], 0, t * 128);
        }
      }
    }
  } else {
    // =========================== builders / epilogue (8 warps) ===========================
    const int gid = lane >> 2, tig = lane & 3;
    uint32_t n_slab = 0;      // slabs pushed through the ring so far
    uint32_t acc_phase = 0;

    // ---- per-thread gather constants: thread = row (TMEM lane) brow of every slab, column half bhh (32 of the
    //      slab's 64 k-values = 64 contiguous bytes of one source pixel)
    const int bq = warp & 3, bhh = warp >> 2;
    const int brow = bq * 32 + lane;
    const uint32_t ring_lane = tmem_ring + (static_cast<uint32_t>(bq * 32) << 16) + bhh * 16;   // + slot * 32
    // conv2 (row = (f, y2, x2) of a pair, k half = tap 2j + bhh, 32 channels): source act1 (2 pixels per swizzled line)
    int xo2[3], s02[3];
    bool vx2[3];
    const int y2 = (brow >> 3) & 7, f2 = brow >> 6;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int xx = 2 * (brow & 7) + kx - 1;
      vx2[kx] = xx >= 0 && xx < 16;
      xo2[kx] = (xx >> 1) * 128;
      s02[kx] = (((xx & 1) << 2) ^ ((xx >> 1) & 7));          // chunk slot of channel chunk c is s02 ^ c
    }
    const int rowbase2 = (f2 * 256 + (2 * y2 - 1) * 16) * 64;   // + ky*1024 + xo2[kx] + ((s02[kx] ^ c) << 4)
    const bool top2 = (y2 == 0);                                // tap row ky = 0 falls above the frame
    // conv3 (row = (g, y3, x3) of the group, k half = channels 32*bhh ..): source act2 (one pixel per swizzled line)
    int xo3[3], s03[3];
    bool vx3[3];
    const int y3 = (brow >> 2) & 3;
    const bool top3 = (y3 == 0);
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int xx = 2 * (brow & 3) + kx - 1;
      vx3[kx] = xx >= 0 && xx < 8;
      xo3[kx] = xx * 128;
      s03[kx] = xx & 7;                                         // chunk slot of chunk c is c ^ s03
    }
    const int rowbase3 = ((brow >> 4) * 64 + (2 * y3 - 1) * 8) * 128;   // + ky*1024 + xo3[kx] + ((c ^ s03[kx]) << 4)

    // conv1 B fragments and bias (constant, registers)
    uint32_t bw1[4][2];
    float bias1[4][2];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      bw1[nt][0] = __ldg(p.w1 + nt * 64 + lane * 2);
      bw1[nt][1] = __ldg(p.w1 + nt * 64 + lane * 2 + 1);
      bias1[nt][0] = __ldg(p.b1 + nt * 8 + 2 * tig);
      bias1[nt][1] = __ldg(p.b1 + nt * 8 + 2 * tig + 1);
    }
    const int k0 = 2 * tig, k1 = 2 * tig + 1;
    const int off0 = (k0 / 3) * 34 + (k0 % 3), off1 = (k1 / 3) * 34 + (k1 % 3), off8 = 2 * 34 + 2;

    // Input prefetch: each thread keeps the next pair's two float4 pieces (2 frames x 1024 px / 256 threads) in
    // registers, so the global-load latency hides behind the current pair's conv1/conv2.
    float4 pre[2];
    auto prefetch_pair = [&](int first_frame) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int id = tid + TC_BUILDERS * i;
        const int f = id >> 8, rem = id & 255;
        const int fr = first_frame + f;
        pre[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (fr < p.M && frame_live(p.frame_lens, p.N, fr)) pre[i] = __ldg(reinterpret_cast<const float4*>(p.frames + static_cast<size_t>(fr) * 1024) + rem);
      }
    };
    // hand a finished slab to the MMA issuer
    // write this thread's 16 columns of slab `slot` and hand the slab to the MMA issuer
    auto publish_slab = [&](uint32_t slot, const uint32_t (&cols)[16]) {
      tmem_st_32x32b_x16(ring_lane + slot * 32, cols);
      tmem_st_wait();
      tc_fence_before();            // the stores (and earlier tcgen05.ld) are ordered before the MMAs this unblocks
      __syncwarp();
      if (lane == 0) mbar_arrive(&ring_full[slot]);
    };
    // conv2 epilogue of one pair: acc (128 px x 64 ch) -> bias + ReLU -> act2
    auto conv2_epilogue = [&](int pair_idx) {
      mbar_wait(bar_acc, acc_phase);
      acc_phase ^= 1;
      tc_fence_after();
      const int q = warp & 3, hh = warp >> 2;              // lane quarter, 32-column half
      const int r = q * 32 + lane;                          // row = (f, y2, x2) of this pair
      uint32_t v[32];
      tmem_ld_32x32b_x32(tmem_acc2 + (static_cast<uint32_t>(q * 32) << 16) + hh * 32, v);
      tmem_ld_wait();
      const int pixel = pair_idx * 128 + r;                 // pixel index inside the 8-frame act2 block
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        uint4 u;
        const float4 ba = __ldg(reinterpret_cast<const float4*>(p.b2 + hh * 32 + ch * 8));
        const float4 bc = __ldg(reinterpret_cast<const float4*>(p.b2 + hh * 32 + ch * 8 + 4));
        u.x = pack_bf16x2(fmaxf(__uint_as_float(v[ch * 8 + 0]) + ba.x, 0.f), fmaxf(__uint_as_float(v[ch * 8 + 1]) + ba.y, 0.f));
        u.y = pack_bf16x2(fmaxf(__uint_as_float(v[ch * 8 + 2]) + ba.z, 0.f), fmaxf(__uint_as_float(v[ch * 8 + 3]) + ba.w, 0.f));
        u.z = pack_bf16x2(fmaxf(__uint_as_float(v[ch * 8 + 4]) + bc.x, 0.f), fmaxf(__uint_as_float(v[ch * 8 + 5]) + bc.y, 0.f));
        u.w = pack_bf16x2(fmaxf(__uint_as_float(v[ch * 8 + 6]) + bc.z, 0.f), fmaxf(__uint_as_float(v[ch * 8 + 7]) + bc.w, 0.f));
        *reinterpret_cast<uint4*>(act2 + act2_chunk_off(pixel, hh * 4 + ch)) = u;
      }
      tc_fence_before();
      named_bar_sync(1, TC_BUILDERS);     // act2 rows of this pair visible; acc2 drained
    };

    // conv3 epilogue of the CTA's g_lt-th group (frames g_frame0 ..): acc (8 frames x 16 px, 128 ch) -> bias + ReLU ->
    // mean over 16 px -> pooled.  Deferred: it runs after conv1 of the next group's second pair, when the MMAs have
    // long completed, instead of waiting for them at the end of the group.
    auto conv3_epilogue = [&](uint32_t g_lt, int g_frame0) {
      mbar_wait(&bar_acc3[g_lt & 1], (g_lt >> 1) & 1);
      tc_fence_after();
      {
        const int q = warp & 3, hh = warp >> 2;                  // lane quarter (2 frames), 64-column half
        const int fr = g_frame0 + q * 2 + (lane >> 4);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          uint32_t v[32];
          const int col0 = hh * 64 + cc * 32;
          tmem_ld_32x32b_x32(tmem_acc3 + (g_lt & 1) * 128 + (static_cast<uint32_t>(q * 32) << 16) + col0, v);
          tmem_ld_wait();
          // bias + ReLU, then sum the 16 pixel rows of each frame (lanes 0-15 / 16-31) with a transposing butterfly:
          // every step halves the number of live columns per lane, 30 shuffles instead of 4 per column.
          float x[32];
#pragma unroll
          for (int jx = 0; jx < 32; ++jx) x[jx] = fmaxf(__uint_as_float(v[jx]) + __ldg(p.b3 + col0 + jx), 0.f);
#pragma unroll
          for (int jx = 0; jx < 16; ++jx) {            // lanes with bit3 clear keep columns 0-15, set keep 16-31
            const bool up = (lane & 8) != 0;
            const float send = up ? x[jx] : x[jx + 16];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 8);
            x[jx] = (up ? x[jx + 16] : x[jx]) + recv;
          }
#pragma unroll
          for (int jx = 0; jx < 8; ++jx) {
            const bool up = (lane & 4) != 0;
            const float send = up ? x[jx] : x[jx + 8];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 4);
            x[jx] = (up ? x[jx + 8] : x[jx]) + recv;
          }
#pragma unroll
          for (int jx = 0; jx < 4; ++jx) {
            const bool up = (lane & 2) != 0;
            const float send = up ? x[jx] : x[jx + 4];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 2);
            x[jx] = (up ? x[jx + 4] : x[jx]) + recv;
          }
#pragma unroll
          for (int jx = 0; jx < 2; ++jx) {
            const bool up = (lane & 1) != 0;
            const float send = up ? x[jx] : x[jx + 2];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
            x[jx] = (up ? x[jx + 2] : x[jx]) + recv;
          }
          // lane l (within its 16-lane half) now holds the frame sums of columns cbase, cbase+1 with
          // cbase = 16*bit3 + 8*bit2 + 4*bit1 + 2*bit0
          if (fr < p.M) {
            const int cbase = ((lane & 8) ? 16 : 0) + ((lane & 4) ? 8 : 0) + ((lane & 2) ? 4 : 0) + ((lane & 1) ? 2 : 0);
            *reinterpret_cast<uint32_t*>(p.pooled + static_cast<size_t>(fr) * 128 + col0 + cbase) =
                pack_bf16x2(x[0] * (1.f / 16.f), x[1] * (1.f / 16.f));
          }
        }
      }
      tc_fence_before();
    };
    prefetch_pair(blockIdx.x * GROUP);
    uint32_t lt = 0;
    int prev_frame0 = 0;

    for (int grp = blockIdx.x; grp < p.num_groups; grp += gridDim.x, ++lt) {
      const int frame0 = grp * GROUP;
      CTRACE(0);
      for (int pair = 0; pair < GROUP / 2; ++pair) {
        // ---- stage 2 input frames (interior of the zero-bordered 34x34 tiles) from the prefetch registers ----
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int id = tid + TC_BUILDERS * i;
          const int f = id >> 8, rem = id & 255;
          const int y = rem >> 3, x4 = (rem & 7) * 4;
          float* d = sIn + f * 34 * 34 + (y + 1) * 34 + (x4 + 1);
          d[0] = pre[i].x; d[1] = pre[i].y; d[2] = pre[i].z; d[3] = pre[i].w;
        }
        named_bar_sync(1, TC_BUILDERS);
        CTRACE(1 + pair * 5);          // input staged
        {
          const int next_first = (pair + 1 < GROUP / 2) ? frame0 + (pair + 1) * 2 : (grp + static_cast<int>(gridDim.x)) * GROUP;
          prefetch_pair(next_first);
        }

        // ---- conv1: rows = 2 x 256 output pixels, K = 9 (padded to 16), N = 32 ----
#pragma unroll
        for (int t = warp; t < 32; t += TC_BUILDERS / 32) {   // 4 independent m-tiles per warp: unrolled for ILP
          uint32_t a[4] = {0, 0, 0, 0};
          int pix[2];
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int r = t * 16 + gid + 8 * hf;
            const int f = r >> 8, rem = r & 255, y = rem >> 4, x = rem & 15;
            pix[hf] = r;
            const float* base = sIn + f * 34 * 34 + (2 * y) * 34 + 2 * x;
            a[hf] = pack_bf16x2(base[off0], base[off1]);
            if (tig == 0) a[2 + hf] = pack_bf16x2(base[off8], 0.f);
          }
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) {
            float cacc[4] = {0.f, 0.f, 0.f, 0.f};
            mma_bf16_16816(cacc, a[0], a[1], a[2], a[3], bw1[nt][0], bw1[nt][1]);
            const float bb0 = bias1[nt][0], bb1 = bias1[nt][1];
            *reinterpret_cast<uint32_t*>(act1 + act1_chunk_off(pix[0], nt) + tig * 4) =
                pack_bf16x2(fmaxf(cacc[0] + bb0, 0.f), fmaxf(cacc[1] + bb1, 0.f));
            *reinterpret_cast<uint32_t*>(act1 + act1_chunk_off(pix[1], nt) + tig * 4) =
                pack_bf16x2(fmaxf(cacc[2] + bb0, 0.f), fmaxf(cacc[3] + bb1, 0.f));
          }
        }
        named_bar_sync(1, TC_BUILDERS);
        CTRACE(2 + pair * 5);          // conv1 done

        // deferred epilogues: the previous pair's conv2 (its MMAs had the staging + conv1 above to complete) and,
        // in the second pair, the previous group's conv3
        if (pair > 0) conv2_epilogue(pair - 1);
        if (pair == 1 && lt > 0) conv3_epilogue(lt - 1, prev_frame0);
        CTRACE(3 + pair * 5);          // deferred conv2 epilogue done

        // ---- conv2: 5 slabs of two taps, gathered from act1 ----
        for (int j = 0; j < W2_SLABS; ++j, ++n_slab) {
          const uint32_t slot = n_slab % NSLOT, use = n_slab / NSLOT;
          if (use > 0) mbar_wait(&ring_free[slot], (use - 1) & 1);
          const int tap = 2 * j + bhh;
          const int ky = (tap * 11) >> 5, kx = tap - 3 * ky;                 // tap / 3, tap % 3 for tap < 16
          const bool ok = (tap < 9) && (kx == 0 ? vx2[0] : (kx == 1 ? vx2[1] : vx2[2])) && !(ky == 0 && top2);
          const int src = rowbase2 + ky * 1024 + (kx == 0 ? xo2[0] : (kx == 1 ? xo2[1] : xo2[2]));
          const int s0 = kx == 0 ? s02[0] : (kx == 1 ? s02[1] : s02[2]);
          uint32_t cols[16];
#pragma unroll
          for (int cch = 0; cch < 4; ++cch) {
            uint4 val = make_uint4(0, 0, 0, 0);
            if (ok) val = *reinterpret_cast<const uint4*>(act1 + src + ((s0 ^ cch) << 4));
            cols[4 * cch] = val.x; cols[4 * cch + 1] = val.y; cols[4 * cch + 2] = val.z; cols[4 * cch + 3] = val.w;
          }
          tc_fence_after();
          publish_slab(slot, cols);
        }
        CTRACE(4 + pair * 5);          // conv2 slabs built
      }
      conv2_epilogue(GROUP / 2 - 1);
      CTRACE(21);                      // last conv2 epilogue done

      // ---- conv3: one slab per tap gathered from act2; weights streamed by TMA ----
      for (int t = 0; t < 9; ++t, ++n_slab) {
        const uint32_t slot = n_slab % NSLOT, use = n_slab / NSLOT;
        if (use > 0) mbar_wait(&ring_free[slot], (use - 1) & 1);
        const int ky = (t * 11) >> 5, kx = t - 3 * ky;
        const bool ok = (kx == 0 ? vx3[0] : (kx == 1 ? vx3[1] : vx3[2])) && !(ky == 0 && top3);
        const int src = rowbase3 + ky * 1024 + (kx == 0 ? xo3[0] : (kx == 1 ? xo3[1] : xo3[2]));
        const int s0 = kx == 0 ? s03[0] : (kx == 1 ? s03[1] : s03[2]);
        uint32_t cols[16];
#pragma unroll
        for (int cch = 0; cch < 4; ++cch) {
          uint4 val = make_uint4(0, 0, 0, 0);
          if (ok) val = *reinterpret_cast<const uint4*>(act2 + src + (((4 * bhh + cch) ^ s0) << 4));
          cols[4 * cch] = val.x; cols[4 * cch + 1] = val.y; cols[4 * cch + 2] = val.z; cols[4 * cch + 3] = val.w;
        }
        tc_fence_after();
        publish_slab(slot, cols);
      }
      CTRACE(22);                      // conv3 slabs built
      CTRACE(23);
      CTRACE(24);                      // group done
      prev_frame0 = frame0;
    }
    if (lt > 0) conv3_epilogue(lt - 1, prev_frame0);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == TC_BUILDERS / 32) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

size_t visual_cnn_tc_w2_bytes() { return W2_SLABS * W2_SLAB_BYTES; }
size_t visual_cnn_tc_w3_bytes() { return 9 * SLAB_BYTES; }

// w2 [64][9*32], w3 [128][9*64] fp32, BN-folded, K index = tap*Cin + c  ->
//   w2_slabs: 5 slabs [64 rows][64 k] bf16, k = (tap&1)*32 + c of taps (2j, 2j+1), 128B-swizzled (chunk ^= row&7)
//   w3_rows : [9 taps][128 rows][64 k] bf16 row-major (TMA applies the swizzle)
void visual_cnn_tc_pack(const float* w2, const float* w3, uint8_t* w2_slabs, uint8_t* w3_rows) {
  memset(w2_slabs, 0, visual_cnn_tc_w2_bytes());
  for (int j = 0; j < W2_SLABS; ++j)
    for (int n = 0; n < 64; ++n)
      for (int k = 0; k < 64; ++k) {
        const int tap = 2 * j + (k >> 5), c = k & 31;
        const float val = tap < 9 ? w2[static_cast<size_t>(n) * 288 + tap * 32 + c] : 0.f;
        const int chunk = (k >> 3) ^ (n & 7);
        uint16_t* dst = reinterpret_cast<uint16_t*>(w2_slabs + j * W2_SLAB_BYTES + n * 128 + chunk * 16) + (k & 7);
        *dst = f2bf(val);
      }
  uint16_t* o = reinterpret_cast<uint16_t*>(w3_rows);
  for (int t = 0; t < 9; ++t)
    for (int n = 0; n < 128; ++n)
      for (int c = 0; c < 64; ++c) o[(static_cast<size_t>(t) * 128 + n) * 64 + c] = f2bf(w3[static_cast<size_t>(n) * 576 + t * 64 + c]);
}

const char* launch_visual_cnn_tc(cudaStream_t s, const float* frames, int M, const CnnWeights& w, const uint8_t* w2_slabs,
                                 const uint8_t* w3_rows, void* pooled, int num_sms, unsigned long long* trace,
                                 const int* frame_lens, int N) {
  if (M <= 0) return "visual_cnn_tc: empty problem";
  CUtensorMap tm;   // w3_rows as [9 * 128 rows][64] bf16
  if (const char* e = tma_encode_2d(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w3_rows, 64, 9 * 128, 64, 64, 128)) return e;
  if (!smem_opt_in(visual_cnn_tc_kernel, TC_SMEM)) return "visual_cnn_tc: cudaFuncSetAttribute failed";
  CnnTcDev d;
  d.frames = frames; d.pooled = reinterpret_cast<__nv_bfloat16*>(pooled);
  d.w1 = w.w1; d.b1 = w.b1; d.w2_slabs = w2_slabs; d.b2 = w.b2; d.b3 = w.b3;
  d.M = M; d.num_groups = (M + GROUP - 1) / GROUP;
  d.trace = trace;
  d.frame_lens = frame_lens; d.N = N;
  const int grid = d.num_groups < num_sms ? d.num_groups : num_sms;
  launch_pdl(visual_cnn_tc_kernel, dim3(grid), dim3(TC_THREADS), TC_SMEM, s, tm, d);
  return cudaGetLastError() == cudaSuccess ? nullptr : "visual_cnn_tc: launch failed";
}

}  // namespace avsep
