// SeparationDecoder.separate (model.py:210-220) as a stand-alone kernel, and the arrival / acknowledge flags of the
// masks-only gather (avsep_b200/sharded.py): every rank pushes only its `masks` shard into the root's global buffer
// over NVLink, then raises a ticket in the root's memory; the root waits for the tickets in stream order and rebuilds
// `separated = masks * mixed` for the remote shards from the mixture it already holds -- bit for bit what the remote
// decoder epilogue wrote (one fp32 multiply), with half of the bytes on the wire.
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

// separated[b,s,f,t] = masks[b,s,f,t] * mixed[b,f,t]; both planes are flat (F*T) arrays, so the kernel walks the flat
// output index: thread = 4 consecutive elements (16-byte loads / stores of masks / separated; the 4 mixture values are
// scalar loads because an (F*T)-float plane is not a multiple of 16 bytes: 257 x 63 floats).  `head` elements in front
// of the first 16-byte boundary (masks and separated share their misalignment, e.g. the two halves of one allocation)
// and the ragged tail are handled element-wise by the first threads.  HBM-bound: 4 * F * T * (2 S + 1) algorithmic
// bytes per utterance (masks in, separated out, the mixture once).
// Variable-length batch (VARLEN): utterance b owns the frames t < T_b = lens[b] clamped to [1, T] (utt_len, as in the
// forward); there the product is the same single multiply, past T_b the kernel stores 0 and reads neither masks nor
// mixed, so NaN / Inf in the padding cannot reach the output (0 x NaN would).  A 4-element group can straddle T_b (T is
// odd at the benchmark shape): its 16-byte masks load is taken only when all four elements are live, else the live
// ones are loaded one by one.
template <bool VARLEN>
__device__ __forceinline__ void separate_one(const float* masks, const float* mixed, float* out, long long i, int plane,
                                             int S, const int* lens, int T) {
  const long long pbs = i / plane;
  if constexpr (VARLEN) {
    const int r = static_cast<int>(i - pbs * plane);
    out[i] = r % T < utt_len(lens, static_cast<int>(pbs / S), T) ? masks[i] * mixed[(pbs / S) * plane + r] : 0.f;
  } else {
    out[i] = masks[i] * mixed[(pbs / S) * plane + (i - pbs * plane)];
  }
}

template <bool VEC, bool VARLEN>
__global__ void __launch_bounds__(256)
separate_kernel(const float* __restrict__ masks, const float* __restrict__ mixed, float* __restrict__ out,
                long long total, int plane, int S, int head, const int* __restrict__ lens, int T) {
  const long long tid = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if constexpr (!VEC) {
    if (tid < total) separate_one<VARLEN>(masks, mixed, out, tid, plane, S, lens, T);
    return;
  }
  const long long groups = (total - head) / 4;
  if (tid < groups) {
    const long long i0 = head + tid * 4;
    long long bs = i0 / plane;                     // (b, s) plane of the first element
    int r = static_cast<int>(i0 - bs * plane);     // offset inside the plane
    long long mbase = (bs / S) * plane;            // mixture plane of utterance b
    if constexpr (VARLEN) {
      int t = r % T, tb = utt_len(lens, static_cast<int>(bs / S), T);
      int live = 0;                                // bit k: element k lies inside its utterance's length
      long long mi[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (r == plane) {                          // crossed into the next (b, s) plane: t restarts, b may change
          r = 0;
          t = 0;
          ++bs;
          mbase = (bs / S) * plane;
          tb = utt_len(lens, static_cast<int>(bs / S), T);
        }
        if (t < tb) live |= 1 << k;
        mi[k] = mbase + r;
        ++r;
        if (++t == T) t = 0;
      }
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (live == 15) {
        const float4 m = __ldcs(reinterpret_cast<const float4*>(masks + i0));
        v[0] = m.x; v[1] = m.y; v[2] = m.z; v[3] = m.w;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (live >> k & 1) v[k] = __ldcs(masks + i0 + k);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (live >> k & 1) v[k] *= __ldg(mixed + mi[k]);
      __stcs(reinterpret_cast<float4*>(out + i0), make_float4(v[0], v[1], v[2], v[3]));
    } else {
      const float4 m = __ldcs(reinterpret_cast<const float4*>(masks + i0));
      float v[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (r == plane) {                            // crossed into the next (b, s) plane
          r = 0;
          ++bs;
          mbase = (bs / S) * plane;
        }
        v[k] *= __ldg(mixed + mbase + r);
        ++r;
      }
      __stcs(reinterpret_cast<float4*>(out + i0), make_float4(v[0], v[1], v[2], v[3]));
    }
  }
  if (tid < 8) {                                   // <= 3 head + <= 3 tail elements
    const long long tail0 = head + groups * 4;
    const long long i = tid < head ? tid : tail0 + (tid - head);
    if (i < total && (tid < head || i >= tail0)) separate_one<VARLEN>(masks, mixed, out, i, plane, S, lens, T);
  }
}

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// One CTA, thread i raises flag i (its own memory or a peer's).  Stream order puts it after the copies it announces.
__global__ void flag_signal_kernel(FlagSet f, unsigned value) {
  const int i = threadIdx.x;
  if (i < f.n) {
    __threadfence_system();
    st_release_sys(f.ptr[i], value);
  }
}

// One CTA, thread i waits until flag i (local memory, written by a peer over NVLink or by this GPU) reaches `value`.
// Tickets only grow, so >= is the test (wrap-safe through the signed difference).  A flag that does not arrive within
// the time limit traps: the caller sees a launch failure instead of a hang.
__global__ void flag_wait_kernel(FlagSet f, unsigned value, unsigned long long timeout_ns) {
  const int i = threadIdx.x;
  if (i < f.n) {
    const unsigned long long t0 = globaltimer();
    while (static_cast<int>(ld_acquire_sys(f.ptr[i]) - value) < 0) {
      __nanosleep(200);
      if (globaltimer() - t0 > timeout_ns) {
        printf("avsep flag wait: flag %d stuck at %u, waiting for %u\n", i, ld_acquire_sys(f.ptr[i]), value);
        __trap();
      }
    }
  }
  __syncthreads();
  __threadfence_system();
}

// With lazy module loading (the CUDA 12 default) the first launch of a kernel loads it, and loading may have to wait
// for running kernels -- a waiter spinning for a signal kernel that is not loaded yet would never see it.  Every entry
// point of this file therefore loads all of the file's kernels first (once per device).
const char* preload_kernels() {
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return "peer_gather: bad device";
  if (done[dev]) return nullptr;
  cudaFuncAttributes a;
  if (cudaFuncGetAttributes(&a, flag_signal_kernel) != cudaSuccess || cudaFuncGetAttributes(&a, flag_wait_kernel) != cudaSuccess ||
      cudaFuncGetAttributes(&a, separate_kernel<true, false>) != cudaSuccess ||
      cudaFuncGetAttributes(&a, separate_kernel<false, false>) != cudaSuccess ||
      cudaFuncGetAttributes(&a, separate_kernel<true, true>) != cudaSuccess ||
      cudaFuncGetAttributes(&a, separate_kernel<false, true>) != cudaSuccess)
    return "peer_gather: kernel image not loadable on this device";
  done[dev] = true;
  return nullptr;
}

}  // namespace

const char* launch_separate(cudaStream_t s, const float* masks, const float* mixed, float* out, long long B, int S,
                            int F, int T, const int* lens) {
  if (B <= 0) return nullptr;
  if (const char* e = preload_kernels()) return e;
  const long long plane = static_cast<long long>(F) * T;
  if (plane > 0x7fffffffLL) return "separate: F*T too large";
  const long long total = B * S * plane;
  const uintptr_t am = reinterpret_cast<uintptr_t>(masks), ao = reinterpret_cast<uintptr_t>(out);
  if ((am | ao | reinterpret_cast<uintptr_t>(mixed)) & 3) return "separate: buffers must be 4-byte aligned";
  const bool vec = ((am ^ ao) & 15) == 0 && total >= 8;      // same misalignment: one shifted vector walk serves both
  const int head = vec ? static_cast<int>(((16 - (am & 15)) & 15) / 4) : 0;
  const long long threads = vec ? (total - head) / 4 + 8 : total;
  const long long blocks = (threads + 255) / 256;
  if (blocks > 0x7fffffffLL) return "separate: batch too large";
  auto kernel = vec ? (lens ? separate_kernel<true, true> : separate_kernel<true, false>)
                    : (lens ? separate_kernel<false, true> : separate_kernel<false, false>);
  kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(masks, mixed, out, total, static_cast<int>(plane), S, head, lens, T);
  return cudaGetLastError() == cudaSuccess ? nullptr : "separate: launch failed";
}

const char* launch_flag_signal(cudaStream_t s, const FlagSet& f, unsigned value) {
  if (f.n <= 0) return nullptr;
  if (f.n > FlagSet::MAX) return "flag_signal: too many flags";
  if (const char* e = preload_kernels()) return e;
  flag_signal_kernel<<<1, 32, 0, s>>>(f, value);
  return cudaGetLastError() == cudaSuccess ? nullptr : "flag_signal: launch failed";
}

const char* launch_flag_wait(cudaStream_t s, const FlagSet& f, unsigned value, double timeout_s) {
  if (f.n <= 0) return nullptr;
  if (f.n > FlagSet::MAX) return "flag_wait: too many flags";
  if (const char* e = preload_kernels()) return e;
  flag_wait_kernel<<<1, 32, 0, s>>>(f, value, static_cast<unsigned long long>(timeout_s * 1e9));
  return cudaGetLastError() == cudaSuccess ? nullptr : "flag_wait: launch failed";
}

}  // namespace avsep
