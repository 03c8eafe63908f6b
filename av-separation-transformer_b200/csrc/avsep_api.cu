// C-ABI layer of libavsep.so (see include/avsep.h): handle, weight prepack, workspace plan and the forward
// orchestration of AVSeparationTransformer.forward (reference: model.py:268-276 and everything it calls).
#include "../../include/avsep.h"
#include "kernels.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <functional>
#include <map>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

using namespace avsep;

namespace {

std::string g_create_error;

__global__ void op_to_f32_kernel(const __nv_bfloat16* in, float* out, size_t n) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}

// out[b, t, :] = lerp of x[b, i0(t), :], x[b, i1(t), :]   (F.interpolate linear, align_corners=False; model.py:115)
__global__ void interp_rows_kernel(const float* __restrict__ x, float* __restrict__ out, int N, int T, int d) {
  const int t = blockIdx.x, b = blockIdx.y;
  const LerpTap k = lerp_tap(t, N, lerp_scale(N, T));
  const float* r0 = x + (static_cast<size_t>(b) * N + k.i0) * d;
  const float* r1 = x + (static_cast<size_t>(b) * N + k.i1) * d;
  float* o = out + (static_cast<size_t>(b) * T + t) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) o[c] = k.w0 * r0[c] + k.w1 * r1[c];
}
const char* launch_interp_rows(cudaStream_t s, const float* x, float* out, int B, int N, int T, int d) {
  interp_rows_kernel<<<dim3(T, B), 128, 0, s>>>(x, out, N, T, d);
  return cudaGetLastError() == cudaSuccess ? nullptr : "interp_rows: launch failed";
}

// Profiling aid: keeps the GPU busy while the host enqueues a whole forward, so that the per-kernel event pairs
// measure device time and not host launch latency.
__global__ void spin_kernel(unsigned long long ns) {
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
  do {
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  } while (t - t0 < ns);
}

// ---- owners of the handle's CUDA resources: each releases its resource when it is replaced or destroyed ----
template <typename H, cudaError_t (*Release)(H)>
struct Releaser {
  void operator()(H x) const { Release(x); }
};
template <typename H, cudaError_t (*Release)(H)>
using Owned = std::unique_ptr<std::remove_pointer_t<H>, Releaser<H, Release>>;
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using GraphExec = Owned<cudaGraphExec_t, cudaGraphExecDestroy>;

// Creates the (non-blocking) stream or the event unless it exists.
cudaError_t make_stream(Stream& s) {
  if (s) return cudaSuccess;
  cudaStream_t x;
  const cudaError_t e = cudaStreamCreateWithFlags(&x, cudaStreamNonBlocking);
  if (e == cudaSuccess) s.reset(x);
  return e;
}
cudaError_t make_event(Event& ev, unsigned flags = cudaEventDisableTiming) {
  if (ev) return cudaSuccess;
  cudaEvent_t x;
  const cudaError_t e = cudaEventCreateWithFlags(&x, flags);
  if (e == cudaSuccess) ev.reset(x);
  return e;
}

// cap elements of device memory (PINNED: page-locked host memory).  alloc() frees the current block before it makes the
// new one, so its caller first makes sure that no queued work and no cached graph still uses the old one.
template <typename T, bool PINNED = false>
struct Buf {
  struct Free {
    void operator()(T* p) const { PINNED ? cudaFreeHost(p) : cudaFree(p); }
  };
  std::unique_ptr<T, Free> ptr;
  size_t cap = 0;
  T* get() const { return ptr.get(); }
  cudaError_t alloc(size_t n) {
    ptr.reset();
    T* p = nullptr;
    const cudaError_t e = PINNED ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
    ptr.reset(e == cudaSuccess ? p : nullptr);
    cap = e == cudaSuccess ? n : 0;
    return e;
  }
};

struct GraphKey {
  int B, T, N, Hh, Ww;
  const void *mixed, *frames, *sep, *masks, *ws;
  const int *lens, *frame_lens;   // the kernels read the lengths at run time: their contents are not part of the key
  bool xp_ready;                  // the forward of avsep_separate_waveforms (forward_device): never shares a graph
  bool operator==(const GraphKey& o) const {
    return B == o.B && T == o.T && N == o.N && Hh == o.Hh && Ww == o.Ww && mixed == o.mixed && frames == o.frames &&
           sep == o.sep && masks == o.masks && ws == o.ws && lens == o.lens && frame_lens == o.frame_lens &&
           xp_ready == o.xp_ready;
  }
};
struct GraphEntry {
  GraphKey key;
  GraphExec exec;
  int64_t launches = 0;
  uint64_t last_use = 0;
};

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

// One encoder or fusion layer on the device.  w_in / b_in: the attention input projection, Q|K|V rows in an encoder
// layer, Q rows only in a fusion layer (the K|V rows of all fusion layers are one concatenated matrix).
struct LayerW {
  const void *w_in, *wo, *w1, *w2;
  const float *b_in, *bo, *b1, *b2, *n1g, *n1b, *n2g, *n2b;
};

struct Workspace {   // carved from one base pointer; all offsets 1 KB aligned
  int B = 0, T = 0, N = 0, Hh = 0, Ww = 0;
  // variable-length batch (avsep_forward_varlen): device int32 [B] audio frames / lip frames per utterance, or null
  // (all T / all N).  Every kernel where rows of different lengths meet reads them.
  const int *lens = nullptr, *frame_lens = nullptr;
  size_t bytes = 0;
  // audio side
  void *xp, *h1, *a_op, *qkv_a, *attn_a, *ffn_a;
  float *x_a, *y_a;
  // visual side
  void *pooled, *v_op, *qkv_v, *attn_v, *ffn_v;
  float *x_v, *y_v, *kvn;
  void* kvb;   // fused fusion stack: K|V rows of every fusion layer, projected from the interpolated visual rows (bf16)
};

}  // namespace

struct avsep_handle {
  avsep_config cfg{};
  int Fp = 0;
  int num_sms = 148;
  std::string err;
  std::map<std::string, HostTensor> host_w;
  bool finalized = false;
  bool use_graph = true; // replay the forward as a CUDA graph (captured per shape + buffer set on its 2nd use)
  int attn_tc = 1;       // AttnProblem::tc_mode of every attention launch
  bool two_stream = true; // audio and visual branches on two streams (fork/join), so partial waves overlap
  Stream aux_stream;
  Event ev_fork, ev_join;
  std::vector<GraphEntry> graphs;
  uint64_t graph_clock = 0;
  Stream cap_stream;
  int profile_spin_us = 3000;
  Buf<uint8_t> weights;
  // device views into weights
  const void *wc1 = nullptr, *wc2 = nullptr, *wproj = nullptr, *wkv_all = nullptr, *wdec0 = nullptr, *wdec3 = nullptr;
  const float *bc1 = nullptr, *bc2 = nullptr, *bproj = nullptr, *bkv_all = nullptr, *bdec0 = nullptr, *bdec3 = nullptr;
  const float *pe_a = nullptr, *pe_v = nullptr, *fng = nullptr, *fnb = nullptr;
  CnnWeights cnn{};
  const uint8_t *cnn_w2_slabs = nullptr, *cnn_w3_rows = nullptr;   // tcgen05 CNN operands
  std::vector<LayerW> enc_a, enc_v, fus;
  // prepacked weight streams / vector blocks of the fused transformer-stack kernel (null when the config cannot use it)
  const uint8_t *xs_a = nullptr, *xs_v = nullptr, *xs_f = nullptr;
  bool xs_f_decoder = false;   // the fusion stream continues with the SeparationDecoder block
  const uint8_t *xs_a_np = nullptr, *xs_v_np = nullptr;   // encoder streams past their input-projection items
  bool xs_v_kvp = false;       // the visual stream ends with the fusion layers' K | V projection block
  // cached library-owned workspace
  Buf<uint8_t> own_ws;
  // host-path staging
  // host-buffer entry point: two independent I/O slots so that consecutive calls can overlap (copy-in of call i+1
  // with the kernels and copy-out of call i); slot 0 serves the synchronous avsep_forward_host
  struct HostSlot {
    Buf<float> io[4];                // mixed, frames, separated, masks (device)
    std::vector<Event> ev;           // 2 per chunk: copy-in done, kernels done
    Event ev_start, ev_end;          // ev_end: last copy-out done
    Event ev_lane[3];                // last kernels of this slot on each compute lane
    // packed batches (avsep_forward_host_packed*): the call's lengths, then its frame lengths, uploaded once per call
    Buf<int32_t, true> lens_host;
    Buf<int32_t> lens_dev;
    Event ev_lens;                   // upload of lens_host done
  } slot[AVSEP_HOST_SLOTS];
  std::vector<void*> shared_owned, shared_mapped;   // avsep_shared_alloc / avsep_shared_open
  Buf<float> synth_waves;   // scratch of avsep_synth_batch
  Stream hs[3];
  int host_chunk = 0;    // utterances per pipeline chunk of the host path; 0 = auto (see host_submit)
  bool pdl = true;       // programmatic dependent launch between consecutive kernels of a stream
  int host_lanes = 0;    // chunks whose kernels may be in flight at once (own stream + workspace each); 0 = auto
  Buf<uint8_t> host_ws;
  Stream host_comp[3];
  // debug
  bool debug = false;
  struct Snapshot {
    Buf<float> buf;
    size_t count = 0;
  };
  std::map<std::string, Snapshot> snaps;
  int64_t launches = 0;
  // per-launch profiling (cudaEvent pairs on the launching stream)
  bool profile = false;
  std::vector<Event> ev_pool;
  size_t ev_used = 0;
  std::vector<std::pair<const char*, size_t>> ev_marks;   // label, index of the start event (stop = +1)
  std::map<std::string, std::pair<int64_t, double>> prof;  // label -> (launches, total ms)

  // every other resource has an owner above; the buffers shared with other processes are released here at the latest
  ~avsep_handle() {
    for (void* ptr : shared_mapped) cudaIpcCloseMemHandle(ptr);
    for (void* ptr : shared_owned) cudaFree(ptr);
  }
};

namespace {

int fail(avsep_handle* h, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return 1;
}

// Selects `device` unless it is current, and selects the caller's device again when it goes out of scope.
struct DeviceScope {
  int caller = 0;
  bool switched = false;
  cudaError_t err;
  explicit DeviceScope(int device) : err(cudaGetDevice(&caller)) {
    if (err == cudaSuccess && caller != device) {
      err = cudaSetDevice(device);
      switched = err == cudaSuccess;
    }
  }
  ~DeviceScope() {
    if (switched) cudaSetDevice(caller);
  }
};
// The rest of the calling C-ABI function runs on `device`, and no call changes which device the calling thread has
// current, on any return path.
#define ON_DEVICE(h, device)              \
  const DeviceScope device_scope(device); \
  if (device_scope.err != cudaSuccess)    \
    return fail(h, std::string("cannot select the device: ") + cudaGetErrorString(device_scope.err))

int prof_begin(avsep_handle* h, const char* label, cudaStream_t s) {
  if (h->ev_used + 2 > h->ev_pool.size()) {
    for (int i = 0; i < 64; ++i) {
      Event e;
      if (make_event(e, cudaEventDefault) != cudaSuccess) return 1;
      h->ev_pool.push_back(std::move(e));
    }
  }
  h->ev_marks.emplace_back(label, h->ev_used);
  cudaEventRecord(h->ev_pool[h->ev_used].get(), s);
  return 0;
}
void prof_end(avsep_handle* h, cudaStream_t s) {
  cudaEventRecord(h->ev_pool[h->ev_used + 1].get(), s);
  h->ev_used += 2;
}

cudaStream_t stream_of(LaunchCtx lc) { return lc.stream; }
cudaStream_t stream_of(cudaStream_t s) { return s; }

// Launcher call fn(on, ...), where `on` is the LaunchCtx of a launch_pdl launcher or the stream of a <<<>>> one, counted
// as one launch of the call.  With profiling on, the call is bracketed by an event pair on that same stream.
#define CKL(label, on, fn, ...)                                         \
  do {                                                                  \
    const cudaStream_t _s = stream_of(on);                              \
    if (h->profile && prof_begin(h, label, _s)) return fail(h, "profiling: cudaEventCreate failed"); \
    const char* _e = fn(on, __VA_ARGS__);                               \
    if (_e != nullptr) return fail(h, std::string(_e) + " [" #fn "(" #on ", " #__VA_ARGS__ ")]"); \
    if (h->profile) prof_end(h, _s);                                    \
    ++h->launches;                                                      \
  } while (0)
#define CK(on, fn, ...) CKL("other", on, fn, __VA_ARGS__)

#define CUDA_OK(expr)                                                                           \
  do {                                                                                          \
    cudaError_t _c = (expr);                                                                    \
    if (_c != cudaSuccess) return fail(h, std::string(#expr ": ") + cudaGetErrorString(_c));    \
  } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

void drop_graphs(avsep_handle* h) { h->graphs.clear(); }   // cached graphs hold raw pointers to weights / workspace

// The launch settings of h's forward-path kernels on stream s: per-launch event pairs (profiling) must time the kernels
// one at a time, so profiling turns PDL off.
LaunchCtx launch_ctx(const avsep_handle* h, cudaStream_t s) { return {s, h->pdl && !h->profile}; }

// The entry of every C-ABI call that enqueues device work on the caller's stream: the call runs on h's device, the
// launch count starts again from 0, and `lc` holds h's launch settings on that stream.
#define ENTER(h, stream)                                                 \
  if (!h) return 1;                                                      \
  ON_DEVICE(h, h->cfg.device);                                           \
  h->launches = 0;                                                       \
  const LaunchCtx lc = launch_ctx(h, static_cast<cudaStream_t>(stream))

size_t op_size(const avsep_handle* h) { return h->cfg.precision == AVSEP_PREC_TF32 ? 4 : 2; }

// ---- workspace -------------------------------------------------------------------------------
size_t carve_workspace(const avsep_handle* h, Workspace& w, uint8_t* base, int B, int T, int N, int Hh, int Ww) {
  const size_t d = h->cfg.d_model, os = op_size(h);
  const size_t Ma = static_cast<size_t>(B) * T, Map = static_cast<size_t>(B) * (T + 2), Mv = static_cast<size_t>(B) * N;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? base + off : nullptr;
    off += align_up(bytes, 1024);
    return p;
  };
  w.B = B; w.T = T; w.N = N; w.Hh = Hh; w.Ww = Ww;
  w.xp = take(Map * h->Fp * os);
  w.h1 = take(Map * d * os);
  w.x_a = static_cast<float*>(take(Ma * d * 4));
  w.y_a = static_cast<float*>(take(Ma * d * 4));
  w.a_op = take(Ma * d * os);
  w.qkv_a = take(Ma * 3 * d * os);
  w.attn_a = take(Ma * d * os);
  w.ffn_a = take(Ma * 4 * d * os);
  w.pooled = take(Mv * 128 * os);
  w.x_v = static_cast<float*>(take(Mv * d * 4));
  w.y_v = static_cast<float*>(take(Mv * d * 4));
  w.v_op = take(Mv * d * os);
  w.qkv_v = take(Mv * 3 * d * os);
  w.attn_v = take(Mv * d * os);
  w.ffn_v = take(Mv * 4 * d * os);
  w.kvn = static_cast<float*>(take(Mv * h->cfg.num_fusion_layers * 2 * d * 4));
  w.kvb = take(Ma * h->cfg.num_fusion_layers * 2 * d * os);
  w.bytes = off;
  return off;
}

int check_shape(avsep_handle* h, int B, int T, int N, int Hh, int Ww) {
  if (!h->finalized) return fail(h, "weights not finalized: call avsep_finalize_weights first");
  if (B < 1 || T < 1 || N < 1 || Hh < 1 || Ww < 1) return fail(h, "empty input: B, T, N, H, W must be >= 1");
  if (T > 5000 || N > 5000) return fail(h, "sequence longer than the positional table (max_len=5000, model.py:286)");
  if (B > 65535) return fail(h, "batch above 65535 utterances per call (grid dimension of the per-utterance kernels): split it");
  return 0;
}

// The caller's workspace when given (checked against `need`), else the library-owned one grown to `need`.
int workspace_base(avsep_handle* h, void* user_ws, size_t user_bytes, size_t need, const char* sizer, uint8_t*& base) {
  if (user_ws != nullptr) {
    if (user_bytes < need) return fail(h, std::string("workspace too small: see ") + sizer);
    if ((reinterpret_cast<uintptr_t>(user_ws) & 1023) != 0) return fail(h, "workspace must be 1024-byte aligned");
    base = static_cast<uint8_t*>(user_ws);
  } else {
    if (h->own_ws.cap < need) {
      drop_graphs(h);   // the cached graphs hold pointers into the old workspace
      CUDA_OK(h->own_ws.alloc(need));
    }
    base = h->own_ws.get();
  }
  return 0;
}

int get_workspace(avsep_handle* h, Workspace& w, void* user_ws, size_t user_bytes, int B, int T, int N, int Hh, int Ww) {
  uint8_t* base = nullptr;
  if (workspace_base(h, user_ws, user_bytes, carve_workspace(h, w, nullptr, B, T, N, Hh, Ww), "avsep_workspace_bytes",
                     base))
    return 1;
  carve_workspace(h, w, base, B, T, N, Hh, Ww);
  return 0;
}

// avsep_separate_waveforms: behind the forward's own workspace the complex spectrum (B, F, T), the masks (B, S, F, T)
// of a call without a masks buffer, the per-utterance frame counts T_b of a variable-length batch (int32 [B]), and the
// magnitude (B, F, T) and `separated` (B, S, F, T) that the fused fusion + decoder kernel reads and writes.
struct WaveStaging {
  float *spec, *masks;
  int32_t* tlens;
  float *mag, *sep;
};
size_t carve_waves(const avsep_handle* h, Workspace& w, WaveStaging& st, uint8_t* base, int B, int T, int N, int Hh,
                   int Ww) {
  size_t off = carve_workspace(h, w, base, B, T, N, Hh, Ww);
  auto take = [&](size_t bytes) {
    void* p = base ? base + off : nullptr;
    off += align_up(bytes, 1024);
    return p;
  };
  const size_t FT = static_cast<size_t>(h->cfg.freq_bins) * T;
  st.spec = static_cast<float*>(take(B * FT * 8));
  st.masks = static_cast<float*>(take(B * h->cfg.num_speakers * FT * 4));
  st.tlens = static_cast<int32_t*>(take(static_cast<size_t>(B) * 4));
  st.mag = static_cast<float*>(take(B * FT * 4));
  st.sep = static_cast<float*>(take(B * h->cfg.num_speakers * FT * 4));
  return off;
}

// Padded staging of a packed batch: the varlen forward's inputs and outputs, (B, F, T), (B, N, Hh, Ww) and 2 x
// (B, S, F, T), carved behind the forward's own workspace.  Returns the bytes of both.
struct Staging {
  float *mixed, *frames, *sep, *masks;
};
size_t carve_packed(const avsep_handle* h, Workspace& w, Staging& st, uint8_t* base, int B, int T, int N, int Hh,
                    int Ww) {
  size_t off = carve_workspace(h, w, base, B, T, N, Hh, Ww);
  auto take = [&](size_t floats) {
    float* p = base ? reinterpret_cast<float*>(base + off) : nullptr;
    off += align_up(floats * 4, 1024);
    return p;
  };
  const size_t F = h->cfg.freq_bins, S = h->cfg.num_speakers;
  st.mixed = take(B * F * T);
  st.frames = take(static_cast<size_t>(B) * N * Hh * Ww);
  st.sep = take(B * S * F * T);
  st.masks = take(B * S * F * T);
  return off;
}

// ---- debug snapshots ---------------------------------------------------------------------------
int snapshot(avsep_handle* h, cudaStream_t s, const char* name, const void* ptr, size_t count, bool is_op) {
  if (!h->debug) return 0;
  auto& snap = h->snaps[name];
  if (snap.buf.cap < count) CUDA_OK(snap.buf.alloc(count));
  snap.count = count;
  if (is_op && h->cfg.precision == AVSEP_PREC_BF16) {
    op_to_f32_kernel<<<static_cast<unsigned>((count + 255) / 256), 256, 0, s>>>(
        static_cast<const __nv_bfloat16*>(ptr), snap.buf.get(), count);
  } else {
    CUDA_OK(cudaMemcpyAsync(snap.buf.get(), ptr, count * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return 0;
}

// ---- stage helpers -----------------------------------------------------------------------------
const char* run_visual_cnn(LaunchCtx lc, const avsep_handle* h, const float* frames, int M, int Hh, int Ww,
                           void* pooled, unsigned long long* trace = nullptr, const int* frame_lens = nullptr,
                           int N = 1) {
  if (Hh == 32 && Ww == 32 && h->cfg.precision == AVSEP_PREC_BF16)
    return launch_visual_cnn_tc(lc, frames, M, h->cnn, h->cnn_w2_slabs, h->cnn_w3_rows, pooled, h->num_sms, trace,
                                frame_lens, N);
  return launch_visual_cnn(lc.stream, h->cfg.precision, frames, M, Hh, Ww, h->cnn, pooled, h->num_sms, frame_lens, N);
}

// out[M, N] = A[M, K] W[N, K]^T: one tap, densely packed operands
GemmProblem dense(const void* A, int M, int K, const void* W, int N) {
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
  return p;
}

int linear(avsep_handle* h, LaunchCtx lc, const char* label, const void* A, int M, int K, const void* W,
           const float* bias, int N, int act, float* out_f32, void* out_op) {
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.bias = bias; e.act = act;
  // a GELU whose only consumer is a bf16 operand does not need the fp32-grade erf
  if (act == ACT_GELU && h->cfg.precision == AVSEP_PREC_BF16 && out_f32 == nullptr) e.act = ACT_GELU_BF16;
  e.out_f32 = out_f32; e.ld_f32 = N;
  e.out_op = out_op; e.ld_op = N;
  CKL(label, lc, launch_gemm, h->cfg.precision, p, e, h->num_sms);
  return 0;
}

// GEMM (epilogue fields of `e` already set: bias/act/pe/rowmap) followed by
//   x_out = value (+ resid);  out_op = LayerNorm_{g,b}(x_out)   (g == null: out_op = cast(x_out))
// Fused into the GEMM epilogue when the row fits one tile (EPI_LN), otherwise GEMM -> y, then the warp-shuffle
// add+LayerNorm kernel.  rows_out = number of output rows; y = scratch [rows_out, N] fp32.
int gemm_resid_ln(avsep_handle* h, LaunchCtx lc, const char* label, const GemmProblem& p, GemmEpilogue e,
                  const float* resid, float* x_out, const float* g, const float* b, void* out_op, int rows_out,
                  float* y) {
  const int prec = h->cfg.precision;
  if (gemm_ln_fusable(p.N)) {
    e.kind = EPI_LN;
    e.resid = resid;
    e.out_f32 = x_out; e.ld_f32 = p.N;
    e.ln_gamma = g; e.ln_beta = b;
    e.out_op = out_op; e.ld_op = p.N;
    CKL(label, lc, launch_gemm, prec, p, e, h->num_sms);
    return 0;
  }
  e.kind = EPI_STD;
  e.out_op = nullptr;
  if (resid != nullptr) {
    e.out_f32 = y; e.ld_f32 = p.N;
    CKL(label, lc, launch_gemm, prec, p, e, h->num_sms);
    CKL("add_layernorm", lc, launch_add_layernorm, prec, resid, y, g, b, x_out, out_op, rows_out, p.N);
  } else {
    e.out_f32 = x_out; e.ld_f32 = p.N;
    CKL(label, lc, launch_gemm, prec, p, e, h->num_sms);
    CKL("add_layernorm", lc, launch_add_layernorm, prec, x_out, nullptr, g, b, nullptr, out_op, rows_out, p.N);
  }
  return 0;
}

int linear_resid_ln(avsep_handle* h, LaunchCtx lc, const char* label, const void* A, int M, int K, const void* W,
                    const float* bias, int N, float* x, const float* g, const float* b, void* out_op, float* y) {
  GemmEpilogue e;
  e.bias = bias;
  return gemm_resid_ln(h, lc, label, dense(A, M, K, W, N), e, x, x, g, b, out_op, M, y);
}

bool stack_fusable(const avsep_handle* h, int len) {
  return h->xs_a != nullptr && xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, len);
}

// Which kernels a forward of T audio and N lip frames per utterance launches.  Computed on every call: set_debug,
// set_profile and set_option change it.  A default Plan is the per-layer path of the sub-module entry points.
struct Plan {
  bool stack_a = false, stack_v = false;   // the audio / visual encoder stack in one kernel, else per-layer kernels
  bool stack_f = false;   // the fusion stack in one kernel (it reads the fp32 residual rows of both encoders)
  bool pro = false;       // the encoder stack kernels also run the input projection (Conv1d #2 / frame_proj, + PE)
  bool kvp = false;       // the visual stack kernel also writes the fusion layers' K|V rows
  bool dec = false;       // the fusion stack kernel also runs the SeparationDecoder
  bool fork = false;      // audio and visual branches on two streams (fork / join), so that partial waves overlap
};

Plan forward_plan(const avsep_handle* h, int T, int N) {
  Plan p;
  p.stack_a = stack_fusable(h, T);
  p.stack_v = stack_fusable(h, N);
  p.stack_f = p.stack_a && p.stack_v;
  // stage snapshots (debug) read the embeddings, the K|V rows and the fused rows from memory
  p.pro = !h->debug;
  // the fused K|V projection needs the audio frames inside a visual tile slot
  p.kvp = p.stack_f && h->xs_v_kvp && !h->debug &&
          xformer_kvp_usable(h->cfg.num_fusion_layers * 2 * h->cfg.d_model, N, T);
  p.dec = p.stack_f && h->xs_f_decoder && !h->debug;
  // per-kernel profiling and stage snapshots need a single ordered stream
  p.fork = h->two_stream && !h->profile && !h->debug;
  return p;
}

// A whole stack in one kernel (xformer_stack_sm100.cu).  which: 0 audio encoder, 1 visual encoder, 2 fusion.  The
// caller sets the buffers and the optional stages of `sp`; this fills what follows from the stack: the weight stream
// (from the input-projection items on when sp.pro_a is set), layer count, attention kind, activation, decoder geometry.
int run_stack(avsep_handle* h, LaunchCtx lc, int which, StackProblem sp) {
  const bool pro = sp.pro_a != nullptr;
  sp.wstream = which == 0 ? (pro ? h->xs_a : h->xs_a_np) : which == 1 ? (pro ? h->xs_v : h->xs_v_np) : h->xs_f;
  sp.n_layers = which == 2 ? h->cfg.num_fusion_layers : h->cfg.num_encoder_layers;
  sp.cross = which == 2;
  if (sp.cross) sp.kv_ld = sp.n_layers * 2 * h->cfg.d_model;
  sp.act = sp.cross ? ACT_GELU : ACT_RELU;
  sp.F = h->cfg.freq_bins; sp.S = h->cfg.num_speakers;
  CKL(which == 0 ? "layer.audio_enc" : which == 1 ? "layer.visual_enc" : sp.masks ? "layer.fusion_decoder" : "layer.fusion",
      lc, launch_xformer_stack, sp, h->num_sms);
  return 0;
}

// One fused kernel per feed-forward sub-layer (ffn_fused_sm100.cu) from this many rows on; below it the unfused GEMM
// pair spreads over more CTAs and wins.
constexpr int FFN_FUSED_MIN_ROWS = 2048;

// Feed-forward sub-layer of layer w: x += W2 act(W1 a_op + b1) + b2; a_op = LN_{g,b}(x).  ffn [M, 4d], y [M, d]: scratch.
int ffn_sublayer(avsep_handle* h, LaunchCtx lc, const LayerW& w, int act, int M, float* x, void* a_op, void* ffn,
                 float* y, const float* g, const float* b) {
  const int d = h->cfg.d_model;
  if (ffn_fusable(h->cfg.precision, d) && M >= FFN_FUSED_MIN_ROWS) {
    CKL("ffn.fused", lc, launch_ffn_fused, a_op, w.w1, w.b1, w.w2, w.b2, act, x, x, g, b, a_op, M, h->num_sms,
        nullptr);
    return 0;
  }
  if (linear(h, lc, "gemm.ffn1", a_op, M, d, w.w1, w.b1, 4 * d, act, nullptr, ffn)) return 1;
  return linear_resid_ln(h, lc, "gemm.ffn2", ffn, M, 4 * d, w.w2, w.b2, d, x, g, b, a_op, y);
}

// nn.TransformerEncoderLayer x L (pre-norm, ReLU FFN; model.py:48-52,59; torch transformer.py:946-950).
// In: x (fp32 residual stream), a_op = LN_{layer0.norm1}(x).  Out: x, a_op = LN_{final}(x) (or cast when final_g == null).
// lens: keys per utterance of a variable-length batch, or null.
int encoder_stack(avsep_handle* h, LaunchCtx lc, const std::vector<LayerW>& layers, int B, int L, float* x,
                  float* y, void* a_op, void* qkv, void* attn, void* ffn, const float* final_g, const float* final_b,
                  const int* lens = nullptr) {
  const int d = h->cfg.d_model, H = h->cfg.nhead, M = B * L, prec = h->cfg.precision;
  const size_t os = op_size(h);
  for (size_t l = 0; l < layers.size(); ++l) {
    const LayerW& w = layers[l];
    if (linear(h, lc, "gemm.qkv", a_op, M, d, w.w_in, w.b_in, 3 * d, ACT_NONE, nullptr, qkv)) return 1;
    AttnProblem ap{};
    ap.q = qkv; ap.ldq = 3 * d;
    ap.k = static_cast<const uint8_t*>(qkv) + static_cast<size_t>(d) * os;
    ap.v = static_cast<const uint8_t*>(qkv) + static_cast<size_t>(2 * d) * os;
    ap.ldkv = 3 * d;
    ap.out = attn; ap.ldo = d;
    ap.B = B; ap.H = H; ap.hd = d / H; ap.Lq = L; ap.Lk = L; ap.lerp_src = 0; ap.tc_mode = h->attn_tc;
    ap.k_lens = lens;
    CKL("attn.self", lc, launch_attention, prec, ap);
    if (linear_resid_ln(h, lc, "gemm.out_proj", attn, M, d, w.wo, w.bo, d, x, w.n2g, w.n2b, a_op, y)) return 1;
    const bool last = (l + 1 == layers.size());
    if (ffn_sublayer(h, lc, w, ACT_RELU, M, x, a_op, ffn, y, last ? final_g : layers[l + 1].n1g,
                     last ? final_b : layers[l + 1].n1b))
      return 1;
  }
  return 0;
}

// AudioEncoder up to (not including) the transformer: Conv1d+ReLU x2, +PE (model.py:56-58), then the first
// layer's LayerNorm: x_a (fp32) and a_op = LN_{layer0.norm1}(x_a).
// pl.stack_a: the stack kernel computes the first LayerNorm itself, so only the fp32 residual rows are written, and with
// pl.pro it runs Conv1d #2 + ReLU + PE too, on h1.  xp_ready: the STFT has already written w.xp.
int audio_frontend(avsep_handle* h, LaunchCtx lc, Workspace& w, const float* mixed, const Plan& pl,
                   bool xp_ready = false) {
  const int d = h->cfg.d_model, F = h->cfg.freq_bins, B = w.B, T = w.T, prec = h->cfg.precision;
  const int Map = B * (T + 2);
  if (!xp_ready) CKL("prep_audio", lc, launch_prep_audio, prec, mixed, w.xp, B, F, T, h->Fp, w.lens);
  {
    GemmProblem p{};
    p.A = w.xp; p.lda = h->Fp; p.rowsA = Map; p.M = Map; p.W = h->wc1; p.ldw = 3 * h->Fp; p.N = d; p.K = h->Fp;
    p.taps = 3; p.tap_stride = h->Fp; p.row_shift = -1;
    GemmEpilogue e;
    e.bias = h->bc1; e.act = ACT_RELU; e.rowmap = ROW_PAD2PAD; e.Lp = T + 2;
    e.lens = w.lens;
    e.out_op = w.h1; e.ld_op = d;
    CKL("gemm.conv1d_0", lc, launch_gemm, prec, p, e, h->num_sms);
  }
  if (pl.stack_a && pl.pro) return 0;
  {
    GemmProblem p{};
    p.A = w.h1; p.lda = d; p.rowsA = Map; p.M = Map; p.W = h->wc2; p.ldw = 3 * d; p.N = d; p.K = d;
    p.taps = 3; p.tap_stride = d; p.row_shift = -1;
    GemmEpilogue e;
    e.bias = h->bc2; e.act = ACT_RELU; e.rowmap = ROW_PAD2COMPACT; e.Lp = T + 2;
    e.pe = h->pe_a;
    if (pl.stack_a) {
      e.out_f32 = w.x_a; e.ld_f32 = d;
      CKL("gemm.conv1d_2", lc, launch_gemm, prec, p, e, h->num_sms);
    } else if (gemm_resid_ln(h, lc, "gemm.conv1d_2", p, e, nullptr, w.x_a, h->enc_a[0].n1g, h->enc_a[0].n1b, w.a_op,
                             B * T, w.y_a)) {
      return 1;
    }
  }
  return snapshot(h, lc.stream, "audio_embed", w.x_a, static_cast<size_t>(B) * T * d, false);
}

// VisualEncoder up to (not including) the transformer: CNN, pool, frame_proj, +PE (model.py:106-110), then the
// first layer's LayerNorm: x_v (fp32) and v_op = LN_{layer0.norm1}(x_v).  pl.stack_v / pl.pro as in audio_frontend.
int visual_frontend(avsep_handle* h, LaunchCtx lc, Workspace& w, const float* frames, const Plan& pl) {
  const int d = h->cfg.d_model, B = w.B, N = w.N;
  const int Mv = B * N;
  CKL("visual_cnn", lc, run_visual_cnn, h, frames, Mv, w.Hh, w.Ww, w.pooled, nullptr, w.frame_lens, N);
  if (snapshot(h, lc.stream, "visual_pool", w.pooled, static_cast<size_t>(Mv) * 128, true)) return 1;
  if (pl.stack_v && pl.pro) return 0;
  const GemmProblem p = dense(w.pooled, Mv, 128, h->wproj, d);
  GemmEpilogue e;
  e.bias = h->bproj; e.pe = h->pe_v; e.pe_period = N;
  if (pl.stack_v) {
    e.out_f32 = w.x_v; e.ld_f32 = d;
    CKL("gemm.frame_proj", lc, launch_gemm, h->cfg.precision, p, e, h->num_sms);
  } else if (gemm_resid_ln(h, lc, "gemm.frame_proj", p, e, nullptr, w.x_v, h->enc_v[0].n1g, h->enc_v[0].n1b, w.v_op, Mv,
                           w.y_v)) {
    return 1;
  }
  return snapshot(h, lc.stream, "visual_embed", w.x_v, static_cast<size_t>(Mv) * d, false);
}

// CrossModalFusion (model.py:145-149,166-173) as one kernel: the visual rows are interpolated to the audio frame rate
// first, exactly where the reference does it (model.py:114-116, before the K/V projection), and the K|V rows of every
// fusion layer come from one GEMM on those T rows (bf16) unless the visual stack kernel has written them (pl.kvp).
// In: x_a (fp32 residual), x_v (fp32 visual encoder output, N rows per utterance).  Out: a_op = fusion.norm(x) in bf16,
// or with pl.dec separated / masks from the SeparationDecoder inside the same kernel.
int fusion_stack_fused(avsep_handle* h, LaunchCtx lc, Workspace& w, const Plan& pl, const float* mixed,
                       float* separated, float* masks) {
  const int d = h->cfg.d_model, B = w.B, T = w.T;
  const int Ma = B * T, Lf = h->cfg.num_fusion_layers;
  if (!pl.kvp) {
    CKL("lerp_kv", lc, launch_lerp_rows, w.x_v, d, B, w.N, T, d, w.attn_a, d, w.frame_lens, w.lens);
    if (linear(h, lc, "gemm.cross_kv", w.attn_a, Ma, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, nullptr, w.kvb)) return 1;
  }
  StackProblem sp{};
  sp.x_in = w.x_a; sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; sp.kv = w.kvb;
  sp.B = B; sp.L = T; sp.lens = w.lens;
  if (pl.dec) {
    sp.mixed = mixed; sp.separated = separated; sp.masks = masks;
    return run_stack(h, lc, 2, sp);
  }
  sp.out_x = h->debug ? w.x_a : nullptr; sp.out_op = w.a_op;
  if (run_stack(h, lc, 2, sp)) return 1;
  return snapshot(h, lc.stream, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

// CrossModalFusion, one kernel per layer.  In: x_a residual stream, a_op = LN_{layer0.norm1}(x_a), v_op = visual rows
// (L_src per utterance).  Out: a_op = fusion.norm(x) in operand precision.
int fusion_stack(avsep_handle* h, LaunchCtx lc, Workspace& w, int L_src) {
  const int d = h->cfg.d_model, H = h->cfg.nhead, B = w.B, T = w.T, prec = h->cfg.precision;
  const int Ma = B * T, Mv = B * L_src, Lf = h->cfg.num_fusion_layers;
  // K/V projection of every fusion layer in one GEMM on the un-interpolated visual rows
  if (linear(h, lc, "gemm.cross_kv", w.v_op, Mv, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, w.kvn, nullptr)) return 1;
  for (int l = 0; l < Lf; ++l) {
    const LayerW& fw = h->fus[l];
    if (linear(h, lc, "gemm.cross_q", w.a_op, Ma, d, fw.w_in, fw.b_in, d, ACT_NONE, nullptr, w.qkv_a)) return 1;
    AttnProblem ap{};
    ap.q = w.qkv_a; ap.ldq = d;
    ap.k = w.kvn + static_cast<size_t>(l) * 2 * d;
    ap.v = w.kvn + static_cast<size_t>(l) * 2 * d + d;
    ap.ldkv = Lf * 2 * d;
    ap.out = w.attn_a; ap.ldo = d;
    ap.B = B; ap.H = H; ap.hd = d / H; ap.Lq = T; ap.Lk = T; ap.lerp_src = L_src; ap.tc_mode = h->attn_tc;
    ap.k_lens = w.lens; ap.src_lens = w.frame_lens;
    {
      // Long sequences: materialise the interpolated K/V rows once (bf16, in the unused 2d columns' worth of the
      // Q buffer) so the tcgen05 kernel can stage them by TMA; short ones interpolate on load inside the kernel.
      AttnProblem tp = ap;
      tp.lerp_src = 0;
      __nv_bfloat16* kvi = static_cast<__nv_bfloat16*>(w.qkv_a) + static_cast<size_t>(Ma) * d;
      tp.k = kvi; tp.v = kvi + d; tp.ldkv = 2 * d;
      if (attention_tc_wanted(prec, tp)) {
        CKL("lerp_kv", lc, launch_lerp_rows, w.kvn + static_cast<size_t>(l) * 2 * d, Lf * 2 * d, B, L_src, T, 2 * d,
            kvi, 2 * d, w.frame_lens, w.lens);
        ap = tp;
      }
    }
    CKL("attn.cross", lc, launch_attention, prec, ap);
    if (linear_resid_ln(h, lc, "gemm.out_proj", w.attn_a, Ma, d, fw.wo, fw.bo, d, w.x_a, fw.n2g, fw.n2b, w.a_op, w.y_a))
      return 1;
    const bool last = (l + 1 == Lf);
    if (ffn_sublayer(h, lc, fw, ACT_GELU, Ma, w.x_a, w.a_op, w.ffn_a, w.y_a, last ? h->fng : h->fus[l + 1].n1g,
                     last ? h->fnb : h->fus[l + 1].n1b))
      return 1;
  }
  return snapshot(h, lc.stream, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

// SeparationDecoder.forward + .separate (model.py:201-220): a_op = fused rows in operand precision.
int decoder_stage(avsep_handle* h, LaunchCtx lc, Workspace& w, const float* mixed, float* separated, float* masks) {
  const int d = h->cfg.d_model, F = h->cfg.freq_bins, S = h->cfg.num_speakers, B = w.B, T = w.T;
  const int Ma = B * T;
  if (linear(h, lc, "gemm.dec0", w.a_op, Ma, d, h->wdec0, h->bdec0, 2 * d, ACT_GELU, nullptr, w.ffn_a)) return 1;
  GemmEpilogue e;
  e.kind = EPI_TAIL;
  e.bias = h->bdec3;
  e.mixed = mixed; e.masks = masks; e.separated = separated; e.F = F; e.S = S; e.T = T;
  e.lens = w.lens;
  CKL("gemm.dec3_tail", lc, launch_gemm, h->cfg.precision, dense(w.ffn_a, Ma, 2 * d, h->wdec3, S * F), e,
      h->num_sms);
  return 0;
}

// xp_ready (avsep_separate_waveforms): w.xp already holds the Conv1d operand, so prep_audio is not launched, and the
// per-layer decoder (EPI_TAIL) writes masks only.  The fused fusion + decoder kernel keeps reading `mixed` and writing
// `separated` (staging): its masks-only variant measured 3x slower on a B200.  The Plan is the same either way.
int forward_device(avsep_handle* h, LaunchCtx lc, Workspace& w, const float* mixed, const float* frames,
                   float* separated, float* masks, bool xp_ready = false) {
  const int d = h->cfg.d_model;
  const int Ma = w.B * w.T, Mv = w.B * w.N;
  const Plan pl = forward_plan(h, w.T, w.N);
  if (h->profile && h->profile_spin_us > 0) spin_kernel<<<1, 1, 0, lc.stream>>>(1000ull * h->profile_spin_us);
  // The audio and visual branches are independent until the fusion.
  LaunchCtx sv = lc;
  if (pl.fork) {
    CUDA_OK(make_stream(h->aux_stream));
    CUDA_OK(make_event(h->ev_fork));
    CUDA_OK(make_event(h->ev_join));
    sv.stream = h->aux_stream.get();
    CUDA_OK(cudaEventRecord(h->ev_fork.get(), lc.stream));
    CUDA_OK(cudaStreamWaitEvent(sv.stream, h->ev_fork.get(), 0));
  }
  // --- visual branch (enqueued first: its CNN is the longest kernel) ---
  if (visual_frontend(h, sv, w, frames, pl)) return 1;
  if (pl.stack_v) {
    // out: x_v (fp32) for the interpolation in front of the K/V projection; v_op (bf16 cast) only for the per-layer fusion
    StackProblem sp{};
    sp.x_in = w.x_v; sp.B = w.B; sp.L = w.N; sp.lens = w.frame_lens; sp.kvp_lens = w.lens;
    if (pl.pro) {
      sp.pro_a = w.pooled; sp.pro_taps = 1; sp.pro_k = 128; sp.pro_pitch = w.N; sp.pro_rows = Mv; sp.pe = h->pe_v;
    }
    if (pl.kvp) {
      sp.kvp_out = w.kvb; sp.kvp_L = w.T; sp.kvp_n = sp.kvp_ld = h->cfg.num_fusion_layers * 2 * d;
    } else {
      sp.out_x = w.x_v; sp.out_op = pl.stack_f ? nullptr : w.v_op;
    }
    if (run_stack(h, sv, 1, sp)) return 1;
  } else if (encoder_stack(h, sv, h->enc_v, w.B, w.N, w.x_v, w.y_v, w.v_op, w.qkv_v, w.attn_v, w.ffn_v, nullptr, nullptr,
                           w.frame_lens)) {
    return 1;
  }
  if (snapshot(h, sv.stream, "visual_enc", w.x_v, static_cast<size_t>(Mv) * d, false)) return 1;
  // --- audio branch ---
  if (audio_frontend(h, lc, w, mixed, pl, xp_ready)) return 1;
  if (pl.stack_a) {
    StackProblem sp{};
    sp.x_in = w.x_a; sp.out_x = w.x_a; sp.out_op = pl.stack_f ? nullptr : w.a_op;
    sp.fin_gamma = h->fus[0].n1g; sp.fin_beta = h->fus[0].n1b;
    sp.B = w.B; sp.L = w.T; sp.lens = w.lens;
    if (pl.pro) {
      sp.pro_a = w.h1; sp.pro_relu = 1; sp.pro_taps = 3; sp.pro_k = d; sp.pro_pitch = w.T + 2;
      sp.pro_rows = w.B * (w.T + 2); sp.pe = h->pe_a;
    }
    if (run_stack(h, lc, 0, sp)) return 1;
  } else if (encoder_stack(h, lc, h->enc_a, w.B, w.T, w.x_a, w.y_a, w.a_op, w.qkv_a, w.attn_a, w.ffn_a, h->fus[0].n1g,
                           h->fus[0].n1b, w.lens)) {
    return 1;
  }
  if (snapshot(h, lc.stream, "audio_enc", w.x_a, static_cast<size_t>(Ma) * d, false)) return 1;
  if (pl.fork) {
    CUDA_OK(cudaEventRecord(h->ev_join.get(), sv.stream));
    CUDA_OK(cudaStreamWaitEvent(lc.stream, h->ev_join.get(), 0));
  }
  // --- fusion + decoder ---
  if (pl.stack_f ? fusion_stack_fused(h, lc, w, pl, mixed, separated, masks) : fusion_stack(h, lc, w, w.N)) return 1;
  return pl.dec ? 0 : decoder_stage(h, lc, w, xp_ready ? nullptr : mixed, xp_ready ? nullptr : separated, masks);
}

// Eager on the first use of a (shape, buffer set); captured into a CUDA graph on the second; replayed afterwards.
// The graph bakes in the kernel parameters (tensor maps included), so a replay costs one host call.
int forward_cached(avsep_handle* h, LaunchCtx lc, Workspace& w, const void* ws_base, const float* mixed,
                   const float* frames, float* separated, float* masks, bool xp_ready = false) {
  if (!h->use_graph || h->profile || h->debug)
    return forward_device(h, lc, w, mixed, frames, separated, masks, xp_ready);
  const GraphKey key{w.B, w.T, w.N, w.Hh, w.Ww, mixed, frames, separated, masks, ws_base, w.lens, w.frame_lens,
                     xp_ready};
  GraphEntry* ent = nullptr;
  for (auto& g : h->graphs)
    if (g.key == key) { ent = &g; break; }
  if (ent == nullptr) {
    if (h->graphs.size() >= 64) {          // evict the least recently used entry
      size_t victim = 0;
      for (size_t i = 1; i < h->graphs.size(); ++i)
        if (h->graphs[i].last_use < h->graphs[victim].last_use) victim = i;
      h->graphs.erase(h->graphs.begin() + victim);
    }
    GraphEntry g;
    g.key = key;
    g.last_use = ++h->graph_clock;
    h->graphs.push_back(std::move(g));
    return forward_device(h, lc, w, mixed, frames, separated, masks, xp_ready);   // warm-up, also sets kernel attributes
  }
  ent->last_use = ++h->graph_clock;
  if (ent->exec == nullptr) {   // the capture counts the launches it records; a replay adds them
    const int64_t before = h->launches;
    CUDA_OK(make_stream(h->cap_stream));
    CUDA_OK(cudaStreamBeginCapture(h->cap_stream.get(), cudaStreamCaptureModeRelaxed));
    const int rc = forward_device(h, {h->cap_stream.get(), lc.pdl}, w, mixed, frames, separated, masks, xp_ready);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(h->cap_stream.get(), &graph);
    if (rc != 0) {
      if (graph) cudaGraphDestroy(graph);
      return 1;
    }
    if (ce != cudaSuccess) return fail(h, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ci = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ci != cudaSuccess) return fail(h, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ci));
    ent->exec.reset(exec);
    ent->launches = h->launches - before;
  } else {
    h->launches += ent->launches;
  }
  CUDA_OK(cudaGraphLaunch(ent->exec.get(), lc.stream));
  return 0;
}

// Utterances b0 .. b0 + w.B - 1 of a packed batch (include/avsep.h) through the staging: unpack, the varlen forward
// (cached graph) on the staging, pack.  lens / flens: DEVICE lengths of the whole packed batch (or null), from whose
// first b0 entries the kernels find the chunk's packed offsets.  Sets w.lens / w.frame_lens.
int forward_packed_run(avsep_handle* h, LaunchCtx lc, Workspace& w, const Staging& st, const void* ws_base,
                       const float* mixed_p, const float* frames_p, const int* lens, const int* flens, int b0,
                       float* sep_p, float* masks_p) {
  const int F = h->cfg.freq_bins, S = h->cfg.num_speakers;
  CKL("unpack", lc, launch_unpack, mixed_p, frames_p, lens, flens, b0, w.B, F, w.T, w.N, w.Hh * w.Ww, st.mixed,
      st.frames);
  w.lens = lens ? lens + b0 : nullptr;
  w.frame_lens = flens ? flens + b0 : nullptr;
  if (forward_cached(h, lc, w, ws_base, st.mixed, st.frames, st.sep, st.masks)) return 1;
  CKL("pack", lc, launch_pack, st.sep, st.masks, lens, b0, w.B, S, F, w.T, sep_p, masks_p);
  return 0;
}

// Waveforms in, waveforms out on the device (avsep_separate_waveforms): the STFT writes the complex spectrum and the
// magnitude to the staging and the Conv1d operand to w.xp (and T_b to st.tlens when lens is given), the forward (cached
// graph) runs without prep_audio (forward_device's xp_ready), the masked inverse writes waves_out.  masks == null: the
// masks go to the staging.  lens: DEVICE sample lengths, flens: DEVICE lip-frame lengths, or null.  Sets w.lens /
// w.frame_lens.
int waves_run(avsep_handle* h, LaunchCtx lc, Workspace& w, const WaveStaging& st, const void* ws_base,
              const float* waves, const float* frames, const int* lens, const int* flens, int L, int n_fft, int hop,
              float* waves_out, float* masks) {
  float* const mk = masks ? masks : st.masks;
  CKL("stft", lc.stream, launch_stft, waves, lens, w.B, 0, L, n_fft, hop, st.spec, st.mag, nullptr,
      lens ? st.tlens : nullptr, w.xp, h->Fp, h->cfg.precision);
  w.lens = lens ? st.tlens : nullptr;
  w.frame_lens = flens;
  if (forward_cached(h, lc, w, ws_base, st.mag, frames, st.sep, mk, true)) return 1;
  CKL("istft", lc.stream, launch_istft_masked, st.spec, mk, lens, w.B, h->cfg.num_speakers, w.T, n_fft, hop, L,
      waves_out);
  return 0;
}

// Geometry of a waveform call: sets T = 1 + L / hop and checks it as check_shape does.
int check_waves(avsep_handle* h, const char* who, int B, int L, int N, int Hh, int Ww, int n_fft, int hop, int& T) {
  if (B < 1 || L < 1) return fail(h, std::string(who) + ": empty input: B and L must be >= 1");
  if (n_fft != 2 * (h->cfg.freq_bins - 1))
    return fail(h, std::string(who) + ": n_fft must be 2 * (freq_bins - 1) = " + std::to_string(2 * (h->cfg.freq_bins - 1)));
  if (!fft_geometry_ok(n_fft, hop))
    return fail(h, std::string(who) + ": n_fft must be a power of two in [8, 2048], 1 <= hop <= n_fft");
  T = 1 + L / hop;
  return check_shape(h, B, T, N, Hh, Ww);
}

// ---- weight access helpers ---------------------------------------------------------------------
const HostTensor* find_w(avsep_handle* h, const std::string& key, std::initializer_list<int64_t> shape) {
  auto it = h->host_w.find(key);
  if (it == h->host_w.end()) {
    h->err = "missing weight: " + key;
    return nullptr;
  }
  std::vector<int64_t> want(shape);
  if (it->second.shape != want) {
    h->err = "bad shape for weight: " + key;
    return nullptr;
  }
  return &it->second;
}

// The 12 tensors of one encoder layer (nn.TransformerEncoderLayer) or fusion layer (model.py:136-149), shape-checked.
// The two kinds differ only in their key names.
struct HostLayer {
  const HostTensor *w_in, *b_in, *wo, *bo, *w1, *b1, *w2, *b2, *n1g, *n1b, *n2g, *n2b;
};
bool find_layer(avsep_handle* h, const std::string& p, bool cross, int64_t d, HostLayer& t) {
  const std::string at = p + (cross ? ".cross_attn." : ".self_attn."), f1 = p + (cross ? ".ff.0." : ".linear1."),
                    f2 = p + (cross ? ".ff.3." : ".linear2.");
  return (t.w_in = find_w(h, at + "in_proj_weight", {3 * d, d})) && (t.b_in = find_w(h, at + "in_proj_bias", {3 * d})) &&
         (t.wo = find_w(h, at + "out_proj.weight", {d, d})) && (t.bo = find_w(h, at + "out_proj.bias", {d})) &&
         (t.w1 = find_w(h, f1 + "weight", {4 * d, d})) && (t.b1 = find_w(h, f1 + "bias", {4 * d})) &&
         (t.w2 = find_w(h, f2 + "weight", {d, 4 * d})) && (t.b2 = find_w(h, f2 + "bias", {d})) &&
         (t.n1g = find_w(h, p + ".norm1.weight", {d})) && (t.n1b = find_w(h, p + ".norm1.bias", {d})) &&
         (t.n2g = find_w(h, p + ".norm2.weight", {d})) && (t.n2b = find_w(h, p + ".norm2.bias", {d}));
}

// Host image of the weight arena.  Every item names the device-pointer field that views it; patch() sets those fields
// once the image is uploaded.
struct ArenaBuilder {
  std::vector<uint8_t> bytes;
  std::vector<std::function<void(const uint8_t*)>> fills;
  template <typename T>
  void add(const T*& field, const void* src, size_t n) {
    const size_t off = align_up(bytes.size(), 256);
    bytes.resize(off + n);
    memcpy(bytes.data() + off, src, n);
    fills.push_back([&field, off](const uint8_t* base) { field = reinterpret_cast<const T*>(base + off); });
  }
  void add_f32(const float*& field, const float* src, size_t n) { add(field, src, n * 4); }
  void add_f32(const float*& field, const HostTensor* t) { add_f32(field, t->data.data(), t->data.size()); }
  void add_op(const void*& field, const float* src, size_t n, bool tf32) {
    if (tf32) {   // round to tf32 (10-bit mantissa, nearest, ties away) so the tensor core's truncation is exact
      std::vector<float> tmp(n);
      for (size_t i = 0; i < n; ++i) {
        uint32_t u;
        memcpy(&u, &src[i], 4);
        if ((u & 0x7f800000u) != 0x7f800000u) u = (u + 0x1000u) & 0xffffe000u;
        memcpy(&tmp[i], &u, 4);
      }
      return add(field, tmp.data(), n * 4);
    }
    std::vector<uint16_t> tmp(n);
    for (size_t i = 0; i < n; ++i) tmp[i] = f2bf(src[i]);
    add(field, tmp.data(), n * 2);
  }
  void add_op(const void*& field, const HostTensor* t, bool tf32) { add_op(field, t->data.data(), t->data.size(), tf32); }
  void patch(const uint8_t* base) {
    for (auto& f : fills) f(base);
  }
};

// Arena items of one layer: the weights, then the vectors.  A fusion layer keeps the Q rows of its input projection
// (the first d), with their bias right behind them.
void add_layer(ArenaBuilder& ar, LayerW& w, const HostLayer& t, bool cross, int64_t d, bool tf32) {
  ar.add_op(w.w_in, t.w_in->data.data(), static_cast<size_t>(cross ? d : 3 * d) * d, tf32);
  if (cross) ar.add_f32(w.b_in, t.b_in->data.data(), d);
  ar.add_op(w.wo, t.wo, tf32);
  ar.add_op(w.w1, t.w1, tf32);
  ar.add_op(w.w2, t.w2, tf32);
  if (!cross) ar.add_f32(w.b_in, t.b_in);
  ar.add_f32(w.bo, t.bo);
  ar.add_f32(w.b1, t.b1);
  ar.add_f32(w.b2, t.b2);
  ar.add_f32(w.n1g, t.n1g);
  ar.add_f32(w.n1b, t.n1b);
  ar.add_f32(w.n2g, t.n2g);
  ar.add_f32(w.n2b, t.n2b);
}

// One layer of a stack-kernel weight stream: its vector block, then its weight items.  b0: bias of the input
// projection in front of layer 0, which rides in that layer's vector block (or null).
void pack_stream_layer(const HostLayer& t, bool cross, int d, const float* b0, std::vector<float>& vecs, uint8_t* dst) {
  xformer_pack_vecs(t.b_in->data.data(), cross ? d : 3 * d, t.bo->data.data(), t.b1->data.data(), t.b2->data.data(),
                    t.n1g->data.data(), t.n1b->data.data(), t.n2g->data.data(), t.n2b->data.data(), vecs.data(), b0);
  (cross ? xformer_pack_cross : xformer_pack_self)(t.w_in->data.data(), t.wo->data.data(), t.w1->data.data(),
                                                   t.w2->data.data(), vecs.data(), dst);
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int avsep_create(const avsep_config* cfg, avsep_handle** out) {
  if (!cfg || !out) return fail(nullptr, "avsep_create: null argument");
  *out = nullptr;
  if (cfg->freq_bins < 1 || cfg->d_model < 8 || cfg->nhead < 1 || cfg->num_encoder_layers < 1 ||
      cfg->num_fusion_layers < 1 || cfg->num_speakers < 1)
    return fail(nullptr, "avsep_create: all sizes must be positive (at least one encoder and one fusion layer)");
  if (cfg->d_model % cfg->nhead != 0) return fail(nullptr, "avsep_create: d_model must be divisible by nhead");
  const int hd = cfg->d_model / cfg->nhead;
  if (hd != 16 && hd != 32 && hd != 64 && hd != 128)
    return fail(nullptr, "avsep_create: head dim (d_model/nhead) must be 16, 32, 64 or 128");
  if (cfg->d_model % 8 != 0 || cfg->d_model > 1024)
    return fail(nullptr, "avsep_create: d_model must be a multiple of 8 and <= 1024");
  if (cfg->precision != AVSEP_PREC_BF16 && cfg->precision != AVSEP_PREC_TF32)
    return fail(nullptr, "avsep_create: unknown precision");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(nullptr, "avsep_create: no CUDA device (this library has no CPU path)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, "avsep_create: bad device ordinal");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return fail(nullptr, "avsep_create: device query failed");
  if (prop.major != 10) return fail(nullptr, "avsep_create: kernels are built for sm_100a (B200) only");
  ON_DEVICE(nullptr, cfg->device);
  if (const char* e = tma_init()) return fail(nullptr, e);
  if (const char* e = fft512_init_tables()) return fail(nullptr, e);
  avsep_handle* h = new avsep_handle();
  h->cfg = *cfg;
  h->Fp = (cfg->freq_bins + 7) / 8 * 8;
  h->num_sms = prop.multiProcessorCount;
  *out = h;
  // A/B switches for measurement runs: AVSEP_OPTS="name=value,name=value" goes through avsep_set_option
  if (const char* e = getenv("AVSEP_OPTS")) {
    std::string opts(e);
    size_t pos = 0;
    while (pos < opts.size()) {
      size_t end = opts.find(',', pos);
      if (end == std::string::npos) end = opts.size();
      const std::string kv = opts.substr(pos, end - pos);
      const size_t eq = kv.find('=');
      if (eq != std::string::npos && avsep_set_option(h, kv.substr(0, eq).c_str(), atoi(kv.c_str() + eq + 1)) != 0)
        fprintf(stderr, "avsep: AVSEP_OPTS: option '%s' not accepted\n", kv.c_str());
      pos = end + 1;
    }
  }
  return 0;
}

void avsep_destroy(avsep_handle* h) {
  if (!h) return;
  const DeviceScope device_scope(h->cfg.device);   // the handle's resources belong to its device
  delete h;
}

const char* avsep_last_error(const avsep_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int avsep_set_weight(avsep_handle* h, const char* key, const void* host_data, int32_t dtype, const int64_t* shape,
                     int32_t ndim) {
  if (!h || !key || (!host_data && ndim >= 0) || ndim < 0 || ndim > 8) return fail(h, "avsep_set_weight: bad argument");
  if (dtype == AVSEP_DTYPE_I64) return 0;   // num_batches_tracked: unused in eval mode
  if (dtype != AVSEP_DTYPE_F32) return fail(h, "avsep_set_weight: only fp32 tensors are accepted");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    if (shape[i] < 0) return fail(h, "avsep_set_weight: negative dimension");
    t.shape.push_back(shape[i]);
    n *= static_cast<size_t>(shape[i]);
  }
  t.data.assign(static_cast<const float*>(host_data), static_cast<const float*>(host_data) + n);
  h->host_w[key] = std::move(t);
  h->finalized = false;
  return 0;
}

int avsep_finalize_weights(avsep_handle* h, void* cuda_stream) {
  ENTER(h, cuda_stream);
  const int64_t d = h->cfg.d_model, F = h->cfg.freq_bins, S = h->cfg.num_speakers, Fp = h->Fp;
  const int Le = h->cfg.num_encoder_layers, Lf = h->cfg.num_fusion_layers;
  const bool tf32 = h->cfg.precision == AVSEP_PREC_TF32;
  // --- look up every tensor once
#define GETW(var, key, ...)                                  \
  const HostTensor* var = find_w(h, key, {__VA_ARGS__});     \
  if (!var) return 1;
  GETW(c0w, "audio_encoder.input_proj.0.weight", d, F, 3);
  GETW(c0b, "audio_encoder.input_proj.0.bias", d);
  GETW(c2w, "audio_encoder.input_proj.2.weight", d, d, 3);
  GETW(c2b, "audio_encoder.input_proj.2.bias", d);
  GETW(pea, "audio_encoder.pos_enc.pe", 1, 5000, d);
  GETW(pev, "visual_encoder.pos_enc.pe", 1, 5000, d);
  GETW(projw, "visual_encoder.frame_proj.weight", d, 128);
  GETW(projb, "visual_encoder.frame_proj.bias", d);
  GETW(fng, "fusion.norm.weight", d);
  GETW(fnb, "fusion.norm.bias", d);
  GETW(dec0w, "decoder.decoder.0.weight", 2 * d, d);
  GETW(dec0b, "decoder.decoder.0.bias", 2 * d);
  GETW(dec3w, "decoder.decoder.3.weight", S * F, 2 * d);
  GETW(dec3b, "decoder.decoder.3.bias", S * F);
  std::vector<HostLayer> enc[2] = {std::vector<HostLayer>(Le), std::vector<HostLayer>(Le)}, fus(Lf);
  for (int l = 0; l < Le; ++l)
    if (!find_layer(h, "audio_encoder.transformer.layers." + std::to_string(l), false, d, enc[0][l]) ||
        !find_layer(h, "visual_encoder.transformer.layers." + std::to_string(l), false, d, enc[1][l]))
      return 1;
  for (int l = 0; l < Lf; ++l)
    if (!find_layer(h, "fusion.layers." + std::to_string(l), true, d, fus[l])) return 1;
  // VisualEncoder CNN: fold BatchNorm (eval) into conv weight/bias, repack tap-major
  const int cins[3] = {1, 32, 64}, couts[3] = {32, 64, 128}, idx[3] = {0, 3, 6};
  std::vector<float> folded[3], fbias[3];
  for (int c = 0; c < 3; ++c) {
    const std::string cp = "visual_encoder.conv." + std::to_string(idx[c]);
    const std::string bp = "visual_encoder.conv." + std::to_string(idx[c] + 1);
    GETW(w, cp + ".weight", couts[c], cins[c], 3, 3);
    GETW(b, cp + ".bias", couts[c]);
    GETW(g, bp + ".weight", couts[c]);
    GETW(be, bp + ".bias", couts[c]);
    GETW(mu, bp + ".running_mean", couts[c]);
    GETW(var, bp + ".running_var", couts[c]);
    const int K = 9 * cins[c];
    folded[c].assign(static_cast<size_t>(couts[c]) * K, 0.f);
    fbias[c].assign(couts[c], 0.f);
    for (int o = 0; o < couts[c]; ++o) {
      const float scale = g->data[o] / sqrtf(var->data[o] + 1e-5f);
      fbias[c][o] = (b->data[o] - mu->data[o]) * scale + be->data[o];
      for (int ci = 0; ci < cins[c]; ++ci)
        for (int tap = 0; tap < 9; ++tap)
          folded[c][static_cast<size_t>(o) * K + tap * cins[c] + ci] =
              w->data[(static_cast<size_t>(o) * cins[c] + ci) * 9 + tap] * scale;
    }
  }
#undef GETW
  // fusion: the K|V rows of every layer's in_proj, concatenated
  const int n_kv = static_cast<int>(Lf * 2 * d);
  std::vector<float> wkv(static_cast<size_t>(n_kv) * d), bkv(n_kv);
  for (int l = 0; l < Lf; ++l) {
    memcpy(wkv.data() + static_cast<size_t>(l) * 2 * d * d, fus[l].w_in->data.data() + d * d, sizeof(float) * 2 * d * d);
    memcpy(bkv.data() + static_cast<size_t>(l) * 2 * d, fus[l].b_in->data.data() + d, sizeof(float) * 2 * d);
  }

  // --- the GEMM path's arena items
  ArenaBuilder ar;
  h->enc_a.assign(Le, LayerW{});
  h->enc_v.assign(Le, LayerW{});
  h->fus.assign(Lf, LayerW{});
  {
    // AudioEncoder Conv1d weights: (Cout, Cin, 3) -> (Cout, 3*Cin_pad), k = tap*Cin_pad + c
    std::vector<float> p0(static_cast<size_t>(d) * 3 * Fp, 0.f), p2(static_cast<size_t>(d) * 3 * d, 0.f);
    for (int64_t o = 0; o < d; ++o)
      for (int64_t c = 0; c < F; ++c)
        for (int tap = 0; tap < 3; ++tap) p0[(o * 3 + tap) * Fp + c] = c0w->data[(o * F + c) * 3 + tap];
    for (int64_t o = 0; o < d; ++o)
      for (int64_t c = 0; c < d; ++c)
        for (int tap = 0; tap < 3; ++tap) p2[(o * 3 + tap) * d + c] = c2w->data[(o * d + c) * 3 + tap];
    ar.add_op(h->wc1, p0.data(), p0.size(), tf32);
    ar.add_op(h->wc2, p2.data(), p2.size(), tf32);
  }
  ar.add_f32(h->bc1, c0b);
  ar.add_f32(h->bc2, c2b);
  ar.add_f32(h->pe_a, pea);
  ar.add_f32(h->pe_v, pev);
  for (int l = 0; l < Le; ++l) add_layer(ar, h->enc_a[l], enc[0][l], false, d, tf32);
  for (int l = 0; l < Le; ++l) add_layer(ar, h->enc_v[l], enc[1][l], false, d, tf32);
  {
    // CNN operands: tcgen05 slabs, fragment order (hi, then the lo parts of the fp32-grade split path)
    std::vector<uint32_t> p1(visual_cnn_pack_sizes(1)), p2(visual_cnn_pack_sizes(2)), p3(visual_cnn_pack_sizes(3));
    visual_cnn_pack(folded[0].data(), folded[1].data(), folded[2].data(), p1.data(), p2.data(), p3.data());
    std::vector<uint8_t> tc2(visual_cnn_tc_w2_bytes()), tc3(visual_cnn_tc_w3_bytes());
    visual_cnn_tc_pack(folded[1].data(), folded[2].data(), tc2.data(), tc3.data());
    ar.add(h->cnn_w2_slabs, tc2.data(), tc2.size());
    ar.add(h->cnn_w3_rows, tc3.data(), tc3.size());
    ar.add(h->cnn.w1, p1.data(), p1.size() * 4);
    ar.add(h->cnn.w2, p2.data(), p2.size() * 4);
    ar.add(h->cnn.w3, p3.data(), p3.size() * 4);
    visual_cnn_pack(folded[0].data(), folded[1].data(), folded[2].data(), p1.data(), p2.data(), p3.data(), true);
    ar.add(h->cnn.w1l, p1.data(), p1.size() * 4);
    ar.add(h->cnn.w2l, p2.data(), p2.size() * 4);
    ar.add(h->cnn.w3l, p3.data(), p3.size() * 4);
    ar.add_f32(h->cnn.b1, fbias[0].data(), 32);
    ar.add_f32(h->cnn.b2, fbias[1].data(), 64);
    ar.add_f32(h->cnn.b3, fbias[2].data(), 128);
  }
  ar.add_op(h->wproj, projw, tf32);
  ar.add_f32(h->bproj, projb);
  for (int l = 0; l < Lf; ++l) add_layer(ar, h->fus[l], fus[l], true, d, tf32);
  ar.add_op(h->wkv_all, wkv.data(), wkv.size(), tf32);
  ar.add_f32(h->bkv_all, bkv.data(), bkv.size());
  ar.add_f32(h->fng, fng);
  ar.add_f32(h->fnb, fnb);
  ar.add_op(h->wdec0, dec0w, tf32);
  ar.add_op(h->wdec3, dec3w, tf32);
  ar.add_f32(h->bdec0, dec0b);
  ar.add_f32(h->bdec3, dec3b);

  // --- fused transformer-stack kernel: weight streams in consumption order + per-layer vector blocks.  The encoder
  // streams start with the input projection (Conv1d #2 as 3 taps x d / frame_proj as 1 x 128), whose bias rides in
  // layer 0's vector block; the visual one ends with the fusion K|V projection, the fusion one with the decoder.
  h->xs_a = h->xs_v = h->xs_f = nullptr;
  if (xformer_stack_usable(h->cfg.precision, static_cast<int>(d), h->cfg.nhead, 1)) {
    const size_t sb = xformer_stream_bytes(false), cb = xformer_stream_bytes(true);
    const size_t pro_a = xformer_pro_bytes(3, static_cast<int>(d)), pro_v = xformer_pro_bytes(1, 128);
    h->xs_v_kvp = xformer_kvp_usable(n_kv, 1, 1);
    h->xs_f_decoder = xformer_decoder_usable(static_cast<int>(S), static_cast<int>(F));
    std::vector<uint8_t> xa(pro_a + Le * sb), xv(pro_v + Le * sb + (h->xs_v_kvp ? xformer_kvp_bytes(n_kv) : 0)),
        xf(Lf * cb + (h->xs_f_decoder ? xformer_decoder_bytes(static_cast<int>(S), static_cast<int>(F)) : 0));
    std::vector<float> vecs(xformer_vec_floats());
    xformer_pack_pro(c2w->data.data(), static_cast<int>(3 * d), 3, 3, static_cast<int>(d), xa.data());
    xformer_pack_pro(projw->data.data(), 128, 1, 1, 128, xv.data());
    for (int l = 0; l < Le; ++l) {
      pack_stream_layer(enc[0][l], false, d, l == 0 ? c2b->data.data() : nullptr, vecs, xa.data() + pro_a + l * sb);
      pack_stream_layer(enc[1][l], false, d, l == 0 ? projb->data.data() : nullptr, vecs, xv.data() + pro_v + l * sb);
    }
    if (h->xs_v_kvp) xformer_pack_kvp(wkv.data(), bkv.data(), n_kv, xv.data() + pro_v + Le * sb);
    for (int l = 0; l < Lf; ++l) pack_stream_layer(fus[l], true, d, nullptr, vecs, xf.data() + l * cb);
    if (h->xs_f_decoder)
      xformer_pack_decoder(dec0w->data.data(), dec0b->data.data(), dec3w->data.data(), dec3b->data.data(),
                           static_cast<int>(S), static_cast<int>(F), xf.data() + Lf * cb);
    ar.add(h->xs_a, xa.data(), xa.size());
    ar.add(h->xs_v, xv.data(), xv.size());
    ar.add(h->xs_f, xf.data(), xf.size());
  }
  // upload
  drop_graphs(h);
  CUDA_OK(h->weights.alloc(ar.bytes.size()));
  CUDA_OK(cudaMemcpyAsync(h->weights.get(), ar.bytes.data(), ar.bytes.size(), cudaMemcpyHostToDevice, lc.stream));
  CUDA_OK(cudaStreamSynchronize(lc.stream));
  ar.patch(h->weights.get());
  if (h->xs_a != nullptr) {
    h->xs_a_np = h->xs_a + xformer_pro_bytes(3, h->cfg.d_model);
    h->xs_v_np = h->xs_v + xformer_pro_bytes(1, 128);
  }
  h->finalized = true;
  return 0;
}

size_t avsep_workspace_bytes(avsep_handle* h, int32_t B, int32_t T, int32_t N, int32_t Hh, int32_t Ww) {
  if (!h || B < 1 || T < 1 || N < 1) return 0;
  Workspace w;
  return carve_workspace(h, w, nullptr, B, T, N, Hh, Ww);
}

int avsep_forward(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T, int32_t N,
                  int32_t Hh, int32_t Ww, float* separated, float* masks, void* workspace, size_t workspace_bytes,
                  void* cuda_stream) {
  return avsep_forward_varlen(h, mixed_spec, lip_frames, nullptr, nullptr, B, T, N, Hh, Ww, separated, masks, workspace,
                              workspace_bytes, cuda_stream);
}

int avsep_forward_varlen(avsep_handle* h, const float* mixed_spec, const float* lip_frames, const int32_t* lengths,
                         const int32_t* frame_lengths, int32_t B, int32_t T, int32_t N, int32_t Hh, int32_t Ww,
                         float* separated, float* masks, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!mixed_spec || !lip_frames || !separated || !masks) return fail(h, "avsep_forward: null buffer");
  if (check_shape(h, B, T, N, Hh, Ww)) return 1;
  Workspace w;
  if (get_workspace(h, w, workspace, workspace_bytes, B, T, N, Hh, Ww)) return 1;
  w.lens = lengths; w.frame_lens = frame_lengths;
  return forward_cached(h, lc, w, workspace ? workspace : h->own_ws.get(), mixed_spec, lip_frames, separated, masks);
}

size_t avsep_packed_workspace_bytes(avsep_handle* h, int32_t B, int32_t T, int32_t N, int32_t Hh, int32_t Ww) {
  if (!h || B < 1 || T < 1 || N < 1 || Hh < 1 || Ww < 1) return 0;
  Workspace w;
  Staging st;
  return carve_packed(h, w, st, nullptr, B, T, N, Hh, Ww);
}

int avsep_forward_packed(avsep_handle* h, const float* mixed_packed, const float* frames_packed, const int32_t* lengths,
                         const int32_t* frame_lengths, int32_t B, int32_t T, int32_t N, int32_t Hh, int32_t Ww,
                         float* separated_packed, float* masks_packed, void* workspace, size_t workspace_bytes,
                         void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!mixed_packed || !frames_packed || !separated_packed || !masks_packed)
    return fail(h, "avsep_forward_packed: null buffer");
  if ((reinterpret_cast<uintptr_t>(mixed_packed) | reinterpret_cast<uintptr_t>(frames_packed) |
       reinterpret_cast<uintptr_t>(separated_packed) | reinterpret_cast<uintptr_t>(masks_packed)) & 3)
    return fail(h, "avsep_forward_packed: buffers must be 4-byte aligned");
  if (check_shape(h, B, T, N, Hh, Ww)) return 1;
  Workspace w;
  Staging st;
  uint8_t* base = nullptr;
  if (workspace_base(h, workspace, workspace_bytes, carve_packed(h, w, st, nullptr, B, T, N, Hh, Ww),
                     "avsep_packed_workspace_bytes", base))
    return 1;
  carve_packed(h, w, st, base, B, T, N, Hh, Ww);
  return forward_packed_run(h, lc, w, st, base, mixed_packed, frames_packed, lengths, frame_lengths, 0,
                            separated_packed, masks_packed);
}

namespace {
// A host tensor of a host-buffer call and the element offsets of its utterances: utterances [b0, b1) are the span
// [at[b0], at[b1]) (packed or padded).
struct HostIn {
  const float* host;
  std::vector<size_t> at;
};
struct HostOut {
  float* host;
  std::vector<size_t> at;
};
std::vector<size_t> padded_at(int B, size_t per) {
  std::vector<size_t> at(B + 1);
  for (int b = 0; b <= B; ++b) at[b] = b * per;
  return at;
}

// What distinguishes the host-buffer forms (padded, packed and waveform forward): the spans each chunk copies in and
// out - input i is mirrored by the slot's device buffer io[i], output j by io[in.size() + j] - and the chunk's device
// step.  Slots, events, lanes and the chunk / lane choice are host_submit's.
struct HostCall {
  std::string who;
  int B = 0;
  std::vector<HostIn> in;
  std::vector<HostOut> out;
  std::vector<int32_t> lens;   // uploaded once per call to the slot's lens_dev (empty: nothing to upload)
  // workspace bytes of one compute lane that runs chunks of up to Bc utterances
  std::function<size_t(int Bc)> lane_bytes;
  // enqueues utterances [b0, b0 + bc) on lc with the lane's workspace ws (carved for Bc), the slot's device buffers io
  // and the uploaded lengths (or null)
  std::function<int(LaunchCtx lc, uint8_t* ws, int Bc, int b0, int bc, float* const* io, const int32_t* lens)> step;
};

int host_submit(avsep_handle* h, const HostCall& c, int slot_id, cudaStream_t s, bool streaming) {
  // Software pipeline over chunks of the batch: H2D of chunk i+1, kernels of chunk i and D2H of chunk i-1 run
  // concurrently on separate streams (PCIe is full duplex), so a call costs ~max(copy-in, compute, copy-out); the
  // slots extend the same pipeline across consecutive calls.
  if (slot_id < 0 || slot_id >= AVSEP_HOST_SLOTS) return fail(h, c.who + "_async: slot must be 0 .. AVSEP_HOST_SLOTS - 1");
  const int B = c.B;
  avsep_handle::HostSlot& sl = h->slot[slot_id];
  const size_t nin = c.in.size(), nio = nin + c.out.size();
  for (size_t i = 0; i < nio; ++i) {
    const size_t need = i < nin ? c.in[i].at[B] : c.out[i - nin].at[B];
    if (sl.io[i].cap < need) {
      if (sl.ev_end) CUDA_OK(cudaEventSynchronize(sl.ev_end.get()));   // the slot's previous call still owns the buffer
      CUDA_OK(sl.io[i].alloc(need));
    }
  }
  float* io[4];
  for (int i = 0; i < 4; ++i) io[i] = sl.io[i].get();
  for (Stream& st : h->hs) CUDA_OK(make_stream(st));
  CUDA_OK(make_event(sl.ev_start));
  CUDA_OK(make_event(sl.ev_end));
  const bool upload = !c.lens.empty();
  if (upload) {
    const size_t n = c.lens.size();
    if (sl.lens_dev.cap < n || sl.lens_host.cap < n) {
      CUDA_OK(cudaEventSynchronize(sl.ev_end.get()));     // the slot's previous call still reads them
      CUDA_OK(sl.lens_dev.alloc(n));
      CUDA_OK(sl.lens_host.alloc(n));
    }
    CUDA_OK(make_event(sl.ev_lens));
    CUDA_OK(cudaEventSynchronize(sl.ev_lens.get()));      // the previous upload from lens_host has been read
    memcpy(sl.lens_host.get(), c.lens.data(), n * sizeof(int32_t));
  }
  // Chunk size: a stack kernel takes as long for 64 utterances as for 256 (one tile per CTA either way), so chunks are
  // a trade between pipelining inside one call and kernel time.  Measured at B = 256 (tools/e2e_probe.py): the one-call
  // form is fastest with ~56-utterance chunks on two compute lanes (copy-in of chunk i+1 under the kernels of chunk i),
  // the streaming form - where consecutive calls overlap anyway - with 128-utterance chunks on one lane (161 k against
  // 140 k utt-s/s with 64 x 2).
  const int auto_chunk = streaming ? 128 : 56;
  const int want_chunk = h->host_chunk > 0 ? h->host_chunk : auto_chunk;
  const int Bc = want_chunk < B ? want_chunk : B;
  const int nchunks = (B + Bc - 1) / Bc;
  while (static_cast<int>(sl.ev.size()) < 2 * nchunks) {
    Event e;
    CUDA_OK(make_event(e));
    sl.ev.push_back(std::move(e));
  }
  // one workspace + compute stream per lane: with small chunks a single forward cannot fill the GPU, so the kernels
  // of consecutive chunks are allowed to overlap
  const int want_lanes = h->host_lanes > 0 ? h->host_lanes : (streaming ? 1 : 2);
  const int lanes = want_lanes > 3 ? 3 : want_lanes;
  const size_t per_lane = c.lane_bytes(Bc);
  if (h->host_ws.cap < per_lane * lanes) {
    CUDA_OK(cudaDeviceSynchronize());          // the other slot may still be using the old workspace
    drop_graphs(h);                            // the cached graphs hold pointers into it
    CUDA_OK(h->host_ws.alloc(per_lane * lanes));
  }
  for (int l = 0; l < lanes; ++l) {
    CUDA_OK(make_stream(h->host_comp[l]));
    CUDA_OK(make_event(sl.ev_lane[l]));
  }
  cudaStream_t s_in = h->hs[0].get(), s_out = h->hs[2].get();
  // order after whatever the caller queued on its stream, and after this slot's previous use: its kernels have read
  // the input buffers (before they are overwritten) and its copy-out has read the output buffers
  CUDA_OK(cudaEventRecord(sl.ev_start.get(), s));
  CUDA_OK(cudaStreamWaitEvent(s_in, sl.ev_start.get(), 0));
  for (const Event& e : sl.ev_lane)
    if (e) CUDA_OK(cudaStreamWaitEvent(s_in, e.get(), 0));
  for (int l = 0; l < lanes; ++l) {
    CUDA_OK(cudaStreamWaitEvent(h->host_comp[l].get(), sl.ev_start.get(), 0));
    CUDA_OK(cudaStreamWaitEvent(h->host_comp[l].get(), sl.ev_end.get(), 0));
  }
  CUDA_OK(cudaStreamWaitEvent(s_out, sl.ev_start.get(), 0));
  if (upload) {
    CUDA_OK(cudaMemcpyAsync(sl.lens_dev.get(), sl.lens_host.get(), sizeof(int32_t) * c.lens.size(),
                            cudaMemcpyHostToDevice, s_in));
    CUDA_OK(cudaEventRecord(sl.ev_lens.get(), s_in));
  }
  for (int ci = 0; ci < nchunks; ++ci) {
    const int b0 = ci * Bc, bc = B - b0 < Bc ? B - b0 : Bc;
    const int lane = ci % lanes;
    const LaunchCtx comp = launch_ctx(h, h->host_comp[lane].get());
    for (size_t i = 0; i < nin; ++i) {
      const std::vector<size_t>& at = c.in[i].at;
      CUDA_OK(cudaMemcpyAsync(io[i] + at[b0], c.in[i].host + at[b0], (at[b0 + bc] - at[b0]) * 4,
                              cudaMemcpyHostToDevice, s_in));
    }
    CUDA_OK(cudaEventRecord(sl.ev[2 * ci].get(), s_in));
    CUDA_OK(cudaStreamWaitEvent(comp.stream, sl.ev[2 * ci].get(), 0));
    if (c.step(comp, h->host_ws.get() + lane * per_lane, Bc, b0, bc, io, upload ? sl.lens_dev.get() : nullptr))
      return 1;
    CUDA_OK(cudaEventRecord(sl.ev[2 * ci + 1].get(), comp.stream));
    CUDA_OK(cudaStreamWaitEvent(s_out, sl.ev[2 * ci + 1].get(), 0));
    for (size_t j = 0; j < c.out.size(); ++j) {
      const std::vector<size_t>& at = c.out[j].at;
      CUDA_OK(cudaMemcpyAsync(c.out[j].host + at[b0], io[nin + j] + at[b0], (at[b0 + bc] - at[b0]) * 4,
                              cudaMemcpyDeviceToHost, s_out));
    }
  }
  for (int l = 0; l < lanes; ++l) CUDA_OK(cudaEventRecord(sl.ev_lane[l].get(), h->host_comp[l].get()));
  // The caller's stream is deliberately NOT made to wait for the results: that would chain call i+1 (which is ordered
  // after the caller's stream) behind call i's copy-out.  Results are consumed on the host after avsep_host_wait.
  CUDA_OK(cudaEventRecord(sl.ev_end.get(), s_out));
  return 0;
}

// The spectrogram forms.  packed: the buffers hold packed batches (include/avsep.h) with HOST lengths lens / flens
// (null: all T / all N); each chunk's copies then cover its packed span and its kernels are forward_packed_run's.
int host_spec_call(avsep_handle* h, HostCall& c, const float* mixed_spec, const float* lip_frames, int B, int T, int N,
                   int Hh, int Ww, float* separated, float* masks, bool packed = false, const int32_t* lens = nullptr,
                   const int32_t* flens = nullptr) {
  c.who = packed ? "avsep_forward_host_packed" : "avsep_forward_host";
  if (!mixed_spec || !lip_frames || !separated || !masks) return fail(h, c.who + ": null buffer");
  if (check_shape(h, B, T, N, Hh, Ww)) return 1;
  // packed spans: utterances [0, b) hold pt[b] audio and pn[b] lip frames; host lengths size the copies, so a value
  // out of range is an error here, not clamped
  std::vector<size_t> pt = padded_at(B, T), pn = padded_at(B, N);
  if (packed) {
    for (int b = 0; b < B; ++b) {
      const int tb = lens ? lens[b] : T, nb = flens ? flens[b] : N;
      if (tb < 1 || tb > T || nb < 1 || nb > N)
        return fail(h, c.who + ": lengths[" + std::to_string(b) + "] = " + std::to_string(tb) + ", frame_lengths[" +
                           std::to_string(b) + "] = " + std::to_string(nb) + " outside [1, T] / [1, N]");
      pt[b + 1] = pt[b] + tb;
      pn[b + 1] = pn[b] + nb;
    }
    if (lens || flens) {   // the call's lengths, then its frame lengths
      c.lens.resize(2 * static_cast<size_t>(B));
      for (int b = 0; b < B; ++b) {
        c.lens[b] = lens ? lens[b] : T;
        c.lens[B + b] = flens ? flens[b] : N;
      }
    }
  }
  auto scaled = [](std::vector<size_t> at, size_t k) {
    for (size_t& v : at) v *= k;
    return at;
  };
  const size_t F = h->cfg.freq_bins, SF = h->cfg.num_speakers * F, HW = static_cast<size_t>(Hh) * Ww;
  c.B = B;
  c.in = {{mixed_spec, scaled(pt, F)}, {lip_frames, scaled(pn, HW)}};
  c.out = {{separated, scaled(pt, SF)}, {masks, scaled(pt, SF)}};
  const bool has_lens = lens != nullptr, has_flens = flens != nullptr;
  if (packed) {
    c.lane_bytes = [=](int Bc) {
      Workspace w;
      Staging st;
      return carve_packed(h, w, st, nullptr, Bc, T, N, Hh, Ww);
    };
    c.step = [=](LaunchCtx lc, uint8_t* ws, int Bc, int b0, int bc, float* const* io, const int32_t* d_lens) {
      Workspace w;
      Staging st;
      carve_packed(h, w, st, ws, Bc, T, N, Hh, Ww);
      w.B = bc;
      return forward_packed_run(h, lc, w, st, ws, io[0], io[1], has_lens ? d_lens : nullptr,
                                has_flens ? d_lens + B : nullptr, b0, io[2], io[3]);
    };
  } else {
    c.lane_bytes = [=](int Bc) {
      Workspace w;
      return carve_workspace(h, w, nullptr, Bc, T, N, Hh, Ww);
    };
    c.step = [=](LaunchCtx lc, uint8_t* ws, int Bc, int b0, int bc, float* const* io, const int32_t*) {
      Workspace w;
      carve_workspace(h, w, ws, Bc, T, N, Hh, Ww);
      w.B = bc;
      const size_t o = SF * T * b0;
      return forward_cached(h, lc, w, ws, io[0] + F * T * b0, io[1] + HW * N * b0, io[2] + o, io[3] + o);
    };
  }
  return 0;
}

// The waveform form (full batches): samples and lip frames in, separated samples (and the masks when masks != null) out.
int host_wave_call(avsep_handle* h, HostCall& c, const float* waves, const float* lip_frames, int B, int L, int N,
                   int Hh, int Ww, int n_fft, int hop, float* waves_out, float* masks) {
  c.who = "avsep_separate_waveforms_host";
  if (!waves || !lip_frames || !waves_out) return fail(h, c.who + ": null buffer");
  int T = 0;
  if (check_waves(h, c.who.c_str(), B, L, N, Hh, Ww, n_fft, hop, T)) return 1;
  const size_t S = h->cfg.num_speakers, SFT = S * h->cfg.freq_bins * T, HW = static_cast<size_t>(Hh) * Ww;
  c.B = B;
  c.in = {{waves, padded_at(B, L)}, {lip_frames, padded_at(B, N * HW)}};
  c.out = {{waves_out, padded_at(B, S * L)}};
  if (masks) c.out.push_back({masks, padded_at(B, SFT)});
  c.lane_bytes = [=](int Bc) {
    Workspace w;
    WaveStaging st;
    return carve_waves(h, w, st, nullptr, Bc, T, N, Hh, Ww);
  };
  const bool want_masks = masks != nullptr;
  c.step = [=](LaunchCtx lc, uint8_t* ws, int Bc, int b0, int bc, float* const* io, const int32_t*) {
    Workspace w;
    WaveStaging st;
    carve_waves(h, w, st, ws, Bc, T, N, Hh, Ww);
    w.B = bc;
    return waves_run(h, lc, w, st, ws, io[0] + static_cast<size_t>(L) * b0, io[1] + N * HW * b0, nullptr, nullptr, L,
                     n_fft, hop, io[2] + S * L * b0, want_masks ? io[3] + SFT * b0 : nullptr);
  };
  return 0;
}
}  // namespace

int avsep_forward_host(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T,
                       int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks, void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_spec_call(h, c, mixed_spec, lip_frames, B, T, N, Hh, Ww, separated, masks) ||
      host_submit(h, c, 0, lc.stream, false))
    return 1;
  CUDA_OK(cudaEventSynchronize(h->slot[0].ev_end.get()));
  return 0;
}

int avsep_forward_host_async(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T,
                             int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks, int32_t slot,
                             void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_spec_call(h, c, mixed_spec, lip_frames, B, T, N, Hh, Ww, separated, masks)) return 1;
  return host_submit(h, c, slot, lc.stream, true);
}

int avsep_forward_host_packed(avsep_handle* h, const float* mixed_packed, const float* frames_packed,
                              const int32_t* lengths, const int32_t* frame_lengths, int32_t B, int32_t T, int32_t N,
                              int32_t Hh, int32_t Ww, float* separated_packed, float* masks_packed, void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_spec_call(h, c, mixed_packed, frames_packed, B, T, N, Hh, Ww, separated_packed, masks_packed, true, lengths,
                     frame_lengths) ||
      host_submit(h, c, 0, lc.stream, false))
    return 1;
  CUDA_OK(cudaEventSynchronize(h->slot[0].ev_end.get()));
  return 0;
}

int avsep_forward_host_packed_async(avsep_handle* h, const float* mixed_packed, const float* frames_packed,
                                    const int32_t* lengths, const int32_t* frame_lengths, int32_t B, int32_t T,
                                    int32_t N, int32_t Hh, int32_t Ww, float* separated_packed, float* masks_packed,
                                    int32_t slot, void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_spec_call(h, c, mixed_packed, frames_packed, B, T, N, Hh, Ww, separated_packed, masks_packed, true, lengths,
                     frame_lengths))
    return 1;
  return host_submit(h, c, slot, lc.stream, true);
}

size_t avsep_waveform_workspace_bytes(avsep_handle* h, int32_t B, int32_t L, int32_t N, int32_t Hh, int32_t Ww,
                                      int32_t n_fft, int32_t hop_length) {
  if (!h || B < 1 || L < 1 || N < 1 || Hh < 1 || Ww < 1 || !fft_geometry_ok(n_fft, hop_length) ||
      n_fft != 2 * (h->cfg.freq_bins - 1))
    return 0;
  Workspace w;
  WaveStaging st;
  return carve_waves(h, w, st, nullptr, B, 1 + L / hop_length, N, Hh, Ww);
}

int avsep_separate_waveforms(avsep_handle* h, const float* waves, const float* lip_frames, const int32_t* lengths,
                             const int32_t* frame_lengths, int32_t B, int32_t L, int32_t N, int32_t Hh, int32_t Ww,
                             int32_t n_fft, int32_t hop_length, float* waves_out, float* masks, void* workspace,
                             size_t workspace_bytes, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!waves || !lip_frames || !waves_out) return fail(h, "avsep_separate_waveforms: null buffer");
  int T = 0;
  if (check_waves(h, "avsep_separate_waveforms", B, L, N, Hh, Ww, n_fft, hop_length, T)) return 1;
  Workspace w;
  WaveStaging st;
  uint8_t* base = nullptr;
  if (workspace_base(h, workspace, workspace_bytes, carve_waves(h, w, st, nullptr, B, T, N, Hh, Ww),
                     "avsep_waveform_workspace_bytes", base))
    return 1;
  carve_waves(h, w, st, base, B, T, N, Hh, Ww);
  return waves_run(h, lc, w, st, base, waves, lip_frames, lengths, frame_lengths, L, n_fft, hop_length, waves_out,
                   masks);
}

int avsep_separate_waveforms_host(avsep_handle* h, const float* waves, const float* lip_frames, int32_t B, int32_t L,
                                  int32_t N, int32_t Hh, int32_t Ww, int32_t n_fft, int32_t hop_length,
                                  float* waves_out, float* masks, void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_wave_call(h, c, waves, lip_frames, B, L, N, Hh, Ww, n_fft, hop_length, waves_out, masks) ||
      host_submit(h, c, 0, lc.stream, false))
    return 1;
  CUDA_OK(cudaEventSynchronize(h->slot[0].ev_end.get()));
  return 0;
}

int avsep_separate_waveforms_host_async(avsep_handle* h, const float* waves, const float* lip_frames, int32_t B,
                                        int32_t L, int32_t N, int32_t Hh, int32_t Ww, int32_t n_fft,
                                        int32_t hop_length, float* waves_out, float* masks, int32_t slot,
                                        void* cuda_stream) {
  ENTER(h, cuda_stream);
  HostCall c;
  if (host_wave_call(h, c, waves, lip_frames, B, L, N, Hh, Ww, n_fft, hop_length, waves_out, masks)) return 1;
  return host_submit(h, c, slot, lc.stream, true);
}

int avsep_host_wait(avsep_handle* h, int32_t slot) {
  if (!h) return 1;
  if (slot < 0 || slot >= AVSEP_HOST_SLOTS) return fail(h, "avsep_host_wait: slot must be 0 .. AVSEP_HOST_SLOTS - 1");
  if (!h->slot[slot].ev_end) return 0;       // nothing was ever submitted on this slot
  ON_DEVICE(h, h->cfg.device);
  CUDA_OK(cudaEventSynchronize(h->slot[slot].ev_end.get()));
  return 0;
}

int avsep_synth_batch(avsep_handle* h, const avsep_synth_config* cfg, int32_t B, const double* amps, const double* freqs,
                      const double* phases, const float* noise, float* mixed_spec, float* lip_frames,
                      float* clean_specs, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!cfg || !amps || !freqs || !phases || !mixed_spec || !lip_frames) return fail(h, "avsep_synth_batch: null argument");
  if (B < 1) return fail(h, "avsep_synth_batch: empty batch");
  SynthProblem p{};
  p.B = B; p.S = cfg->num_speakers; p.n = cfg->num_samples_audio; p.nfft = cfg->n_fft; p.hop = cfg->hop_length;
  p.nf = cfg->num_frames; p.Hh = cfg->frame_h; p.Ww = cfg->frame_w; p.duration = cfg->duration;
  p.amps = amps; p.freqs = freqs; p.phases = phases; p.noise = noise;
  p.mixed_spec = mixed_spec; p.lip_frames = lip_frames; p.clean_specs = clean_specs;
  if (p.S < 1 || p.n < 1) return fail(h, "avsep_synth_batch: bad geometry");
  const size_t need = static_cast<size_t>(B) * (p.S + 1) * p.n;
  if (h->synth_waves.cap < need) CUDA_OK(h->synth_waves.alloc(need));
  p.waves = h->synth_waves.get();
  CK(lc.stream, launch_synth_waves, p);
  CK(lc.stream, launch_stft, p.waves, nullptr, B, p.S + 1, p.n, p.nfft, p.hop, nullptr, mixed_spec, clean_specs,
     nullptr);
  CK(lc.stream, launch_synth_lips, p);
  return 0;
}

int avsep_eval_snr(avsep_handle* h, const float* separated, const float* targets, const float* mixed, int32_t B,
                   int32_t S, int32_t F, int32_t T, double* input_snr, double* output_snr, int32_t* best_perm,
                   double* si_snr, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!separated || !targets) return fail(h, "avsep_eval_snr: null argument");
  if (B < 1 || F < 1 || T < 1) return fail(h, "avsep_eval_snr: empty problem");
  CK(lc.stream, launch_eval_snr, separated, targets, mixed, B, S, F * T, input_snr, output_snr, best_perm, si_snr);
  return 0;
}

int avsep_stft(avsep_handle* h, const float* waves, int32_t B, int32_t L, int32_t n_fft, int32_t hop_length,
               float* spec, float* mag, void* cuda_stream) {
  return avsep_stft_varlen(h, waves, nullptr, B, L, n_fft, hop_length, spec, mag, nullptr, cuda_stream);
}

int avsep_stft_varlen(avsep_handle* h, const float* waves, const int32_t* lengths, int32_t B, int32_t L, int32_t n_fft,
                      int32_t hop_length, float* spec, float* mag, int32_t* frame_lengths_out, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!waves || !spec) return fail(h, "avsep_stft: null argument");
  if (B <= 0 || L <= 0) return fail(h, "stft: empty problem");
  if (!fft_geometry_ok(n_fft, hop_length))
    return fail(h, "stft: n_fft must be a power of two in [8, 2048], 1 <= hop <= n_fft");
  CK(lc.stream, launch_stft, waves, lengths, B, 0, L, n_fft, hop_length, spec, mag, nullptr, frame_lengths_out);
  return 0;
}

int avsep_istft(avsep_handle* h, const float* spec, const float* masks, int32_t B, int32_t S, int32_t T,
                int32_t n_fft, int32_t hop_length, int32_t L, float* waves, void* cuda_stream) {
  return avsep_istft_varlen(h, spec, masks, nullptr, B, S, T, n_fft, hop_length, L, waves, cuda_stream);
}

int avsep_istft_varlen(avsep_handle* h, const float* spec, const float* masks, const int32_t* lengths, int32_t B,
                       int32_t S, int32_t T, int32_t n_fft, int32_t hop_length, int32_t L, float* waves,
                       void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!spec || !waves) return fail(h, "avsep_istft: null argument");
  CK(lc.stream, launch_istft_masked, spec, masks, lengths, B, S, T, n_fft, hop_length, L, waves);
  return 0;
}

int64_t avsep_last_launch_count(const avsep_handle* h) { return h ? h->launches : 0; }

// ---- batch sharding over the GPUs of one box: peer-mapped buffers + copy-engine transfers (SURVEY 8e) ----------
int avsep_shared_alloc(avsep_handle* h, size_t bytes, void** dev_ptr, unsigned char handle_out[AVSEP_IPC_HANDLE_BYTES]) {
  if (!h) return 1;
  if (!dev_ptr || !handle_out || bytes == 0) return fail(h, "avsep_shared_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == AVSEP_IPC_HANDLE_BYTES, "IPC handle size");
  ON_DEVICE(h, h->cfg.device);
  void* ptr = nullptr;
  CUDA_OK(cudaMalloc(&ptr, bytes));       // a dedicated allocation: an IPC handle always names a whole cudaMalloc block
  cudaIpcMemHandle_t ih;
  const cudaError_t ce = cudaIpcGetMemHandle(&ih, ptr);
  if (ce != cudaSuccess) {
    cudaFree(ptr);
    return fail(h, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(ce));
  }
  memcpy(handle_out, &ih, sizeof ih);
  h->shared_owned.push_back(ptr);
  *dev_ptr = ptr;
  return 0;
}

int avsep_shared_free(avsep_handle* h, void* dev_ptr) {
  if (!h) return 1;
  ON_DEVICE(h, h->cfg.device);
  for (size_t i = 0; i < h->shared_owned.size(); ++i)
    if (h->shared_owned[i] == dev_ptr) {
      h->shared_owned.erase(h->shared_owned.begin() + i);
      CUDA_OK(cudaFree(dev_ptr));
      return 0;
    }
  return fail(h, "avsep_shared_free: pointer was not allocated by avsep_shared_alloc on this handle");
}

int avsep_shared_open(avsep_handle* h, const unsigned char handle[AVSEP_IPC_HANDLE_BYTES], void** dev_ptr) {
  if (!h) return 1;
  if (!handle || !dev_ptr) return fail(h, "avsep_shared_open: bad argument");
  ON_DEVICE(h, h->cfg.device);
  cudaIpcMemHandle_t ih;
  memcpy(&ih, handle, sizeof ih);
  void* ptr = nullptr;
  CUDA_OK(cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess));
  h->shared_mapped.push_back(ptr);
  *dev_ptr = ptr;
  return 0;
}

int avsep_shared_close(avsep_handle* h, void* dev_ptr) {
  if (!h) return 1;
  ON_DEVICE(h, h->cfg.device);
  for (size_t i = 0; i < h->shared_mapped.size(); ++i)
    if (h->shared_mapped[i] == dev_ptr) {
      h->shared_mapped.erase(h->shared_mapped.begin() + i);
      CUDA_OK(cudaIpcCloseMemHandle(dev_ptr));
      return 0;
    }
  return fail(h, "avsep_shared_close: pointer was not mapped by avsep_shared_open on this handle");
}

int avsep_copy_async(avsep_handle* h, void* dst, const void* src, size_t bytes, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!dst || !src) return fail(h, "avsep_copy_async: null buffer");
  if (bytes == 0) return 0;
  CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, lc.stream));
  return 0;
}

int avsep_separate(avsep_handle* h, const float* masks, const float* mixed_spec, int32_t B, int32_t T, float* separated,
                   void* cuda_stream) {
  return avsep_separate_varlen(h, masks, mixed_spec, nullptr, B, T, separated, cuda_stream);
}

int avsep_separate_varlen(avsep_handle* h, const float* masks, const float* mixed_spec, const int32_t* lengths,
                          int32_t B, int32_t T, float* separated, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!masks || !mixed_spec || !separated) return fail(h, "avsep_separate: null buffer");
  if (B < 1 || T < 1) return fail(h, "avsep_separate: B and T must be >= 1");
  CK(lc.stream, launch_separate, masks, mixed_spec, separated, B, h->cfg.num_speakers, h->cfg.freq_bins, T, lengths);
  return 0;
}

namespace {
int make_flag_set(avsep_handle* h, uint32_t* const* flags, int32_t n, FlagSet& f, const char* who) {
  if (!flags || n < 1 || n > FlagSet::MAX) return fail(h, std::string(who) + ": 1 .. 16 flags");
  f.n = n;
  for (int i = 0; i < n; ++i) {
    if (!flags[i] || (reinterpret_cast<uintptr_t>(flags[i]) & 3)) return fail(h, std::string(who) + ": bad flag pointer");
    f.ptr[i] = flags[i];
  }
  return 0;
}
}  // namespace

int avsep_flag_signal(avsep_handle* h, uint32_t* const* flags, int32_t n, uint32_t value, void* cuda_stream) {
  ENTER(h, cuda_stream);
  FlagSet f;
  if (make_flag_set(h, flags, n, f, "avsep_flag_signal")) return 1;
  CK(lc.stream, launch_flag_signal, f, value);
  return 0;
}

int avsep_flag_wait(avsep_handle* h, uint32_t* const* flags, int32_t n, uint32_t value, double timeout_s,
                    void* cuda_stream) {
  ENTER(h, cuda_stream);
  FlagSet f;
  if (make_flag_set(h, flags, n, f, "avsep_flag_wait")) return 1;
  if (!(timeout_s > 0.0) || timeout_s > 3600.0) return fail(h, "avsep_flag_wait: timeout_s must be in (0, 3600]");
  CK(lc.stream, launch_flag_wait, f, value, timeout_s);
  return 0;
}

// ---- sub-module forwards ------------------------------------------------------------------------
int avsep_audio_encoder(avsep_handle* h, const float* mixed_spec, int32_t B, int32_t T, float* out_BTd,
                        void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!mixed_spec || !out_BTd) return fail(h, "avsep_audio_encoder: null buffer");
  if (check_shape(h, B, T, 1, 1, 1)) return 1;
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, 1, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T;
  if (audio_frontend(h, lc, w, mixed_spec, Plan{})) return 1;
  if (encoder_stack(h, lc, h->enc_a, B, T, w.x_a, w.y_a, w.a_op, w.qkv_a, w.attn_a, w.ffn_a, nullptr, nullptr)) return 1;
  CUDA_OK(cudaMemcpyAsync(out_BTd, w.x_a, static_cast<size_t>(Ma) * d * 4, cudaMemcpyDeviceToDevice, lc.stream));
  return 0;
}

int avsep_visual_encoder(avsep_handle* h, const float* lip_frames, int32_t B, int32_t N, int32_t Hh, int32_t Ww,
                         int32_t target_len, float* out_BTd, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!lip_frames || !out_BTd) return fail(h, "avsep_visual_encoder: null buffer");
  if (check_shape(h, B, 1, N, Hh, Ww)) return 1;
  if (target_len < 1) return fail(h, "avsep_visual_encoder: target_len must be >= 1");
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, 1, N, Hh, Ww)) return 1;
  const int d = h->cfg.d_model;
  if (visual_frontend(h, lc, w, lip_frames, Plan{})) return 1;
  if (encoder_stack(h, lc, h->enc_v, B, N, w.x_v, w.y_v, w.v_op, w.qkv_v, w.attn_v, w.ffn_v, nullptr, nullptr)) return 1;
  CKL("interp_rows", lc.stream, launch_interp_rows, w.x_v, out_BTd, B, N, target_len, d);
  return 0;
}

int avsep_fusion(avsep_handle* h, const float* audio_BTd, const float* visual_BLd, int32_t B, int32_t T, int32_t L,
                 float* out_BTd, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!audio_BTd || !visual_BLd || !out_BTd) return fail(h, "avsep_fusion: null buffer");
  if (check_shape(h, B, T, L, 1, 1)) return 1;
  if (L != T) return fail(h, "avsep_fusion: audio and visual must have the same length (model.py:131-133)");
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, L, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T, Mv = B * L, prec = h->cfg.precision;
  CUDA_OK(cudaMemcpyAsync(w.x_a, audio_BTd, static_cast<size_t>(Ma) * d * 4, cudaMemcpyDeviceToDevice, lc.stream));
  CKL("add_layernorm", lc, launch_add_layernorm, prec, w.x_a, nullptr, h->fus[0].n1g, h->fus[0].n1b, nullptr, w.a_op,
      Ma, d);
  // cast only
  CKL("add_layernorm", lc, launch_add_layernorm, prec, visual_BLd, nullptr, nullptr, nullptr, nullptr, w.v_op, Mv, d);
  const bool dbg = h->debug;
  h->debug = false;
  const int rc = fusion_stack(h, lc, w, L);   // identity interpolation (L == T)
  h->debug = dbg;
  if (rc) return 1;
  // fused rows in fp32: recompute the final LayerNorm from the fp32 residual stream straight into the caller's buffer
  CKL("add_layernorm", lc, launch_add_layernorm, PREC_TF32, w.x_a, nullptr, h->fng, h->fnb, nullptr, out_BTd, Ma, d);
  return 0;
}

int avsep_decoder(avsep_handle* h, const float* fused_BTd, const float* mixed_spec, int32_t B, int32_t T,
                  float* separated, float* masks, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!fused_BTd || !mixed_spec || !separated || !masks) return fail(h, "avsep_decoder: null buffer");
  if (check_shape(h, B, T, 1, 1, 1)) return 1;
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, 1, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T;
  CKL("add_layernorm", lc, launch_add_layernorm, h->cfg.precision, fused_BTd, nullptr, nullptr, nullptr, nullptr,
      w.a_op, Ma, d);
  return decoder_stage(h, lc, w, mixed_spec, separated, masks);
}

// ---- debug ---------------------------------------------------------------------------------------
int avsep_set_debug(avsep_handle* h, int32_t enable) {
  if (!h) return 1;
  h->debug = enable != 0;
  return 0;
}

int avsep_debug_get_stage(avsep_handle* h, const char* name, float* host_out, size_t capacity, size_t* count) {
  if (!h || !name || !count) return fail(h, "avsep_debug_get_stage: bad argument");
  auto it = h->snaps.find(name);
  if (it == h->snaps.end()) return fail(h, std::string("no snapshot named ") + name);
  const auto& snap = it->second;
  *count = snap.count;
  if (host_out == nullptr) return 0;
  if (capacity < snap.count) return fail(h, "avsep_debug_get_stage: buffer too small");
  ON_DEVICE(h, h->cfg.device);
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(host_out, snap.buf.get(), snap.count * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int avsep_set_profile(avsep_handle* h, int32_t enable) {
  if (!h) return 1;
  h->profile = enable != 0;
  return 0;
}

// Folds the pending event pairs into the per-label totals (synchronises) and writes
// "label count total_ms\n" lines into buf.  reset != 0 clears the totals afterwards.
int avsep_profile_report(avsep_handle* h, char* buf, size_t capacity, int32_t reset) {
  if (!h || !buf || capacity == 0) return fail(h, "avsep_profile_report: bad argument");
  ON_DEVICE(h, h->cfg.device);
  CUDA_OK(cudaDeviceSynchronize());
  for (auto& mk : h->ev_marks) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_pool[mk.second].get(), h->ev_pool[mk.second + 1].get()) == cudaSuccess) {
      auto& slot = h->prof[mk.first];
      slot.first += 1;
      slot.second += ms;
    }
  }
  h->ev_marks.clear();
  h->ev_used = 0;
  std::string out;
  for (auto& kv : h->prof) {
    char line[160];
    snprintf(line, sizeof line, "%s %lld %.6f\n", kv.first.c_str(), static_cast<long long>(kv.second.first), kv.second.second);
    out += line;
  }
  if (out.size() + 1 > capacity) return fail(h, "avsep_profile_report: buffer too small");
  memcpy(buf, out.c_str(), out.size() + 1);
  if (reset) h->prof.clear();
  return 0;
}

// ---- kernel-level test hooks -----------------------------------------------------------------------
int avsep_test_gemm(avsep_handle* h, const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N,
                    int32_t K, int32_t act, int32_t force_bn, void* cuda_stream) {
  ENTER(h, cuda_stream);
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.bias = bias; e.act = act; e.out_f32 = out; e.ld_f32 = N;
  CK(lc, launch_gemm, h->cfg.precision, p, e, h->num_sms, force_bn);
  return 0;
}

// out-proj/FFN2-style GEMM with the fused residual + LayerNorm epilogue: x (in/out, fp32 [M,N]) += A W^T + bias;
// out_op = LN_{gamma,beta}(x) in operand precision.
int avsep_test_gemm_ln(avsep_handle* h, const void* A, const void* W, const float* bias, float* x, const float* gamma,
                       const float* beta, void* out_op, int32_t M, int32_t N, int32_t K, void* cuda_stream) {
  ENTER(h, cuda_stream);
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.kind = EPI_LN;
  e.bias = bias; e.resid = x; e.out_f32 = x; e.ld_f32 = N; e.ln_gamma = gamma; e.ln_beta = beta;
  e.out_op = out_op; e.ld_op = N;
  CK(lc, launch_gemm, h->cfg.precision, p, e, h->num_sms);
  return 0;
}

// Debug: same GEMM as avsep_test_gemm / avsep_test_gemm_ln (ln != 0) with a per-CTA phase trace:
// trace_dev[cta*8 + k] = globaltimer (ns) at k = 0 entry, 1 setup done, 2 first operands landed, 3 MMAs issued,
// 4 accumulator ready, 5 accumulator drained (LN), 6 first tile's epilogue done, 7 CTA done.
int avsep_test_gemm_trace(avsep_handle* h, const void* A, const void* W, const float* bias, float* x_or_out,
                          const float* gamma, const float* beta, void* out_op, int32_t M, int32_t N, int32_t K,
                          int32_t ln, int32_t act, unsigned long long* trace_dev, void* cuda_stream) {
  ENTER(h, cuda_stream);
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.bias = bias; e.act = act;
  if (ln == 7) {
    // decoder head (EPI_TAIL) for the trace tool: S = 2, F = N / 2, T = act; mixed = gamma, masks = x_or_out,
    // separated = out_op (all float32)
    e.kind = EPI_TAIL; e.act = ACT_NONE;
    e.S = 2; e.F = N / 2; e.T = act;
    e.mixed = gamma; e.masks = x_or_out; e.separated = static_cast<float*>(out_op);
  } else if (ln) {
    e.kind = EPI_LN;
    e.resid = x_or_out; e.out_f32 = x_or_out; e.ld_f32 = N; e.ln_gamma = gamma; e.ln_beta = beta;
    e.out_op = out_op; e.ld_op = N;
    if (ln == 2) e.resid = nullptr;            // ablations for the trace tool
    if (ln == 3) e.out_f32 = nullptr;
    if (ln == 4) e.out_op = nullptr;
    if (ln == 5) { e.resid = nullptr; e.out_f32 = nullptr; }
    if (ln == 6) { e.ln_gamma = nullptr; }
  } else {
    e.out_op = out_op; e.ld_op = N;
    e.out_f32 = out_op ? nullptr : x_or_out; e.ld_f32 = N;
  }
  CK(lc, launch_gemm, h->cfg.precision, p, e, h->num_sms, 0, trace_dev);
  return 0;
}

// Fused FFN sub-layer (d_model = 256, bf16): x (fp32, in place) += W2 act(W1 a + b1) + b2; out_op = LN(x) (bf16).
int avsep_test_ffn_fused(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                         const float* b2, int32_t act, float* x_inout, const float* gamma, const float* beta,
                         void* out_op, int32_t M, void* cuda_stream) {
  ENTER(h, cuda_stream);
  CK(lc, launch_ffn_fused, a, w1, b1, w2, b2, act, x_inout, x_inout, gamma, beta, out_op, M, h->num_sms, nullptr);
  return 0;
}

// Debug: the same with a phase trace ([grid][64] globaltimer stamps of each CTA's first tile: [0] entry, [1] A landed,
// [2] acc2 complete, [3] epilogue-2 done, per chunk j at 8+4j: GEMM1 issued, GEMM2 issued, acc1 ready, H published).
int avsep_test_ffn_fused_trace(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                               const float* b2, int32_t act, float* x_inout, const float* gamma, const float* beta,
                               void* out_op, int32_t M, unsigned long long* trace_dev, void* cuda_stream) {
  ENTER(h, cuda_stream);
  CK(lc, launch_ffn_fused, a, w1, b1, w2, b2, act, x_inout, x_inout, gamma, beta, out_op, M, h->num_sms, trace_dev);
  return 0;
}

// One whole stack through the fused kernel (xformer_stack_sm100.cu) on the handle's weights.  which: 0 audio encoder,
// 1 visual encoder, 2 fusion (kv = bf16 [B*L, num_fusion_layers*2*d] K|V rows).  x_in fp32 [B*L, d]; out_x fp32 and /
// or out_op bf16 (final_ln != 0: the LayerNorm that follows the stack in the model -- fusion layer 0 norm1 after the
// audio encoder, fusion.norm after the fusion stack; the visual encoder has none -- else a plain cast).
int avsep_test_xformer_stack(avsep_handle* h, int32_t which, const float* x_in, const void* kv, int32_t B, int32_t L,
                             float* out_x, void* out_op, int32_t final_ln, long long* trace_dev, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!h->finalized) return fail(h, "weights not finalized");
  if (which < 0 || which > 2) return fail(h, "test_xformer_stack: which must be 0, 1 or 2");
  if (h->xs_a == nullptr || !xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, L))
    return fail(h, "test_xformer_stack: the fused stack kernel does not support this configuration");
  StackProblem sp{};
  sp.x_in = x_in; sp.out_x = out_x; sp.out_op = out_op; sp.kv = kv; sp.B = B; sp.L = L; sp.trace = trace_dev;
  if (final_ln && which == 0) { sp.fin_gamma = h->fus[0].n1g; sp.fin_beta = h->fus[0].n1b; }
  if (final_ln && which == 2) { sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; }
  return run_stack(h, lc, which, sp);
}

int avsep_test_fusion_decoder(avsep_handle* h, const float* x_in, const void* kv, int32_t B, int32_t L, const float* mixed,
                              float* separated, float* masks, long long* trace_dev, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!h->finalized) return fail(h, "weights not finalized");
  if (h->xs_f == nullptr || !h->xs_f_decoder || !xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, L))
    return fail(h, "test_fusion_decoder: the fused stack kernel does not support this configuration");
  if (!mixed || !separated || !masks) return fail(h, "test_fusion_decoder: null buffer");
  StackProblem sp{};
  sp.x_in = x_in; sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; sp.kv = kv; sp.B = B; sp.L = L; sp.trace = trace_dev;
  sp.mixed = mixed; sp.separated = separated; sp.masks = masks;
  return run_stack(h, lc, 2, sp);
}

int avsep_set_option(avsep_handle* h, const char* name, int32_t value) {
  if (!h || !name) return 1;
  ON_DEVICE(h, h->cfg.device);   // drop_graphs destroys graph execs of h's device
  if (strcmp(name, "host_chunk") == 0) { h->host_chunk = value; return 0; }
  if (strcmp(name, "host_lanes") == 0) { h->host_lanes = value; return 0; }
  if (strcmp(name, "pdl") == 0) { h->pdl = value != 0; drop_graphs(h); return 0; }
  if (strcmp(name, "use_graph") == 0) { h->use_graph = value != 0; return 0; }
  if (strcmp(name, "two_stream") == 0) { h->two_stream = value != 0; drop_graphs(h); return 0; }
  if (strcmp(name, "attn_tc") == 0) { h->attn_tc = value; drop_graphs(h); return 0; }
  if (strcmp(name, "profile_spin_us") == 0) { h->profile_spin_us = value; return 0; }
  return fail(h, std::string("unknown option ") + name);
}

int avsep_test_conv1d(avsep_handle* h, const void* A_padded, const void* W3, const float* bias, float* out, int32_t B,
                      int32_t L, int32_t N, int32_t K, void* cuda_stream) {
  ENTER(h, cuda_stream);
  GemmProblem p{};
  const int Mp = B * (L + 2);
  p.A = A_padded; p.lda = K; p.rowsA = Mp; p.M = Mp; p.W = W3; p.ldw = 3 * K; p.N = N; p.K = K;
  p.taps = 3; p.tap_stride = K; p.row_shift = -1;
  GemmEpilogue e;
  e.bias = bias; e.rowmap = ROW_PAD2COMPACT; e.Lp = L + 2; e.out_f32 = out; e.ld_f32 = N;
  CK(lc, launch_gemm, h->cfg.precision, p, e, h->num_sms);
  return 0;
}

int avsep_test_attention(avsep_handle* h, const void* q, const void* k, const void* v, void* out, int32_t B, int32_t H,
                         int32_t hd, int32_t Lq, int32_t Lk, int32_t lerp_src, void* cuda_stream) {
  ENTER(h, cuda_stream);
  AttnProblem ap{};
  ap.q = q; ap.ldq = H * hd; ap.k = k; ap.v = v; ap.ldkv = H * hd; ap.out = out; ap.ldo = H * hd;
  ap.B = B; ap.H = H; ap.hd = hd; ap.Lq = Lq; ap.Lk = Lk; ap.lerp_src = lerp_src; ap.tc_mode = h->attn_tc;
  Buf<__nv_bfloat16> scratch;
  const int rc = [&] {
    if (lerp_src > 0) {   // same routing as fusion_stack: K then V columns side by side in one interpolated buffer
      AttnProblem tp = ap;
      tp.lerp_src = 0; tp.ldkv = 2 * H * hd;
      if (attention_tc_wanted(h->cfg.precision, tp)) {
        const int dm = H * hd;
        if (scratch.alloc(static_cast<size_t>(B) * Lk * 2 * dm) != cudaSuccess)
          return fail(h, "test_attention: cudaMalloc failed");
        tp.k = scratch.get(); tp.v = scratch.get() + dm;
        CK(lc, launch_lerp_rows, static_cast<const float*>(k), dm, B, lerp_src, Lk, dm, scratch.get(), 2 * dm);
        CK(lc, launch_lerp_rows, static_cast<const float*>(v), dm, B, lerp_src, Lk, dm, scratch.get() + dm, 2 * dm);
        ap = tp;
      }
    }
    CK(lc, launch_attention, h->cfg.precision, ap);
    return 0;
  }();
  if (scratch.get()) cudaStreamSynchronize(lc.stream);   // before scratch is freed, on every return path
  return rc;
}

int avsep_test_add_layernorm(avsep_handle* h, const float* x, const float* y, const float* gamma, const float* beta,
                             float* x_out, void* out_op, int32_t M, int32_t d, void* cuda_stream) {
  ENTER(h, cuda_stream);
  CKL("add_layernorm", lc, launch_add_layernorm, h->cfg.precision, x, y, gamma, beta, x_out, out_op, M, d);
  return 0;
}

int avsep_test_visual_cnn(avsep_handle* h, const float* frames, int32_t M, int32_t Hh, int32_t Ww, void* pooled,
                          void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!h->finalized) return fail(h, "weights not finalized");
  CK(lc, run_visual_cnn, h, frames, M, Hh, Ww, pooled);
  return 0;
}

// Debug: tcgen05 CNN with a phase trace ([grid][64] globaltimer stamps of each CTA's second frame group).
int avsep_test_visual_cnn_trace(avsep_handle* h, const float* frames, int32_t M, void* pooled,
                                unsigned long long* trace_dev, void* cuda_stream) {
  ENTER(h, cuda_stream);
  if (!h->finalized) return fail(h, "weights not finalized");
  CK(lc, run_visual_cnn, h, frames, M, 32, 32, pooled, trace_dev);
  return 0;
}

}  // extern "C"
